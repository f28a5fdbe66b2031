"""Regenerates tests/golden/*.npz.  Runs ONLY in the authoring container (needs /root/reference):

* dense_sums.npz   -- outputs of the reference's own mshadow arithmetic (oracle/_ref/libkvref.so,
                      built from /root/reference/3rdparty/mshadow by oracle/Makefile) for the
                      CommDevice and CommCPU reduce orders;
* compression.npz  -- outputs of the reference's bit-level simulator `compute_1bit` /
                      `compute_2bit` (tests/nightly/test_kvstore.py:35-98), executed from the
                      reference file itself (nothing is copied into this repository).

* layerwise.npz    -- weights produced by the reference's own non-fused ``step`` methods of LAMB / LANS /
                      LARS (python/mxnet/optimizer/{lamb,lans,lars}.py), executed from the reference files
                      on a float32 numpy stand-in for NDArray (nothing is copied into this repository).

* optimizer_steps.npz -- the same for SGD / SGD-momentum / Adam / Test (sgd.py, adam.py, optimizer.py).

* sparse_steps.npz -- row_sparse gradients: the reference's OWN Python references for its sparse kernels,
                      ``PySparseSGD.step`` / ``PySparseAdam.step`` (tests/python/unittest/test_optimizer.py:90-159,
                      372-437; lazy and standard), and ``SGD.step`` on the densified gradient for the standard SGD
                      update (test_std_sparse_sgd, :183-203), executed from the reference files the same way.

* tree_topology.npz -- MXNET_KVSTORE_USETREE: the trees the reference's OWN solver (src/kvstore/gpu_topology.h,
                      compiled where it lies into oracle/_ref/libkvref_topo.so by oracle/ref_topology.cc) builds
                      from link matrices -- one switch (uniform weights, 2 ... 8 GPUs), the NVLink hybrid cube
                      mesh of its comments, random matrices of 2 ... 16 GPUs with and without missing links --
                      by Kernighan-Lin and by the exhaustive search; plus the outcome of one Kernighan-Lin pass.

* reference_sums.npz, tree_draw.npz, c_api_prototypes.json -- what the reference's arithmetic, its tree solver and
                      its C header give for the inputs of three tests that compare with them (see each function).

The GPU box has no /root/reference; tests read the committed fixtures instead.
"""
import ast
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference"


def dense_sums():
    from oracle import oracle as O
    assert O.ref_lib() is not None, "build oracle/_ref first (make -C oracle)"
    out = {}
    rng = np.random.default_rng(20260921)
    for n in (2, 3, 4, 5, 7, 8):
        for E in (1, 33, 4099):
            vals = [rng.uniform(-1, 1, E).astype(np.float32) for _ in range(n)]
            tag = "n%d_E%d" % (n, E)
            out["in_" + tag] = np.stack(vals)
            out["device_f32_" + tag] = O.ref_sum_device(vals)
            out["commcpu_f32_" + tag] = O.ref_sum_cpu(vals)
            out["device_f16_" + tag] = O.ref_sum_device([v.astype(np.float16) for v in vals])
    # big enough to take CommCPU's OpenMP branch (>= 1e6 elements, 4096-element tasks)
    vals = [rng.uniform(-1, 1, 1000003).astype(np.float32) for _ in range(5)]
    out["seed_big"] = np.array([777], np.int64)
    big_rng = np.random.default_rng(777)
    vals = [big_rng.uniform(-1, 1, 1000003).astype(np.float32) for _ in range(5)]
    s = O.ref_sum_cpu(vals)
    out["commcpu_f32_big_head"] = s[:4096]
    out["commcpu_f32_big_tail"] = s[-4096:]
    out["commcpu_f32_big_xor"] = np.bitwise_xor.reduce(s.view(np.uint32)).reshape(1)
    np.savez_compressed(os.path.join(HERE, "dense_sums.npz"), **out)


def compression():
    src = open(os.path.join(REF, "tests/nightly/test_kvstore.py")).read()
    tree = ast.parse(src)
    ns = {"np": np}
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in ("compute_1bit", "compute_2bit"):
            exec(compile(ast.Module([node], []), "reference:tests/nightly/test_kvstore.py", "exec"), ns)

    def pack(bits):
        # compute_expected_quantization (:81-98) reverses the four bytes of every 32-bit group and
        # stores the word little-endian, i.e. memory byte j holds bits[8j:8j+8] MSB first
        by = [int(bits[i:i + 8], 2) for i in range(0, len(bits), 8)]
        return np.array(by, np.uint8)

    out = {}
    rng = np.random.default_rng(4242)
    for kind, fn, thr in (("2bit", ns["compute_2bit"], 0.5), ("1bit", ns["compute_1bit"], 0.0)):
        for E in (32, 64, 160):
            res = np.zeros(E, np.float32)
            for it in range(3):
                arr = rng.uniform(-1.2, 1.2, E).astype(np.float32)
                bits, new_res, dec = fn(arr.copy(), res, thr)
                tag = "%s_E%d_it%d" % (kind, E, it)
                out["grad_" + tag] = arr
                out["res_in_" + tag] = res.copy()
                out["bytes_" + tag] = pack(bits)[: ((E + (31 if kind == "1bit" else 15)) // (32 if kind == "1bit" else 16)) * 4]
                out["res_out_" + tag] = np.array(new_res, np.float32)
                out["dec_" + tag] = np.array(dec, np.float32)
                res = np.array(new_res, np.float32)
    np.savez_compressed(os.path.join(HERE, "compression.npz"), **out)


# ---------------------------------------------------------------------------------------------
# LAMB / LANS / LARS: run the reference's Python `step` (the "use_fused_step=False" implementation the
# reference's own tests compare its fused kernels against, tests/python/unittest/test_optimizer.py:232-312)
# ---------------------------------------------------------------------------------------------
class _F32(np.ndarray):
    """float32 ndarray that answers the few NDArray methods `step` calls."""

    def norm(self):
        return np.sqrt(np.sum(np.square(np.asarray(self, np.float32)), dtype=np.float32, keepdims=False)
                       ).astype(np.float32).reshape(1).view(_F32)

    def asscalar(self):
        return np.asarray(self).reshape(-1)[0]

    def astype(self, dtype, copy=True):       # noqa: D401 -- NDArray.astype always copies
        return np.array(np.asarray(self), dtype=dtype).view(_F32)


def _nd(a):
    return np.array(a, dtype=np.float32).view(_F32)


def _step_functions(fname, cls, names):
    """The named methods of class `cls` in the reference file, compiled from the reference source."""
    src = open(os.path.join(REF, "python/mxnet/optimizer", fname)).read()
    tree = ast.parse(src)
    import math
    shim = {
        "math": math,
        "clip": lambda x, lo, hi: np.clip(x, np.float32(lo), np.float32(hi)).view(_F32),
        "sqrt": lambda x, out=None: np.sqrt(x, out=out),
        "square": lambda x: np.square(x),
        "maximum": lambda a, b: np.maximum(a, np.float32(b)).view(_F32),
        "minimum": lambda a, b: np.minimum(a, np.float32(b)).view(_F32),
        "where": lambda c, x, y: np.where(np.asarray(c) != 0, x, y).view(_F32),   # NaN counts as true
        "ones_like": lambda x: np.ones_like(x),
        "NDnorm": lambda v: v.norm(),
    }
    fns = {}
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name == cls:
            for item in node.body:
                if isinstance(item, ast.FunctionDef) and item.name in names:
                    ns = dict(shim)
                    exec(compile(ast.Module([item], []), "reference:python/mxnet/optimizer/" + fname, "exec"), ns)
                    fns[item.name] = ns[item.name]
    assert set(fns) == set(names), (fname, sorted(fns))
    return fns


class _FakeOptimizer(object):
    """The attributes `step` reads from `self` (python/mxnet/optimizer/optimizer.py)."""

    def __init__(self, fns, lr, wd, **attrs):
        self.lr, self.wd = lr, wd
        self.rescale_grad, self.clip_gradient = 1.0, None
        self._index_update_count = {}
        self.idx2name = {}
        self.__dict__.update(attrs)
        for name, fn in fns.items():
            setattr(self, name, fn.__get__(self))

    def _update_count(self, index):
        self._index_update_count[index] = self._index_update_count.get(index, 0) + 1

    def _get_lr(self, index):
        return self.lr

    def _get_wd(self, index):
        return self.wd


def layerwise():
    out = {}
    shapes = [(3, 4, 5), (10, 4), (7,)]                       # test_optimizer.py:235,261,291
    lamb = _step_functions("lamb.py", "LAMB", ["step"])
    lans = _step_functions("lans.py", "LANS", ["step"])
    lars = _step_functions("lars.py", "LARS", ["step", "_get_lars", "_l2norm"])
    cases = []
    for bc in (True, False):
        for extra in (dict(), dict(beta1=0.5, beta2=0.8, clip_gradient=0.4, rescale_grad=0.14, wd=0.03,
                                   lower_bound=1e-3, upper_bound=10.0)):
            cases.append(("lamb", lamb, dict(bias_correction=bc, **extra)))
    for extra in (dict(), dict(beta1=0.5, beta2=0.8, clip_gradient=0.4, rescale_grad=0.14, wd=0.03,
                               lower_bound=1e-3, upper_bound=10.0)):
        cases.append(("lans", lans, dict(extra)))
    for mom in (0.0, 0.9):
        for extra in (dict(), dict(eta=0.01, clip_gradient=0.4, rescale_grad=0.14, wd=0.05)):
            cases.append(("lars", lars, dict(momentum=mom, **extra)))
    rng = np.random.default_rng(20260922)
    meta = []
    for ci, (name, fns, kw) in enumerate(cases):
        kw = dict(kw)
        wd = kw.pop("wd", 0.0)
        lr = 0.1 if name == "lars" else 0.01
        attrs = dict(beta1=0.9, beta2=0.999, epsilon=1e-8 if name == "lars" else 1e-6, lower_bound=None,
                     upper_bound=None, bias_correction=True, momentum=0.0, eta=0.001)
        attrs.update(kw)
        for si, shape in enumerate(shapes):
            opt = _FakeOptimizer(fns, lr, wd, **attrs)
            w = _nd(rng.uniform(-1, 1, shape))
            if name == "lars":
                state = _nd(np.zeros(shape)) if attrs["momentum"] != 0.0 else None
            else:
                state = (_nd(np.zeros(shape)), _nd(np.zeros(shape)))
            tag = "c%d_s%d" % (ci, si)
            out["w0_" + tag] = np.asarray(w).copy()
            for t in range(4):
                g = rng.uniform(-1, 1, shape).astype(np.float32)
                out["g%d_%s" % (t, tag)] = g
                opt.step([0], [w], [_nd(g)], [state])
                out["w%d_%s" % (t + 1, tag)] = np.asarray(w).copy()
        meta.append(repr((name, lr, wd, {k: v for k, v in attrs.items()})))
    out["cases"] = np.array(meta)
    np.savez_compressed(os.path.join(HERE, "layerwise.npz"), **out)


def plain_steps():
    """SGD / SGD-momentum / Adam / AdamW / Test: the reference's `step` methods (sgd.py:118-154,
    adam.py:107-147, adamW.py:98-140, optimizer.py:570-577) executed the same way -> optimizer_steps.npz."""
    out = {}
    sgd = _step_functions("sgd.py", "SGD", ["step"])
    adam = _step_functions("adam.py", "Adam", ["step"])
    test = _step_functions("optimizer.py", "Test", ["step"])
    adamw = _step_functions("adamW.py", "AdamW", ["step"])
    cases = [("adamw", adamw, 0.01, dict(beta1=0.9, beta2=0.999, epsilon=1e-6, wd=0.03, correct_bias=True)),
             ("adamw", adamw, 0.01, dict(beta1=0.7, beta2=0.9, epsilon=1e-6, wd=0.05, correct_bias=False,
                                         rescale_grad=0.8, clip_gradient=0.5)),
             ("sgd", sgd, 0.1, dict(momentum=0.0, wd=1e-3, rescale_grad=0.5)),
             ("sgd", sgd, 0.1, dict(momentum=0.9, wd=1e-3, rescale_grad=0.5)),
             ("sgd", sgd, 0.05, dict(momentum=0.9, wd=1e-4, rescale_grad=0.25, clip_gradient=0.4)),
             ("adam", adam, 0.01, dict(beta1=0.9, beta2=0.999, epsilon=1e-8, wd=1e-3, rescale_grad=0.5,
                                       clip_gradient=0.8)),
             ("adam", adam, 0.001, dict(beta1=0.5, beta2=0.8, epsilon=1e-8, wd=0.0)),
             ("test", test, 0.01, dict(wd=0.01, rescale_grad=0.5))]
    cases = cases[2:] + cases[:2]      # keep the indices of the earlier cases stable
    rng = np.random.default_rng(20260923)
    meta = []
    for ci, (name, fns, lr, kw) in enumerate(cases):
        kw = dict(kw)
        wd = kw.pop("wd", 0.0)
        for si, shape in enumerate([(3, 4, 5), (10, 4), (1001,)]):
            opt = _FakeOptimizer(fns, lr, wd, **kw)
            w = _nd(rng.uniform(0, 1, shape))
            if name == "sgd":
                state = _nd(np.zeros(shape)) if kw["momentum"] != 0.0 else None
            elif name in ("adam", "adamw"):
                state = (_nd(np.zeros(shape)), _nd(np.zeros(shape)))
            else:
                state = None
            tag = "c%d_s%d" % (ci, si)
            out["w0_" + tag] = np.asarray(w).copy()
            for t in range(5):
                g = rng.uniform(-1, 1, shape).astype(np.float32)
                out["g%d_%s" % (t, tag)] = g
                opt.step([0], [w], [_nd(g)], [state])
                out["w%d_%s" % (t + 1, tag)] = np.asarray(w).copy()
        meta.append(repr((name, lr, wd, kw)))
    out["cases"] = np.array(meta)
    np.savez_compressed(os.path.join(HERE, "optimizer_steps.npz"), **out)


def sparse_steps():
    """sparse_steps.npz -- pins the restatement of the sparse (lazy and standard) kernels (SURVEY 8 row a28):
    the classes the reference's tests compare those kernels with are executed from the reference's test file."""
    import math
    src = open(os.path.join(REF, "tests/python/unittest/test_optimizer.py")).read()
    tree = ast.parse(src)

    class _NDShim(object):
        @staticmethod
        def clip(x, lo, hi, out=None):
            r = np.clip(np.asarray(x), np.float32(lo), np.float32(hi))
            if out is not None:
                out[...] = r
                return out
            return r.view(_F32)

        @staticmethod
        def square(x, out=None):
            r = np.square(np.asarray(x))
            if out is not None:
                out[...] = r
                return out
            return r.view(_F32)

        @staticmethod
        def sqrt(x, out=None):
            return np.sqrt(np.asarray(x)).view(_F32)

    class _TestUtils(object):
        @staticmethod
        def almost_equal(a, b, rtol=None, atol=None):      # python/mxnet/test_utils.py:629-635,171-177 (float64 defaults)
            return bool(np.allclose(a, b, rtol=1e-5 if rtol is None else rtol, atol=1e-20 if atol is None else atol))

    class _MX(object):
        nd = _NDShim
        test_utils = _TestUtils

    def grab(cls):
        for node in tree.body:
            if isinstance(node, ast.ClassDef) and node.name == cls:
                for item in node.body:
                    if isinstance(item, ast.FunctionDef) and item.name == "step":
                        ns = {"mx": _MX, "np": np, "math": math}
                        exec(compile(ast.Module([item], []), "reference:tests/python/unittest/test_optimizer.py", "exec"), ns)
                        return {"step": ns["step"]}
        raise KeyError(cls)

    class _RowView(_F32):
        """`x[row]` of an NDArray is a writable view with .asnumpy()"""
        def asnumpy(self):
            return np.asarray(self)

    def nd(a):
        return np.array(a, dtype=np.float32).view(_RowView)

    py_sgd, py_adam = grab("PySparseSGD"), grab("PySparseAdam")
    dense_sgd = _step_functions("sgd.py", "SGD", ["step"])
    out, meta = {}, []
    rng = np.random.default_rng(20260924)
    cases = []
    for mom in (0.0, 0.9):
        for extra in (dict(), dict(clip_gradient=0.4, rescale_grad=0.14, wd=0.03)):
            cases.append(("sgd_lazy", py_sgd, 0.1, dict(momentum=mom, **extra)))
            cases.append(("sgd_std", dense_sgd, 0.1, dict(momentum=mom, **extra)))
    for lazy in (True, False):
        for extra in (dict(), dict(beta1=0.5, beta2=0.8, clip_gradient=0.4, rescale_grad=0.14, wd=0.03)):
            cases.append(("adam_lazy" if lazy else "adam_std", py_adam, 0.01, dict(lazy_update=lazy, **extra)))
    for ci, (name, fns, lr, kw) in enumerate(cases):
        kw = dict(kw)
        wd = kw.pop("wd", 0.0)
        attrs = dict(beta1=0.9, beta2=0.999, epsilon=1e-8, momentum=0.0, lazy_update=False)
        attrs.update(kw)
        for si, shape in enumerate([(10, 4), (37, 6)]):
            opt = _FakeOptimizer(fns, lr, wd, **attrs)
            w = nd(rng.uniform(-1, 1, shape))
            if name.startswith("sgd"):
                state = nd(np.zeros(shape)) if attrs["momentum"] != 0.0 else None
            else:
                state = (nd(np.zeros(shape)), nd(np.zeros(shape)))
            tag = "c%d_s%d" % (ci, si)
            out["w0_" + tag] = np.asarray(w).copy()
            for t in range(4):
                rows = np.sort(rng.choice(shape[0], max(1, shape[0] // 3), replace=False))
                g = np.zeros(shape, np.float32)
                g[rows] = rng.uniform(-1, 1, (len(rows),) + shape[1:]).astype(np.float32)
                # keep every present row clearly non-zero: the references skip rows that are `almost_equal` to zero
                g[rows, 0] = np.where(np.abs(g[rows, 0]) < 0.05, 0.5, g[rows, 0])
                out["rows%d_%s" % (t, tag)] = rows.astype(np.int64)
                out["g%d_%s" % (t, tag)] = g.copy()
                opt.step([0], [w], [nd(g)], [state])
                out["w%d_%s" % (t + 1, tag)] = np.asarray(w).copy()
        meta.append(repr((name, lr, wd, attrs)))
    out["cases"] = np.array(meta)
    np.savez_compressed(os.path.join(HERE, "sparse_steps.npz"), **out)


LR_CASES = [
    ("FactorScheduler", dict(step=7, factor=0.5, base_lr=0.3)),
    ("FactorScheduler", dict(step=3, factor=0.1, stop_factor_lr=1e-4, base_lr=0.1, warmup_steps=5, warmup_begin_lr=0.01)),
    ("MultiFactorScheduler", dict(step=[4, 9, 30], factor=0.3, base_lr=0.2)),
    ("MultiFactorScheduler", dict(step=[10, 20], factor=0.5, base_lr=1.0, warmup_steps=6, warmup_mode="constant",
                                  warmup_begin_lr=0.1)),
    ("PolyScheduler", dict(max_update=40, base_lr=0.05, pwr=2, final_lr=1e-4)),
    ("PolyScheduler", dict(max_update=30, base_lr=0.4, pwr=1, warmup_steps=8)),
    ("CosineScheduler", dict(max_update=45, base_lr=0.1, final_lr=0.001)),
    ("CosineScheduler", dict(max_update=25, base_lr=0.7, warmup_steps=5, warmup_begin_lr=0.2)),
]


def lr_schedules():
    """lr_schedules.npz: python/mxnet/lr_scheduler.py imported from the reference tree and called with
    num_update = 0..59 (and once more out of order, for the stateful classes)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_lr_scheduler", os.path.join(REF, "python/mxnet/lr_scheduler.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    out = {}
    for i, (cls, kw) in enumerate(LR_CASES):
        s = getattr(ref, cls)(**kw)
        out["seq_%d" % i] = np.array([s(n) for n in range(60)], np.float64)
        s2 = getattr(ref, cls)(**kw)                      # a resumed run jumps straight to a late update
        out["jump_%d" % i] = np.array([s2(37), s2(38), s2(59)], np.float64)
    np.savez_compressed(os.path.join(HERE, "lr_schedules.npz"), **out)


P3_16XLARGE = [[0, 2, 2, 3, 3, 1, 1, 1], [2, 0, 3, 2, 1, 3, 1, 1], [2, 3, 0, 3, 1, 1, 2, 1], [3, 2, 3, 0, 1, 1, 1, 2],
               [3, 1, 1, 1, 0, 2, 2, 3], [1, 3, 1, 1, 2, 0, 3, 2], [1, 1, 2, 1, 2, 3, 0, 3], [1, 1, 1, 2, 3, 2, 3, 0]]


def tree_topology():
    """Link matrices and what the reference's solver makes of them.  case_i_W / _alpha / _backtrack -> _topo / _scan
    (or _fails = 1 where the reference aborts: no balanced binary tree over those links)."""
    import ctypes
    from oracle import oracle as O
    lib = O.ref_topology_lib()
    assert lib is not None, "build oracle/_ref first (make -C oracle)"
    rng = np.random.default_rng(20260921)
    cases = []
    for n in range(2, 9):                                   # behind one switch: every pair alike
        for w in (1.0, 2.0, 3.0):
            for bt in (0, 1):
                cases.append((w * (np.ones((n, n)) - np.eye(n)), 0.7, bt))
    p3 = np.array(P3_16XLARGE, np.float64)
    for bt in (0, 1):                                       # gpu_topology.h:181-190, PCI-E kept (1) and dropped (0)
        cases.append((p3, 0.7, bt))
        cases.append((np.where(p3 == 1, 0.0, p3), 0.7, bt))
        cases.append((p3, 0.5, bt))
    for n in range(2, 17):                                  # the shape of TestComputeTrees1/2's random matrices
        for rep in range(4):
            u = rng.uniform(0, 1, (n, n))
            W = np.where(u < 0.33, 1.0, np.where(u < 0.66, 2.0, 3.0))
            if rep == 3:
                W = np.where(rng.uniform(0, 1, (n, n)) < 0.25, 0.0, W)
            W = np.triu(W, 1)
            W = W + W.T
            for bt in ((0, 1) if n <= 8 else (0,)):
                cases.append((W, 0.7, bt))
    out = {"n_cases": np.array(len(cases))}
    fails = 0
    for i, (W, alpha, bt) in enumerate(cases):
        out["case_%d_W" % i] = W.astype(np.float32)
        out["case_%d_alpha" % i] = np.float32(alpha)
        out["case_%d_backtrack" % i] = np.array(bt)
        r = O.ref_compute_trees(W, alpha, bool(bt))
        if r is None:
            out["case_%d_fails" % i] = np.array(1)
            fails += 1
        else:
            out["case_%d_topo" % i], out["case_%d_scan" % i] = r[0].astype(np.int16), r[1].astype(np.int16)
    # one Kernighan-Lin pass from a single cluster, seeds 1 ... 4 (TestKernighanLin1/2 call it with seed 1)
    kl = []
    for n in (5, 6, 8, 11, 16):
        for seed in (1, 2, 3, 4):
            u = rng.uniform(0, 1, (n, n))
            W = np.triu(np.where(u < 0.4, 1.0, np.where(u < 0.7, 2.0, 4.0)), 1)
            W = (W + W.T).astype(np.float32)
            P = np.zeros(n, np.int32)
            npart = ctypes.c_int(1)
            pairs = np.zeros(4 * n, np.int32)
            npairs = ctypes.c_int()
            stop = lib.kvref_topo_kernighan_lin(ctypes.c_void_p(W.ctypes.data), n, ctypes.c_void_p(P.ctypes.data),
                                                ctypes.byref(npart), ctypes.c_void_p(pairs.ctypes.data),
                                                ctypes.byref(npairs), ctypes.c_uint32(seed))
            kl.append((W, seed, P.copy(), npart.value, pairs[:2 * npairs.value].copy(), stop))
    out["n_kl"] = np.array(len(kl))
    for i, (W, seed, P, npart, pairs, stop) in enumerate(kl):
        out["kl_%d_W" % i], out["kl_%d_seed" % i], out["kl_%d_P" % i] = W, np.array(seed), P
        out["kl_%d_npart" % i], out["kl_%d_pairs" % i], out["kl_%d_stop" % i] = np.array(npart), pairs, np.array(stop)
    np.savez_compressed(os.path.join(HERE, "tree_topology.npz"), **out)
    print("tree_topology: %d matrices (%d without a tree), %d Kernighan-Lin passes" % (len(cases), fails, len(kl)))


def _digest(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def reference_sums():
    """The reference's CommDevice / CommCPU sums of the inputs test_dense_sum_against_live_reference_arithmetic draws
    (seed 5, n = 2 ... 13 values of E elements).  `<kind>_E<E>` [case, i]: the value at idx_E<E>[i] (every element
    up to 64, a seeded sample above); `<kind>_E<E>_sha256` [case]: the SHA-256 of the whole output, so that the test
    still compares every bit."""
    from oracle import oracle as O
    assert O.ref_lib() is not None, "build oracle/_ref first (make -C oracle)"
    rng = np.random.default_rng(5)
    out = {}
    for n in (2, 3, 4, 5, 6, 8, 9, 13):
        for E in (1, 17, 5000):
            idx = out.setdefault("idx_E%d" % E, (np.arange(E) if E <= 64 else np.sort(
                np.random.default_rng(E).choice(E, 64, replace=False))).astype(np.int64))
            vals = [rng.uniform(-1, 1, E).astype(np.float32) for _ in range(n)]
            for kind, s in (("device_f32", O.ref_sum_device(vals)), ("commcpu_f32", O.ref_sum_cpu(vals)),
                            ("device_f64", O.ref_sum_device([v.astype(np.float64) for v in vals])),
                            ("device_i32", O.ref_sum_device([(v * 1000).astype(np.int32) for v in vals]))):
                out.setdefault("%s_E%d" % (kind, E), []).append(s[idx])
                out.setdefault("%s_E%d_sha256" % (kind, E), []).append(_digest(s))
    np.savez_compressed(os.path.join(HERE, "reference_sums.npz"), **{k: np.stack(v) if isinstance(v, list) else v
                                                                     for k, v in out.items()})


def tree_draw():
    """The trees the reference's solver builds for the fixed draw of link matrices in
    test_trees_match_the_reference_header_compiled_in_place (seed 20260921), case after case: W, alpha, backtrack,
    and topo / scan, each case's rows of topo_len / scan_len elements, flattened; a case the reference aborts on
    (no balanced binary tree) has lengths 0."""
    from oracle import oracle as O
    assert O.ref_topology_lib() is not None, "build oracle/_ref first (make -C oracle)"
    sys.path.insert(0, os.path.dirname(HERE))
    from test_topology import link_matrix_draw
    cols = {k: [] for k in ("W", "alpha", "backtrack", "topo", "scan", "topo_len", "scan_len")}
    for W, alpha, bt in link_matrix_draw(np.random.default_rng(20260921)):
        r = O.ref_compute_trees(W, alpha, bt)
        topo, scan = (np.zeros((0, 0), np.int16),) * 2 if r is None else (r[0].astype(np.int16), r[1].astype(np.int16))
        for k, v in (("W", W.ravel()), ("alpha", [alpha]), ("backtrack", [bt]), ("topo", topo.ravel()),
                     ("scan", scan.ravel()), ("topo_len", [topo.shape[1]]), ("scan_len", [scan.shape[1]])):
            cols[k].append(np.asarray(v))
    np.savez_compressed(os.path.join(HERE, "tree_draw.npz"), **{k: np.concatenate(v) for k, v in cols.items()})


def c_api_prototypes():
    """Parameter types of every entry point the reference's include/mxnet/c_api.h declares (test_abi.py::c_prototypes),
    so that an entry point include/mxkv_b200.h adds later is checked too."""
    sys.path.insert(0, os.path.dirname(HERE))
    from test_abi import c_prototypes
    ref = c_prototypes(os.path.join(REF, "include", "mxnet", "c_api.h"), "MXNET_DLL")
    with open(os.path.join(HERE, "c_api_prototypes.json"), "w") as f:
        json.dump(ref, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    if len(sys.argv) > 1:                 # e.g. `make_golden.py tree_topology`: only the named fixtures
        for name in sys.argv[1:]:
            globals()[name]()
        sys.exit(0)
    dense_sums()
    compression()
    layerwise()
    plain_steps()
    sparse_steps()
    lr_schedules()
    tree_topology()
    reference_sums()
    tree_draw()
    c_api_prototypes()
    print("wrote", sorted(f for f in os.listdir(HERE) if f.endswith((".npz", ".json"))))

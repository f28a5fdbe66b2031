"""CPU tests that pin the oracle (test infrastructure) to the reference:
golden vectors produced by the reference's own arithmetic / simulators, the reference's
scenario-level known answers, and an independent restatement of the reference's non-fused
Python optimizer steps (the reference's own oracle for its fused kernels)."""
import hashlib
import os

import numpy as np
import pytest

from oracle import oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _eq_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    v = {2: np.uint16, 4: np.uint32, 8: np.uint64, 1: np.uint8}[a.dtype.itemsize]
    return np.array_equal(a.view(v), b.view(v))


def test_dense_sum_golden_vectors():
    g = np.load(os.path.join(GOLD, "dense_sums.npz"))
    tags = sorted(k[3:] for k in g.files if k.startswith("in_"))
    assert len(tags) == 18
    for tag in tags:
        vals = [np.ascontiguousarray(v) for v in g["in_" + tag]]
        assert _eq_bits(O.sum_device(vals), g["device_f32_" + tag]), tag
        assert _eq_bits(O.sum_cpu(vals), g["commcpu_f32_" + tag]), tag
        assert _eq_bits(O.sum_device([v.astype(np.float16) for v in vals]), g["device_f16_" + tag]), tag
    rng = np.random.default_rng(int(g["seed_big"][0]))
    vals = [rng.uniform(-1, 1, 1000003).astype(np.float32) for _ in range(5)]
    s = O.sum_cpu(vals)       # takes the OpenMP branch (>= MXNET_KVSTORE_BIGARRAY_BOUND)
    assert _eq_bits(s[:4096], g["commcpu_f32_big_head"])
    assert _eq_bits(s[-4096:], g["commcpu_f32_big_tail"])
    assert np.bitwise_xor.reduce(s.view(np.uint32)) == g["commcpu_f32_big_xor"][0]


def test_dense_sum_against_live_reference_arithmetic():
    """tests/golden/reference_sums.npz: what the reference's own arithmetic (oracle/_ref/libkvref.so,
    make_golden.py::reference_sums) returned for these inputs -- sampled values and the SHA-256 of every output."""
    g = np.load(os.path.join(GOLD, "reference_sums.npz"))
    rng = np.random.default_rng(5)
    for case, n in enumerate((2, 3, 4, 5, 6, 8, 9, 13)):
        for E in (1, 17, 5000):
            vals = [rng.uniform(-1, 1, E).astype(np.float32) for _ in range(n)]
            idx = g["idx_E%d" % E]
            for kind, s in (("device_f32", O.sum_device(vals)), ("commcpu_f32", O.sum_cpu(vals)),
                            ("device_f64", O.sum_device([v.astype(np.float64) for v in vals])),
                            ("device_i32", O.sum_device([(v * 1000).astype(np.int32) for v in vals]))):
                assert _eq_bits(s[idx], g["%s_E%d" % (kind, E)][case]), (kind, n, E)
                digest = hashlib.sha256(np.ascontiguousarray(s).tobytes()).digest()
                assert digest == g["%s_E%d_sha256" % (kind, E)][case].tobytes(), (kind, n, E)


def test_compression_golden_vectors():
    g = np.load(os.path.join(GOLD, "compression.npz"))
    for kind, thr in (("2bit", 0.5), ("1bit", 0.0)):
        for E in (32, 64, 160):
            for it in range(3):
                tag = "%s_E%d_it%d" % (kind, E, it)
                grad = np.ascontiguousarray(g["grad_" + tag])
                res = np.ascontiguousarray(g["res_in_" + tag]).copy()
                if kind == "2bit":
                    comp = O.quantize_2bit(grad, res, thr)
                    dec = O.dequantize_2bit(comp, E, thr)
                else:
                    comp = O.quantize_1bit(grad, res, thr)
                    dec = O.dequantize_1bit(comp, E, thr)
                assert np.array_equal(comp, g["bytes_" + tag]), tag
                assert _eq_bits(res, g["res_out_" + tag]), tag
                assert _eq_bits(dec, g["dec_" + tag]), tag


# ---- reference scenario KATs against the oracle KVStore model --------------------------------
SHAPE = (4, 4)
KEYS = [5, 7, 11]
STR_KEYS = ["b", "c", "d"]


def _init_kv(kind="local", str_keys=False):
    kv = O.OracleKVStore(kind)
    if str_keys:
        kv.init("a", np.zeros(SHAPE, np.float32))
        kv.init(STR_KEYS, [np.zeros(SHAPE, np.float32)] * 3)
    else:
        kv.init(3, np.zeros(SHAPE, np.float32))
        kv.init(KEYS, [np.zeros(SHAPE, np.float32)] * 3)
    return kv


def test_kat_single_kv_pair_and_init():
    # tests/python/unittest/test_kvstore.py:55-66, 96-105
    for s in (False, True):
        kv = _init_kv(str_keys=s)
        key = "a" if s else 3
        kv.push(key, np.ones(SHAPE, np.float32))
        val = np.empty(SHAPE, np.float32)
        kv.pull(key, val)
        assert np.all(val == 1)
    kv = O.OracleKVStore("local")
    kv.init(3, np.ones(SHAPE, np.float32) * 4)
    a = np.zeros(SHAPE, np.float32)
    kv.pull(3, a)
    assert np.all(a == 4)


def test_kat_pull_and_list():
    # test_kvstore.py:107-136
    for kind in ("device", "local"):
        kv = O.OracleKVStore(kind)
        a, b = np.ones(SHAPE, np.float32), np.zeros(SHAPE, np.float32)
        kv.init("1", np.zeros(SHAPE, np.float32))
        kv.push("1", [a, a, a, a])
        kv.pull("1", b)
        assert np.all(b == 4)
        kv.init("2", np.zeros(SHAPE, np.float32))
        kv.pull("2", b)
        assert np.all(b == 0)
    kv = _init_kv()
    kv.push(KEYS, [np.ones(SHAPE, np.float32) * 4] * 3)
    val = [np.empty(SHAPE, np.float32) for _ in KEYS]
    kv.pull(KEYS, val)
    assert all(np.all(v == 4) for v in val)


def test_kat_updater():
    # test_kvstore.py:222-274: updater local += recv, 4 devices, 4 pushes -> num_devs * num_push
    for s in (False, True):
        kv = _init_kv(str_keys=s)
        kv.set_updater(lambda k, recv, local: np.add(local, recv, out=local))
        key, klist = ("a", STR_KEYS) if s else (3, KEYS)
        vals = [np.ones(SHAPE, np.float32) for _ in range(4)]
        kv.push(key, vals)
        outs = [np.empty(SHAPE, np.float32) for _ in range(4)]
        kv.pull(key, outs)
        assert all(np.all(o == 4) for o in outs)
        for _ in range(4):
            kv.push(klist, [vals] * 3)
        outs = [[np.empty(SHAPE, np.float32) for _ in range(4)] for _ in klist]
        kv.pull(klist, outs)
        assert all(np.all(o == 16) for oo in outs for o in oo)


def test_kat_key_type_mixing_and_duplicates():
    # test_kvstore.py:281-339, kvstore_local.h:230-233,344-347
    kv = _init_kv()
    with pytest.raises(ValueError):
        kv.init("a", np.zeros(SHAPE, np.float32))
    with pytest.raises(ValueError):
        kv.push("a", np.zeros(SHAPE, np.float32))
    with pytest.raises(ValueError):
        kv.init(3, np.zeros(SHAPE, np.float32))
    kv = _init_kv(str_keys=True)
    with pytest.raises(ValueError):
        kv.pull(3, np.zeros(SHAPE, np.float32))


def test_kat_row_sparse_pull():
    # test_kvstore.py:68-94 and the docstring of kvstore.py:row_sparse_pull
    kv = O.OracleKVStore("local")
    kv.init("e", O.RowSparse.from_dense(np.ones(SHAPE, np.float32)))
    rng = np.random.default_rng(0)
    for _ in range(5):
        row_id = rng.integers(0, SHAPE[0], SHAPE[0])
        out = O.RowSparse(np.zeros(0, np.int64), np.zeros((0, SHAPE[1]), np.float32), SHAPE)
        kv.row_sparse_pull("e", out, row_id.reshape(2, -1))
        dense = out.todense()
        for r in range(SHAPE[0]):
            assert np.all(dense[r] == (1 if r in row_id else 0))


def test_kat_nightly_test_optimizer():
    # tests/nightly/test_kvstore.py:100-119,297-343: 4 workers, random uniform[-1,1), the 'test'
    # optimizer; expectation restated from python/mxnet/optimizer/optimizer.py:570-577
    rng = np.random.default_rng(1)
    lr = 0.01  # Optimizer default learning_rate
    rescale = 0.1
    for shape in ((4, 4), (100, 100), (2000, 2000)):
        kv = O.OracleKVStore("device")
        kv.init(9, np.zeros(shape, np.float32))
        kv.set_optimizer(O.OracleOptimizer("test", rescale_grad=rescale))
        res = np.zeros(shape, np.float64)
        for _ in range(3):
            data = [rng.uniform(-1, 1, shape).astype(np.float32) for _ in range(4)]
            kv.push(9, data)
            res = res - lr * rescale * sum(d.astype(np.float64) for d in data)
        out = np.empty(shape, np.float32)
        kv.pull(9, out)
        err = np.sum(np.abs(out - res)) / np.sum(np.abs(res))
        assert err < 1e-6, (err, shape)


# ---- optimizer kernels vs. an independent restatement of the reference's Python step() ---------
def _np_sgd_step(w, g, mom, lr, wd, momentum, rescale, clip):
    # python/mxnet/optimizer/sgd.py:118-154 (NDArray ops = separate fp32 elementwise ops)
    g = (g * np.float32(rescale)).astype(np.float32)
    if clip is not None:
        g = np.clip(g, -clip, clip).astype(np.float32)
    g = (g + np.float32(wd) * w).astype(np.float32)
    if mom is not None:
        mom *= np.float32(momentum)
        mom -= np.float32(lr) * g
        w += mom
    else:
        w += -np.float32(lr) * g


def _np_adam_step(w, g, mean, var, lr, wd, b1, b2, eps, rescale, clip, t):
    # python/mxnet/optimizer/adam.py:107-147
    import math
    g = (g * np.float32(rescale)).astype(np.float32)
    if clip is not None:
        g = np.clip(g, -clip, clip).astype(np.float32)
    g = (g + np.float32(wd) * w).astype(np.float32)
    lr = lr * math.sqrt(1. - b2 ** t) / (1. - b1 ** t)
    mean *= np.float32(b1)
    mean += np.float32(1. - b1) * g
    var *= np.float32(b2)
    var += np.float32(1. - b2) * np.square(g)
    w -= np.float32(lr) * (mean / (np.sqrt(var) + np.float32(eps)))


@pytest.mark.parametrize("momentum,clip", [(0.0, None), (0.9, None), (0.9, 0.4)])
def test_sgd_kernel_vs_python_step(momentum, clip):
    # tolerances of tests/python/unittest/test_optimizer.py:75-84 (rtol 1e-3 / atol 1e-4) -- the
    # restatements in fact agree to ~1 ulp
    rng = np.random.default_rng(11)
    E = 10007
    w = rng.uniform(0, 1, E).astype(np.float32); w2 = w.copy()
    mom = np.zeros(E, np.float32) if momentum else None
    opt = O.OracleOptimizer("sgd", learning_rate=0.1, wd=1e-3, momentum=momentum, rescale_grad=0.5,
                            clip_gradient=clip)
    for _ in range(5):
        g = rng.uniform(-1, 1, E).astype(np.float32)
        opt.update(0, w, g.copy())
        _np_sgd_step(w2, g.copy(), mom, 0.1, 1e-3, momentum, 0.5, clip)
        np.testing.assert_allclose(w, w2, rtol=1e-3, atol=1e-4)
        assert np.max(np.abs(w - w2)) < 1e-6


def test_adam_kernel_vs_python_step():
    # tolerances of test_optimizer.py:461-463 (rtol 1e-4 / atol 2e-5)
    rng = np.random.default_rng(12)
    E = 10007
    w = rng.uniform(0, 1, E).astype(np.float32); w2 = w.copy()
    mean, var = np.zeros(E, np.float32), np.zeros(E, np.float32)
    opt = O.OracleOptimizer("adam", learning_rate=0.01, wd=1e-3, rescale_grad=0.5, clip_gradient=0.8)
    for t in range(1, 6):
        g = rng.uniform(-1, 1, E).astype(np.float32)
        opt.update(0, w, g.copy())
        _np_adam_step(w2, g.copy(), mean, var, 0.01, 1e-3, 0.9, 0.999, 1e-8, 0.5, 0.8, t)
        np.testing.assert_allclose(w, w2, rtol=1e-4, atol=2e-5)


# ---- LAMB / LANS / LARS: the fused-kernel restatement against a transcription of the reference's
# ---- non-fused Python ``step`` -- the comparison tests/python/unittest/test_optimizer.py:232-312 makes
def _norm32(x):
    return np.sqrt(np.sum(np.square(x.astype(np.float32)), dtype=np.float32), dtype=np.float32)


def _trust(r1, r2):
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.float32(r1) / np.float32(r2)
    return np.float32(1.0) if (not np.isfinite(ratio) or ratio == 0) else ratio


def _np_lamb_step(w, g, mean, var, lr, wd, t, b1, b2, eps, rescale, clip, bias_correction, lb, ub):
    """lamb.py:93-150 on float32 arrays."""
    f = np.float32
    g = g * f(rescale)
    if clip is not None:
        g = np.clip(g, -f(clip), f(clip))
    mean *= f(b1); mean += f(1. - b1) * g
    var *= f(b2); var += f(1. - b2) * np.square(g)
    r1 = _norm32(w)
    if lb is not None:
        r1 = max(r1, f(lb))
    if ub is not None:
        r1 = min(r1, f(ub))
    if bias_correction:
        mean_hat = mean / f(1. - b1 ** t)
        var_hat = var / f(1. - b2 ** t)
        var_hat = np.sqrt(var_hat) + f(eps)
        mean_hat = mean_hat / var_hat + f(wd) * w
    else:
        mean_hat = mean / (np.sqrt(var) + f(eps)) + f(wd) * w
    r = _trust(r1, _norm32(mean_hat))
    w -= mean_hat * f(lr * r)


def _np_lans_step(w, g, mean, var, lr, wd, t, b1, b2, eps, rescale, clip, lb, ub):
    """lans.py:86-150."""
    f = np.float32
    g = g * f(rescale)
    g = g / _norm32(g)
    if clip is not None:
        g = np.clip(g, -f(clip), f(clip))
    mean *= f(b1); mean += f(1. - b1) * g
    var *= f(b2); var += f(1. - b2) * np.square(g)
    r1 = _norm32(w)
    if lb is not None:
        r1 = max(r1, f(lb))
    if ub is not None:
        r1 = min(r1, f(ub))
    mean_hat = mean / f(1. - b1 ** t)
    var_hat = np.sqrt(var / f(1. - b2 ** t)) + f(eps)
    m = mean_hat / var_hat + f(wd) * w
    r_m = _trust(r1, _norm32(m))
    # the reference's step() applies the two halves one after the other (the second sees the
    # already-updated weight in wd * weight); the fused kernel uses the old weight for both -- the
    # reference test accepts the difference at rtol/atol 1e-3
    w -= m * f(lr * r_m * b1)
    gg = g / var_hat + f(wd) * w
    r_g = _trust(r1, _norm32(gg))
    w -= gg * f(lr * r_g * (1 - b1))


def _np_lars_step(w, g, mom, lr, wd, momentum, eta, eps, rescale, clip, use_lars=True):
    """lars.py:117-133,135-175."""
    f = np.float32
    if use_lars:
        w_norm = _norm32(w)
        g_norm = _norm32(g * f(rescale))
        with np.errstate(divide="ignore", invalid="ignore"):
            ratio = w_norm / g_norm
        lars = f(eta) * w_norm / (g_norm + f(wd) * w_norm + f(eps))
        if not np.isfinite(ratio) or ratio == 0:
            lars = f(1.0)
        lr = lr * float(lars)
    g = g * f(rescale)
    if clip is not None:
        g = np.clip(g, -f(clip), f(clip))
    g = g + f(wd) * w
    if mom is not None:
        mom *= f(momentum); mom -= f(lr) * g
        w += mom
    else:
        w += -f(lr) * g


_SHAPES = [(3, 4, 5), (10, 4), (7,)]     # test_optimizer.py:235,261,291


@pytest.mark.parametrize("bias_correction", [False, True])
@pytest.mark.parametrize("bounds", [(None, None), (1e-3, 10)])
def test_lamb_kernel_vs_python_step(bias_correction, bounds):
    lb, ub = bounds
    for opts in (dict(), dict(beta1=0.5, beta2=0.8, clip_gradient=0.4, rescale_grad=0.14, wd=0.03)):
        for shape in _SHAPES:
            rng = np.random.default_rng(31)
            w = rng.uniform(-1, 1, shape).astype(np.float32); w2 = w.copy()
            mean, var = np.zeros(shape, np.float32), np.zeros(shape, np.float32)
            opt = O.OracleOptimizer("lamb", learning_rate=0.01, bias_correction=bias_correction, lower_bound=lb,
                                    upper_bound=ub, **opts)
            for t in range(1, 5):
                g = rng.uniform(-1, 1, shape).astype(np.float32)
                opt.update(0, w, g.copy())
                _np_lamb_step(w2, g.copy(), mean, var, 0.01, opts.get("wd", 0.0), t, opts.get("beta1", 0.9),
                              opts.get("beta2", 0.999), 1e-6, opts.get("rescale_grad", 1.0),
                              opts.get("clip_gradient"), bias_correction, lb, ub)
                np.testing.assert_allclose(w, w2, rtol=1e-3, atol=1e-3)
                assert np.max(np.abs(w - w2)) < 1e-5      # in fact the two restatements agree to ~1e-7
                np.testing.assert_allclose(opt.states[0][0], mean, rtol=1e-5, atol=1e-7)
                np.testing.assert_allclose(opt.states[0][1], var, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("bounds", [(None, None), (1e-3, 10)])
def test_lans_kernel_vs_python_step(bounds):
    lb, ub = bounds
    for opts in (dict(), dict(beta1=0.5, beta2=0.8, clip_gradient=0.4, rescale_grad=0.14, wd=0.03)):
        for shape in _SHAPES:
            rng = np.random.default_rng(32)
            w = rng.uniform(-1, 1, shape).astype(np.float32); w2 = w.copy()
            mean, var = np.zeros(shape, np.float32), np.zeros(shape, np.float32)
            opt = O.OracleOptimizer("lans", learning_rate=0.01, lower_bound=lb, upper_bound=ub, **opts)
            for t in range(1, 5):
                g = rng.uniform(-1, 1, shape).astype(np.float32)
                opt.update(0, w, g.copy())
                _np_lans_step(w2, g.copy(), mean, var, 0.01, opts.get("wd", 0.0), t, opts.get("beta1", 0.9),
                              opts.get("beta2", 0.999), 1e-6, opts.get("rescale_grad", 1.0),
                              opts.get("clip_gradient"), lb, ub)
                np.testing.assert_allclose(w, w2, rtol=1e-3, atol=1e-3)     # test_optimizer.py:310-312


@pytest.mark.parametrize("momentum", [0.0, 0.9])
def test_lars_kernel_vs_python_step(momentum):
    for opts in (dict(), dict(eta=0.01, clip_gradient=0.4, rescale_grad=0.14, wd=0.05)):
        for shape in _SHAPES:
            rng = np.random.default_rng(33)
            w = rng.uniform(-1, 1, shape).astype(np.float32); w2 = w.copy()
            mom = np.zeros(shape, np.float32) if momentum else None
            opt = O.OracleOptimizer("lars", learning_rate=0.1, momentum=momentum, **opts)
            for t in range(1, 5):
                g = rng.uniform(-1, 1, shape).astype(np.float32)
                opt.update(0, w, g.copy())
                _np_lars_step(w2, g.copy(), mom, 0.1, opts.get("wd", 0.0), momentum, opts.get("eta", 0.001), 1e-8,
                              opts.get("rescale_grad", 1.0), opts.get("clip_gradient"))
                np.testing.assert_allclose(w, w2, rtol=1e-3, atol=1e-3)     # test_optimizer.py:251-253
                assert np.max(np.abs(w - w2)) < 1e-6
    # names ending in gamma / beta / bias keep the plain learning rate (lars.py:121-123)
    rng = np.random.default_rng(34)
    w = rng.uniform(-1, 1, 50).astype(np.float32); w2 = w.copy()
    g = rng.uniform(-1, 1, 50).astype(np.float32)
    O.OracleOptimizer("lars", learning_rate=0.1, no_trust=[3]).update(3, w, g.copy())
    _np_lars_step(w2, g.copy(), None, 0.1, 0.0, 0.0, 0.001, 1e-8, 1.0, None, use_lars=False)
    assert np.max(np.abs(w - w2)) < 1e-6


def test_sum_sq_and_trust_ratio_edge_cases():
    rng = np.random.default_rng(35)
    x = rng.uniform(-1, 1, 100003).astype(np.float32)
    exact = float(np.sum(x.astype(np.float64) ** 2))
    assert abs(float(O.sum_sq(x, mode="f64")) - exact) <= 1e-7 * exact
    assert abs(float(O.sum_sq(x, mode="seq")) - exact) <= 1e-4 * exact      # sequential float sum drifts
    assert abs(float(O.sum_sq(x, 0.5, mode="f64")) - exact / 4) <= 1e-6 * exact
    assert O.count_nonfinite(np.array([1, np.inf, -np.inf, np.nan, 0], np.float32)) == 3
    # zero weight or zero update direction: ratio 1 (multi_lamb.cc:104-107)
    w = np.zeros(16, np.float32); g = np.ones(16, np.float32)
    opt = O.OracleOptimizer("lamb", learning_rate=0.5)
    opt.update(0, w, g)
    # step 1: m = 0.1 g, v = 0.001 g^2, bias-corrected -> ghat = 1/(1+eps); lr * 1 * ghat
    np.testing.assert_allclose(w, -0.5 / (1 + 1e-6), rtol=1e-6)
    # LARS with a zero gradient: ratio inf -> lars 1 -> plain sgd step (which is a no-op on g = 0, wd = 0)
    w = np.ones(8, np.float32)
    O.OracleOptimizer("lars", learning_rate=0.1).update(0, w, np.zeros(8, np.float32))
    assert np.all(w == 1)


def test_plain_optimizers_vs_reference_step_golden():
    """tests/golden/optimizer_steps.npz: weights produced by the reference's own `step` of SGD / Adam / AdamW /
    Test (sgd.py:118-154, adam.py:107-147, adamW.py:98-140, optimizer.py:570-577; make_golden.py::plain_steps).  Tolerances of
    tests/python/unittest/test_optimizer.py (:75-84 SGD rtol 1e-3 / atol 1e-4, :461-463 Adam rtol 1e-4 /
    atol 2e-5); the kernel restatement in fact agrees to a few ulp."""
    gold = np.load(os.path.join(GOLD, "optimizer_steps.npz"))
    cases = [eval(c) for c in gold["cases"]]
    for ci, (name, lr, wd, kw) in enumerate(cases):
        for si in range(3):
            tag = "c%d_s%d" % (ci, si)
            w = gold["w0_" + tag].copy()
            opt = O.OracleOptimizer(name, learning_rate=lr, wd=wd, **kw)
            for t in range(5):
                opt.update(0, w, gold["g%d_%s" % (t, tag)].copy())
                want = gold["w%d_%s" % (t + 1, tag)]
                if name == "adamw":
                    # AdamW.step applies `w -= lr*d` and then `w -= lr*wd*w` to the already-updated weight
                    # (adamW.py:135-140); the operator uses the old weight for the decay term
                    # (adamw-inl.h:118-120): they differ by lr^2 * wd * d.  The reference's own comparison of
                    # the two grants rtol/atol 1e-4 (test_contrib_optimizer.py:163-168)
                    np.testing.assert_allclose(w, want, rtol=1e-4, atol=1e-4, err_msg=str((name, ci, si, t)))
                    continue
                if name == "adam":
                    np.testing.assert_allclose(w, want, rtol=1e-4, atol=2e-5, err_msg=str((name, ci, si, t)))
                else:
                    np.testing.assert_allclose(w, want, rtol=1e-3, atol=1e-4, err_msg=str((name, ci, si, t)))
                assert np.max(np.abs(w - want)) < 2e-6, (name, ci, si, t, np.max(np.abs(w - want)))


def test_layerwise_oracle_vs_reference_step_golden():
    """tests/golden/layerwise.npz holds weights produced by the reference's OWN `step` methods of LAMB /
    LANS / LARS, executed from python/mxnet/optimizer/{lamb,lans,lars}.py (make_golden.py::layerwise).
    The fused-kernel restatement in oracle/ must agree with them within the tolerance the reference's
    tests grant its fused kernels against that same `step` (rtol = atol = 1e-3, test_optimizer.py:251-312);
    LAMB and LARS perform the same operations in both forms and agree to ~1e-7."""
    gold = np.load(os.path.join(GOLD, "layerwise.npz"))
    cases = [eval(c) for c in gold["cases"]]        # (name, lr, wd, attrs) literals written by make_golden.py
    shapes = 3
    worst = {"lamb": 0.0, "lans": 0.0, "lars": 0.0}
    for ci, (name, lr, wd, attrs) in enumerate(cases):
        for si in range(shapes):
            tag = "c%d_s%d" % (ci, si)
            w = gold["w0_" + tag].copy()
            kw = dict(learning_rate=lr, wd=wd, rescale_grad=attrs.get("rescale_grad", 1.0),
                      clip_gradient=attrs.get("clip_gradient"), epsilon=attrs["epsilon"])
            if name == "lars":
                kw.update(momentum=attrs["momentum"], eta=attrs["eta"])
            else:
                kw.update(beta1=attrs["beta1"], beta2=attrs["beta2"], lower_bound=attrs["lower_bound"],
                          upper_bound=attrs["upper_bound"])
                if name == "lamb":
                    kw.update(bias_correction=attrs["bias_correction"])
            opt = O.OracleOptimizer(name, **kw)
            for t in range(4):
                opt.update(0, w, gold["g%d_%s" % (t, tag)].copy())
                want = gold["w%d_%s" % (t + 1, tag)]
                np.testing.assert_allclose(w, want, rtol=1e-3, atol=1e-3, err_msg=str((name, ci, si, t)))
                worst[name] = max(worst[name], float(np.max(np.abs(w - want))))
    assert worst["lamb"] < 1e-5 and worst["lars"] < 1e-5, worst
    assert worst["lans"] < 1e-3, worst


def test_rsp_sum_and_retain_oracle_properties():
    rng = np.random.default_rng(2)
    rows, L = 50, 8
    rsps = []
    dense_sum = np.zeros((rows, L), np.float64)
    for _ in range(4):
        idx = np.sort(rng.choice(rows, 12, replace=False)).astype(np.int64)
        val = rng.uniform(-1, 1, (12, L)).astype(np.float32)
        rsps.append(O.RowSparse(idx, val, (rows, L)))
        dense_sum[idx] += val
    s = O.rsp_sum(rsps)
    assert np.all(np.diff(s.indices) > 0)
    np.testing.assert_allclose(s.todense(), dense_sum, rtol=1e-6, atol=1e-6)
    # order of accumulation = input order starting from zero (ndarray_function.cu:176-187)
    r = int(s.indices[0])
    acc = np.zeros(L, np.float32)
    for x in rsps:
        pos = np.where(x.indices == r)[0]
        if len(pos):
            acc = acc + x.data[pos[0]]
    assert _eq_bits(acc, s.data[0])
    ret = O.sparse_retain(s, O.unique([3, 3, 1, 49]))
    assert list(ret.indices) == [1, 3, 49]


def test_sparse_optimizers_vs_reference_python_references_golden():
    """tests/golden/sparse_steps.npz (SURVEY 8 row a28): weights produced by the classes the reference's OWN tests
    hold its sparse kernels to -- `PySparseSGD.step`, `PySparseAdam.step` (lazy and standard;
    tests/python/unittest/test_optimizer.py:90-159,372-437) and `SGD.step` on the densified gradient
    (test_std_sparse_sgd :183-203) -- executed from the reference files by make_golden.py::sparse_steps.  The
    restatements of SGDDnsRspKernel / SGDMomDnsRspDnsKernel / AdamDnsRspDnsKernel / the *Std* kernels in oracle/
    must agree within the tolerances of those tests (SGD: compare_optimizer defaults rtol 1e-4 / atol 1e-5; Adam
    rtol 1e-4 / atol 2e-5, :486-499); they in fact agree to a few ulp."""
    gold = np.load(os.path.join(GOLD, "sparse_steps.npz"))
    cases = [eval(c) for c in gold["cases"]]
    worst = 0.0
    seen = set()
    for ci, (name, lr, wd, attrs) in enumerate(cases):
        seen.add(name)
        for si in range(2):
            tag = "c%d_s%d" % (ci, si)
            w = gold["w0_" + tag].copy()
            kw = dict(learning_rate=lr, wd=wd, rescale_grad=attrs.get("rescale_grad", 1.0),
                      clip_gradient=attrs.get("clip_gradient"), lazy_update=name.endswith("lazy"))
            if name.startswith("sgd"):
                opt = O.OracleOptimizer("sgd", momentum=attrs["momentum"], **kw)
            else:
                opt = O.OracleOptimizer("adam", beta1=attrs["beta1"], beta2=attrs["beta2"], epsilon=attrs["epsilon"], **kw)
            for t in range(4):
                rows = gold["rows%d_%s" % (t, tag)]
                g = gold["g%d_%s" % (t, tag)]
                grad = O.RowSparse(rows, g[rows].copy(), g.shape)
                opt.update(0, w, grad)
                want = gold["w%d_%s" % (t + 1, tag)]
                if name.startswith("adam"):
                    np.testing.assert_allclose(w, want, rtol=1e-4, atol=2e-5, err_msg=str((name, ci, si, t)))
                else:
                    np.testing.assert_allclose(w, want, rtol=1e-4, atol=1e-5, err_msg=str((name, ci, si, t)))
                worst = max(worst, float(np.max(np.abs(w - want))))
    assert seen == {"sgd_lazy", "sgd_std", "adam_lazy", "adam_std"}
    assert worst < 2e-6, worst

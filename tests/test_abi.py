"""The C-ABI library loads without a GPU and exports every symbol include/mxkv_b200.h declares;
host-only entry points behave; device entry points fail loudly (no CPU fallback)."""
import ctypes
import json
import os
import re

import numpy as np
import pytest

import mxnet_b200 as mx
from mxnet_b200.base import _LIB, check_call

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "mxkv_b200.h")).read()
    return sorted(set(re.findall(r"MXKV_DLL\s+(?:const\s+)?[\w\*]+\s+\*?(\w+)\s*\(", text)))


def test_every_declared_symbol_is_exported():
    syms = declared_symbols()
    assert len(syms) >= 70, syms
    for s in syms:
        assert hasattr(_LIB, s), "symbol %s declared in mxkv_b200.h but not exported" % s
    for must in ("MXKVStoreCreate", "MXKVStorePushPullEx", "MXKVStorePullRowSparse", "MXKVStoreSetUpdaterEx",
                 "MXNDArrayFromDLPack", "MXKVB200CommInit", "MXGetLastError"):
        assert must in syms


def test_library_contains_sm100a_code():
    import subprocess
    so = os.path.join(ROOT, "incubator-mxnet_b200", "libmxkv_b200.so")
    out = subprocess.run(["cuobjdump", "-lelf", so], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in out.stdout


def test_host_only_entry_points():
    v = ctypes.c_int()
    check_call(_LIB.MXGetVersion(ctypes.byref(v)))
    assert v.value == 20000
    for t in ("local", "device", "local_allreduce_cpu", "local_allreduce_device"):
        kv = mx.kv.create(t)
        assert kv.type == t                 # tests/python/unittest/test_kvstore.py:276-279
        assert kv.rank == 0 and kv.num_workers == 1
    assert mx.kv.create("Device").type == "device"          # src/kvstore/kvstore.cc:43-44,83: lower-cased
    with pytest.raises(mx.MXNetError):
        mx.kv.create("dist_sync")
    w = ctypes.c_int()
    check_call(_LIB.MXKVStoreIsWorkerNode(ctypes.byref(w)))
    assert w.value == 1
    # server-side entry points are no-ops of a single-node store (include/mxnet/kvstore.h:432,466)
    kv = mx.kv.create("device")
    kv._send_command_to_servers(0, "")
    check_call(_LIB.MXKVStoreRunServer(kv.handle, None, None))
    n = ctypes.c_int(-1)
    check_call(_LIB.MXKVStoreGetNumDeadNode(kv.handle, 0, ctypes.byref(n), 60))
    assert n.value == 0


def test_error_contract_and_key_rules_without_gpu():
    kv = mx.kv.create("device")
    a = mx.nd.zeros((4, 4))
    kv.init(3, a)
    with pytest.raises(mx.MXNetError, match="duplicate init of key 3"):
        kv.init(3, a)
    with pytest.raises(mx.MXNetError, match="Mixed key types"):
        kv.init("a", a)
    with pytest.raises(mx.MXNetError, match="has not been inited"):
        kv.pull(99, out=a)
    skv = mx.kv.create("device")
    skv.init("a", a)
    with pytest.raises(mx.MXNetError, match="doesn't exist"):
        skv.pull("zz", out=a)
    with pytest.raises(mx.MXNetError, match="Mixed key types"):
        skv.push(3, a)
    # host-resident value, host-resident output: plumbing only, no GPU needed (BASELINE configs[0] shape)
    kv2 = mx.kv.create("local")
    big = mx.nd.array(np.arange(1024 * 1024, dtype=np.float32).reshape(1024, 1024))
    kv2.init(0, big)
    out = mx.nd.zeros((1024, 1024))
    kv2.pull(0, out=out)
    assert np.array_equal(out.asnumpy(), big.asnumpy())


@pytest.mark.skipif(mx.num_gpus() > 0, reason="the no-GPU plumbing case")
@pytest.mark.parametrize("kv_type", ["local", "device"])
def test_baseline_config0_push_pull_of_one_cpu_array_without_gpu(kv_type):
    """BASELINE.json configs[0]: kv.create('local') push / pull of one 1024 x 1024 float32 array on the CPU, world
    size 1 -- the reference's own CPU-runnable case.  One value and no updater is a copy in the reference too
    (comm.h:128-131, kvstore_local.h:279-284): served without a device, compared with the oracle store; a second
    value (a sum) or an optimizer (an update) is compute and still refuses to run without a GPU."""
    from oracle import oracle as O
    rng = np.random.default_rng(0)
    w0 = rng.uniform(-1, 1, (1024, 1024)).astype(np.float32)
    g = rng.uniform(-1, 1, (1024, 1024)).astype(np.float32)
    kv = mx.kv.create(kv_type)
    okv = O.OracleKVStore(kv_type)
    kv.init(0, mx.nd.array(w0))
    okv.init(0, w0.copy())
    out = mx.nd.zeros((1024, 1024))
    for val in (g, 2 * g):
        kv.push(0, mx.nd.array(val))
        okv.push(0, val)
        kv.pull(0, out=out)
        want = np.empty_like(w0)
        okv.pull(0, want)
        assert np.array_equal(out.asnumpy().view(np.uint32), want.view(np.uint32))
    kv.pushpull(0, mx.nd.array(g), out=out)                 # push then pull (kvstore_local.h:358-365)
    assert np.array_equal(out.asnumpy(), g)
    with pytest.raises(mx.MXNetError, match="dtype mismatch"):
        kv.push(0, mx.nd.array(g.astype(np.float64), dtype=np.float64))
    with pytest.raises(mx.MXNetError, match="no CPU fallback"):
        kv.push(0, [mx.nd.array(g), mx.nd.array(g)])
    kv.set_optimizer(mx.optimizer.SGD(learning_rate=0.1))
    with pytest.raises(mx.MXNetError, match="no CPU fallback"):
        kv.push(0, mx.nd.array(g))


@pytest.mark.skipif(mx.num_gpus() > 0, reason="checks the no-GPU failure mode")
def test_compute_fails_loudly_without_gpu():
    kv = mx.kv.create("device")
    kv.init(1, mx.nd.zeros((8,)))
    with pytest.raises(mx.MXNetError, match="no CPU fallback"):
        kv.push(1, [mx.nd.ones((8,)), mx.nd.ones((8,))])
    with pytest.raises(mx.MXNetError, match="no CPU fallback"):
        mx.nd.zeros((2,), mx.gpu(0))


def test_shard_ranges_cover_and_align():
    for size in (0, 1, 127, 128, 1000, 65536, (1 << 26) + 5, 25_557_032):
        for world in (1, 2, 3, 4, 8):
            prev = 0
            for r in range(world):
                b, e = mx.dist.shard_range(size, world, r)
                assert b == prev and b <= e <= size
                assert b % 128 == 0 or b == size
                prev = e
            assert prev == size


def test_optimizer_descriptors():
    o = mx.optimizer.create("sgd", learning_rate=0.1, momentum=0.9, wd=1e-4, rescale_grad=0.5, clip_gradient=2.0)
    kw = o.fused_kwargs()
    assert o.fused_name == "sgd" and kw["momentum"] == 0.9 and kw["clip_gradient"] == 2.0
    kv = mx.kv.create("device")
    kv.set_optimizer(o)           # accepted by the native registry without touching a device
    with pytest.raises(mx.MXNetError, match="unknown optimizer argument"):
        check_call(_LIB.MXKVB200SetOptimizer(kv.handle, b"sgd", 1, (ctypes.c_char_p * 1)(b"bogus"),
                                             (ctypes.c_char_p * 1)(b"1")))
    kv.set_gradient_compression({"type": "2bit", "threshold": 0.5})
    with pytest.raises(mx.MXNetError, match="Unknown type for gradient compression"):
        kv.set_gradient_compression({"type": "3bit"})
    # gradient_compression.cc:40-52: no type means "none", which is refused; 2bit needs a positive threshold (given
    # in any order); arguments the parameter struct does not know are allowed; kvstore.py:551-557: other store types
    # refuse compression altogether
    with pytest.raises(mx.MXNetError, match="Unknown type for gradient compression none"):
        kv.set_gradient_compression({"threshold": 0.5})
    with pytest.raises(mx.MXNetError, match="threshold must be greater than 0"):
        kv.set_gradient_compression({"threshold": 0, "type": "2bit"})
    kv.set_gradient_compression({"type": "1bit", "threshold": 0, "some_future_option": 3})
    with pytest.raises(Exception, match="not supported for this type of kvstore"):
        mx.kv.create("local").set_gradient_compression({"type": "2bit", "threshold": 0.5})
    assert mx.kv.KVStore.is_capable("optimizer")
    assert isinstance(mx.kv.create("b200device"), mx.kv.KVStore)      # registry path, base.py:450-452


def test_dlpack_roundtrip_on_host():
    """MXNDArrayFromDLPack / MXNDArrayToDLPack (c_api.h:976-1002) with host tensors: zero copy both ways."""
    import torch
    t = torch.arange(12, dtype=torch.float32).reshape(3, 4)
    a = mx.nd.from_dlpack(t)
    assert a.shape == (3, 4) and a.context.device_type == "cpu"
    assert a.data_ptr == t.data_ptr()
    assert np.array_equal(a.asnumpy(), t.numpy())
    back = a.as_torch()
    back[0, 0] = 42.0
    assert t[0, 0].item() == 42.0            # same memory
    kv = mx.kv.create("local")
    kv.init("w", a)                           # host value parked in the store (no GPU needed)
    out = mx.nd.zeros((3, 4))
    kv.pull("w", out=out)
    assert out.asnumpy()[0, 0] == 42.0


def test_native_library_is_current():
    """The in-tree .so must have been rebuilt after the last source edit (it travels to the GPU box
    as built; __graft_entry__.build() does this)."""
    import importlib.util, os
    spec = importlib.util.spec_from_file_location(
        "mxkv_build", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                   "incubator-mxnet_b200", "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    assert not b.needs_build(), "libmxkv_b200.so is older than its sources: run python __graft_entry__.py"


def test_store_types_of_the_reference_factory():
    """KVStore::Create (src/kvstore/kvstore.cc:42-85): local / device / nccl names are served, dist is not."""
    for name in ("local", "device", "local_update_cpu", "local_allreduce_cpu", "local_allreduce_device", "nccl"):
        kv = mx.kv.create(name)
        assert kv.type == name and kv.rank == 0 and kv.num_workers == 1
    with pytest.raises(mx.MXNetError):
        mx.kv.create("dist_sync")


def test_loss_scaler_schedule():
    """loss_scaler.py:67-79: halve on overflow (effective one step later), double after scale_seq_len clean steps."""
    s = mx.amp.LossScaler(init_scale=1024., scale_seq_len=3, max_loss_scale=4096.)
    assert s.update(True) is True and s.loss_scale == 1024. and s._next_loss_scale == 512.
    assert s.update(False) is False and s.loss_scale == 512.
    s.update(False)
    s.update(False)                       # third clean step: schedule a doubling
    assert s._next_loss_scale == 1024.
    s.update(False)
    assert s.loss_scale == 1024.
    for _ in range(12):
        s.update(False)
    assert s.loss_scale <= 4096. and s._next_loss_scale == 4096.


def test_layerwise_optimizer_descriptors():
    """hyper-parameter names handed to MXKVB200SetOptimizer follow python/mxnet/optimizer/{lamb,lans,lars}.py."""
    kw = mx.optimizer.create("lamb", learning_rate=0.01, lower_bound=0.1, skip_nonfinite=True).fused_kwargs()
    assert kw["bias_correction"] is True and kw["lower_bound"] == 0.1 and "upper_bound" not in kw
    assert kw["skip_nonfinite"] is True and kw["epsilon"] == 1e-6
    lars = mx.optimizer.create("lars", momentum=0.9, param_idx2name={0: "fc_weight", 1: "fc_bias", 2: "bn_gamma"})
    assert lars.fused_kwargs()["eta"] == 0.001 and sorted(lars.no_trust_ratio_indices()) == [1, 2]
    kv = mx.kv.create("device")
    kv.set_optimizer(lars)               # descriptors reach the engine without a GPU
    kv.set_optimizer(mx.optimizer.create("lans"))
    with pytest.raises(mx.MXNetError):   # skip_nonfinite is a layer-wise-optimizer feature
        from mxnet_b200.base import _LIB, check_call, c_str, c_str_array
        check_call(_LIB.MXKVB200SetOptimizer(kv.handle, c_str("sgd"), 1, c_str_array(["skip_nonfinite"]),
                                             c_str_array(["True"])))
    assert isinstance(mx.optimizer.get_updater(mx.optimizer.create("adam")), mx.optimizer.NativeUpdater)

    class Custom(mx.optimizer.Optimizer):
        pass
    assert isinstance(mx.optimizer.get_updater(Custom()), mx.optimizer.Updater)


def test_lr_schedulers_match_the_reference_module():
    """tests/golden/lr_schedules.npz was produced by importing python/mxnet/lr_scheduler.py out of the
    reference tree (make_golden.py::lr_schedules); the schedules here must return the same doubles."""
    import importlib.util, os
    here = os.path.dirname(os.path.abspath(__file__))
    spec = importlib.util.spec_from_file_location("mk", os.path.join(here, "golden", "make_golden.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    gold = np.load(os.path.join(here, "golden", "lr_schedules.npz"))
    for i, (cls, kw) in enumerate(mk.LR_CASES):
        s = getattr(mx.lr_scheduler, cls)(**kw)
        got = np.array([s(n) for n in range(60)], np.float64)
        assert np.array_equal(got, gold["seq_%d" % i]), (cls, kw)
        s2 = getattr(mx.lr_scheduler, cls)(**kw)
        assert np.array_equal(np.array([s2(37), s2(38), s2(59)]), gold["jump_%d" % i]), (cls, kw)
    with pytest.raises(ValueError):
        mx.lr_scheduler.FactorScheduler(step=0)
    with pytest.raises(ValueError):
        mx.lr_scheduler.MultiFactorScheduler(step=[5, 5])


def test_scheduler_is_consulted_after_counting_the_update():
    """fused_step counts first and reads the learning rate afterwards (sgd.py:184-186): the first update
    runs at lr_scheduler(1), and every key of one call sees the same rate."""
    sched = mx.lr_scheduler.FactorScheduler(step=2, factor=0.5, base_lr=1.0)
    opt = mx.optimizer.SGD(learning_rate=1.0, lr_scheduler=sched)
    kv = mx.kv.create("device")
    kv.set_optimizer(opt)
    seen = []
    for step in range(1, 7):
        kv._advance_counts([0, 1, 0])          # two keys, one of them pushed from two devices
        seen.append(kv._last_lr)
        assert opt._index_update_count == {0: step, 1: step} and opt.num_update == step
    assert seen == [sched_ref for sched_ref in [1.0, 1.0, 0.5, 0.5, 0.25, 0.25]]


def test_multipliers_follow_the_reference_precedence():
    """Optimizer._get_lrs / _get_wds (optimizer.py:461-526): Parameter object, then index, then name."""
    class P(object):
        lr_mult, wd_mult = 3.0, 0.0
    opt = mx.optimizer.SGD(learning_rate=0.1, wd=0.01, param_idx2name={0: "fc_weight", 1: "fc_bias", 2: "bn_gamma"},
                           param_dict={2: P()})
    opt.set_lr_mult({"fc_bias": 2.0, 0: 0.5})
    opt.set_wd_mult({"fc_bias": 0.0})
    assert opt._get_lr(0) == 0.05 and opt._get_lr(1) == 0.2 and abs(opt._get_lr(2) - 0.3) < 1e-15
    assert opt._get_wd(0) == 0.01 and opt._get_wd(1) == 0.0 and opt._get_wd(2) == 0.0
    assert opt.key_multipliers() == {0: (0.5, 1.0), 1: (2.0, 0.0), 2: (3.0, 0.0)}
    kv = mx.kv.create("device")
    kv.set_optimizer(opt)                     # reaches MXKVB200SetOptimizerMult by index


def test_plain_c_consumer(tmp_path):
    """include/mxkv_b200.h is valid C99 and the library links from plain C; the host-only part of the
    contract (handles, host arrays, key-type rules, 0 / -1 + MXGetLastError) runs without a GPU."""
    import os, shutil, subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "incubator-mxnet_b200")
    exe = str(tmp_path / "abi_consumer")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(root, "include"),
                    os.path.join(root, "tests", "c", "abi_consumer.c"), "-o", exe, "-L", libdir, "-lmxkv_b200",
                    "-Wl,-rpath," + libdir], check=True, capture_output=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "abi_consumer ok" in r.stdout


def test_trainer_update_requires_local_updates():
    """trainer.py:436-439: update() is refused when the kvstore applies the optimizer."""
    class P(object):                       # stands in for a torch Parameter: never touched before the assert
        pass
    tr = mx.Trainer([P()], "sgd", {"learning_rate": 0.1}, kvstore="device")
    tr._kv_initialized, tr._kvstore, tr._update_on_kvstore = True, object(), True
    with pytest.raises(AssertionError):
        tr.update(4)


def _key_hyper(kv, key):
    import ctypes
    from mxnet_b200.base import _LIB, check_call
    lr, wd, eta = ctypes.c_float(), ctypes.c_float(), ctypes.c_float()
    check_call(_LIB.MXKVB200GetKeyHyper(kv.handle, int(key), None, ctypes.byref(lr), ctypes.byref(wd), ctypes.byref(eta)))
    return np.float32(lr.value), np.float32(wd.value), np.float32(eta.value)


def _set_count(kv, key, t):
    import ctypes
    from mxnet_b200.base import _LIB, check_call
    check_call(_LIB.MXKVB200SetUpdateCount(kv.handle, int(key), None, ctypes.c_int64(t)))


def test_per_key_hyper_parameters_follow_the_python_optimizers():
    """What the fused kernel receives per key, checked on the host against the reference's Python
    bookkeeping: lr/wd multipliers (optimizer.py:461-526), Adam's bias correction folded into lr in double
    (adam.py:172-175), AdamW driving its operator with lr = 1 and eta = lr_t (adamW.py:158-200)."""
    import math
    from oracle import oracle as O
    kv = mx.kv.create("device")
    kv.init([0, 1], [mx.nd.zeros((4,)), mx.nd.zeros((4,))])
    # SGD with multipliers
    opt = mx.optimizer.SGD(learning_rate=0.1, wd=0.01)
    opt.set_lr_mult({1: 0.5}); opt.set_wd_mult({1: 0.0})
    kv.set_optimizer(opt)
    assert _key_hyper(kv, 0) == (np.float32(0.1), np.float32(0.01), np.float32(1.0))
    assert _key_hyper(kv, 1) == (np.float32(0.05), np.float32(0.0), np.float32(1.0))
    # Adam: lr * sqrt(1 - b2^t) / (1 - b1^t), rounded once
    kv.set_optimizer(mx.optimizer.Adam(learning_rate=0.003, beta1=0.8, beta2=0.95, wd=0.02))
    for t in (1, 2, 7, 1000):
        _set_count(kv, 0, t)
        want = 0.003 * math.sqrt(1. - 0.95 ** t) / (1. - 0.8 ** t)
        lr, wd, eta = _key_hyper(kv, 0)
        assert lr == np.float32(want) == np.float32(O.adam_lr(0.003, 0.8, 0.95, t)) and wd == np.float32(0.02)
    # AdamW: operator lr = 1, eta = (bias-corrected) learning rate [* the engine's own eta multiplier]
    for correct_bias, mult in ((True, 1.0), (False, 0.7)):
        kv.set_optimizer(mx.optimizer.AdamW(learning_rate=0.01, beta1=0.9, beta2=0.98, wd=0.05,
                                            correct_bias=correct_bias, eta=mult))
        for t in (1, 3, 50):
            _set_count(kv, 0, t)
            lr_t = 0.01 * math.sqrt(1. - 0.98 ** t) / (1. - 0.9 ** t) if correct_bias else 0.01
            lr, wd, eta = _key_hyper(kv, 0)
            assert lr == np.float32(1.0) and wd == np.float32(0.05) and eta == np.float32(lr_t * mult)
    # LAMB / LARS keep the plain learning rate (their ratios are taken on the device)
    kv.set_optimizer(mx.optimizer.LAMB(learning_rate=0.02))
    assert _key_hyper(kv, 0)[0] == np.float32(0.02)


def test_engine_defaults_are_the_reference_optimizers():
    """A C consumer that names an optimizer without arguments gets the reference classes' defaults: learning rates
    sgd 0.1 (sgd.py:95), adam / adamw / lamb / lans 0.001 (adam.py:85, adamW.py:80, lamb.py:66, lans.py:62),
    lars 0.1 (lars.py:77), test 0.01 (optimizer.py:100-101); and so do the Python classes of this package."""
    kv = mx.kv.create("device")
    kv.init(0, mx.nd.zeros((4,)))
    for name, lr in (("sgd", 0.1), ("adam", 0.001), ("lamb", 0.001), ("lans", 0.001), ("lars", 0.1), ("test", 0.01)):
        check_call(_LIB.MXKVB200SetOptimizer(kv.handle, name.encode(), 0, None, None))
        _set_count(kv, 0, 10 ** 6)                              # Adam's bias correction -> 1
        got = _key_hyper(kv, 0)
        assert got[0] == np.float32(lr) and got[1] == 0.0, (name, got)
        assert mx.optimizer.create(name).learning_rate == lr, name
    check_call(_LIB.MXKVB200SetOptimizer(kv.handle, b"adamw", 0, None, None))
    _set_count(kv, 0, 10 ** 6)
    lr, wd, eta = _key_hyper(kv, 0)
    assert lr == np.float32(1.0) and eta == np.float32(0.001), (lr, eta)     # operator lr = 1, eta = learning rate
    assert mx.optimizer.create("adamw").epsilon == 1e-6 and mx.optimizer.create("adam").epsilon == 1e-8


def c_prototypes(path, macro):
    """{entry point: parameter types} of the `macro int name(...);` declarations of a C header."""
    t = open(path).read()
    t = re.sub(r"/\*.*?\*/", " ", t, flags=re.S)
    t = re.sub(r"//[^\n]*", " ", t)
    out = {}
    for m in re.finditer(macro + r"\s+int\s+(\w+)\s*\((.*?)\)\s*;", t, flags=re.S):
        parts = []
        for a in re.sub(r"DEFAULT\([^)]*\)", "", m.group(2)).split(","):
            a = " ".join(a.split())
            if a in ("void", ""):
                continue
            if not a.endswith("*"):
                a = re.sub(r"\s*\b\w+\s*$", "", a)            # drop the parameter name
            a = a.replace("const ", "").replace(" *", "*").replace("* ", "*").strip()
            for alias, canon in (("mx_uint", "uint32_t"), ("unsigned int", "uint32_t"), ("dim_t", "int64_t")):
                a = a.replace(alias, canon)
            parts.append(a)
        out[m.group(1)] = parts
    return out


def test_prototypes_match_the_reference_header():
    """Every entry point this library shares with include/mxnet/c_api.h has the reference's parameter types, in
    order (names and `const` aside; `dim_t` is `int64_t`, `mx_uint` is `uint32_t`).  The reference's side is
    tests/golden/c_api_prototypes.json (make_golden.py::c_api_prototypes)."""
    with open(os.path.join(ROOT, "tests", "golden", "c_api_prototypes.json")) as f:
        ref = json.load(f)
    mine = c_prototypes(os.path.join(ROOT, "include", "mxkv_b200.h"), "MXKV_DLL")
    shared = [n for n in mine if n in ref]
    assert len(shared) >= 50, len(shared)
    for n in shared:
        assert mine[n] == ref[n], (n, mine[n], ref[n])


def test_engine_ops_run_in_order_on_the_calling_thread():
    """MXEnginePushSync[ND] / MXEnginePushAsync[ND] (include/mxnet/c_api.h:3010-3127; what the Horovod-style plug-ins
    wrap their work in): served conservatively -- drain, then run on the calling thread; the Async flavours return
    only after the function has called on_complete (here from another thread)."""
    import ctypes
    import threading
    import mxnet_b200  # noqa: F401
    from mxnet_b200.base import _LIB
    seen = []
    SYNC = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_void_p)
    ASYNC = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p)
    DEL = ctypes.CFUNCTYPE(None, ctypes.c_void_p)
    ctx = (ctypes.c_int * 2)(1, 0)                       # {dev_type = cpu, dev_id = 0}

    sync_fn = SYNC(lambda rctx, param: seen.append(("sync", param)))
    deleter = DEL(lambda param: seen.append(("deleted", param)))
    rc = _LIB.MXEnginePushSyncND(sync_fn, ctypes.c_void_p(7), deleter, ctx, None, 0, None, 0, None, 0, b"op")
    assert rc == 0 and seen == [("sync", 7), ("deleted", 7)]

    def later(on_complete):
        seen.append("worker")
        _LIB.MXKVB200EngineOnComplete(ctypes.c_void_p(on_complete))

    def async_body(rctx, on_complete, param):
        seen.append(("async", param))
        threading.Thread(target=later, args=(on_complete,)).start()
    _LIB.MXKVB200EngineOnComplete.restype = None
    async_fn = ASYNC(async_body)
    rc = _LIB.MXEnginePushAsync(async_fn, ctypes.c_void_p(9), None, ctx, None, 0, None, 0, None, 0, None, False)
    assert rc == 0 and seen[2:] == [("async", 9), "worker"]
    assert _LIB.MXEnginePushSync(None, None, None, ctx, None, 0, None, 0, None, 0, None) != 0     # null function: an error, not a crash

#!/usr/bin/env python
"""bench.py -- KVStore push+pull throughput on B200 (BASELINE.json metric).

A *step* is one pass of the hot path over one batch of synthetic gradients: `pushpull` of the
whole key set (sum over the ranks' gradients, fused SGD-momentum update of the stored fp32
weights, new weights delivered to every rank).  Workload (config.workload):

  sweep     BASELINE.json configs[1]: one fp32 key per size 2^10, 2^12, ..., 2^26 elements
            (4 KB ... 256 MB; 89.5 M elements, 358 MB per rank) -- the default
  resnet50  configs[2]'s key set: the 193 gradient-carrying arrays of Gluon ResNet-50-v1 (25.6 M elements)
  bert      configs[3]'s key set: BERT-base (synthetic shape list), Adam

One process per GPU (torchrun for N > 1); every rank contributes its own gradient for every key
(weak scaling: per-GPU work is fixed).  `value` = N * 2 * S / t  [GB/s]: bytes pushed plus bytes
pulled by all ranks per second, S = key-set bytes.  Inputs are larger than L2 (358 MB of
gradients + 358 MB of weights + state per step vs 126 MB of L2), so no flush is needed.

Besides the contract's keys the line carries
  parity     the timed configuration (same arrays, same kernel variant) run once from a fresh store and compared
             with the CPU oracle; the run FAILS when it does not match
  sweep      BASELINE.json configs[1] as a sweep: per key size, all-reduce only and with the fused update, us per
             call, bus bandwidth, kernel variant, next to NCCL's all-reduce timed in the same process
  secondary  BASELINE.json configs[2..4]: ResNet-50 / BERT-base bf16 training steps (samples/sec) through
             Trainer(kvstore='device'), row_sparse push + row_sparse_pull

Usage: python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...]
                       [--dump-outputs DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


# ---------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------
def keyset(workload):
    if workload == "sweep":
        return [(1 << p,) for p in range(10, 27, 2)]
    if workload == "resnet50":
        # python/mxnet/gluon/model_zoo/vision/resnet.py:345-422 (BottleneckV1, layers [3,4,6,3],
        # channels [64,256,512,1024,2048]); conv weights, the biases Gluon leaves on the 1x1
        # convs, BN gamma/beta, FC weight/bias
        shapes = [(64, 3, 7, 7), (64,), (64,)]
        inp = 64
        for stage, (blocks, ch) in enumerate(zip([3, 4, 6, 3], [256, 512, 1024, 2048])):
            mid = ch // 4
            for b in range(blocks):
                shapes += [(mid, inp, 1, 1), (mid,), (mid,), (mid,)]          # conv1x1 + bias + BN
                shapes += [(mid, mid, 3, 3), (mid,), (mid,)]                  # conv3x3 + BN
                shapes += [(ch, mid, 1, 1), (ch,), (ch,), (ch,)]              # conv1x1 + bias + BN
                if b == 0:
                    shapes += [(ch, inp, 1, 1), (ch,), (ch,)]                 # downsample conv + BN
                inp = ch
        shapes += [(1000, 2048), (1000,)]
        return shapes
    if workload == "bert":
        H, FF = 768, 3072
        shapes = [(30522, H), (512, H), (2, H), (H,), (H,)]
        for _ in range(12):
            shapes += [(H, H), (H,)] * 3 + [(H, H), (H,), (H,), (H,), (FF, H), (FF,), (H, FF), (H,), (H,), (H,)]
        shapes += [(H, H), (H,)]
        return shapes
    raise ValueError(workload)


def nelem(shape):
    n = 1
    for d in shape:
        n *= d
    return n


def tile_fill(rng, lo, hi, shape):
    """Synthetic float32 data.  Arrays above 1 M elements repeat a random block of 1 000 003 elements (a period
    no tile, chunk or shard boundary is a multiple of): numpy draws ~20 M values/s, the sweep needs 90 M per array
    and the parity check regenerates every rank's arrays."""
    e = nelem(shape)
    if e <= (1 << 20):
        return rng.uniform(lo, hi, e).astype(np.float32).reshape(shape)
    return np.resize(rng.uniform(lo, hi, 1000003).astype(np.float32), e).reshape(shape)


def rank_grads(rank, shapes):
    rng = np.random.default_rng(1234 + rank)
    return [tile_fill(rng, -1, 1, s) for s in shapes]


def initial_weights(shapes):
    rng = np.random.default_rng(99)
    return [tile_fill(rng, 0, 1, s) for s in shapes]


OPTIMIZERS = {   # name -> (mx class name, kwargs, oracle name, algorithmic 4-byte streams per element at N=1)
    "sgd": ("SGD", dict(learning_rate=0.01, momentum=0.9, wd=1e-4), "sgd", 6),     # read g, w, mom; write w(store), mom, w(out)
    "adam": ("Adam", dict(learning_rate=0.001), "adam", 8),                         # read g, w, m, v; write w, m, v, out
    # first: read g, w, m, v; write m, v, ghat.  apply: read w, ghat; write w(store), out
    "lamb": ("LAMB", dict(learning_rate=0.001, wd=0.01), "lamb", 11),
    # first: read g, w; write g.  mid: read g, w, m, v; write m, v, temp_m, temp_g.  apply: read w, temp_m, temp_g; write w, out
    "lans": ("LANS", dict(learning_rate=0.001, wd=0.01), "lans", 16),
    # first: read g, w; write g.  apply: read w, g, mom; write w(store), mom, out
    "lars": ("LARS", dict(learning_rate=0.1, momentum=0.9, wd=1e-4), "lars", 9),
    "none": (None, {}, None, 3),                                                    # read g; write store, out
}


# ---------------------------------------------------------------------------
# host placement: one rank per GPU, each bound to the CPUs (and so the memory) of its GPU's NUMA node
# ---------------------------------------------------------------------------
def bind_to_gpu_numa(gpu_index):
    """Restrict this process to the CPUs of the NUMA node the GPU hangs off, BEFORE pinned buffers are allocated
    (first touch places them on that node): host<->device copies then never cross the socket interconnect.
    Returns a description for the JSON line; does nothing when the topology cannot be read."""
    info = {"gpu": gpu_index, "numa_node": None, "cpus": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        bdf = pynvml.nvmlDeviceGetPciInfo(h).busId
        bdf = bdf.decode() if isinstance(bdf, bytes) else bdf
        bdf = bdf.lower()
        if len(bdf.split(":")[0]) == 8:           # nvml prints an 8-digit domain, sysfs a 4-digit one
            bdf = bdf[4:]
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read())
        info["numa_node"] = node
        if node < 0:
            return info
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["cpus"] = len(allowed)
    except Exception as e:          # noqa: BLE001 -- containers without sysfs / nvml: run unbound
        info["error"] = repr(e)[:100]
    return info


# ---------------------------------------------------------------------------
# NVLink traffic as the hardware counts it (NVML field values, no profiler): DATA = payload bytes, RAW = payload +
# protocol overhead, both directions, summed over the GPU's 18 links.  Read before and after the timed region,
# the difference per step is the `traffic` of the N > 1 roofline (ncu cannot profile a kernel that rendezvous
# with kernels on other GPUs: profiles/README.md).
# ---------------------------------------------------------------------------
_NVL_FIELDS = {"data_tx": 138, "data_rx": 139, "raw_tx": 140, "raw_rx": 141}     # NVML_FI_DEV_NVLINK_THROUGHPUT_*, KiB


def nvlink_counters(gpu_index):
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ids = list(_NVL_FIELDS.values())
        try:
            vals = pynvml.nvmlDeviceGetFieldValues(h, [(f, 0xFFFFFFFF) for f in ids])     # scope: all links
        except Exception:
            vals = pynvml.nvmlDeviceGetFieldValues(h, ids)
        out = {}
        for name, v in zip(_NVL_FIELDS, vals):
            if v.nvmlReturn != 0:
                return {"error": "nvml field %s: return %d" % (name, v.nvmlReturn)}
            vt = v.valueType
            val = {0: v.value.dVal, 1: v.value.uiVal, 2: v.value.ulVal, 3: v.value.ullVal, 4: v.value.sllVal}.get(vt, v.value.ullVal)
            out[name] = float(val) * 1024.0
        return out
    except Exception as e:          # noqa: BLE001
        return {"error": repr(e)[:120]}


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler(object):
    """SM clock, max clock and throttle reasons of one GPU while the timed region runs.

    The samples come from NVML calls made by a thread of this process (clock info + current clocks-event reasons,
    every 100 ms) -- NOT from an `nvidia-smi -lms` loop: on 8 GPUs that loop, at the 20 ms period round 2 first
    used, slowed the NVSwitch-multicast exchange from 0.79 to 1.21 ms per step (profiles/r02_diag_n8_sampler.txt;
    one GPU's queries stall all eight through the rendezvous), while at N = 1 / 2 it cost nothing.  Only when
    pynvml is missing does the sampler fall back to `nvidia-smi -lms 250`."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    PERIOD_S = 0.1

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []        # (host time, sm MHz, max sm MHz, set of reasons)
        self.proc = None
        self.thread = None
        self.stop_flag = False
        self.how = None

    def _nvml_loop(self, pynvml, h):
        masks = [("hw_slowdown", getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8)),
                 ("hw_thermal_slowdown", getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
                 ("sw_thermal_slowdown", getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)),
                 ("sw_power_cap", getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4))]
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
        try:
            mx_clock = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            mx_clock = None
        while not self.stop_flag:
            try:
                sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                bits = int(get_reasons(h))
                self.samples.append((time.time(), sm, mx_clock, {n for n, m in masks if bits & m}))
            except Exception:
                pass
            time.sleep(self.PERIOD_S)

    def _smi_loop(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm, mxc = float(f[1]), float(f[2])
            except ValueError:
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            self.samples.append((time.time(), sm, mxc, {n for n, v in zip(names, f[5:9]) if v.lower().startswith("active")}))

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.how = "NVML calls from a thread of this process, every %d ms" % int(self.PERIOD_S * 1e3)
            self.thread = threading.Thread(target=self._nvml_loop, args=(pynvml, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "250"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.how = "nvidia-smi -lms 250"
            self.thread = threading.Thread(target=self._smi_loop, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def active(self):
        return self.thread is not None

    def wait_first(self, timeout=10.0):
        """do not start the timed region before the sampler delivers (nvidia-smi needs ~1 s for its first line)"""
        t0 = time.time()
        while self.active() and not self.samples and time.time() - t0 < timeout:
            time.sleep(0.02)

    def count(self, t0, t1):
        return sum(1 for s in self.samples if t0 <= s[0] <= t1)

    def stop(self, t0, t1):
        if not self.active():
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock sampler available"], "samples": 0}
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        win = [s for s in self.samples if t0 <= s[0] <= t1]
        sm = [s[1] for s in win]
        mxc = [s[2] for s in win if s[2] is not None]
        reasons = set()
        for s in win:
            reasons |= s[3]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mxc) if mxc else None,
                "reasons": sorted(reasons), "samples": len(sm), "how": self.how}


# ---------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's CPU KVStore ('local': CommCPU reduce +
# CPU updater + ParallelCopy broadcast) restated in oracle/kv_oracle.c, all host cores
# ---------------------------------------------------------------------------
def cpu_kvstore_step_factory(shapes, n_values, threads, optimizer):
    from oracle import oracle as O
    rng = np.random.default_rng(1234)
    sizes = [nelem(s) for s in shapes]
    grads = [[rng.uniform(-1, 1, e).astype(np.float32) for _ in range(n_values)] for e in sizes]
    stage = [[np.empty(e, np.float32) for _ in range(n_values)] for e in sizes]    # pinned merge/copy bufs
    weights = [rng.uniform(0, 1, e).astype(np.float32) for e in sizes]
    mom = [np.zeros(e, np.float32) for e in sizes]
    mean = [np.zeros(e, np.float32) for e in sizes] if optimizer in ("adam", "lamb", "lans") else None
    outs = [[np.empty(e, np.float32) for _ in range(n_values)] for e in sizes]
    lib = O.lib()
    import ctypes
    state = {"t": 0}
    lib.kvo_set_threads(ctypes.c_int(threads))     # the optimizer loops use the OpenMP default team

    def step():
        state["t"] += 1
        for k, e in enumerate(sizes):
            if n_values == 1:
                merged = grads[k][0]                                  # comm.h:128-131
            else:
                for j in range(n_values):                             # CopyFromTo(src[j], &buf) comm.h:147,162
                    lib.kvo_parallel_copy_f32(stage[k][j].ctypes.data_as(O.c_f32p),
                                              grads[k][j].ctypes.data_as(O.c_f32p), ctypes.c_int64(e),
                                              ctypes.c_int(threads))
                O.sum_cpu_inplace(stage[k], nthreads=threads)         # ReduceSumCPU comm.h:359-411
                merged = stage[k][0]
            if optimizer == "adam":
                O.adam_update(weights[k], merged, mean[k], mom[k], O.adam_lr(0.001, 0.9, 0.999, state["t"]))
            elif optimizer == "sgd":
                O.sgd_mom_update(weights[k], merged, mom[k], 0.01, 1e-4, 0.9)
            elif optimizer == "lamb":        # multi_lamb_update on the CPU: sequential norms + two passes
                O.lamb_update(weights[k], merged, mean[k], mom[k], 0.001, 0.01, state["t"])
            elif optimizer == "lans":
                O.lans_update(weights[k], merged, mean[k], mom[k], 0.001, 0.01, state["t"])
            elif optimizer == "lars":
                O.sgd_mom_update(weights[k], merged, mom[k], O.lars_lr(0.1, weights[k], merged, 1e-4), 1e-4, 0.9)
            else:
                weights[k][...] = merged
            for j in range(n_values):                                 # Broadcast: CopyFromTo(local, out_j)
                lib.kvo_parallel_copy_f32(outs[k][j].ctypes.data_as(O.c_f32p),
                                          weights[k].ctypes.data_as(O.c_f32p), ctypes.c_int64(e),
                                          ctypes.c_int(threads))
    return step


def ncu_dram_bytes(path):
    """dram__bytes_read.sum + dram__bytes_write.sum of the first kernel in an `ncu --page raw` text dump
    (`metric  unit  value` or `metric  value  unit` columns)."""
    units = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    got = {}
    try:
        with open(path) as f:
            for line in f:
                parts = line.split()
                if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") \
                        and parts[0] not in got:
                    unit = [x for x in parts[1:] if x in units]
                    num = [x for x in parts[1:] if x.replace(",", "").replace(".", "", 1).isdigit()]
                    if unit and num:
                        got[parts[0]] = float(num[-1].replace(",", "")) * units[unit[0]]
    except OSError:
        return None
    return sum(got.values()) if len(got) == 2 else None


def host_cpus():
    """CPUs this process may actually use: affinity mask, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:            # cgroup v2
            q, per = f.read().split()
            if q != "max":
                n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:   # cgroup v1
                q = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = int(f.read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


def run_cpu_reference(args, shapes, as_baseline=False):
    """Times the reference's CPU KVStore algorithm (oracle port).  A step is a BOUNDED SAMPLE of the workload:
    every key is cut to the same leading fraction so that the whole --steps/--warmup run stays within ~2 minutes
    (GB/s is intensive, so the sample is comparable).  Threads: every host core this process may use --
    torchrun's OMP_NUM_THREADS=1 is NOT honoured (it is torchrun's default for its workers, not a property of
    the box); the reference's own default of 4 reduce threads (MXNET_KVSTORE_REDUCTION_NTHREADS,
    src/kvstore/comm.h:107-108) is timed beside it and reported in `reference_default_4_threads`."""
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")     # oversubscribed spinning would only hurt the CPU arm
    try:                                                    # a NUMA binding of this rank must not cap the CPU arm
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    except Exception:
        pass
    avail = max(1, host_cpus())
    n_values = max(1, args.gpus)
    warm = 1 if as_baseline else args.warmup
    steps = 3 if as_baseline else args.steps
    budget_s = 15.0 if as_baseline else 100.0
    sizes = [nelem(s) for s in shapes]
    probe_frac = min(1.0, 64e6 / max(1, sum(sizes)) / n_values * 4)     # probe on <= ~64 M elements of traffic
    probe_shapes = [(max(256, int(e * probe_frac)),) for e in sizes]
    # give the CPU arm its best thread count (all usable cores, or fewer when memory-bound)
    threads, t_probe, t_four = avail, None, None
    for cand in sorted({avail, max(1, avail // 2), max(1, avail // 4), min(4, avail)}, reverse=True):
        probe = cpu_kvstore_step_factory(probe_shapes, n_values, cand, args.optimizer)
        probe()
        t0 = time.perf_counter(); probe(); tp = time.perf_counter() - t0
        if cand == min(4, avail):
            t_four = tp
        if t_probe is None or tp < t_probe:
            threads, t_probe = cand, tp
    t_full = t_probe / probe_frac
    frac = min(1.0, budget_s / (steps + warm) / t_full)
    sample_shapes = [(max(256, int(e * frac)),) for e in sizes]
    S = 4 * sum(nelem(s) for s in sample_shapes)
    step = cpu_kvstore_step_factory(sample_shapes, n_values, threads, args.optimizer)
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    value = n_values * 2 * S / dt / 1e9
    sample = ("%d step(s), each over the leading %.1f%% of every key of the %s key set (%.1f MB x %d value(s) per key), "
              "%d OpenMP threads of %d usable cores" % (steps, 100 * frac, args.workload, S / 1e6, n_values, threads, avail))
    Sp = 4 * sum(nelem(s) for s in probe_shapes)
    base = {"value": value, "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample,
            "reference_default_4_threads": {"value": n_values * 2 * Sp / t_four / 1e9, "unit": "GB/s",
                                            "cores": min(4, avail), "sample": "one probe step over %.1f MB" % (Sp / 1e6)}
            if t_four else None}
    return value, dt, base


# ---------------------------------------------------------------------------
# process environment shared by the main measurement and the secondary workloads
# ---------------------------------------------------------------------------
class Env(object):
    def __init__(self, args):
        import torch
        import mxnet_b200 as mx
        self.torch, self.mx = torch, mx
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", self.rank)) if self.world > 1 else 0
        assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
        torch.cuda.set_device(self.local)
        self.hier = False
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.hier = 0 < args.local_world < self.world
            mx.dist.init_process_group(device=self.local, local_world=args.local_world if self.hier else self.world)
        else:
            assert args.gpus == 1, "launch with torchrun for --gpus > 1"
        self.ctx = mx.gpu(self.local)
        # multicast-capable arrays: the engine's own arena (VMM allocations bound to a multicast object,
        # csrc/vmm_arena.cc) when the GPUs support it, else torch's symmetric-memory allocator, else none
        self.multicast = None
        if self.world > 1 and not self.hier:
            if args.no_nvls:
                mx.kv.set_nvls(0)
            elif mx.nd.has_multicast(mx.nd.empty_symmetric((1024,))):
                self.multicast = "engine"
            else:
                try:
                    if mx.nd.has_multicast(mx.nd.empty_multicast((1024,))):
                        self.multicast = "torch"
                except Exception as e:                     # noqa: BLE001 -- torch symmetric memory unavailable
                    sys.stderr.write("multicast allocation unavailable (%r): peer-load kernels\n" % (e,))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def allgather_int(self, x):
        if self.world == 1:
            return [int(x)]
        t = self.torch.tensor([int(x)], dtype=self.torch.int64, device="cuda")
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [int(o) for o in out]

    def engine_stream(self):
        import ctypes
        from mxnet_b200.base import _LIB, check_call
        sp = ctypes.c_void_p()
        check_call(_LIB.MXKVB200GetEngineStream(self.local, ctypes.byref(sp)))
        return self.torch.cuda.ExternalStream(sp.value, device=self.torch.device("cuda", self.local))

    def variant_counts(self):
        return {v: self.mx.kv.launch_count(v) for v in ("per_thread", "bulk", "nvls", "tree")}

    def finish(self):
        self.mx.nd.waitall()
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


KERNEL_NAMES = {"per_thread": "kv_dense_kernel", "bulk": "kv_dense_bulk_kernel", "nvls": "kv_dense_nvls_kernel",
                "tree": "kv_dense_tree_kernel"}


def oracle_tree(env, kvtype):
    """MXNET_KVSTORE_USETREE=1 in the environment (three ranks or more, a `device` store): the trees the engine builds
    for this job's GPUs, in the form the oracle store takes (DESIGN.md section 7f); None otherwise."""
    if os.environ.get("MXNET_KVSTORE_USETREE", "0") in ("", "0") or env.world < 3 or "device" not in kvtype or \
            getattr(env, "hier", False):
        return None
    T = env.mx.topology
    topo, scan, depth = T.compute_trees(T.query_links(env.allgather_int(env.local)),
                                        float(os.environ.get("MXNET_KVSTORE_TREE_LINK_USAGE_PENALTY", 0.7)),
                                        os.environ.get("MXNET_KVSTORE_TREE_BACKTRACK", "0") not in ("", "0"))
    return dict(topo=topo, scan=scan, depth=depth, bound=int(os.environ.get("MXNET_KVSTORE_TREE_ARRAY_BOUND", 10000000)))


def variant_since(env, before):
    now = env.variant_counts()
    used = [v for v in now if now[v] > before[v]]
    return "+".join(used) if used else "none"


def make_optimizer(mx, name):
    cls, kw, _, _ = OPTIMIZERS[name]
    return getattr(mx.optimizer, cls)(**kw) if cls else None


# ---------------------------------------------------------------------------
# parity: what was timed is compared with the oracle once (VERDICT r1 item 1c)
# ---------------------------------------------------------------------------
def parity_check(env, args, shapes, keys, grads, weights, kvtype, keep=False):
    """A fresh store, the SAME gradient / output arrays and kernel selection as the timed loop, one pushpull,
    compared on rank 0 with the CPU oracle fed every rank's gradients (regenerated from their seeds); every rank's
    outputs must carry the same bits as rank 0's.  Bit-exact on the peer-memory kernels; the NVSwitch reduction
    (multimem.ld_reduce) and the layer-wise optimizers' tree-shaped norms are held to the reference's own bound,
    relative L1 <= 1e-6 (tests/nightly/test_kvstore.py:117-119)."""
    from oracle import oracle as O
    mx = env.mx
    w0 = initial_weights(shapes)
    kvp = mx.kv.create(kvtype)
    kvp.init(keys, [mx.nd.array(w, env.ctx) for w in w0])
    opt = make_optimizer(mx, args.optimizer)
    if opt is not None:
        kvp.set_optimizer(opt)
    before = env.variant_counts()
    env.torch.cuda.synchronize(); env.barrier()
    kvp.pushpull(keys, grads, out=weights)
    mx.nd.waitall(); env.torch.cuda.synchronize()
    variant = variant_since(env, before)
    sums = [int(w.asnumpy().view(np.int32).astype(np.int64).sum()) for w in weights] if env.world > 1 else []
    chk = sum(sums) & 0x7FFFFFFFFFFFFFFF
    replicas_equal = len(set(env.allgather_int(chk))) == 1
    res = {"checked": True, "variant": variant, "replicas_bit_identical": replicas_equal, "keys": len(keys)}
    kept = None
    tree = oracle_tree(env, kvtype)
    if tree is not None:
        res["sum_order"] = "MXNET_KVSTORE_USETREE"
    if env.rank == 0:
        _, kw, oname, _ = OPTIMIZERS[args.optimizer]
        all_g = [rank_grads(r, shapes) for r in range(env.world)]
        okv = O.OracleKVStore("device", tree=tree)
        okv.init(keys, [w.copy() for w in w0])
        layerwise = oname in ("lamb", "lans", "lars")
        if oname:
            okv.set_optimizer(O.OracleOptimizer(oname, **(dict(kw, norm_mode="f64") if layerwise else kw)))
        okv.push(keys, [[all_g[r][k] for r in range(env.world)] for k in keys])
        worst, exact = 0.0, True
        wants = []
        for k, s in zip(keys, shapes):
            want = np.empty(s, np.float32)
            okv.pull(k, want)
            got = weights[k].asnumpy().reshape(s)
            if not np.array_equal(got.view(np.uint32), want.view(np.uint32)):
                exact = False
                den = max(float(np.abs(want).sum(dtype=np.float64)), 1e-30)
                worst = max(worst, float(np.abs(got.astype(np.float64) - want).sum() / den))
            wants.append(want)
        must_be_exact = "nvls" not in variant and not layerwise
        res.update({"max_rel_l1": worst, "bit_exact": exact, "tolerance": 0.0 if must_be_exact else 1e-6,
                    "ok": bool(replicas_equal and (exact or (not must_be_exact and worst <= 1e-6)))})
        if keep:
            gsum = [okv._reduce([all_g[r][k] for r in range(env.world)]).reshape(shapes[k]) if env.world > 1
                    else all_g[0][k] for k in keys]
            kept = {"fused": wants, "allreduce": gsum}
    ok = env.allgather_int(1 if (env.rank != 0 or res.get("ok")) else 0)
    res["ok"] = all(ok) and replicas_equal
    del kvp
    return res, kept


# ---------------------------------------------------------------------------
# BASELINE.json configs[1] as a sweep (tools/bandwidth/measure.py:113-138): per key size
# ---------------------------------------------------------------------------
def sweep_points(env, args, shapes, grads, weights, kept):
    """Per key size E = 2^10 ... 2^26 and per mode (all-reduce only / with the fused SGD-momentum update): one key
    per call, back-to-back calls, device time per call from CUDA events on the engine stream (max over ranks),
    bus bandwidth 2S(n-1)/n/t, the kernel variant the engine chose -- next to NCCL's all-reduce of the same
    buffer size timed in the same process.  The first call of every point is checked against the oracle."""
    mx, torch = env.mx, env.torch
    n = env.world
    stream = env.engine_stream()
    twoshot = int(os.environ.get("MXKV_B200_TWOSHOT_BYTES", 256 * 1024))
    stores = {}
    for mode in ("allreduce", "fused"):
        kv = mx.kv.create("device")
        kv.init(list(range(len(shapes))), [mx.nd.array(w, env.ctx) for w in initial_weights(shapes)])
        if mode == "fused":
            kv.set_optimizer(make_optimizer(mx, "sgd"))
        stores[mode] = kv
    points = []
    for k, s in enumerate(shapes):
        E = nelem(s)
        row = {"elements": E, "bytes": 4 * E, "path": ("two-shot" if (n > 1 and 4 * E >= twoshot and E >= 128 * n) else
                                                       ("one-shot" if n > 1 else "local"))}
        for mode in ("allreduce", "fused"):
            kv = stores[mode]
            before = env.variant_counts()
            env.torch.cuda.synchronize(); env.barrier()
            kv.pushpull(k, grads[k], out=weights[k])                  # first call: verified
            mx.nd.waitall()
            ok = None
            if env.rank == 0 and kept is not None and (mode == "allreduce" or args.optimizer == "sgd"):
                ok = True
                want = kept[mode][k]
                got = weights[k].asnumpy().reshape(want.shape)
                if not np.array_equal(got.view(np.uint32), want.view(np.uint32)):
                    den = max(float(np.abs(want).sum(dtype=np.float64)), 1e-30)
                    ok = float(np.abs(got.astype(np.float64) - want).sum() / den) <= 1e-6
            variant = variant_since(env, before)
            for _ in range(3):
                kv.pushpull(k, grads[k], out=weights[k])
            torch.cuda.synchronize(); env.barrier()
            est_ms = max(0.01, 4.0 * E * (1 if n == 1 else 2) / 600e6)
            steps = int(min(200, max(20, 40.0 / est_ms)))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                kv.pushpull(k, grads[k], out=weights[k])
            e1.record(stream)
            torch.cuda.synchronize()
            us = env.max_over_ranks([e0.elapsed_time(e1) / steps * 1e3])[0]
            ent = {"us_per_call": us, "variant": variant, "verified": ok, "calls": steps}
            if n > 1:
                ent["busbw_gbs"] = 2.0 * 4 * E * (n - 1) / n / (us * 1e-6) / 1e9
            else:
                streams = OPTIMIZERS["sgd"][3] if mode == "fused" else OPTIMIZERS["none"][3]
                ent["hbm_gbs"] = 4.0 * E * streams / (us * 1e-6) / 1e9
            row[mode] = ent
        if n > 1:
            t = torch.empty(E, device="cuda", dtype=torch.float32).uniform_(-1, 1)
            for _ in range(3):
                env.dist.all_reduce(t)
            torch.cuda.synchronize(); env.barrier()
            steps = row["allreduce"]["calls"]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                env.dist.all_reduce(t)
            e1.record()
            torch.cuda.synchronize()
            us = env.max_over_ranks([e0.elapsed_time(e1) / steps * 1e3])[0]
            row["nccl_allreduce"] = {"us_per_call": us, "busbw_gbs": 2.0 * 4 * E * (n - 1) / n / (us * 1e-6) / 1e9,
                                     "note": "torch.distributed.all_reduce (NCCL %s), in place, same process" %
                                             ".".join(str(x) for x in torch.cuda.nccl.version())}
            del t
        points.append(row)
    for kv in stores.values():
        del kv
    return points


# ---------------------------------------------------------------------------
# samples/sec: BASELINE.json configs[2] -- ResNet-50 bf16, synthetic 3x224x224, SGD-momentum
# (multi-precision) through Trainer(kvstore='device'); torch does forward/backward, the engine does
# the gradient exchange + fused update.
# ---------------------------------------------------------------------------
def gluon_resnet50(torch):
    """torchvision's resnet50 re-shaped into Gluon's resnet50_v1 (python/mxnet/gluon/model_zoo/vision/resnet.py:
    106-116): BottleneckV1 keeps the BIAS on both 1x1 convolutions and puts the stride on the first one -- 193
    parameter arrays instead of torchvision's 161."""
    import torchvision
    model = torchvision.models.resnet50(weights=None)
    for layer in (model.layer1, model.layer2, model.layer3, model.layer4):
        for blk in layer:
            stride = blk.conv2.stride
            c1, c2, c3 = blk.conv1, blk.conv2, blk.conv3
            blk.conv1 = torch.nn.Conv2d(c1.in_channels, c1.out_channels, 1, stride=stride, bias=True)
            blk.conv2 = torch.nn.Conv2d(c2.in_channels, c2.out_channels, 3, stride=1, padding=1, bias=False)
            blk.conv3 = torch.nn.Conv2d(c3.in_channels, c3.out_channels, 1, bias=True)
    return model


def bert_base(torch, seq):
    """BERT-base (12 x 768, 12 heads, vocabulary 30522) with a masked-LM head, random init."""
    import transformers
    cfg = transformers.BertConfig(max_position_embeddings=512)
    try:
        cfg._attn_implementation = "sdpa"
    except Exception:
        pass
    return transformers.BertForMaskedLM(cfg)


def train_steps(env, args, which, steps, dump=None):
    """One JSON-able dict: samples/sec of `steps` timed `which` ('resnet50' | 'bert') training steps -- torch
    forward/backward in bf16, Trainer(kvstore='device') exchanging + updating (fused, multi-precision: fp32 master
    weights and state in the engine) every parameter in one launch per step.  dump: --dump-outputs directory."""
    torch, mx = env.torch, env.mx
    torch.manual_seed(0)
    if which == "resnet50":
        model = gluon_resnet50(torch).cuda().to(memory_format=torch.channels_last).to(torch.bfloat16)
        B = args.batch
        x = torch.randn(B, 3, 224, 224, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
        y = torch.randint(0, 1000, (B,), device="cuda")
        lossf = torch.nn.CrossEntropyLoss()
        optname, okw = "sgd", {"learning_rate": 0.1, "momentum": 0.9, "wd": 1e-4, "multi_precision": True}

        def fwd():
            return lossf(model(x).float(), y)
        metric = "samples/sec (Gluon ResNet-50-v1 bf16, synthetic 3x224x224, Trainer(kvstore='device'))"
        desc = "resnet50-train: Gluon resnet50_v1 layout (1x1-conv biases kept), batch %d per GPU, SGD momentum 0.9 wd 1e-4 multi-precision"
    else:
        seq = 128
        model = bert_base(torch, seq).cuda().to(torch.bfloat16)
        B = args.bert_batch
        x = torch.randint(0, 30522, (B, seq), device="cuda")
        y = torch.randint(0, 30522, (B, seq), device="cuda")
        optname, okw = "adam", {"learning_rate": 1e-4, "wd": 0.01, "multi_precision": True}

        def fwd():
            return model(input_ids=x, labels=y).loss
        metric = "samples/sec (BERT-base bf16, seq 128, synthetic tokens, fused multi-precision Adam, Trainer(kvstore='device'))"
        desc = "bert-train: BERT-base masked-LM (random init), seq 128, batch %d per GPU, Adam multi-precision"
    params = [p for p in model.parameters() if p.requires_grad]
    trainer = mx.Trainer(params, optname, okw, kvstore="device", symmetric=True, overlap=bool(args.overlap))
    world = env.world
    if not trainer._kv_initialized:
        trainer._init_kvstore()              # binds p.data / p.grad to the peer-mapped arena
    gl = [p.grad for p in params]

    def step(ev=None):
        loss = fwd()
        loss.backward()
        if ev is not None:
            ev[0].record()
        trainer.step(B * world)
        if ev is not None:
            ev[1].record()
        torch._foreach_zero_(gl)
        return loss

    warm = max(3, args.warmup)
    for _ in range(warm):
        step()
    torch.cuda.synchronize(); env.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ec = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    launches0 = mx.kv.launch_count()
    e0.record()
    for i in range(steps):
        loss = step(ec[i])
    e1.record()
    torch.cuda.synchronize()
    ms, comm_ms = env.max_over_ranks([e0.elapsed_time(e1) / steps, sum(a.elapsed_time(b) for a, b in ec) / steps])
    if dump and env.rank == 0:          # before the traced step below updates the parameters again
        mx.nd.waitall()
        dump_outputs(dump, [("param_%03d" % i, p.numel(), lambda p=p: p.detach().float().cpu().numpy())
                            for i, p in enumerate(params)])
    nparam = sum(p.numel() for p in params)
    # one traced step: where the buckets' exchange ran relative to backward (CUDA events on the engine stream
    # against events on the framework stream; stands in for an nsys timeline, which this image does not have)
    trace = None
    if args.overlap and getattr(trainer, "_buckets", None):
        trainer.trace = []
        eb0, eb1, eb2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        loss = fwd()
        eb0.record()
        loss.backward()
        eb1.record()
        trainer.step(B * world)
        eb2.record()
        torch._foreach_zero_(gl)
        torch.cuda.synchronize()
        bw = eb0.elapsed_time(eb1)
        # per bucket: when its gradients were ready (framework stream) and when its exchange + update had
        # finished (engine stream), ms from the start of backward; an exchange can start at max(ready, previous end)
        rows = [[b, eb0.elapsed_time(s), eb0.elapsed_time(e)] for b, s, e in trainer.trace]
        busy, prev_end = 0.0, None
        for _, ready, end in rows:
            start = ready if prev_end is None else max(ready, prev_end)
            busy += max(0.0, end - start)
            prev_end = end
        trace = {"backward_ms": bw, "step_call_ms_after_backward": eb1.elapsed_time(eb2),
                 "buckets_ready_end_ms_from_backward_start": [[b, round(s, 3), round(e, 3)] for b, s, e in rows],
                 "exchange_busy_ms_upper_bound": busy,
                 "exchange_exposed_ms_after_backward": max(0.0, max(e for _, _, e in rows) - bw) if rows else None}
        trainer.trace = None
    out = {"metric": metric, "value": world * B / (ms * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": steps,
           "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16", "data": "synthetic",
           "config": {"workload": (desc % B) + ", %d keys / %.1f M params" % (len(params), nparam / 1e6),
                      "exchange_ms_per_step_after_backward": comm_ms, "keys": len(params),
                      "overlap_with_backward": bool(args.overlap), "overlap_trace": trace},
           "gpu_launches": mx.kv.launch_count() - launches0, "loss": float(loss)}
    del trainer, model
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------
# BASELINE.json configs[4]: one row_sparse key (1 M x 256 fp32), 10 k distinct rows per GPU;
# step = row_sparse push (union + gather-sum + lazy SGD-momentum on the touched rows) followed by
# row_sparse_pull of the same ids.
# ---------------------------------------------------------------------------
def bench_rsp(env, args, steps, dump=None):
    torch, mx = env.torch, env.mx
    rank, world, ctx = env.rank, env.world, env.ctx
    R, L, nnz = 1_000_000, 256, 10_000
    rng = np.random.default_rng(1234 + rank)
    idx = np.sort(rng.choice(R, nnz, replace=False)).astype(np.int64)
    val = rng.uniform(-1, 1, (nnz, L)).astype(np.float32)
    grad = mx.nd.row_sparse_array((val, idx), shape=(R, L), ctx=ctx)
    ids = mx.nd.array(idx, ctx, dtype=np.int64)
    out = mx.nd.empty((R, L), ctx, stype="row_sparse", capacity=nnz)
    kv = mx.kv.create("device")
    kv.init("emb", mx.nd.row_sparse_array((np.zeros((1, L), np.float32), np.zeros(1, np.int64)), shape=(R, L), ctx=ctx))
    kv.set_optimizer(mx.optimizer.SGD(learning_rate=0.01, momentum=0.9, wd=0.0, lazy_update=True))

    def step():
        kv.push("emb", grad)
        kv.row_sparse_pull("emb", out=out, row_ids=ids)

    warm = max(3, args.warmup)
    for _ in range(warm):
        step()
    torch.cuda.synchronize(); env.barrier()
    launches0 = mx.kv.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = env.max_over_ranks([e0.elapsed_time(e1) / steps])[0]
    union = int(out.indices.shape[0])
    if dump and env.rank == 0:          # the rows the last pull returned, and their row ids
        dump_outputs(dump, [("out_data", out.data.size, out.data.asnumpy),
                            ("out_indices", union, lambda: out.indices.asnumpy().astype(np.float64))])
    # parity of exactly this shape: the pulled rows against the oracle's lazy SGD-momentum after warm+steps pushes
    # is the job of tests/test_gpu_rsp.py::test_c5_shape; here the union size is cross-checked
    all_idx = np.unique(np.concatenate([np.sort(np.random.default_rng(1234 + r).choice(R, nnz, replace=False))
                                        for r in range(world)]))
    row_bytes = L * 4
    # algorithmic bytes per GPU per step: read every rank's nnz rows (+ ids), read-modify-write weight and momentum
    # rows of the union (2 reads + 2 writes), then gather nnz rows out (read + write)
    alg = world * nnz * (row_bytes + 8) + int(all_idx.size) * row_bytes * 4 + nnz * row_bytes * 2
    peak = measured_peaks().get("hbm_gbs", 6650.0)
    res = {"metric": "row_sparse push + row_sparse_pull rows/s", "value": world * nnz / (ms * 1e-3),
           "unit": "rows/s", "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": ms,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "rsp: 1 key 1000000x256 fp32 row_sparse, %d rows per GPU, lazy SGD-momentum, "
                                  "push + row_sparse_pull" % nnz, "union_rows": int(all_idx.size),
                      "pulled_rows": union},
           "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_step": alg, "traffic": None,
                        "note": "latency-bound: %d launches per step move %.1f MB" % (
                            (mx.kv.launch_count() - launches0) // steps, alg / 1e6)},
           "gpu_launches": mx.kv.launch_count() - launches0}
    del kv
    return res


# timed steps of the secondaries the sweep runs: fixed, so that --steps sets the headline's count alone
SECONDARY_TRAIN_STEPS = 30
SECONDARY_RSP_STEPS = 100

DUMP_LIMIT_ELEMS = 8 << 20      # --dump-outputs writes at most 8 Mi elements (32 MiB of float32)


def dump_counts(sizes, limit=DUMP_LIMIT_ELEMS):
    """How many elements of each array --dump-outputs writes: every array whole while the total fits in `limit`,
    else every array whole up to one common cap, the larger ones sampled down to it."""
    counts, left = {}, limit
    order = sorted(range(len(sizes)), key=lambda k: sizes[k])
    for i, k in enumerate(order):
        counts[k] = min(sizes[k], left // (len(order) - i))
        left -= counts[k]
    return [counts[k] for k in range(len(sizes))]


def dump_outputs(path, arrays):
    """arrays: (name, elements, fetch) per array, fetch() returning it as a numpy array.  Writes DIR/<name>.npy --
    float64 arrays as float64, everything else as float32 -- the whole array, or (beyond the dump_counts budget) the
    flattened array at a sorted sample of positions drawn with seed <index in arrays>, so that two runs with the same
    arguments write the same positions."""
    os.makedirs(path, exist_ok=True)
    counts = dump_counts([n for _, n, _ in arrays])
    for k, ((name, n, fetch), c) in enumerate(zip(arrays, counts)):
        a = fetch()
        if c < n:
            a = a.reshape(-1)[np.sort(np.random.default_rng(k).choice(n, c, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


_PEAKS = None


def measured_peaks():
    global _PEAKS
    if _PEAKS is None:
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                _PEAKS = json.load(f)
        except Exception:
            _PEAKS = {}
    return _PEAKS


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sweep", choices=["sweep", "resnet50", "bert", "resnet50-train", "bert-train", "rsp"])
    ap.add_argument("--batch", type=int, default=128, help="per-GPU batch of resnet50-train")
    ap.add_argument("--bert-batch", type=int, default=32, help="per-GPU batch of bert-train")
    ap.add_argument("--optimizer", default=None, choices=[None, "sgd", "adam", "lamb", "lans", "lars", "none"])
    ap.add_argument("--overlap", type=int, default=1, help="training workloads: exchange buckets from grad-ready hooks")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-nvls", action="store_true", help="keep gradients/weights out of multicast memory")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the per-size sweep array")
    ap.add_argument("--no-secondary", action="store_true", help="skip the ResNet-50 / BERT / row_sparse secondaries")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="do not run the nvidia-smi clock sampler (diagnosis)")
    ap.add_argument("--no-nvml", action="store_true", help="do not read the NVML NVLink counters (diagnosis)")
    ap.add_argument("--local-world", type=int, default=0,
                    help="split the box into 'nodes' of this many GPUs and use kv.create('dist_device_sync'): NVLink "
                         "peer memory inside a node, NCCL between nodes (not the driver's configuration)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned, to compare two builds: the pulled weights "
                         "(DIR/out_<key>.npy), the trained parameters (DIR/param_<i>.npy) or the pulled row_sparse "
                         "rows (DIR/out_data.npy, DIR/out_indices.npy); float32 (row ids float64), a fixed seeded "
                         "sample of the larger arrays, 8 Mi elements in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.optimizer is None:
        args.optimizer = "adam" if args.workload == "bert" else "sgd"
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", rank)) if world > 1 else 0

    if args.workload in ("resnet50-train", "bert-train", "rsp"):
        numa = bind_to_gpu_numa(local)
        env = Env(args)
        if args.workload == "rsp":
            res = bench_rsp(env, args, args.steps, args.dump_outputs)
        else:
            res = train_steps(env, args, "resnet50" if args.workload == "resnet50-train" else "bert", args.steps,
                              args.dump_outputs)
        res["numa"] = numa
        if env.rank == 0:
            print(json.dumps(res))
        env.finish()
        return

    shapes = keyset(args.workload)
    S = 4 * sum(nelem(s) for s in shapes)
    config = {"workload": "%s: pushpull of %d fp32 keys (%.1f MB per rank), fused %s update" % (
        args.workload, len(shapes), S / 1e6, args.optimizer),
        "keys": len(shapes), "bytes_per_rank": S, "optimizer": args.optimizer,
        "parallelism": "dp%d (one process per GPU, gradient exchange over NVLink peer memory)" % args.gpus,
        "l2": "working set (%.0f MB grads + weights + state per rank) exceeds the 126 MB L2; no flush" % (3 * S / 1e6)}

    if args.impl == "reference":
        if rank != 0:
            return
        value, dt, base = run_cpu_reference(args, shapes)
        line = {"impl": "reference", "metric": "kvstore push+pull GB/s", "value": value, "unit": "GB/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config, "cpu_baseline": base,
                "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    sampler = ClockSampler(local)
    if rank == 0 and not args.no_clocks:
        sampler.start()                      # nvidia-smi needs about a second before its first sample
    numa = bind_to_gpu_numa(local)
    env = Env(args)
    torch, mx = env.torch, env.mx
    hier, ctx = env.hier, env.ctx

    keys = list(range(len(shapes)))
    # gradients / weights live in the peer-mapped arena (zero-copy over NVLink); at N=1 this is
    # plain device memory
    exchange = "nvlink-p2p" if world > 1 else "none (one GPU)"
    alloc = mx.nd.empty_symmetric
    if hier:
        exchange = "hierarchical: nvlink-p2p in nodes of %d, nccl between %d nodes" % (
            args.local_world, world // args.local_world)
    if env.multicast:
        if env.multicast == "torch":
            alloc = mx.nd.empty_multicast      # NVSwitch multicast-capable arrays from torch's allocator
        # the engine switches to the multimem kernel above 4 ranks (MXKVB200SetNvls)
        exchange = ("nvls-multicast" if world > 4 else "nvlink-p2p (multicast-capable arrays)") + \
                   " [%s-owned multicast memory]" % env.multicast
    grads = [alloc(s) for s in shapes]
    weights = [alloc(s) for s in shapes]
    for g, a in zip(grads, rank_grads(rank, shapes)):
        g[:] = a
    kvtype = "dist_device_sync" if hier else "device"
    kv = mx.kv.create(kvtype)
    kv.init(keys, [mx.nd.array(w, ctx) for w in initial_weights(shapes)])
    opt = make_optimizer(mx, args.optimizer)
    if opt is not None:
        kv.set_optimizer(opt)
    bytes_per_elem_n1 = OPTIMIZERS[args.optimizer][3] * 4
    layerwise = args.optimizer in ("lamb", "lans", "lars")

    def step():
        kv.pushpull(keys, grads, out=weights)

    engine_stream = env.engine_stream()
    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    if rank == 0:
        sampler.wait_first()
    env.barrier()

    # ---- timed region: device time (inputs resident in HBM) ----------------------------------
    launches0 = mx.kv.launch_count()
    variants0 = env.variant_counts()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize(); env.barrier()
    nvl0 = nvlink_counters(local) if (world > 1 and not args.no_nvml) else None
    t_host0 = time.time()
    ev0.record()
    for i in range(args.steps):
        kern[i][0].record(engine_stream)
        step()
        kern[i][1].record(engine_stream)
    ev1.record()
    host_issue_ms = (time.time() - t_host0) * 1e3 / args.steps      # the host's share: calls are asynchronous
    torch.cuda.synchronize(); env.barrier()
    nvl1 = nvlink_counters(local) if (world > 1 and not args.no_nvml) else None
    # the untimed steps and the parity check below overwrite `weights`: keep what the last timed step returned
    snapshot = [w.copyto(ctx) for w in weights] if (args.dump_outputs and rank == 0) else None
    launches = mx.kv.launch_count() - launches0
    variant = variant_since(env, variants0)
    ms_total = ev0.elapsed_time(ev1)
    kern_ms = statistics.mean(a.elapsed_time(b) for a, b in kern)
    ms_total, kern_ms = env.max_over_ranks([ms_total, kern_ms])
    ms_step = ms_total / args.steps
    value = world * 2 * S / (ms_step * 1e-3) / 1e9
    # clocks: the timed window is a few hundred ms at most -- every rank keeps the SAME steps running (untimed)
    # until the GPU has been under this load for ~0.6 s, so that the 100 ms sampler sees it several times; the
    # record covers both windows and says so
    soak_steps = int(min(5000, max(0.0, 600.0 - ms_total) / max(ms_step, 1e-3)))
    for _ in range(soak_steps):
        step()
    torch.cuda.synchronize(); env.barrier()
    t_host2 = time.time()
    clocks = None
    if rank == 0:
        clocks = sampler.stop(t_host0, t_host2)
        clocks["window"] = "timed region (%d steps)%s" % (
            args.steps, " + %d identical untimed steps (~0.6 s under load for the 100 ms sampler)" % soak_steps if soak_steps else "")

    # ---- roofline for the dominant (only) kernel ------------------------------------------------
    peaks = measured_peaks()
    nel = S // 4
    kname = "+".join(KERNEL_NAMES.get(v, v) for v in variant.split("+"))
    if world == 1:
        alg = nel * bytes_per_elem_n1
        peak = peaks.get("hbm_gbs", 6650.0)
        roof = {"bound": "hbm", "achieved": alg / (kern_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650",
                "traffic": None, "kernel": "kv_norm_first/(mid)/apply_kernel sequence" if layerwise else kname,
                "kernel_ms": kern_ms, "algorithmic_bytes_per_launch": alg}
        if args.optimizer == "sgd":
            # SURVEY 8d counts the reference's in-place update (read g, w, mom; write w, mom = 5 streams); the
            # sixth stream is the caller's `out` array, which the pushpull contract makes this kernel write
            roof["frac_in_place_5_streams"] = nel * 20 / (kern_ms * 1e-3) / 1e9 / peak
    else:
        if "nvls" in variant:
            # in-switch reduction + replication: per GPU per direction S (own data out / all shards in)
            # plus S/n (its reduced shard in / its updated shard out)
            alg = S * (1.0 + 1.0 / world)
            kname += " (multimem.ld_reduce + fused update + multimem.st)"
        else:
            alg = 2.0 * S * (world - 1) / world      # per GPU per direction (tools/bandwidth/measure.py:138)
            kname += " (peer loads + fused update + peer stores)"
        roof = {"bound": "nvlink", "achieved": alg / (kern_ms * 1e-3) / 1e9, "peak": 770.0, "unit": "GB/s",
                "peak_source": "B200_PROFILING.md measured peer copy 770 GB/s/dir (900 nominal)",
                "traffic": None, "kernel": kname, "kernel_ms": kern_ms,
                "algorithmic_bytes_per_launch": alg,
                "note": "bytes that must cross this GPU's NVLink per direction; busbw_gbs_per_gpu is the "
                        "NCCL-comparable 2S(n-1)/n / t"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    if world > 1:
        if nvl0 and nvl1 and "error" not in nvl0 and "error" not in nvl1:
            per = {k: (nvl1[k] - nvl0[k]) / args.steps for k in _NVL_FIELDS}
            # (the NVML counters tick in coarse units and lag by a sampling period: over 300 steps that is < 1 %)
            roof["traffic"] = per["raw_tx"] + per["raw_rx"]
            roof["traffic_source"] = "NVML NVLINK_THROUGHPUT_RAW_TX + RAW_RX of this rank's GPU over the timed region, per step"
            roof["nvlink_bytes_per_step"] = per
            roof["nvlink_raw_gbs_per_dir"] = {"tx": per["raw_tx"] / (ms_step * 1e-3) / 1e9, "rx": per["raw_rx"] / (ms_step * 1e-3) / 1e9}
            roof["nvlink_payload_efficiency"] = {"tx": per["data_tx"] / max(per["raw_tx"], 1.0), "rx": per["data_rx"] / max(per["raw_rx"], 1.0)}
        else:
            roof["traffic_error"] = (nvl0 or {}).get("error") or (nvl1 or {}).get("error")
    # DRAM / NVLink bytes of the same kernel on the same workload from this round's ncu capture (bench.py
    # cannot run under ncu itself: a number printed under a profiler is never a bench value)
    tsrc = os.path.join(ROOT, "profiles", "r02_n%d_%s_ncu_full.txt" % (world, variant.replace("+", "_")))
    if args.workload == "sweep" and args.optimizer == "sgd" and os.path.exists(tsrc):
        roof["traffic"], roof["traffic_source"] = ncu_dram_bytes(tsrc), os.path.relpath(tsrc, ROOT)

    # ---- parity of what was just timed --------------------------------------------------------------
    parity, kept = {"checked": False}, None
    if not args.no_parity and not hier:
        parity, kept = parity_check(env, args, shapes, keys, grads, weights, kvtype,
                                    keep=(args.workload == "sweep" and not args.no_sweep))

    # ---- e2e: host gradients in, host weights out, through the same public API ---------------------
    e2e = None
    if not args.no_e2e:
        hg = [mx.nd.empty(s, mx.cpu_pinned()) for s in shapes]
        hw = [mx.nd.empty(s, mx.cpu_pinned()) for s in shapes]
        for g, a in zip(hg, rank_grads(rank + 100, shapes)):
            g[:] = a
        for _ in range(2):
            kv.pushpull(keys, hg, out=hw)
        mx.nd.waitall(); torch.cuda.synchronize(); env.barrier()
        n_e2e = max(3, args.steps // 4)
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            kv.pushpull(keys, hg, out=hw)
        mx.nd.waitall(); torch.cuda.synchronize()
        dt = env.max_over_ranks([time.perf_counter() - t0])[0] / n_e2e
        e2e = {"value": world * 2 * S / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": S,
               "d2h_bytes_per_step": S, "ms_per_step": dt * 1e3, "steps": n_e2e,
               "how": "pinned host gradients -> kv.pushpull -> pinned host weights, wall clock incl. both copies"}
        del hg, hw

    # ---- the sweep as a sweep, and the other BASELINE configs ---------------------------------------
    sweep = None
    if args.workload == "sweep" and not args.no_sweep and not hier:
        try:
            sweep = sweep_points(env, args, shapes, grads, weights, kept)
        except Exception as e:          # noqa: BLE001 -- the headline numbers stand on their own
            sweep = {"error": repr(e)[:300]}
    kept = None
    secondary = None
    if args.workload == "sweep" and not args.no_secondary and not hier:
        secondary = {}
        del kv, grads, weights
        torch.cuda.empty_cache()
        for name, fn in (("row_sparse_C5", lambda: bench_rsp(env, args, SECONDARY_RSP_STEPS)),
                         ("resnet50_C3", lambda: train_steps(env, args, "resnet50", SECONDARY_TRAIN_STEPS)),
                         ("bert_base_C4", lambda: train_steps(env, args, "bert", SECONDARY_TRAIN_STEPS))):
            try:
                secondary[name] = fn()
            except Exception as e:          # noqa: BLE001
                secondary[name] = {"error": repr(e)[:300]}
            torch.cuda.synchronize(); env.barrier()

    if rank != 0:
        env.finish()
        return

    cpu_base = None
    if not args.no_cpu_baseline:
        _, _, cpu_base = run_cpu_reference(args, shapes, as_baseline=True)

    line = {"metric": "kvstore push+pull GB/s", "value": value, "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "roofline": roof, "cpu_baseline": cpu_base, "e2e": e2e, "gpu_launches": launches,
            "host_issue_ms_per_step": host_issue_ms,
            "clocks": clocks, "parity": parity,
            "busbw_gbs_per_gpu": (2.0 * S * (world - 1) / world) / (ms_step * 1e-3) / 1e9 if world > 1 else 0.0,
            "exchange": exchange, "numa": numa,      # (not in `config`: the reference arm prints the same config)
            "sweep": sweep, "secondary": secondary}
    if snapshot is not None:
        dump_outputs(args.dump_outputs, [("out_%03d" % k, w.size, w.asnumpy) for k, w in enumerate(snapshot)])
    if parity.get("checked") and not parity.get("ok"):
        sys.stderr.write("PARITY FAILURE: the timed configuration does not match the oracle\n" + json.dumps(line) + "\n")
        env.finish()
        sys.exit(1)
    print(json.dumps(line))
    env.finish()


if __name__ == "__main__":
    main()

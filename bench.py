#!/usr/bin/env python
"""bench.py -- KVStore push+pull throughput on the ResNet-50 gradient set (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload ...]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over the synthetic gradient set: push the gradients of all
157 ResNet-50 tensors (25 549 486 fp32 elements, uniform [-1,1)), reduce them, apply SGD with
momentum ON THE STORE, and pull the new weights back -- one grouped MXKVStorePushPull call, which
the library turns into ONE fused kernel launch per GPU.

Printed JSON (one line, rank 0):
  value      push+pull payload GB/s of the whole job: n_gpus x (bytes pushed + bytes pulled per GPU)
             / step time -- the same definition at every N, so the per-N lines are comparable --
             inputs and outputs resident in HBM, timed with CUDA events on the launching stream
  e2e        same metric through the same C-ABI call with HOST buffers (pinned CPU-context
             NDArrays): the H2D copy of the gradients and the D2H copy of the weights are inside
             the timed region; e2e.roofline = bytes per PCIe direction / time against the pinned
             copy rate measured in the same run with both directions busy
  roofline   dominant kernel: ALGORITHMIC bytes per launch (SURVEY.md 8d: 24 B/element for
             SGD-momentum at N=1; all-reduce bus bandwidth per GPU, tools/bandwidth/measure.py:137-138,
             at N>=2) / mean launch duration (CUDA events) against the measured HBM copy bandwidth
             (MEASURED_PEAKS.json) or 900 GB/s/dir NVLink
  parity     the weights pulled after the first two steps of THIS run compared with the CPU oracle
             (kvstore('local') model fed the same seeded gradients): bit-exact, or <= 1e-6 relative
             L1 when the NVSwitch sums (NVLS mode); a failed check makes the run exit non-zero
  configs    short legs over the other BASELINE.json configs (BERT-base + Adam, row_sparse table
             1M x 512) with their own roofline / parity blocks
  frontends  the same step issued the way the reference's callers do: one call PER KEY with
             priority=-i (gluon/trainer.py:385-396) and push-all-then-pull-all (tools/bandwidth/
             measure.py:112-122), plus the python front-end's grouped call
  cpu_baseline   the reference's CPU kvstore('local') arithmetic (oracle/_ref, else the oracle
             port) on this box's host cores, bounded sample
`--impl reference` times that CPU path as the whole job (the driver's reference arm).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "kvstore_push_pull_GBps"
UNIT = "GB/s"
VALUE_FORMULA = ("n_gpus * (bytes pushed + bytes pulled per GPU) / time = n_gpus * 2 * gradient-set "
                 "bytes / time, identical at every N; roofline.achieved uses the kernel's algorithmic "
                 "bytes (HBM, N=1) or the all-reduce bus bandwidth per GPU (NVLink, N>=2)")
L2_NOTE = "per-GPU working set of a step > 126 MB L2 (inputs larger than L2), no flush between steps"


# ------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------
def resnet50_shapes():
    """Gradient tensors of the reference's ResNet-50 symbol (example/image-classification/symbols/
    resnet.py, num_layers=50: units [3,4,6,3], filters [64,256,512,1024,2048], bottleneck, 1000
    classes): 157 arrays, 25 549 486 elements (SURVEY.md 8a)."""
    shapes = [(3,), (3,), (64, 3, 7, 7), (64,), (64,)]  # bn_data gamma/beta, conv0, bn0
    filters = [64, 256, 512, 1024, 2048]
    units = [3, 4, 6, 3]
    for stage in range(4):
        nf = filters[stage + 1]
        for u in range(units[stage]):
            cin = filters[stage] if u == 0 else nf
            q = nf // 4
            shapes += [(cin,), (cin,), (q, cin, 1, 1), (q,), (q,), (q, q, 3, 3), (q,), (q,),
                       (nf, q, 1, 1)]
            if u == 0:
                shapes.append((nf, cin, 1, 1))  # projection shortcut
    shapes += [(2048,), (2048,), (1000, 2048), (1000,)]
    return shapes


def bert_base_shapes():
    """BERT-base parameter set: 199 arrays, 109 482 240 elements (SURVEY.md 8a)."""
    H, L, FF, V = 768, 12, 3072, 30522
    shapes = [(V, H), (512, H), (2, H), (H,), (H,)]
    for _ in range(L):
        shapes += [(H, H), (H,)] * 4 + [(H,), (H,), (FF, H), (FF,), (H, FF), (H,), (H,), (H,)]
    shapes += [(H, H), (H,)]
    return shapes


WORKLOADS = {
    "resnet50_sgd": dict(shapes=resnet50_shapes, opt="sgd", bytes_per_elem=24,
                         desc="ResNet-50 gradient set, 157 fp32 tensors / 25549486 elements, "
                              "SGD momentum fused on the store"),
    "bert_adam": dict(shapes=bert_base_shapes, opt="adam", bytes_per_elem=32,
                      desc="BERT-base gradient set, 199 fp32 tensors / 109482240 elements, Adam "
                           "fused on the store"),
}
RSP_DESC = ("row_sparse push + row_sparse_pull, embedding table (1000000, 512) fp32, 10000 distinct hot "
            "rows per value (1 %), lazy SGD on the store, pull ids unsorted with 5 % duplicates")

SGD_KW = dict(learning_rate=0.1, momentum=0.9, wd=1e-4)
ADAM_KW = dict(learning_rate=1e-3, beta1=0.9, beta2=0.999, epsilon=1e-8, wd=0.01)


def opt_kwargs(workload, n_gpus):
    if WORKLOADS[workload]["opt"] == "sgd":
        return "SGD", dict(rescale_grad=1.0 / (256 * n_gpus), **SGD_KW)
    return "Adam", dict(rescale_grad=1.0 / n_gpus, **ADAM_KW)


def kernel_label(workload, n_src, nvls=False):
    opt = "SGD" if WORKLOADS[workload]["opt"] == "sgd" else "Adam"
    return "dense_fused_kernel<float,%d,%s>%s" % (1 if nvls else n_src, opt, " [NVLS multimem]" if nvls else "")


def config_block(workload, n_values):
    """`config` is a pure function of (workload, N): both arms of the driver's comparison print the
    same dict; arm-specific descriptors live under `impl_detail`."""
    desc = RSP_DESC if workload == "rsp" else WORKLOADS[workload]["desc"]
    return {"workload": desc, "values_per_key": n_values, "value_formula": VALUE_FORMULA, "l2": L2_NOTE}


def payload_bytes(workload, n_gpus):
    """`value`: bytes PUSHED plus bytes PULLED per step over the whole job -- the same definition at
    every N (each GPU pushes its gradient set and pulls the weights), so the per-N values are
    comparable (weak scaling). The roofline uses the kernel's ALGORITHMIC bytes instead."""
    n_elem = sum(int(np.prod(s)) for s in WORKLOADS[workload]["shapes"]())
    return n_gpus * n_elem * 4 * 2


def algorithmic_bytes(workload, n_gpus):
    n_elem = sum(int(np.prod(s)) for s in WORKLOADS[workload]["shapes"]())
    if n_gpus == 1:
        return n_elem * WORKLOADS[workload]["bytes_per_elem"]
    # all-reduce bus bandwidth, per GPU (tools/bandwidth/measure.py:137-138)
    return int(n_elem * 4 * 2 * (n_gpus - 1) / n_gpus)


# ------------------------------------------------------------------------------------------------
# synthetic data (SURVEY.md 8d: uniform [-1, 1), seeded per role and per GPU) and the oracle check
# ------------------------------------------------------------------------------------------------
def flat_set(seed, sizes):
    """values of every tensor of a set from ONE seeded stream; views of one flat fp32 buffer"""
    rng = np.random.default_rng(seed)
    flat = rng.random(int(sum(sizes)), dtype=np.float32)
    flat *= 2.0
    flat -= 1.0
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return [flat[offs[i]:offs[i + 1]] for i in range(len(sizes))]


def weight_seed():
    return 0xB200 + 777


def grad_seed(rank):
    return 0xB200 + 1000 * rank


def oracle_expected(workload, n_ranks, steps, order="device"):
    """Weights after `steps` pushes of every rank's (constant) seeded gradient set, computed by the
    CPU oracle's kvstore('local') model (oracle/kvoracle.py: LocalKVStoreModel; reduce order of the
    store type, optimizer bookkeeping of python/mxnet/optimizer/optimizer.py). Checker only."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import kvoracle as K
    shapes = WORKLOADS[workload]["shapes"]()
    sizes = [int(np.prod(s)) for s in shapes]
    model = K.LocalKVStoreModel(order)
    w0 = flat_set(weight_seed(), sizes)
    for k in range(len(sizes)):
        model.init(k, w0[k])
    name, kw = opt_kwargs(workload, n_ranks)
    kw = dict(kw)
    kw["lr"] = kw.pop("learning_rate")
    model.set_optimizer(name.lower(), **kw)
    grads = [flat_set(grad_seed(r), sizes) for r in range(n_ranks)]
    for _ in range(steps):
        for k in range(len(sizes)):
            model.push(k, [grads[r][k] for r in range(n_ranks)])
    return [model.pull(k) for k in range(len(sizes))]


def compare_sets(got, want, exact):
    """parity block: bit equality, or the reference's own relative L1 bound
    (tests/nightly/test_kvstore.py:95-98: sum|got - want| / sum|want| < 1e-6)"""
    num = den = 0.0
    bad = 0
    for g, w in zip(got, want):
        g = np.ascontiguousarray(g, dtype=np.float32).reshape(-1)
        w = np.ascontiguousarray(w, dtype=np.float32).reshape(-1)
        if not np.array_equal(g.view(np.uint32), w.view(np.uint32)):
            bad += 1
        num += float(np.sum(np.abs(g.astype(np.float64) - w)))
        den += float(np.sum(np.abs(w.astype(np.float64))))
    rel = num / den if den > 0 else (0.0 if num == 0 else float("inf"))
    ok = (bad == 0) if exact else (rel < 1e-6)
    return {"mode": "bit-exact" if exact else "1e-6 relative L1 (in-switch summation order)",
            "ok": bool(ok), "max_rel": rel, "tensors": len(want), "tensors_differing": bad,
            "checker": "oracle/kvoracle.py LocalKVStoreModel (CPU restatement pinned to oracle/_ref)"}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                for name, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline
# ------------------------------------------------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def best_cpu_threads(workload, n_src):
    """The reference sizes its CPU kernels' OpenMP team from the visible cores
    (engine::OpenMP::GetRecommendedOMPThreadCount); on a big shared host that is far from the
    fastest choice for 157 mostly-small tensors, so the baseline gets the BEST team size of a probe
    (every power of two up to the visible cores, best of three steps each)."""
    best, best_t = 1, float("inf")
    cands = sorted({c for c in (1, 2, 4, 8, 16, 32, 64, 128, host_cores()) if c <= host_cores()})
    for c in cands:
        step, _, _ = cpu_kvstore_step_fn(workload, n_src, c)
        step()
        dt = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            step()
            dt = min(dt, time.perf_counter() - t0)
        if dt < best_t:
            best, best_t = c, dt
        elif dt > 3.0 * best_t:
            break
    return best


def cpu_kvstore_step_fn(workload, n_src, threads=None):
    """One kvstore('local') step on host cores: CommCPU reduce of n_src gradient buffers per key
    (comm.h:357-410), then the optimizer kernel per key (one updater call per key, OMP inside, as
    the reference's callback path does), then the copy to n_src outputs (comm.h:209-224)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import kvoracle as K
    ref = K.ref()
    o = K.get_oracle()
    cores = threads or host_cores()
    shapes = WORKLOADS[workload]["shapes"]()
    rng = np.random.default_rng(0xB200)
    sizes = [int(np.prod(s)) for s in shapes]
    W = [rng.uniform(-1, 1, n).astype(np.float32) for n in sizes]
    G = [[rng.uniform(-1, 1, n).astype(np.float32) for _ in range(n_src)] for n in sizes]
    M = [np.zeros(n, np.float32) for n in sizes]
    V = [np.zeros(n, np.float32) for n in sizes]
    OUT = [[np.empty(n, np.float32) for _ in range(n_src)] for n in sizes]
    kind = "reference" if ref is not None else "port"
    sp, f32 = K.scalar_param, K.f32
    opt = WORKLOADS[workload]["opt"]
    state = {"t": 0}

    def step():
        state["t"] += 1
        t = state["t"]
        for k in range(len(sizes)):
            if n_src > 1:
                bufs = [g for g in G[k]]
                if ref is not None:
                    merged_bufs = [bufs[0].copy()] + bufs[1:]      # CopyFromTo(src[0] -> merged)
                    ref.reduce_inplace(merged_bufs, 4)             # MXNET_KVSTORE_REDUCTION_NTHREADS=4
                    merged = merged_bufs[0]
                else:
                    merged = o.reduce(bufs, "local", 4)
            else:
                merged = G[k][0]
            if opt == "sgd":
                if ref is not None:
                    ref.multi_sgd_update([W[k]], [merged], [M[k]], [f32(0.1)], [f32(1e-4)],
                                         sp(0.9), sp(1.0 / 256), None, cores)
                else:
                    o.multi_sgd_update(W[k], merged, M[k], f32(0.1), sp(0.9), f32(1e-4),
                                       sp(1.0 / 256), None, cores)
            else:
                lr_t = sp(K.adam_lr(1e-3, 0.9, 0.999, t))
                fn = ref.adam_update if ref is not None else o.adam_update
                fn(W[k], merged, M[k], V[k], lr_t, sp(0.9), sp(0.999), sp(1e-8), sp(0.01), 1.0,
                   None, cores)
            for out in OUT[k]:
                np.copyto(out, W[k])
    return step, kind, cores


def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path on this box's cores."""
    if args.workload == "rsp":
        import bench_rsp
        return bench_rsp.run_reference(args)
    n_src = max(1, args.gpus)
    step, kind, cores = cpu_kvstore_step_fn(args.workload, n_src, best_cpu_threads(args.workload, n_src))
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = payload_bytes(args.workload, n_src) / dt / 1e9
    sample = "%d full steps of %s with %d host gradient buffers per key" % (
        args.steps, args.workload, n_src)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block(args.workload, n_src),
            "impl_detail": {"store": "kvstore('local') on CPU: the reference's own CommCPU reduce and "
                                     "optimizer kernels (oracle/_ref, compiled in place from "
                                     "/root/reference) over host buffers",
                            "omp_team": cores, "omp_team_choice": "best of a probe over powers of two"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": sample, "host_cores_visible": host_cores()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def make_optimizer(mx, workload, n_gpus):
    name, kw = opt_kwargs(workload, n_gpus)
    return getattr(mx.optimizer, name)(**kw)


def pcie_pinned_copy_peak(torch, dev, nbytes):
    """Pinned-memory copy rate of this box in GB/s per direction: one direction alone, and with
    H2D and D2H running at the same time on two streams (the denominator of e2e.roofline: a step
    moves the gradient set in and the weight set out, both directions busy)."""
    n = nbytes // 4
    h_in = torch.empty(n, dtype=torch.float32).pin_memory()
    h_out = torch.empty(n, dtype=torch.float32).pin_memory()
    d_in = torch.empty(n, dtype=torch.float32, device=dev)
    d_out = torch.ones(n, dtype=torch.float32, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    reps = 5

    def timed(both):
        best = float("inf")
        for _ in range(reps):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c, d = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(s1):
                a.record()
                d_in.copy_(h_in, non_blocking=True)
                b.record()
            if both:
                with torch.cuda.stream(s2):
                    c.record()
                    h_out.copy_(d_out, non_blocking=True)
                    d.record()
            torch.cuda.synchronize()
            t = a.elapsed_time(b)
            if both:
                t = max(t, c.elapsed_time(d))
            best = min(best, t)
        return nbytes / (best * 1e-3) / 1e9
    uni = timed(False)
    bidir = timed(True)
    return {"h2d_alone_GBps": uni, "per_direction_both_busy_GBps": bidir}


def c_step_fn(mx, kv, keys, vals, outs):
    """the C-ABI entry point itself with prebuilt argument arrays, as a compiled host issues it"""
    from anand_mxnet_b200.kvstore.base import _ctype_key_value
    ckeys, cvals, _ = _ctype_key_value(keys, vals)
    _, couts, _ = _ctype_key_value(keys, outs)
    lib, handle, nkeys, zero = mx.base._LIB, kv.handle, ctypes.c_uint(len(keys)), ctypes.c_int(0)

    def step(_keep=(ckeys, cvals, couts)):
        rc = lib.MXKVStorePushPull(handle, nkeys, ckeys, nkeys, ckeys, cvals, couts, zero)
        if rc != 0:
            raise RuntimeError(lib.MXGetLastError().decode())
    return step


def per_key_step_fns(mx, kv, keys, vals, outs):
    """The reference's callers issue one call per key: Trainer._allreduce_grads
    (python/mxnet/gluon/trainer.py:385-396: pushpull / push+pull of parameter i with priority=-i)
    and tools/bandwidth/measure.py:112-122 (push every key, then pull every key, priority=i).
    Issued from compiled code (B200KVIssuePerKey loops over the MXKVStore* entry points), as a C++
    host would; `python_loop` is the trainer pattern issued call by call through ctypes."""
    lib, handle = mx.base._LIB, kv.handle
    n = ctypes.c_uint(len(keys))
    ck = (ctypes.c_int * len(keys))(*keys)
    cv = (ctypes.c_void_p * len(keys))(*[v._hv for v in vals])
    co = (ctypes.c_void_p * len(keys))(*[o._hv for o in outs])

    def issue(pattern):
        def fn(_keep=(ck, cv, co)):
            if lib.B200KVIssuePerKey(handle, n, ck, cv, co, ctypes.c_int(pattern)) != 0:
                raise RuntimeError(lib.MXGetLastError().decode())
        return fn
    one = ctypes.c_uint(1)
    k1 = [(ctypes.c_int * 1)(k) for k in keys]
    v1 = [(ctypes.c_void_p * 1)(v._hv) for v in vals]
    o1 = [(ctypes.c_void_p * 1)(o._hv) for o in outs]
    pr = [ctypes.c_int(-i) for i in range(len(keys))]

    def python_loop():
        for i in range(len(keys)):
            if lib.MXKVStorePushPull(handle, one, k1[i], one, k1[i], v1[i], o1[i], pr[i]) != 0:
                raise RuntimeError(lib.MXGetLastError().decode())
    return issue(0), issue(1), python_loop


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE_SEED = 0xB200 + 31


def dump_outputs(dump_dir, arrays):
    """Write what the last timed step handed its caller as DIR/<name>.npy, flattened; `arrays` maps
    names to float32 / float64 numpy arrays. Every file keeps at most the byte count that keeps them
    all under DUMP_LIMIT_BYTES; a longer array is written as the values at sorted positions drawn by
    np.random.default_rng(DUMP_SAMPLE_SEED + its index in `arrays`), so the files of two builds run
    with the same arguments compare value for value."""
    arrays = [(name, np.ascontiguousarray(a).reshape(-1)) for name, a in arrays.items()]
    sizes = sorted(a.nbytes for _, a in arrays)
    budget, cap = DUMP_LIMIT_BYTES - 128 * len(arrays), 0      # 128: the .npy header
    for i, n in enumerate(sizes):          # water-filling: the smallest arrays whole, the rest capped
        left = len(sizes) - i
        if n * left > budget:
            cap = budget // left
            break
        budget -= n
    else:
        cap = sizes[-1]
    os.makedirs(dump_dir, exist_ok=True)
    for k, (name, a) in enumerate(arrays):
        assert a.dtype in (np.float32, np.float64), name
        if a.nbytes > cap:
            pos = np.random.default_rng(DUMP_SAMPLE_SEED + k).choice(a.size, cap // a.itemsize, replace=False)
            a = a[np.sort(pos)]
        np.save(os.path.join(dump_dir, name + ".npy"), a)


def time_region(torch, stream, fn, steps, after=None):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(steps):
        fn()
    if after is not None:
        after()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_dense_single(mx, torch, stream, args, workload, steps, warmup, full, dump_dir=None):
    """One dense workload on one GPU: parity, device-resident timing, and (full) the front-end
    variants and the host-buffer arm. dump_dir: where the timed path's outputs go (dump_outputs)."""
    dev = torch.device("cuda", 0)
    shapes = WORKLOADS[workload]["shapes"]()
    sizes = [int(np.prod(s)) for s in shapes]
    keys = list(range(len(shapes)))
    n_elem = sum(sizes)
    w0 = flat_set(weight_seed(), sizes)
    g0 = flat_set(grad_seed(0), sizes)
    # library-owned NDArrays (what the reference's callers hold), one per tensor
    ctx = mx.gpu(0)
    grads = [mx.nd.array(g0[k].reshape(shapes[k]), ctx) for k in keys]
    outs = [mx.nd.empty(s, ctx) for s in shapes]
    kv = mx.kv.create("device")
    kv.init(keys, [mx.nd.array(w0[k].reshape(shapes[k]), ctx) for k in keys])
    kv.set_optimizer(make_optimizer(mx, workload, 1))
    torch.cuda.synchronize()
    # ---- parity: the first two steps of this very store against the CPU oracle
    for _ in range(2):
        kv.pushpull(keys, grads, out=outs)      # python front-end: hands lr / multipliers over
    mx.nd.waitall()
    torch.cuda.synchronize()
    got = [o.asnumpy() for o in outs]
    want = oracle_expected(workload, 1, 2)
    parity = compare_sets(got, want, exact=True)
    parity["after_steps"] = 2

    step = c_step_fn(mx, kv, keys, grads, outs)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    mx.base.reset_kernel_launch_count()
    ms_step = time_region(torch, stream, step, steps)
    launches = mx.base.kernel_launch_count()
    clocks = sampler.stop()
    if dump_dir:
        dump_outputs(dump_dir, {"weight_%03d" % k: o.asnumpy() for k, o in enumerate(outs)})
    # the timed region is exactly K launches of the dominant kernel back to back on this stream:
    # its average launch duration (incl. launch gaps) is the region's duration / K
    alg = algorithmic_bytes(workload, 1)
    pay = payload_bytes(workload, 1)
    peaks, peak_src = measured_peaks()
    achieved = alg / (ms_step * 1e-3) / 1e9
    res = {"workload": WORKLOADS[workload]["desc"], "ms_per_step": ms_step, "steps": steps,
           "value": pay / (ms_step * 1e-3) / 1e9, "unit": UNIT, "gpu_launches": int(launches),
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": achieved / peaks["hbm_gbs"], "traffic": None,
                        "traffic_note": "dram bytes per launch are in the committed ncu capture of this "
                                        "command (profiles/), not re-read at run time",
                        "kernel": kernel_label(workload, 1), "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": alg, "ms_per_launch": ms_step},
           "parity": parity, "clocks": clocks}
    if not full:
        return res

    # ---- front-ends: python grouped call, and the per-key call patterns of the reference's callers
    th = time.perf_counter()
    py_ms = time_region(torch, stream, lambda: kv.pushpull(keys, grads, out=outs), steps)
    host_py_us = (time.perf_counter() - th) / steps * 1e6
    th = time.perf_counter()
    for _ in range(steps):
        step()
    host_c_us = (time.perf_counter() - th) / steps * 1e6
    torch.cuda.synchronize()
    trainer_pattern, measure_pattern, python_loop = per_key_step_fns(mx, kv, keys, grads, outs)
    flush = mx.base.flush_all
    fe = {"python_api_GBps": pay / (py_ms * 1e-3) / 1e9, "python_api_ms_per_step": py_ms,
          "python_api_host_us_per_call": host_py_us, "c_abi_host_us_per_call": host_c_us}
    def flushed(fn):
        # the caller's next read of a weight is what runs a queued bucket; one flush per step
        # stands in for it (a framework reads the weights in its next forward pass)
        def g():
            fn()
            flush()
        return g
    for name, fn, calls in (("per_key_pushpull_priority_minus_i", trainer_pattern, len(keys)),
                            ("per_key_push_all_then_pull_all", measure_pattern, 2 * len(keys)),
                            ("per_key_pushpull_python_ctypes_loop", python_loop, len(keys))):
        try:
            for _ in range(3):
                flushed(fn)()
            torch.cuda.synchronize()
            mx.base.reset_kernel_launch_count()
            th = time.perf_counter()
            ms = time_region(torch, stream, flushed(fn), steps)
            fe[name] = {"ms_per_step": ms, "GBps": pay / (ms * 1e-3) / 1e9,
                        "vs_grouped_call": ms / ms_step,
                        "host_us_per_step": (time.perf_counter() - th) / steps * 1e6,
                        "calls_per_step": calls,
                        "kernel_launches_per_step": mx.base.kernel_launch_count() / steps}
        except Exception as e:  # a front-end variant must not sink the headline
            fe[name] = {"error": str(e)[:200]}
    res["frontends"] = fe

    # ---- end-to-end arm: same C-ABI call, HOST (pinned) gradient and weight buffers
    kv2 = mx.kv.create("device")
    kv2.init(keys, [mx.nd.array(w0[k].reshape(shapes[k]), mx.cpu()) for k in keys])
    kv2.set_optimizer(make_optimizer(mx, workload, 1))
    hgrads = [mx.nd.array(g0[k].reshape(shapes[k]), mx.cpu()) for k in keys]
    houts = [mx.nd.empty(s, mx.cpu()) for s in shapes]
    e2e_steps = max(3, min(steps, 10))
    for _ in range(2):
        kv2.pushpull(keys, hgrads, out=houts)
    mx.nd.waitall()
    e2e_parity = compare_sets([h.asnumpy() for h in houts], want, exact=True)
    hstep = c_step_fn(mx, kv2, keys, hgrads, houts)
    hstep()
    mx.nd.waitall()
    # the last D2H copies run on the copy-out lane: wait for them before stamping the end event
    e2e_ms = time_region(torch, stream, hstep, e2e_steps, after=mx.nd.waitall)
    pcie = pcie_pinned_copy_peak(torch, dev, n_elem * 4)
    per_dir = n_elem * 4 / (e2e_ms * 1e-3) / 1e9
    res["e2e"] = {"value": pay / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": n_elem * 4,
                  "d2h_bytes_per_step": n_elem * 4, "ms_per_step": e2e_ms, "steps": e2e_steps,
                  "parity": e2e_parity,
                  "roofline": {"bound": "pcie", "achieved": per_dir,
                               "peak": pcie["per_direction_both_busy_GBps"], "unit": "GB/s per direction",
                               "frac": per_dir / pcie["per_direction_both_busy_GBps"],
                               "peak_source": "cudaMemcpyAsync pinned<->device, H2D and D2H concurrently, "
                                              "measured in this run", "h2d_alone_GBps": pcie["h2d_alone_GBps"]}}
    return res


def run_single_gpu(args):
    import torch
    import anand_mxnet_b200 as mx
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    # a dedicated non-default stream shared by torch (events, data generation) and the library
    # (B200KVEngineSetStream): the CUDA events below are recorded on the stream the kernels run on
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    mx.base.set_stream(0, stream.cuda_stream)
    assert mx.base.get_stream(0) == stream.cuda_stream

    if args.workload == "rsp":
        import bench_rsp
        line = bench_rsp.run_single_gpu_line(mx, torch, stream, args)
        print(json.dumps(line))
        if not line["parity"]["ok"]:
            sys.exit(3)
        return

    main = run_dense_single(mx, torch, stream, args, args.workload, args.steps, args.warmup, full=True,
                            dump_dir=args.dump_outputs)
    configs = {}
    if not args.no_config_legs:
        other = "bert_adam" if args.workload == "resnet50_sgd" else "resnet50_sgd"
        try:
            leg = run_dense_single(mx, torch, stream, args, other, max(3, min(args.steps, 10)), 3, full=False)
            configs[other] = leg
        except Exception as e:
            configs[other] = {"error": str(e)[:300]}
        try:
            import bench_rsp
            configs["rsp"] = bench_rsp.run_single_gpu_leg(mx, torch, stream, max(5, min(args.steps, 20)))
        except Exception as e:
            configs["rsp"] = {"error": str(e)[:300]}

    # ---- cpu baseline (bounded sample, rank 0, N=1)
    cpu = None
    if not args.no_cpu_baseline:
        pay = payload_bytes(args.workload, 1)
        cstep, kind, cores = cpu_kvstore_step_fn(args.workload, 1, best_cpu_threads(args.workload, 1))
        cstep()
        t0 = time.perf_counter()
        n = 0
        while n < 3 or (time.perf_counter() - t0 < 10.0 and n < 200):
            cstep()
            n += 1
        cdt = (time.perf_counter() - t0) / n
        cpu = {"value": pay / cdt / 1e9, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": "%d full steps of %s (reduce of 1 value + optimizer + copy-out per key), "
                         "%.1f ms/step" % (n, args.workload, cdt * 1e3)}
    line = {"metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block(args.workload, 1),
            "impl_detail": {"store": "kvstore('device')",
                            "call": "one grouped MXKVStorePushPull (C ABI, prebuilt argument arrays) over "
                                    "all keys per step; per-key call patterns and the python front-end "
                                    "under 'frontends'",
                            "optimizer": opt_kwargs(args.workload, 1)[1]},
            "roofline": main["roofline"], "parity": main["parity"], "cpu_baseline": cpu, "e2e": main["e2e"],
            "gpu_launches": main["gpu_launches"], "clocks": main["clocks"], "frontends": main["frontends"],
            "configs": configs}
    print(json.dumps(line))
    ok = main["parity"]["ok"] and main["e2e"]["parity"]["ok"] and all(
        c.get("parity", {}).get("ok", True) for c in configs.values())
    if not ok:
        sys.stderr.write("bench.py: PARITY FAILURE against the oracle\n")
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="resnet50_sgd", choices=sorted(WORKLOADS) + ["rsp"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config-legs", action="store_true",
                    help="skip the short legs over the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned to DIR/*.npy (at most "
                         "64 MB, longer outputs sampled): the pulled weights (dense workloads) or every "
                         "puller's row ids and rows (rsp). One-GPU runs only: with --gpus > 1 each rank is "
                         "a separate torchrun process, and that arm does not dump")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1):
        ap.error("--dump-outputs covers --impl b200 on one GPU")
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is entitled to all host
        # threads (it sizes its OpenMP teams itself), so drop the cap before libgomp loads
        os.environ.pop("OMP_NUM_THREADS", None)
        if rank == 0:
            run_reference(args)
        return
    if args.gpus == 1 and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        run_single_gpu(args)
        return
    from bench_multi import run_multi_gpu
    run_multi_gpu(args)


if __name__ == "__main__":
    main()

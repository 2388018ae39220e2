#!/usr/bin/env python
"""bench_rsp.py -- row_sparse push + row_sparse_pull (BASELINE.json configs[4]): embedding table
(1 000 000, 512) fp32, 10 000 distinct hot rows per value (1 %), lazy SGD on the store, then every
value's owner pulls its own id list (unsorted, 5 % duplicates).

Used three ways:
  * `python bench.py --workload rsp` (N=1: the 8 values of a push all live on the one GPU; N>1 under
    torchrun: one value per rank, the table sharded by row range over the ranks) -> a full bench
    line with roofline, parity, cpu_baseline and e2e;
  * as the `configs.rsp` leg of the default bench line;
  * `python bench_rsp.py --gpus N`: the reference's process model (ONE process driving N GPUs).

Algorithmic bytes (SURVEY.md 8d): push = every source row + id read once, the union's weight rows
read and written once (the summed gradient lives in registers, it is never stored); pull = unique
rows read + written, ids read. The check: pulled ids and rows bit-exact against the CPU oracle
(oracle.rsp_reduce -> sgd_rsp_update -> unique -> sparse_retain; ndarray_function.cc:59-175,
optimizer_op-inl.h:426-450, kvstore_utils.cc:31-44, sparse_retain-inl.h:262-323).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

ROWS, ROW_LEN, HOT = 1000000, 512, 10000
LR = 0.1


def make_inputs(nval, rows=ROWS, row_len=ROW_LEN, hot=HOT):
    """ids / values of every value of the push and every puller's id list, seeded per value"""
    idx, val, pull = [], [], []
    for i in range(nval):
        rng = np.random.default_rng(0xB200 + 1000 * i + 5)
        ids = np.sort(rng.choice(rows, hot, replace=False)).astype(np.int64)
        idx.append(ids)
        v = rng.random((hot, row_len), dtype=np.float32)
        v *= 2.0
        v -= 1.0
        val.append(v)
        p = np.concatenate([ids, rng.choice(ids, hot // 20)])
        rng.shuffle(p)
        pull.append(p)
    return idx, val, pull


def table_init(rows=ROWS, row_len=ROW_LEN):
    rng = np.random.default_rng(0xB200 + 777)
    w = rng.random((rows, row_len), dtype=np.float32)
    w *= 2.0
    w -= 1.0
    return w


def alg_bytes(idx, pull, row_len=ROW_LEN):
    row_bytes = row_len * 4
    union = np.unique(np.concatenate(idx))
    push = sum(len(i) for i in idx) * (row_bytes + 8) + len(union) * row_bytes * 2
    pl = sum(len(np.unique(p)) for p in pull) * row_bytes * 2 + sum(len(p) for p in pull) * 8
    return push, pl, len(union)


def oracle_rows(w, idx, val, steps, nval):
    """`steps` pushes of the same values through the oracle; returns the touched rows' new values"""
    import kvoracle as K
    o = K.get_oracle()
    gi, gv = o.rsp_reduce(idx, val)
    sub = np.ascontiguousarray(w[gi])                       # only the union's rows change (lazy update)
    sp = K.scalar_param
    local = np.arange(len(gi), dtype=np.int64)
    for _ in range(steps):
        o.sgd_rsp_update(sub, local, gv, sp(LR), sp(0.0), sp(1.0 / nval), None)
    return gi, sub


def check_pull(o, gi, sub, w, ids, got_idx, got_val):
    u = o.unique(ids)
    if not np.array_equal(got_idx, u):
        return False
    pos = np.searchsorted(gi, u)
    pos = np.minimum(pos, len(gi) - 1)
    hit = gi[pos] == u
    want = np.where(hit[:, None], sub[pos], w[u])
    return bool(np.array_equal(np.ascontiguousarray(got_val).view(np.uint32).reshape(want.shape),
                               want.view(np.uint32)))


def cpu_reduce_update_ms(idx, val, w, nval):
    """the reference's semantics on the host (oracle port, single thread): union + in-order row sums
    + lazy SGD on the union rows + retain of every puller's rows. Bounded: one pass."""
    import kvoracle as K
    o = K.get_oracle()
    t0 = time.perf_counter()
    gi, gv = o.rsp_reduce(idx, val)
    sub = np.ascontiguousarray(w[gi])
    o.sgd_rsp_update(sub, np.arange(len(gi), dtype=np.int64), gv, K.scalar_param(LR), K.scalar_param(0.0),
                     K.scalar_param(1.0 / nval), None)
    t_push = time.perf_counter() - t0
    return t_push


def _time(torch, stream, fn, steps, after):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(steps):
        fn()
    after()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run_single_gpu_leg(mx, torch, stream, steps, nval=8, host_arm=False, dump_dir=None):
    """nval values on ONE GPU (what BASELINE configs[4] looks like from the store's side on a single
    GPU): timing + roofline + bit-exact check of the pulled rows. dump_dir: where
    the last timed pull's outputs go (bench.dump_outputs; row ids as float64, exact below 2**53)."""
    import kvoracle as K
    from bench import measured_peaks
    shape = (ROWS, ROW_LEN)
    ctx = mx.gpu(0)
    w = table_init()
    idx, val, pull = make_inputs(nval)
    kv = mx.kv.create('device')
    # the stored weight holds every row (a dense weight in row_sparse form, as gluon creates it)
    kv.init('emb', mx.nd.sparse.row_sparse_array((w, np.arange(ROWS, dtype=np.int64)), shape=shape, ctx=ctx))
    kv.set_optimizer(mx.optimizer.SGD(learning_rate=LR, momentum=0.0, wd=0.0, rescale_grad=1.0 / nval))
    grads = [mx.nd.sparse.row_sparse_array((val[i], idx[i]), shape=shape, ctx=ctx) for i in range(nval)]
    pull_ids = [mx.nd.array(p, ctx, np.int64) for p in pull]
    outs = [mx.nd.sparse.zeros('row_sparse', shape, ctx) for _ in range(nval)]

    def push():
        kv.push('emb', grads)

    def pull_fn():
        kv.row_sparse_pull('emb', out=outs, row_ids=pull_ids)

    n_push = 0
    for _ in range(2):
        push()
        n_push += 1
    pull_fn()
    mx.nd.waitall()
    # ---- check: after 2 pushes, every puller's ids and rows against the oracle
    o = K.get_oracle()
    gi, sub = oracle_rows(w, idx, val, n_push, nval)
    ok = all(check_pull(o, gi, sub, w, pull[i], outs[i].indices.asnumpy(), outs[i].data.asnumpy())
             for i in range(nval))
    parity = {"mode": "bit-exact (ids and rows of every puller)", "ok": bool(ok), "after_pushes": n_push,
              "pullers": nval, "checker": "oracle rsp_reduce + sgd_rsp_update + unique + retain"}
    mx.base.reset_kernel_launch_count()
    push_ms = _time(torch, stream, push, steps, mx.nd.waitall)
    launches_push = mx.base.kernel_launch_count() / steps
    mx.base.reset_kernel_launch_count()
    pull_ms = _time(torch, stream, pull_fn, steps, mx.nd.waitall)
    launches_pull = mx.base.kernel_launch_count() / steps
    if dump_dir:
        from bench import dump_outputs
        dumped = {}
        for i, out in enumerate(outs):
            dumped["pull_%d_ids" % i] = out.indices.asnumpy().astype(np.float64)
            dumped["pull_%d_rows" % i] = out.data.asnumpy()
        dump_outputs(dump_dir, dumped)
    pb, lb, union = alg_bytes(idx, pull)
    peaks, peak_src = measured_peaks()
    res = {"workload": "row_sparse push + row_sparse_pull, table (%d, %d) fp32, %d values x %d rows, "
                       "lazy SGD on the store" % (ROWS, ROW_LEN, nval, HOT),
           "union_rows": int(union), "push_ms": push_ms, "pull_ms": pull_ms, "steps": steps,
           "value": (pb + lb) / ((push_ms + pull_ms) * 1e-3) / 1e9, "unit": "GB/s (algorithmic, push+pull)",
           "kernel_launches_per_push": launches_push, "kernel_launches_per_pull": launches_pull,
           "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peaks["hbm_gbs"], "peak_source": peak_src,
                        "push": {"algorithmic_bytes": pb, "achieved": pb / (push_ms * 1e-3) / 1e9,
                                 "frac": pb / (push_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]},
                        "pull": {"algorithmic_bytes": lb, "achieved": lb / (pull_ms * 1e-3) / 1e9,
                                 "frac": lb / (pull_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]},
                        "achieved": (pb + lb) / ((push_ms + pull_ms) * 1e-3) / 1e9,
                        "frac": (pb + lb) / ((push_ms + pull_ms) * 1e-3) / 1e9 / peaks["hbm_gbs"],
                        "traffic": None,
                        "note": "pull includes the one host wait per call for the unique counts "
                                "(the reference blocks once per output, kvstore_utils.cu:95)"},
           "parity": parity}
    if host_arm:
        # e2e: row_sparse gradients and pull targets in HOST memory (CPU-context NDArrays)
        hgrads = [mx.nd.sparse.row_sparse_array((val[i], idx[i]), shape=shape, ctx=mx.cpu()) for i in range(nval)]
        hids = [mx.nd.array(p, mx.cpu(), np.int64) for p in pull]
        houts = [mx.nd.sparse.zeros('row_sparse', shape, mx.cpu()) for _ in range(nval)]

        def hstep():
            kv.push('emb', hgrads)
            kv.row_sparse_pull('emb', out=houts, row_ids=hids)
        hstep()
        mx.nd.waitall()
        n_push += steps * 1 + 1   # timed pushes above + this one
        esteps = max(3, min(steps, 10))
        e_ms = _time(torch, stream, hstep, esteps, mx.nd.waitall)
        n_push += esteps
        gi2, sub2 = oracle_rows(w, idx, val, n_push, nval)
        eok = all(check_pull(o, gi2, sub2, w, pull[i], houts[i].indices.asnumpy(), houts[i].data.asnumpy())
                  for i in range(nval))
        h2d = sum(v.nbytes + i.nbytes for v, i in zip(val, idx)) + sum(p.nbytes for p in pull)
        d2h = sum(len(np.unique(p)) * (ROW_LEN * 4 + 8) for p in pull)
        res["e2e"] = {"value": (pb + lb) / (e_ms * 1e-3) / 1e9, "unit": "GB/s (algorithmic, push+pull)",
                      "ms_per_step": e_ms, "steps": esteps, "h2d_bytes_per_step": int(h2d),
                      "d2h_bytes_per_step": int(d2h), "parity": {"mode": "bit-exact", "ok": bool(eok)}}
    return res


def run_single_gpu_line(mx, torch, stream, args):
    """`bench.py --workload rsp` at N=1: a full bench line."""
    from bench import config_block, ClockSampler
    sampler = ClockSampler(0)
    sampler.start()
    leg = run_single_gpu_leg(mx, torch, stream, args.steps, host_arm=True, dump_dir=args.dump_outputs)
    clocks = sampler.stop()
    w = table_init()
    idx, val, _ = make_inputs(8)
    cpu_s = cpu_reduce_update_ms(idx, val, w, 8)
    pb = leg["roofline"]["push"]["algorithmic_bytes"]
    step_ms = leg["push_ms"] + leg["pull_ms"]
    return {"metric": "kvstore_row_sparse_push_pull_GBps", "value": leg["value"], "unit": "GB/s", "n_gpus": 1,
            "steps": args.steps, "warmup": 2, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block("rsp", 8), "impl_detail": {k: leg[k] for k in (
                "union_rows", "push_ms", "pull_ms", "kernel_launches_per_push", "kernel_launches_per_pull")},
            "roofline": leg["roofline"], "parity": leg["parity"], "e2e": leg["e2e"],
            "cpu_baseline": {"value": pb / cpu_s / 1e9, "unit": "GB/s (push only)", "cores": 1, "kind": "port",
                             "sample": "one push (union of 8 x 10000 ids, in-order row sums, lazy SGD on "
                                       "the union rows), %.1f ms" % (cpu_s * 1e3)},
            "gpu_launches": int(round((leg["kernel_launches_per_push"] + leg["kernel_launches_per_pull"]) * args.steps)),
            "clocks": clocks}


def cpu_step_fn(nval, threads=1):
    """one row_sparse push + nval pulls on host cores: the reference's own ElementwiseSumRsp, lazy
    SGD kernel, UniqueImpl and sparse_retain kernels (oracle/_ref/libmxref.so, OpenMP team of
    `threads`) when that library is present, else the oracle port (one thread)"""
    import kvoracle as K
    w = table_init()
    idx, val, pull = make_inputs(nval)
    r = K.ref()
    sp = K.scalar_param
    if r is not None and r.has_sparse():
        all_rows = np.arange(ROWS, dtype=np.int64)

        def step():
            gi, gv = r.rsp_reduce(idx, val, nthreads=threads)
            r.sgd_rsp_update(w, gi, gv, sp(LR), sp(0.0), sp(1.0 / nval), None, nthreads=threads)
            for p in pull:
                r.sparse_retain(all_rows, w, r.unique(p), src_dense_rows=True, nthreads=threads)
        return step, "reference", idx, pull
    o = K.get_oracle()

    def step():
        gi, gv = o.rsp_reduce(idx, val)
        sub = np.ascontiguousarray(w[gi])
        o.sgd_rsp_update(sub, np.arange(len(gi), dtype=np.int64), gv, sp(LR), sp(0.0), sp(1.0 / nval), None)
        w[gi] = sub
        for p in pull:
            _ = w[o.unique(p)]     # retain from a table that holds every row = gather of the rows
    return step, "port", idx, pull


def run_reference(args):
    """reference arm of `--workload rsp`: the reference's CPU implementation of the path on the host
    cores with the best OpenMP team of a probe (powers of two, best of three steps each)"""
    from bench import config_block, host_cores
    os.environ.pop("OMP_NUM_THREADS", None)          # torchrun sets 1; the team size is passed per call
    nval = 8 if args.gpus <= 1 else args.gpus
    step, kind, idx, pull = cpu_step_fn(nval, 1)
    cores, best = 1, float("inf")
    if kind == "reference":
        for c in sorted({c for c in (1, 2, 4, 8, 16, 32, 64) if c <= host_cores()}):
            fn = cpu_step_fn(nval, c)[0]
            fn()
            dt = min(_timed(fn) for _ in range(3))
            if dt < best:
                cores, best = c, dt
            elif dt > 3.0 * best:
                break
        step = cpu_step_fn(nval, cores)[0]
    pb, lb, _ = alg_bytes(idx, pull)
    for _ in range(min(args.warmup, 1)):
        step()
    n = max(1, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(n):
        step()
    dt = (time.perf_counter() - t0) / n
    value = (pb + lb) / dt / 1e9
    what = "the reference's own CPU kernels (oracle/_ref)" if kind == "reference" else "the oracle port"
    print(json.dumps({"impl": "reference", "metric": "kvstore_row_sparse_push_pull_GBps", "value": value,
                      "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": config_block("rsp", nval),
                      "cpu_baseline": {"value": value, "unit": "GB/s", "cores": cores, "kind": kind,
                                       "sample": "%d steps (push + %d pulls) of %s" % (n, nval, what),
                                       "host_cores_visible": host_cores()},
                      "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}))


def _timed(fn):
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def main():
    """The reference's process model: one process, N GPUs, value i on GPU i % N."""
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=0, help="0 = all visible")
    ap.add_argument("--values", type=int, default=8, help="values per push (GPUs in the reference)")
    ap.add_argument("--steps", type=int, default=50)
    args = ap.parse_args()
    import torch
    import anand_mxnet_b200 as mx
    import kvoracle as K
    ngpu = args.gpus or torch.cuda.device_count()
    nval = args.values
    shape = (ROWS, ROW_LEN)
    ctxs = [mx.gpu(i % ngpu) for i in range(nval)]
    w = table_init()
    idx, val, pull = make_inputs(nval)
    kv = mx.kv.create('device')
    kv.init('emb', mx.nd.sparse.row_sparse_array((w, np.arange(ROWS, dtype=np.int64)), shape=shape, ctx=mx.gpu(0)))
    kv.set_optimizer(mx.optimizer.SGD(learning_rate=LR, momentum=0.0, wd=0.0, rescale_grad=1.0 / nval))
    grads = [mx.nd.sparse.row_sparse_array((val[i], idx[i]), shape=shape, ctx=ctxs[i]) for i in range(nval)]
    pull_ids = [mx.nd.array(pull[i], ctxs[i], np.int64) for i in range(nval)]
    outs = [mx.nd.sparse.zeros('row_sparse', shape, ctxs[i]) for i in range(nval)]

    def push():
        kv.push('emb', grads)

    def pull_fn():
        kv.row_sparse_pull('emb', out=outs, row_ids=pull_ids)

    for _ in range(2):
        push()
    pull_fn()
    mx.nd.waitall()
    o = K.get_oracle()
    gi, sub = oracle_rows(w, idx, val, 2, nval)
    ok = all(check_pull(o, gi, sub, w, pull[i], outs[i].indices.asnumpy(), outs[i].data.asnumpy())
             for i in range(nval))
    mx.base.reset_kernel_launch_count()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        push()
    mx.nd.waitall()
    t_push = (time.perf_counter() - t0) / args.steps
    launches_push = mx.base.kernel_launch_count() / args.steps
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pull_fn()
    mx.nd.waitall()
    t_pull = (time.perf_counter() - t0) / args.steps
    pb, lb, union = alg_bytes(idx, pull)
    print(json.dumps({
        "metric": "row_sparse_push_pull", "process_model": "one process driving %d GPUs" % ngpu,
        "n_gpus": ngpu, "values_per_push": nval, "table": list(shape), "hot_rows_per_value": HOT,
        "union_rows": int(union), "push_ms": t_push * 1e3, "pull_ms": t_pull * 1e3,
        "push_GBps": pb / t_push / 1e9, "pull_GBps": lb / t_pull / 1e9,
        "kernel_launches_per_push": launches_push, "parity": {"mode": "bit-exact", "ok": bool(ok)},
        "note": "host-timed over %d back-to-back calls + waitall" % args.steps}))
    if not ok:
        sys.exit(3)


if __name__ == "__main__":
    main()

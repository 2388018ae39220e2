"""CPU-only checks of host-side policy code: launch-support helpers of anand_mxnet_b200.dist, the
bench's byte accounting, the optimizer front-end's bookkeeping for the LARS / LAMB classes (no
arithmetic runs here -- the operators need a GPU)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_nvls_rule(monkeypatch):
    import anand_mxnet_b200 as mx
    monkeypatch.delenv('B200KV_NVLS', raising=False)
    assert [mx.dist.nvls_wanted(w) for w in (2, 4, 8, 16)] == [False, False, True, True]
    monkeypatch.setenv('B200KV_NVLS', 'auto')
    assert mx.dist.nvls_wanted(8) and not mx.dist.nvls_wanted(4)
    monkeypatch.setenv('B200KV_NVLS', '1')
    assert mx.dist.nvls_wanted(2)
    monkeypatch.setenv('B200KV_NVLS', '0')
    assert not mx.dist.nvls_wanted(8)


def test_numa_binding_is_best_effort(monkeypatch):
    """no GPU here: the helper must leave the affinity alone and return None, never raise"""
    import anand_mxnet_b200 as mx
    before = os.sched_getaffinity(0)
    assert mx.dist.bind_to_gpu_numa_node(0) is None
    assert os.sched_getaffinity(0) == before
    monkeypatch.setenv('B200KV_BIND_NUMA', '0')
    assert mx.dist.bind_to_gpu_numa_node(0) is None


def test_bench_byte_accounting():
    import bench
    n = sum(int(np.prod(s)) for s in bench.resnet50_shapes())
    assert n == 25549486 and len(bench.resnet50_shapes()) == 157          # SURVEY 8a
    nb = sum(int(np.prod(s)) for s in bench.bert_base_shapes())
    assert nb == 109482240 and len(bench.bert_base_shapes()) == 199
    # value: push + pull payload, same definition at every N
    for w in (1, 2, 4, 8):
        assert bench.payload_bytes('resnet50_sgd', w) == w * n * 4 * 2
    # roofline: 24 B / element at N=1 (SGD momentum), bus bandwidth bytes per GPU at N>=2
    assert bench.algorithmic_bytes('resnet50_sgd', 1) == n * 24
    assert bench.algorithmic_bytes('bert_adam', 1) == nb * 32
    assert bench.algorithmic_bytes('resnet50_sgd', 8) == int(n * 4 * 2 * 7 / 8)


def test_lars_and_lamb_bookkeeping():
    from compat import mxnet_optimizer as mxopt      # mirror of the reference's front-end (tests/compat)
    names = {0: 'conv_weight', 1: 'bn_gamma', 2: 'fc_bias'}
    opt = mxopt.create('lars', learning_rate=0.1, momentum=0.9, wd=1e-4, param_idx2name=names)
    opt.set_wd_mult({})
    assert opt._get_wds([0, 1, 2]) == [1e-4, 0.0, 0.0]          # only *_weight parameters decay
    opt._update_count([0, 1, 2])
    assert opt._get_lrs([0, 1, 2]) == [0.1, 0.1, 0.1]
    assert opt.last_lr == 0.1 and opt.cur_lr == 0.1
    opt.lr = 0.05
    opt._get_lrs([0])
    assert (opt.last_lr, opt.cur_lr) == (0.1, 0.05)            # what the momentum correction uses
    lamb = mxopt.create('lamb', learning_rate=0.01)
    assert lamb.aggregate_num == 45 and lamb.epsilon == 1e-6 and lamb.bias_correction
    assert isinstance(mxopt.get_updater(lamb), mxopt.Updater)


def test_every_multi_tensor_operator_is_registered_and_has_golden_cases():
    """the operator names of SURVEY 8f-f1 resolve through NNGetOpHandle (no GPU needed for the
    lookup) and each of them is exercised by a seeded case whose golden output is committed"""
    import ctypes
    import inspect
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import golden_ops as G
    import anand_mxnet_b200 as mx
    ops = ['multi_sum_sq', 'multi_lars', 'preloaded_multi_sgd_update', 'preloaded_multi_sgd_mom_update',
           'preloaded_multi_mp_sgd_update', 'preloaded_multi_mp_sgd_mom_update', '_adamw_update',
           '_mp_adamw_update', '_multi_adamw_update', '_multi_mp_adamw_update', 'lamb_update_phase1',
           'lamb_update_phase2', 'mp_lamb_update_phase1', 'mp_lamb_update_phase2', '_multi_lamb_update',
           '_multi_mp_lamb_update']
    src = inspect.getsource(G)
    gold = np.load(os.path.join(ROOT, "tests", "golden", "multi_tensor_ops.npz"))
    assert {k.split('/')[0] for k in gold.files} == set(G.CASES)
    for name in ops:
        h = ctypes.c_void_p()
        assert mx.base._LIB.NNGetOpHandle(name.encode(), ctypes.byref(h)) == 0 and h.value, name
        assert hasattr(G.OracleOps, '_op_' + name.lstrip('_')), name
        base = name.replace('_mom_', '_%s').replace('_mp_', '_%s') if False else name
        assert ("'%s'" % name in src) or (name.startswith('preloaded_') and "'preloaded_multi_%ssgd_%supdate'" in src), name
    h = ctypes.c_void_p()
    assert mx.base._LIB.NNGetOpHandle(b'no_such_operator', ctypes.byref(h)) != 0


@pytest.mark.parametrize("seed", range(6))
def test_oracle_ops_match_live_reference_on_random_cases(seed):
    """beyond the fixed golden cases: random shapes / hyper-parameters, restatement vs the reference's
    own FCompute<cpu> (its results stored by oracle/refrecord.py)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import golden_ops as G
    import refrecord as R
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(1, 7))
    shapes = [tuple(int(x) for x in rng.integers(1, 40, int(rng.integers(1, 4)))) for _ in range(n)]
    kw = dict(lrs=[float(x) for x in rng.uniform(1e-4, 1e-1, n)], wds=[float(x) for x in rng.uniform(0, 1e-2, n)],
              etas=[float(x) for x in rng.uniform(0.5, 1.0, n)], beta1=float(rng.uniform(0.8, 0.95)),
              beta2=float(rng.uniform(0.9, 0.9999)), epsilon=float(10 ** rng.uniform(-9, -5)), num_weights=n)
    if seed % 2:
        kw['clip_gradient'] = float(rng.uniform(0.1, 2.0))
    lamb = dict(learning_rates=kw['lrs'], wds=kw['wds'], beta1=kw['beta1'], beta2=kw['beta2'],
                epsilon=kw['epsilon'], rescale_grad=float(rng.uniform(0.1, 2.0)), bias_correction=bool(seed % 3),
                num_tensors=n, step_count=[int(x) for x in rng.integers(1, 2000, n)])

    def run(backend):
        r2 = np.random.default_rng(77 + seed)
        ws = [r2.uniform(-1, 1, s).astype(np.float32) for s in shapes]
        gs = [r2.uniform(-3, 3, s).astype(np.float32) for s in shapes]
        ms = [r2.uniform(-0.1, 0.1, s).astype(np.float32) for s in shapes]
        vs = [r2.uniform(0, 0.1, s).astype(np.float32) for s in shapes]
        rs = np.array([0.37], np.float32)
        ins = [x for t in zip(ws, gs, ms, vs) for x in t]
        backend.invoke('_multi_adamw_update', ins + [rs], ws, **kw)
        backend.invoke('_multi_lamb_update', ins, ws, **lamb)
        return [R.digest(a) for a in ws + ms + vs]         # weights, then means, then variances
    want = R.reference("test_host_logic::oracle_ops_random[%d]" % seed, lambda ref: run(G._RefBackend(ref)))
    got = run(G.OracleOps())
    for i, (a, b) in enumerate(zip(got, want)):
        assert a == b, "%s of tensor %d (shape %s)" % (('weight', 'mean', 'var')[i // n], i % n, shapes[i % n])


def test_nccl_fallback_library_binds():
    """kvstore 'nccl' binds libnccl.so.2 at run time (csrc/nccl_dyn.cc): every entry point the
    fallback needs resolves here, without a GPU"""
    import ctypes
    import anand_mxnet_b200 as mx
    lib = mx.base._LIB
    avail = ctypes.c_int(-1)
    ver = ctypes.create_string_buffer(32)
    assert lib.B200KVTestNcclAvailable(ctypes.byref(avail), ver, ctypes.c_size_t(32)) == 0
    assert avail.value == 1, "libnccl.so.2 not loadable in this image"
    major = int(ver.value.decode().split('.')[0])
    assert major >= 2


def test_bench_parity_and_config_helpers():
    """bench.py's checker plumbing: the config block is a pure function of (workload, N) -- the two
    arms of the driver's comparison print the same dict --, the parity block distinguishes
    bit equality from the reference's 1e-6 relative-L1 bound, and the seeded sets are reproducible"""
    import numpy as np
    import bench
    for wl in ('resnet50_sgd', 'bert_adam', 'rsp'):
        for n in (1, 2, 8):
            assert bench.config_block(wl, n) == bench.config_block(wl, n)
            assert set(bench.config_block(wl, n)) == {'workload', 'values_per_key', 'value_formula', 'l2'}
    assert bench.config_block('resnet50_sgd', 2) != bench.config_block('resnet50_sgd', 4)
    a = [np.arange(10, dtype=np.float32), np.ones(5, np.float32)]
    same = bench.compare_sets([x.copy() for x in a], a, exact=True)
    assert same['ok'] and same['max_rel'] == 0.0 and same['tensors_differing'] == 0
    b = [x.copy() for x in a]
    b[0][3] = np.nextafter(b[0][3], np.float32(10))            # one ulp off
    assert not bench.compare_sets(b, a, exact=True)['ok']
    tol = bench.compare_sets(b, a, exact=False)
    assert tol['ok'] and 0 < tol['max_rel'] < 1e-6 and tol['tensors_differing'] == 1
    b[1][0] = 2.0
    assert not bench.compare_sets(b, a, exact=False)['ok']
    s1 = bench.flat_set(bench.grad_seed(3), [7, 1, 100])
    s2 = bench.flat_set(bench.grad_seed(3), [7, 1, 100])
    assert all(np.array_equal(x, y) for x, y in zip(s1, s2)) and [len(x) for x in s1] == [7, 1, 100]
    assert all(np.all((x >= -1) & (x < 1)) for x in s1)
    assert not np.array_equal(bench.flat_set(bench.grad_seed(4), [7])[0], s1[0])
    assert bench.kernel_label('bert_adam', 4) == 'dense_fused_kernel<float,4,Adam>'
    assert 'NVLS' in bench.kernel_label('resnet50_sgd', 8, nvls=True)
    # the oracle model behind the parity block, on a small made-up "workload"
    bench.WORKLOADS['_tiny'] = dict(shapes=lambda: [(5,), (2, 3)], opt='sgd', bytes_per_elem=24, desc='tiny')
    try:
        w1 = bench.oracle_expected('_tiny', 2, 1)
        w2 = bench.oracle_expected('_tiny', 2, 2)
        assert [x.shape for x in w1] == [(5,), (6,)] or [x.size for x in w1] == [5, 6]
        assert not np.array_equal(w1[0], w2[0])
    finally:
        del bench.WORKLOADS['_tiny']


def test_reference_arm_under_torchrun_two_ranks():
    """bench.py --impl reference launched the way the driver launches it for N > 1 (torchrun, one
    process per GPU): rank 0 alone runs the reference's CPU implementation and prints ONE JSON line
    whose `config` is the one the GPU arm prints at that N; the other rank exits 0 without work.
    No GPU involved (gloo-free: the arm needs no process group)."""
    import json
    import socket
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(root, "bench.py"),
                        "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       cwd=root, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    d = json.loads(lines[0])
    sys.path.insert(0, root)
    import bench
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["steps"] == 1
    assert d["config"] == bench.config_block("resnet50_sgd", 2)
    assert d["metric"] == "kvstore_push_pull_GBps" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0

"""Pins the CPU oracle (oracle/kvoracle.c) -- CPU-only tests.

Three anchors, as SURVEY.md 8(c) lists them:
  1. tests/golden/*.npz -- outputs of the reference's own headers (oracle/gen_golden.py), committed;
  2. oracle/_ref/libmxref.so -- the same reference code, live, when it has been built here;
  3. the reference's known-answer values (SURVEY.md 8c) and the exact small-integer identities its
     unit tests use (tests/python/unittest/test_kvstore.py:49-51, tests/python/gpu/test_device.py).
All comparisons are bit-exact.
"""
import numpy as np
import pytest

import kvoracle as K
import refrecord as R


def eq(a, b):
    return np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))


HP = dict(lr=0.1, wd=1e-4, rescale=1.0 / 256, momentum=0.9)
CLIPS = (("noclip", None), ("clip", 0.002))


# ---------------------------------------------------------------- golden fixtures (reference outputs)
def test_reduce_local_golden(oracle, golden):
    g = golden("reduce_local")
    for n in range(1, 10):
        srcs = list(g["n%d_src" % n])
        assert eq(oracle.reduce(srcs, "local"), g["n%d_out" % n]), n
        assert eq(oracle.reduce(srcs, "local", nthreads=3), g["n%d_out" % n]), n
        if n <= 2:  # 'device' (left fold) and 'local' agree bit-for-bit only up to 2 sources
            assert eq(oracle.reduce(srcs, "device"), g["n%d_out" % n])


@pytest.mark.parametrize("tag,clip", CLIPS)
def test_optimizers_golden(oracle, golden, tag, clip):
    g = golden("optimizers")
    w, gr = g["sgd_%s_in" % tag]
    assert eq(oracle.sgd_update(w.copy(), gr, HP["lr"], HP["wd"], HP["rescale"], clip),
              g["sgd_%s_out" % tag])
    w, gr, m = g["sgdmom_%s_in" % tag]
    w2, m2 = w.copy(), m.copy()
    oracle.sgd_mom_update(w2, gr, m2, HP["lr"], HP["momentum"], HP["wd"], HP["rescale"], clip)
    assert eq(np.stack([w2, m2]), g["sgdmom_%s_out" % tag])
    w2, m2 = w.copy(), m.copy()
    oracle.multi_sgd_update(w2, gr, m2, HP["lr"], HP["momentum"], HP["wd"], HP["rescale"], clip)
    assert eq(np.stack([w2, m2]), g["multisgdmom_%s_out" % tag])
    w2 = w.copy()
    oracle.multi_sgd_update(w2, gr, None, HP["lr"], 0.0, HP["wd"], HP["rescale"], clip)
    assert eq(w2, g["multisgd_%s_out" % tag])


@pytest.mark.parametrize("tag,clip", (("noclip", None), ("clip", 0.5)))
def test_adam_golden(oracle, golden, tag, clip):
    g = golden("optimizers")
    w, gr, m, v = [x.copy() for x in g["adam_%s_in" % tag]]
    sp = K.scalar_param
    for t in range(1, 6):
        lr_t = sp(K.adam_lr(1e-3, 0.9, 0.999, t))
        oracle.adam_update(w, gr, m, v, lr_t, sp(0.9), sp(0.999), sp(1e-8), sp(0.01), 1.0, clip)
        assert eq(np.stack([w, m, v]), g["adam_%s_out" % tag][t - 1]), t


def test_scalar_parse_golden(golden):
    """python repr -> dmlc::stof, the hop every scalar hyper-parameter takes: the oracle's
    restatement AND the product library's (csrc/scalar_parse.cc, host-only test hooks) must both
    reproduce the reference's values -- which differ from nearest-float32 for ~6% of inputs."""
    import ctypes
    import anand_mxnet_b200 as mx
    lib = mx.base._LIB
    g = golden("scalar_parse")
    buf = ctypes.create_string_buffer(64)
    out = ctypes.c_float()
    n_not_nearest = 0
    for v, want in zip(g["values"], g["parsed"]):
        v = float(v)
        assert np.float32(K.dmlc_stof(repr(v))) == want, v
        assert lib.B200KVTestPyFloatRepr(ctypes.c_double(v), buf, 64) == 0
        assert buf.value.decode() == repr(v)
        assert lib.B200KVTestDmlcStof(repr(v).encode(), ctypes.byref(out)) == 0
        assert np.float32(out.value) == want, v
        n_not_nearest += int(np.float32(v) != want)
    assert n_not_nearest > 0   # the quirk is real: a correctly rounded parse would NOT be bit-exact
    for v in (0.0, -0.0, 1e16, 1e22, 123456789.125, 5e-324, 1.7976931348623157e308, 1e-5, 0.0001):
        assert lib.B200KVTestPyFloatRepr(ctypes.c_double(v), buf, 64) == 0
        assert buf.value.decode() == repr(v)


@pytest.mark.parametrize("tag,clip", CLIPS)
def test_mixed_precision_golden(oracle, golden, tag, clip):
    g = golden("optimizers")
    w16, g16 = g["mp_%s_in16" % tag]
    w32, m = g["mp_%s_in32" % tag]
    a16, a32, am = w16.copy(), w32.copy(), m.copy()
    oracle.multi_mp_sgd_update(a16, a32, g16, am, 0, HP["lr"], HP["momentum"], HP["wd"],
                               HP["rescale"], clip)
    assert eq(a16, g["mpmom_%s_out16" % tag])
    assert eq(np.stack([a32, am]), g["mpmom_%s_out32" % tag])
    a16, a32 = w16.copy(), w32.copy()
    oracle.mp_sgd_update(a16, a32, g16, 0, HP["lr"], HP["wd"], HP["rescale"], clip)
    assert eq(a16, g["mpsgd_%s_out16" % tag])
    assert eq(a32, g["mpsgd_%s_out32" % tag])


@pytest.mark.parametrize("tag,clip", (("noclip", None), ("clip", 0.3)))
def test_rowsparse_updates_golden(oracle, golden, tag, clip):
    g = golden("rowsparse_updates")
    w, m, v = g["rsp_%s_in" % tag]
    gi, gv = g["rsp_%s_gidx" % tag], g["rsp_%s_gval" % tag]
    assert eq(oracle.sgd_rsp_update(w.copy(), gi, gv, 0.1, 1e-3, 0.5, clip),
              g["rsp_sgd_%s_out" % tag])
    w2, m2 = w.copy(), m.copy()
    oracle.sgd_mom_rsp_update(w2, m2, gi, gv, 0.1, 0.9, 1e-3, 0.5, clip)
    assert eq(np.stack([w2, m2]), g["rsp_sgdmom_%s_out" % tag])
    w2, m2, v2 = w.copy(), m.copy(), v.copy()
    oracle.adam_rsp_update(w2, m2, v2, gi, gv, 1e-3, wd=0.01, clip=clip)
    assert eq(np.stack([w2, m2, v2]), g["rsp_adam_%s_out" % tag])


@pytest.mark.parametrize("tag,clip", (("noclip", None), ("clip", 0.3)))
def test_rowsparse_std_updates_golden_and_live(oracle, golden, tag, clip):
    """non-lazy updates (SURVEY 8f-f3): restatement vs the golden outputs of the reference's
    <req,cpu> std kernels, and vs the live harness when it is built here"""
    g = golden("rowsparse_std_updates")
    w, m, v = g["std_%s_in" % tag]
    gi, gv = g["std_%s_gidx" % tag], g["std_%s_gval" % tag]
    backends = [(oracle, True)]
    if K.ref() is not None and K.ref().has_ops():
        backends.append((K.ref(), False))
    for b, _ in backends:
        assert eq(b.sgd_std_rsp_update(w.copy(), gi, gv, 0.1, 1e-3, 0.5, clip), g["std_sgd_%s_out" % tag])
        w2, m2 = w.copy(), m.copy()
        b.sgd_mom_std_rsp_update(w2, m2, gi, gv, 0.1, 0.9, 1e-3, 0.5, clip)
        assert eq(np.stack([w2, m2]), g["std_sgdmom_%s_out" % tag])
        w2, m2, v2 = w.copy(), m.copy(), v.copy()
        b.adam_std_rsp_update(w2, m2, v2, gi, gv, 1e-3, wd=0.01, clip=clip)
        assert eq(np.stack([w2, m2, v2]), g["std_adam_%s_out" % tag])
        w2, m2 = w.copy(), m.copy()
        b.sgd_mom_std_rsp_update(w2, m2, np.zeros(0, np.int64), np.zeros((0, w.shape[1]), np.float32),
                                 0.1, 0.9, 1e-3, 0.5, clip)
        assert eq(np.stack([w2, m2]), g["std_sgdmom_%s_empty_out" % tag])
    # std SGD / SGD-momentum equal the DENSE kernels on the densified gradient (what the CUDA path uses)
    dense = np.zeros_like(w)
    dense[gi] = gv
    assert eq(oracle.sgd_update(w.copy().ravel(), dense.ravel(), 0.1, 1e-3, 0.5, clip).reshape(w.shape),
              g["std_sgd_%s_out" % tag])
    w2, m2 = w.copy().ravel(), m.copy().ravel()
    oracle.sgd_mom_update(w2, dense.ravel(), m2, 0.1, 0.9, 1e-3, 0.5, clip)
    assert eq(np.stack([w2.reshape(w.shape), m2.reshape(w.shape)]), g["std_sgdmom_%s_out" % tag])


def test_twobit_golden(oracle, golden):
    g = golden("twobit")
    res = np.zeros_like(g["grad"])
    c1 = oracle.quantize_2bit(g["grad"], res, 0.5)
    assert eq(c1, g["comp1"]) and eq(res, g["res1"])
    c2 = oracle.quantize_2bit(g["grad"], res, 0.5)
    assert eq(c2, g["comp2"]) and eq(res, g["res2"])
    assert eq(oracle.dequantize_2bit(c1, g["grad"].size, 0.5), g["deq1"])


# ---------------------------------------------------------------- known answers (SURVEY.md 8c)
def test_known_answers(oracle):
    w = np.array([1, 2, 3, 4], np.float32)
    g = np.array([.1, .2, .3, .4], np.float32)
    o = oracle.sgd_update(np.array([1, 4], np.float32), np.array([.1, .4], np.float32),
                          K.f32(.1), K.f32(.01))
    assert o[0] == np.float32(0.989000022) and o[1] == np.float32(3.95600009)
    m, v = np.zeros(4, np.float32), np.zeros(4, np.float32)
    o = oracle.adam_update(w.copy(), g, m, v, K.f32(1e-3), wd=K.f32(.01))
    assert o[0] == np.float32(0.996837735) and o[3] == np.float32(3.99683762)
    mom = np.full(4, .5, np.float32)
    o = oracle.multi_sgd_update(w.copy(), g, mom, K.f32(.1), K.f32(.9), K.f32(1e-4),
                                K.f32(1 / 256))
    assert o[0] == np.float32(1.44995093) and o[3] == np.float32(4.44980383)
    assert mom[0] == np.float32(0.449950904)
    grad = np.array([(i % 3 - 1) * 0.6 for i in range(16)], np.float32)
    assert oracle.quantize_2bit(grad, np.zeros(16, np.float32), .5)[0] == 0x8ee3388e
    # 8 inputs of 0.1*(i+1) through the CommCPU association -> 3.5999999 (SURVEY 8c)
    srcs = [np.full(3, np.float32(0.1 * (i + 1)), np.float32) for i in range(8)]
    assert oracle.reduce(srcs, "local")[0] == np.float32(3.5999999)


def test_small_integer_identities(oracle):
    # tests/python/gpu/test_device.py:38-71: ones over n devices == n, for both associations
    for n in range(1, 9):
        for shape in ((10,), (100, 50), (2, 3, 4, 5, 6, 7, 8)):
            srcs = [np.ones(shape, np.float32) for _ in range(n)]
            for order in ("local", "device"):
                assert np.all(oracle.reduce(srcs, order) == n)
    # tests/python/unittest/test_kvstore.py:227-279: updater `local += recv`, four pushes of
    # ones over 4 devices -> stored == 1 + 4*4 per push chain
    m = K.LocalKVStoreModel()
    m.init(3, np.ones((4, 4), np.float32))
    m.set_optimizer('test', rescale_grad=1.0)
    for _ in range(4):
        m.push(3, [np.ones((4, 4), np.float32)] * 4)
    assert np.all(m.pull(3) == 17)


def test_half_conversions(oracle):
    allh = np.arange(0x7c00, dtype=np.uint16)  # every finite non-negative fp16
    f = oracle.from_half(allh, 0)
    back = np.array([oracle.lib.kvo_float_to_half(float(x), 0) for x in f], dtype=np.uint16)
    assert eq(back, allh)
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.uniform(-70000, 70000, 4000), rng.uniform(-1e-4, 1e-4, 4000),
                        rng.uniform(-1e-7, 1e-7, 2000)]).astype(np.float32)
    mine = np.array([oracle.lib.kvo_float_to_half(float(t), 0) for t in x], dtype=np.uint16)
    assert eq(mine, x.astype(np.float16).view(np.uint16))
    # bf16: round-to-nearest-even on the upper 16 bits
    import torch
    tb = torch.from_numpy(x).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    mine = np.array([oracle.lib.kvo_float_to_half(float(t), 1) for t in x], dtype=np.uint16)
    assert eq(mine, tb)
    assert eq(oracle.to_half(x, 1), tb) and eq(oracle.to_half(x, 0), x.astype(np.float16).view(np.uint16))


def test_rowsparse_reduce_unique_retain(oracle):
    rng = np.random.default_rng(2)
    R, L = 64, 5
    idxs, vals = [], []
    for s in range(4):
        i = np.sort(rng.choice(R, 20, replace=False)).astype(np.int64)
        idxs.append(i)
        vals.append(rng.integers(-3, 4, (20, L)).astype(np.float32))
    oi, ov = oracle.rsp_reduce(idxs, vals)
    dense = np.zeros((R, L), np.float32)
    for i, v in zip(idxs, vals):
        dense[i] += v
    assert np.array_equal(oi, np.unique(np.concatenate(idxs)))
    assert np.array_equal(ov, dense[oi])  # small integers: exact (test_kvstore.py:178-227)
    # unique: unsorted + duplicates -> ascending unique (kvstore_utils.cc:32-44)
    ids = rng.integers(0, R, 100)
    assert np.array_equal(oracle.unique(ids), np.unique(ids))
    assert oracle.unique(np.array([], np.int64)).size == 0
    # retain: every requested id is emitted; missing rows are zero (sparse_retain-inl.h:121-150)
    req = np.unique(rng.integers(0, R, 30)).astype(np.int64)
    ri, rv = oracle.sparse_retain(oi, ov, req)
    assert np.array_equal(ri, req)
    present = np.isin(req, oi)
    assert np.array_equal(rv[present], dense[req[present]])
    assert np.all(rv[~present] == 0)
    # dense-source fast path: idx used as the row position
    full_i = np.arange(R, dtype=np.int64)
    ri, rv = oracle.sparse_retain(full_i, dense, req, src_dense_rows=True)
    assert np.array_equal(rv, dense[req])


def test_rowsparse_reduce_retain_unique_golden(oracle, golden):
    """oracle vs outputs of the reference's OWN ElementwiseSumRsp / GetUniqueRspRowIdx
    (src/ndarray/ndarray_function.cc:59-176), sparse_retain kernels (sparse_retain-inl.h:121-262) and
    UniqueImpl (kvstore_utils.cc:31-44), generated by oracle/gen_golden.py through oracle/ref_sparse.cc.
    Bit for bit: the sum over sources is taken in list order, rows ascending."""
    from gen_golden import rsp_cases
    g = golden("rowsparse_reduce_retain")
    red, ret, uniq = rsp_cases()
    for tag, (idxs, vals) in red.items():
        oi, ov = oracle.rsp_reduce(idxs, vals)
        assert np.array_equal(oi, g["reduce_%s_idx" % tag]), tag
        assert eq(ov, g["reduce_%s_val" % tag]), tag
    for tag, (si, sv, ids, dense) in ret.items():
        oi, ov = oracle.sparse_retain(si, sv, ids, src_dense_rows=dense)
        assert np.array_equal(oi, g["retain_%s_idx" % tag]), tag
        assert eq(ov, g["retain_%s_val" % tag]), tag
    for tag, ids in uniq.items():
        assert np.array_equal(oracle.unique(ids), g["unique_%s" % tag]), tag


# ---------------------------------------------------------------- the reference's own code (stored results)
def test_reduce_vs_reference_live(oracle):
    rng = np.random.default_rng(3)
    cases = [([rng.uniform(-1, 1, 3001).astype(np.float32) for _ in range(n)], 1)
             for n in (1, 2, 3, 4, 5, 6, 7, 8, 9, 13, 16)]
    # above MXNET_KVSTORE_BIGARRAY_BOUND: 4 threads x 4096-element tasks (comm.h:394-410)
    cases.append(([rng.uniform(-1, 1, 1200007).astype(np.float32) for _ in range(8)], 4))
    want = R.reference("test_oracle::reduce", lambda r: [R.digest(r.reduce(s, nthreads=t)) for s, t in cases])
    for i, ((s, t), w) in enumerate(zip(cases, want)):
        assert R.digest(oracle.reduce(s, "local", nthreads=t)) == w, "%d sources of %d, %d threads" % (
            len(s), s[0].size, t)


def test_dmlc_stof_vs_reference_live():
    import random
    random.seed(7)
    texts = [repr(random.choice([random.uniform(0, 2), 10 ** random.uniform(-12, 6),
                                 0.1 * 0.97 ** random.randint(0, 500), -random.uniform(0, 1e-3)]))
             for _ in range(5000)]
    want = R.reference("test_oracle::dmlc_stof",
                       lambda r: R.digest(np.float32([r.dmlc_stof(t) for t in texts])))
    assert R.digest(np.float32([K.dmlc_stof(t) for t in texts])) == want


@pytest.mark.parametrize("clip", (None, 0.5, 0.002))
def test_optimizers_vs_reference_live(oracle, clip):
    rng = np.random.default_rng(4)
    n = 10007
    w, g, m, v = [rng.uniform(-1, 1, n).astype(np.float32) for _ in range(4)]
    v = np.abs(v)

    def run(sgd, sgd_mom, multi_sgd, adam):
        out = [sgd(w.copy(), g, .1, 1e-4, 1 / 256, clip)]
        b = [w.copy(), m.copy()]
        sgd_mom(b[0], g, b[1], .1, .9, 1e-4, 1 / 256, clip)
        out += b
        b = [w.copy(), m.copy()]
        multi_sgd(b[0], g, b[1])
        out += b
        b = [w.copy(), m.copy(), v.copy()]
        adam(b[0], g, b[1], b[2], 1e-3, wd=.01, clip=clip)
        return dict(zip(('sgd_w', 'sgd_mom_w', 'sgd_mom_mom', 'multi_sgd_w', 'multi_sgd_mom', 'adam_w',
                         'adam_mean', 'adam_var'), [R.digest(x) for x in out + b]))
    want = R.reference("test_oracle::optimizers[%s]" % clip, lambda r: run(
        r.sgd_update, r.sgd_mom_update,
        lambda w_, g_, m_: r.multi_sgd_update([w_], [g_], [m_], [.1], [1e-4], .9, 1 / 256, clip),
        r.adam_update))
    got = run(oracle.sgd_update, oracle.sgd_mom_update,
              lambda w_, g_, m_: oracle.multi_sgd_update(w_, g_, m_, .1, .9, 1e-4, 1 / 256, clip),
              oracle.adam_update)
    for name in want:
        assert got[name] == want[name], name


def test_rowsparse_reduce_retain_vs_reference_live(oracle):
    """random layouts against the reference's own code (oracle/ref_sparse.cc), any thread count"""
    rng = np.random.default_rng(11)
    trials = []
    for trial in range(60):
        rows, rl = int(rng.integers(1, 400)), int(rng.integers(1, 70))
        nsrc = int(rng.integers(1, 10))
        idxs, vals = [], []
        for _ in range(nsrc):
            c = int(rng.integers(0, rows + 1)) if rng.random() < 0.8 else 0
            idxs.append(np.sort(rng.choice(rows, c, replace=False)).astype(np.int64))
            vals.append(rng.uniform(-1, 1, (c, rl)).astype(np.float32))
        nthreads = int(rng.integers(1, 6))
        ids = rng.integers(0, rows, int(rng.integers(0, 2 * rows + 1))).astype(np.int64)
        dense = rng.uniform(-1, 1, (rows, rl)).astype(np.float32)
        trials.append((rows, idxs, vals, nthreads, ids, dense))

    def run(rsp_reduce, unique, retain, retain_row_block):
        out = []
        for rows, idxs, vals, nthreads, ids, dense in trials:
            ri, rv = rsp_reduce(idxs, vals, nthreads)
            u = unique(ids)
            res = [(ri, rv), (u, None)] + [retain(ri, rv, req) for req in (ids, u)]
            res.append(retain_row_block(ri, rv, u))
            res.append(retain(np.arange(rows), dense, ids, src_dense_rows=True))
            out.append([[R.digest(np.asarray(a, np.int64)), None if b is None else R.digest(b)]
                        for a, b in res])
        return out
    # ascending unique ids: the reference's row-block retain kernel is a third witness
    want = R.reference("test_oracle::rowsparse_reduce_retain", lambda r: run(
        lambda i, v, t: r.rsp_reduce(i, v, nthreads=t), r.unique, r.sparse_retain,
        lambda i, v, q: r.sparse_retain(i, v, q, row_block=True)))
    got = run(lambda i, v, t: oracle.rsp_reduce(i, v), oracle.unique, oracle.sparse_retain,
              oracle.sparse_retain)
    steps = ('reduce', 'unique', 'retain', 'retain unique ids', 'retain row-block', 'retain dense rows')
    for trial, (g, w) in enumerate(zip(got, want)):
        for step, a, b in zip(steps, g, w):
            assert a == b, "trial %d: %s (ids, values) differ" % (trial, step)


def _key_lists(rng, trials):
    for t in range(trials):
        n, nk = int(rng.integers(1, 400)), int(rng.integers(1, 60))
        mode = t % 4
        if mode == 0:
            yield rng.integers(0, nk, n)                                   # no structure
        elif mode == 1:
            yield np.repeat(np.arange(nk), rng.integers(1, 9))             # key-major: k0 d0, k0 d1, ...
        elif mode == 2:
            yield np.tile(np.arange(nk), int(rng.integers(1, 9)))          # device-major: d0 k0, d0 k1, ...
        else:
            yield np.sort(rng.integers(0, nk, n))[::-1].copy()             # descending keys


def test_group_order_small_calls_and_hook(oracle):
    """Grouping of a call's (key, value) pairs (kvstore_local.h:377-407). Up to 16 pairs -- every
    per-parameter call of Trainer / Module, every call of the reference's unit tests -- the
    reference's std::sort leaves the values of a key in call order, which is what the product's
    stable grouping yields; the restated libstdc++ order agrees there by construction. The product's
    own sort (host hook) must equal the oracle's in both modes."""
    import ctypes
    import anand_mxnet_b200 as mx
    lib = mx.base._LIB
    rng = np.random.default_rng(21)
    for keys in _key_lists(rng, 400):
        keys = np.ascontiguousarray(keys, np.int32)
        if keys.size <= 16:
            assert K.group_positions(keys, 'reference') == K.group_positions(keys, 'call')
        for flag, order in ((0, 'call'), (1, 'reference')):
            pos = np.zeros(keys.size, np.int32)
            assert lib.B200KVTestGroupOrder(keys.ctypes.data_as(ctypes.c_void_p), int(keys.size), flag,
                                            pos.ctypes.data_as(ctypes.c_void_p)) == 0
            want = [p for grp in K.group_positions(keys, order)[1] for p in grp]
            assert list(pos) == want, (order, keys.size)


def test_group_order_vs_reference_live(oracle):
    """the reference's own GroupKVPairs compiled against libstdc++ (oracle/ref_sparse.cc): equal to
    the restated order for every call; equal to CALL order up to 16 pairs; beyond that the values of a
    key are handed to the reduce in an order only std::sort's internals explain -- the finding
    DESIGN.md section 6 records, and what B200KV_GROUP_ORDER=reference reproduces."""
    rng = np.random.default_rng(22)
    # last: the shape that matters, a list of keys with one value per device (10 keys x 4 GPUs)
    calls = list(_key_lists(rng, 1500)) + [np.repeat(np.arange(10), 4)]
    restated = [list(K.group_positions(k, 'reference')) for k in calls]
    want = R.reference("test_oracle::group_order",
                       lambda r: R.digest_json([list(r.group_positions(k)) for k in calls]))
    assert R.digest_json(restated) == want                     # every call, position for position
    left_call_order = 0
    for keys, live in zip(calls, restated):
        stable = list(K.group_positions(keys, 'call'))
        assert live[0] == stable[0]
        assert [sorted(g) for g in live[1]] == stable[1]          # same members, possibly another order
        if len(keys) <= 16:
            assert live == stable
        left_call_order += int(live != stable)
    assert left_call_order > 0
    assert restated[-1] != list(K.group_positions(calls[-1], 'call'))

"""Host orchestration pinned to the reference's OWN Python front-end.

oracle/ref_python.py loads /root/reference/python/mxnet/optimizer/optimizer.py and lr_scheduler.py
unmodified and runs them over the reference's own compiled operators (oracle/_ref/libmxref.so), so
update counts, schedulers, lr / wd multipliers, Adam's bias correction, SGD's aggregation, mixed
precision states, LARS's layer split and LAMB's step counts are all the reference's code. Against it:

  * ``kvoracle.LocalKVStoreModel`` -- the checker of the GPU store's fused route -- bit for bit;
  * the mirror under tests/compat/ -- the checker of the GPU store's callback route -- bit for bit
    AND call for call (same operators, same parameter strings, same order);
  * tests/golden/updater_trajectories.npz (written from it by oracle/gen_golden.py; the reference
    Python cannot travel to the GPU box, the fixture does) -- checked here against the model, and
    against the CUDA store in tests/test_updater_reference_fixture_gpu.py.

What the reference front-end returned in each comparison -- num_update, its operator calls with their
parameter strings, the weight and state arrays, the learning rates its schedulers gave -- is stored by
oracle/refrecord.py, and the mirror runs over the plain-C operators (golden_ops.OracleOps) and
schedulers that replay those learning rates, so these comparisons need neither the reference tree nor
oracle/_ref. Checks that need a live object of the reference's classes (the fixture recomputed from the
reference, FusedOptimizer records taken from a reference optimizer) are skipped where it is absent."""
import numpy as np
import pytest

import kvoracle as K
import ref_python as RP
import refrecord as R
from gen_golden import updater_cases, run_updater_case

live = pytest.mark.skipif(not RP.available(), reason="needs the reference tree and oracle/_ref/libmxref.so")


def eq(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def model_run(case):
    """the same plan through kvoracle.LocalKVStoreModel: per step, per key, push the gradient"""
    shapes, w0, grads = case['shapes'], case['w0'], case['grads']
    model = K.LocalKVStoreModel('device')
    for k, w in enumerate(w0):
        model.init(k, w)
    model.set_optimizer(lr_mult=case.get('lr_mult'), wd_mult=case.get('wd_mult'), **case['model'])
    for step in range(len(grads)):
        if 'lr_at' in case:
            model.opt['lr'] = case['lr_at'][step]
        for k in range(len(shapes)):
            model.push(k, [grads[step][k]])
    return [model.pull(k) for k in range(len(shapes))]


@pytest.mark.parametrize("name", sorted(n for n, c in updater_cases().items() if c['model']))
def test_model_vs_golden_trajectories(golden, name):
    g = golden("updater_trajectories")
    case = updater_cases()[name]
    got = model_run(case)
    for k, w in enumerate(got):
        assert eq(w, g["%s_w%d" % (name, k)]), (name, k)


@live
@pytest.mark.parametrize("name", sorted(updater_cases()))
def test_golden_trajectories_are_the_live_reference(golden, name):
    g = golden("updater_trajectories")
    case = updater_cases()[name]
    with RP.reference_python() as (opt, sched):
        got = run_updater_case(opt, sched, case)
    for k, w in enumerate(got):
        assert eq(w, g["%s_w%d" % (name, k)]), (name, k)


# ---------------------------------------------------------------- the tests/compat mirror
def _mirror():
    """tests/compat/mxnet_optimizer.py with its operator imports replaced by the harness's, so it
    runs on the same numpy buffers as the reference front-end, over the plain-C operators that
    tests/test_oracle_ops.py pins bit for bit to the reference's own"""
    from compat import mxnet_optimizer as M
    RP.use_oracle_ops()
    saved = dict(M.__dict__)
    M.__dict__.update(RP.op_table())
    M._contrib = type('contrib', (), {'multi_lamb_update': staticmethod(RP.multi_lamb_update),
                                      'multi_mp_lamb_update': staticmethod(RP.multi_mp_lamb_update)})
    return M, saved


NAMES = ['conv0_weight', 'conv0_bias', 'bn0_gamma', 'bn0_beta', 'fc_weight', 'fc_bias', 'emb_weight']
SHAPES = [(8, 3, 3, 3), (8,), (8,), (8,), (10, 72), (10,), (37, 5)]


def _plan(rng, steps, dtype=np.float32):
    w0 = [rng.uniform(-1, 1, s).astype(dtype) for s in SHAPES]
    grads = [[rng.uniform(-1, 1, s).astype(dtype) for s in SHAPES] for _ in range(steps)]
    return w0, grads


def _drive(mod, sched_mod, make, w0, grads, mode, devices=1, lr_changes=None, restart_at=None):
    """mode 'single': updater(index, grad, weight) per key, as the store's callback does;
    mode 'list': updater([indices], [grads], [weights]) as Trainer._update does.
    devices > 1: one Updater per device sharing ONE optimizer (gluon/trainer.py:321-323).
    restart_at: pickle the updater states (dump_optimizer=True) before that step and continue from a
    fresh Updater, as Trainer.save_states / load_states do."""
    RP.LOG[:] = []
    opt = make(mod, sched_mod)
    upds = [mod.get_updater(opt) for _ in range(devices)]
    ws = [[RP.NDArray(w.copy(), RP.Context(d, 'gpu')) for w in w0] for d in range(devices)]
    for step, gs in enumerate(grads):
        if lr_changes and step in lr_changes:
            opt.set_learning_rate(lr_changes[step])
        if restart_at == step:
            blobs = [u.get_states(dump_optimizer=True) for u in upds]
            upds = [mod.get_updater(make(mod, sched_mod)) for _ in range(devices)]
            for u, b in zip(upds, blobs):
                u.set_states(b)
            opt = upds[0].optimizer
            for u in upds:
                u.optimizer = opt
        for d, upd in enumerate(upds):
            garr = [RP.NDArray(g.copy(), RP.Context(d, 'gpu')) for g in gs]
            if mode == 'single':
                for k in range(len(w0)):
                    upd(k, garr[k], ws[d][k])
            else:
                upd(list(range(len(w0))), garr, ws[d])
    states = {}
    for d, upd in enumerate(upds):
        for k, st in upd.states.items():
            flat = RP._flat([st]) if isinstance(st, (list, tuple)) else [st]
            states[(d, k)] = [s.a.copy() for s in flat if s is not None]
    return [[w.a.copy() for w in dev] for dev in ws], states, list(RP.LOG), opt.num_update


CONFIGS = {
    'sgd_mom': lambda m, s: m.SGD(learning_rate=0.1, momentum=0.9, wd=1e-4, rescale_grad=1 / 32,
                                  param_idx2name=dict(enumerate(NAMES))),
    'sgd_plain_clip': lambda m, s: m.SGD(learning_rate=0.05, wd=1e-3, clip_gradient=0.3),
    'sgd_mults': lambda m, s: _with_mults(m.SGD(learning_rate=0.1, momentum=0.9, wd=1e-4,
                                                param_idx2name=dict(enumerate(NAMES)))),
    'sgd_factor_sched': lambda m, s: m.SGD(momentum=0.9, wd=1e-4,
                                           lr_scheduler=s.FactorScheduler(step=2, factor=0.5, base_lr=0.2)),
    'sgd_multifactor_warmup': lambda m, s: m.SGD(
        momentum=0.9, lr_scheduler=s.MultiFactorScheduler(step=[2, 4], factor=0.1, base_lr=0.4,
                                                          warmup_steps=2, warmup_begin_lr=0.01)),
    'sgd_cosine': lambda m, s: m.SGD(learning_rate=0.3, momentum=0.5,
                                     lr_scheduler=s.CosineScheduler(max_update=5, base_lr=0.3, final_lr=0.01)),
    'sgd_begin_num_update': lambda m, s: m.SGD(learning_rate=0.1, begin_num_update=7,
                                               lr_scheduler=s.PolyScheduler(max_update=20, base_lr=0.1, pwr=2)),
    'adam': lambda m, s: m.Adam(learning_rate=1e-3, wd=0.01, rescale_grad=0.5,
                                param_idx2name=dict(enumerate(NAMES))),
    'adam_clip_betas': lambda m, s: m.Adam(learning_rate=3e-4, beta1=0.8, beta2=0.98, epsilon=1e-6,
                                           clip_gradient=0.25),
    'adam_begin_num_update': lambda m, s: m.Adam(learning_rate=1e-3, begin_num_update=100),
    'lars': lambda m, s: m.LARS(learning_rate=0.2, momentum=0.9, wd=1e-4, eta=0.001, eps=1e-9,
                                rescale_grad=1 / 32, param_idx2name=dict(enumerate(NAMES))),
    'lars_sched_correction': lambda m, s: m.LARS(momentum=0.9, wd=1e-4, eta=0.002, rescale_grad=1 / 8,
                                                 param_idx2name=dict(enumerate(NAMES)),
                                                 lr_scheduler=s.FactorScheduler(step=2, factor=0.5, base_lr=0.4)),
    'lars_no_momentum': lambda m, s: m.LARS(learning_rate=0.1, wd=1e-3, eta=0.01, clip_gradient=0.5,
                                            param_idx2name=dict(enumerate(NAMES))),
    'lamb': lambda m, s: m.LAMB(learning_rate=2e-3, wd=0.01, rescale_grad=0.25,
                                param_idx2name=dict(enumerate(NAMES))),
    'lamb_bounds_nobias': lambda m, s: m.LAMB(learning_rate=1e-3, lower_bound=0.01, upper_bound=2.0,
                                              bias_correction=False, clip_gradient=0.4),
    'test': lambda m, s: m.Test(rescale_grad=2.0),
}


def _with_mults(opt):
    opt.set_lr_mult({1: 0.5, 'fc_weight': 2.0, 6: 0.25})
    opt.set_wd_mult({0: 0.0, 'bn0_beta': 0.5})
    return opt


SCHEDULERS = ('FactorScheduler', 'MultiFactorScheduler', 'CosineScheduler', 'PolyScheduler')
SCHEDULE_LEN = 64          # num_update 0..63: beyond every plan below


class _Recorder(object):
    """stand-in lr_scheduler module over the reference's: keeps every scheduler it makes"""

    def __init__(self, sched):
        self.made = []
        for name in SCHEDULERS:
            setattr(self, name, self._maker(getattr(sched, name)))

    def _maker(self, cls):
        def make(**kw):
            self.made.append(cls(**kw))
            return self.made[-1]
        return make


def _schedules(name, build):
    """[base_lr, learning rates for num_update 0..SCHEDULE_LEN-1 asked in increasing order as the
    optimizers do] of each reference scheduler build(opt, sched) returns"""
    def reference(_):
        with RP.reference_python() as (opt, sched):
            return [[s.base_lr, [s(n) for n in range(SCHEDULE_LEN)]] for s in build(opt, sched)]
    return R.reference("test_reference_python::schedule[%s]" % name, reference)


def _config_schedule(cfg):
    def build(opt, sched):
        rec = _Recorder(sched)
        CONFIGS[cfg](opt, rec)          # the optimizer may set the scheduler's base_lr
        return rec.made
    return _schedules(cfg, build)


class ReplayScheduler(object):
    """a scheduler returning the learning rates a reference scheduler gave (_schedules), one table
    per base_lr"""

    def __init__(self, tables, base_lr):
        self.tables = {b: r for b, r in tables}
        self.base_lr = base_lr

    @property
    def base_lr(self):
        return self._base

    @base_lr.setter
    def base_lr(self, v):
        assert v in self.tables, "no learning rates recorded for base_lr %r" % v
        self._base = v

    def __call__(self, num_update):
        return self.tables[self._base][num_update]


class _Replay(object):
    """stand-in lr_scheduler module for the mirror: its schedulers replay the recorded tables"""

    def __init__(self, tables):
        for name in SCHEDULERS:
            setattr(self, name, lambda base_lr=tables[0][0] if tables else None, **kw:
                    ReplayScheduler(tables, base_lr))


def _norm(call):
    """(operator, parameters) with tuple-valued parameters as token lists: the mirror hands python
    tuples to the operators where the reference hands lists -- '(0.1,)' and '[0.1]' are the same
    value to the Tuple<float> parser (include/mxnet/tuple.h); every token must still be identical"""
    name, params = call
    out = {}
    for k, v in params.items():
        out[k] = [t.strip() for t in v.strip('()[]').split(',') if t.strip()] if v[:1] in '([' else v
    return name, out


def _compare(cfg, mode, dtype=np.float32, steps=5, monkeypatch=None, agg=None, mp=False, **kw):
    if agg is not None:
        monkeypatch.setenv('MXNET_OPTIMIZER_AGGREGATION_SIZE', str(agg))
    make = CONFIGS[cfg]
    if mp:
        base = make

        def make(m, s):                     # noqa: E306
            o = base(m, s)
            o.multi_precision = True
            return o
    w0, grads = _plan(np.random.default_rng(len(cfg) + steps), steps, dtype)

    def summary(res):
        """weights and states as digests, every operator call as (operator, parameter tokens)"""
        ws, states, log, num_update = res
        return {'num_update': num_update,
                'calls': [R.digest_json(list(_norm(c))) for c in log],
                'weights': [[R.digest(w) for w in dev] for dev in ws],
                'states': {'%d,%d' % key: [R.digest(a) for a in v] for key, v in sorted(states.items())}}

    def reference(_):
        with RP.reference_python() as (opt, sched):
            return summary(_drive(opt, sched, make, w0, grads, mode, **kw))
    key = "test_reference_python::%s|%s|%s|steps=%d|agg=%s|mp=%s|%s" % (
        cfg, mode, np.dtype(dtype).name, steps, agg, mp, sorted(kw.items()))
    want = R.reference(key, reference)
    M, saved = _mirror()
    try:
        got = summary(_drive(M, _Replay(_config_schedule(cfg)), make, w0, grads, mode, **kw))
    finally:
        RP.use_oracle_ops(False)
        M.__dict__.clear()
        M.__dict__.update(saved)
    assert got['num_update'] == want['num_update']
    assert len(got['calls']) == len(want['calls']) and len(want['calls']) > 0
    for i, (a, b) in enumerate(zip(got['calls'], want['calls'])):   # operator, parameter strings, order
        assert a == b, (cfg, mode, 'operator call %d differs: the mirror called %r' % (i, RP.LOG[i]))
    for d, (dev_g, dev_w) in enumerate(zip(got['weights'], want['weights'])):
        for k, (a, b) in enumerate(zip(dev_g, dev_w)):
            assert a == b, (cfg, mode, 'device %d weight %d (%s) differs' % (d, k, NAMES[k]))
    assert sorted(got['states']) == sorted(want['states']), (cfg, mode)
    for st in want['states']:
        assert got['states'][st] == want['states'][st], (cfg, mode, 'state (device, key) = ' + st)


@pytest.mark.parametrize("mode", ['single', 'list'])
@pytest.mark.parametrize("cfg", sorted(c for c in CONFIGS if c != 'test'))
def test_compat_mirror_vs_reference(cfg, mode):
    _compare(cfg, mode)


def test_compat_mirror_test_optimizer():
    _compare('test', 'single')


@pytest.mark.parametrize("cfg", ['sgd_mom', 'sgd_plain_clip', 'lars', 'lars_no_momentum', 'lamb', 'adam'])
@pytest.mark.parametrize("agg", [1, 3, 45])
def test_compat_mirror_aggregation_sizes(cfg, agg, monkeypatch):
    if cfg == 'lamb' and agg == 1:
        pytest.skip("LAMB's one-tensor form calls NDArray.norm(), an operator outside the harness")
    _compare(cfg, 'list', monkeypatch=monkeypatch, agg=agg)


@pytest.mark.parametrize("cfg", ['sgd_mom', 'sgd_plain_clip', 'lars', 'lars_no_momentum', 'lamb', 'adam'])
@pytest.mark.parametrize("mode", ['single', 'list'])
def test_compat_mirror_multi_precision_fp16(cfg, mode):
    _compare(cfg, mode, dtype=np.float16, mp=True)


@pytest.mark.parametrize("cfg", ['sgd_mom', 'adam', 'lars_sched_correction', 'sgd_factor_sched'])
def test_compat_mirror_shared_optimizer_two_devices(cfg):
    _compare(cfg, 'list', devices=2)


@pytest.mark.parametrize("cfg", ['sgd_mom', 'adam', 'lamb'])
def test_compat_mirror_set_learning_rate_between_steps(cfg):
    _compare(cfg, 'single', lr_changes={2: 0.01, 4: 0.3})


@pytest.mark.parametrize("cfg", ['sgd_mom', 'adam', 'sgd_factor_sched'])
def test_compat_mirror_state_pickle_restart(cfg):
    _compare(cfg, 'list', restart_at=3)


# ---------------------------------------------------------------- the product's hyper-parameter record
class _Param(object):
    def __init__(self, lr_mult, wd_mult):
        self.lr_mult, self.wd_mult = lr_mult, wd_mult


_VARIANTS = [
    dict(),
    dict(param_idx2name=dict(enumerate(NAMES))),
    dict(param_idx2name=dict(enumerate(NAMES)), param_dict={2: _Param(0.3, 0.7), 4: _Param(5.0, 0.0)}),
    dict(param_dict={0: _Param(0.5, 2.0)}),
]
_SETTERS = [
    ({}, {}),
    ({1: 0.5, 'fc_weight': 2.0, 6: 0.25}, {0: 0.0, 'bn0_beta': 0.5, 'fc_bias': 3.0}),
    ({'conv0_weight': 0.1, 0: 0.2}, {'emb_weight': 0.0}),          # index beats name
]
_INDICES = list(range(len(NAMES) + 2)) + ['fc_weight']
_NUM_UPDATES = (0, 1, 3, 4, 7, 20)


def _sched_variants(sched):
    return [lambda: dict(lr_scheduler=sched.FactorScheduler(step=3, factor=0.5, base_lr=0.4)),
            lambda: dict(lr_scheduler=sched.FactorScheduler(step=3, factor=0.5, base_lr=0.4), learning_rate=0.8),
            lambda: dict(learning_rate=0.25), lambda: dict()]


def _optimizers(mod):
    """(class, variant, setter, optimizer) with lr = wd = 1, so _get_lr / _get_wd are the multipliers"""
    for cls in ('SGD', 'Adam', 'Test'):
        for v, kw in enumerate(_VARIANTS):
            for t, (lr_mult, wd_mult) in enumerate(_SETTERS):
                o = getattr(mod, cls)(learning_rate=1.0, wd=1.0, **kw)
                o.set_lr_mult(lr_mult)
                o.set_wd_mult(wd_mult)
                yield cls, v, t, o


def _learning_rates(o):
    """learning_rate at each of _NUM_UPDATES, then whether set_learning_rate(0.03) is refused"""
    rates = []
    for n in _NUM_UPDATES:
        o.num_update = n
        rates.append(o.learning_rate)
    try:
        o.set_learning_rate(0.03)
    except UserWarning:
        return rates, True
    assert o.learning_rate == 0.03
    return rates, False


def test_fused_record_vs_reference_optimizer():
    """anand_mxnet_b200.optimizer.FusedOptimizer (what kv.set_optimizer turns into the native replay's
    inputs) against the reference's Optimizer: multiplier lookup order (Parameter object, index, name),
    default wd_mult of non-weights, scheduler / explicit learning rate precedence -- the reference's
    answers stored by oracle/refrecord.py"""
    from anand_mxnet_b200 import optimizer as P

    def reference(_):
        with RP.reference_python() as (opt, sched):
            mults = [[[o._get_lr(i), o._get_wd(i)] for i in _INDICES] for _, _, _, o in _optimizers(opt)]
            rates = [_learning_rates(opt.SGD(**mk())) for mk in _sched_variants(sched)]
            return {'multipliers': mults, 'learning_rates': rates}
    want = R.reference("test_reference_python::fused_record", reference)
    for (cls, v, t, mine), w in zip(_optimizers(P), want['multipliers']):
        for i, m in zip(_INDICES, w):
            assert list(mine.multipliers(i)) == m, (cls, sorted(_VARIANTS[v]), t, i)
    tables = _schedules('fused_record', lambda opt, sched: [
        sched.FactorScheduler(step=3, factor=0.5, base_lr=b) for b in (0.4, 0.8)])
    for k, (mk, w) in enumerate(zip(_sched_variants(_Replay(tables)), want['learning_rates'])):
        rates, refused = _learning_rates(P.SGD(**mk()))
        assert [rates, refused] == w, k


@live
def test_record_of_reference_optimizer():
    """FusedOptimizer records taken from objects of the reference's own optimizer classes (record_of):
    the same multipliers, learning rates and operator parameters as the reference object"""
    from anand_mxnet_b200 import optimizer as P
    with RP.reference_python() as (opt, sched):
        for cls, v, t, ref in _optimizers(opt):
            assert P.fused_kind(ref) == cls.lower()
            rec = P.record_of(ref)
            for i in _INDICES:
                assert rec.multipliers(i) == (ref._get_lr(i), ref._get_wd(i)), (cls, v, t, i)
        for mk in _sched_variants(sched):
            ref = opt.SGD(**mk())
            for n in _NUM_UPDATES:
                ref.num_update = n
                assert ref.learning_rate == P.record_of(ref).learning_rate
        # operator parameters handed to the library: the reference object's own attribute values
        ref = opt.Adam(learning_rate=2e-3, beta1=0.8, beta2=0.97, epsilon=1e-5, wd=0.1, rescale_grad=0.5,
                       clip_gradient=0.7, begin_num_update=11)
        p = P.record_of(ref).op_params()
        assert (p['learning_rate'], p['beta1'], p['beta2'], p['epsilon'], p['wd'], p['rescale_grad'],
                p['clip_gradient'], p['begin_num_update']) == (2e-3, 0.8, 0.97, 1e-5, 0.1, 0.5, 0.7, 11)
        ref = opt.SGD(momentum=0.9, clip_gradient=None)
        p = P.record_of(ref).op_params()
        assert p['momentum'] == 0.9 and p['clip_gradient'] == 0.0 and p['learning_rate'] == 0.01

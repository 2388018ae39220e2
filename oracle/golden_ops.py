"""TEST INFRASTRUCTURE ONLY.

Seeded cases for the multi-tensor optimizer operators (SURVEY 8f-f1) written once against a tiny
backend interface

    backend.invoke(op_name, inputs, outputs, **params)      # numpy arrays, outputs written in place

which is the calling convention of the reference's imperative front-end (inputs in operator order,
`out=` arrays, keyword parameters stringified). Three backends run the SAME cases:
  * kvoracle.Ref.op_invoke        the reference's own FCompute<cpu> (oracle/ref_ops.cc)
  * OracleOps (below)             the plain-C restatement oracle/kvoracle.c + the parameter plumbing
  * tests' GPU backend            the CUDA library through MXImperativeInvokeEx

`python oracle/golden_ops.py` regenerates tests/golden/multi_tensor_ops.npz from the live reference.
"""
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, _HERE)
import kvoracle as K  # noqa: E402


def _tuple(v):
    """mxnet::Tuple<float> parameter: str(list) parsed by istream >> float (nearest float32)"""
    return [K.f32(x) for x in v]


def _u16(a):
    return a.view(np.uint16) if a.dtype == np.float16 else a


class OracleOps(object):
    """Operator-level front of oracle/kvoracle.c: splits the reference calling convention into the
    per-tensor restatements and applies the parameter plumbing (scalars: python repr -> dmlc::stof;
    tuples: nearest float32)."""

    def __init__(self, oracle=None):
        self.o = oracle or K.get_oracle()

    @staticmethod
    def _s(params, key, default):
        return K.scalar_param(params[key]) if key in params else default

    @staticmethod
    def _clipv(params):
        return K.scalar_param(params['clip_gradient']) if 'clip_gradient' in params else -1.0

    def invoke(self, op, inputs, outputs, **p):
        getattr(self, '_op_' + op.lstrip('_'))(inputs, outputs, p)

    def _op_multi_sum_sq(self, ins, outs, p):
        assert int(p['num_arrays']) == len(ins)
        outs[0][:] = self.o.multi_sum_sq([_u16(a) for a in ins],
                                         kind=None if ins[0].dtype == np.float32 else 0)

    def _op_multi_lars(self, ins, outs, p):
        outs[0][:] = self.o.multi_lars(ins[0], ins[1], ins[2], ins[3], self._s(p, 'eta', None),
                                       self._s(p, 'eps', None), self._s(p, 'rescale_grad', 1.0))

    def _preloaded(self, ins, outs, p, stride, has_mom, mp):
        n = int(p['num_weights'])
        self._multi_sgd(ins, outs, p, stride, has_mom, mp, ins[n * stride], ins[n * stride + 1])

    def _multi_sgd(self, ins, outs, p, stride, has_mom, mp, lrs, wds):
        n = int(p['num_weights'])
        clip, rescale = self._clipv(p), self._s(p, 'rescale_grad', 1.0)
        momentum = self._s(p, 'momentum', 0.0) if has_mom else 0.0
        L = self.o.lib
        for k in range(n):
            t = ins[k * stride:(k + 1) * stride]
            w, g = t[0], t[1]
            mom = t[2] if has_mom else None
            mp_ = K._ptr(mom) if mom is not None else None
            if mp:
                w32 = t[stride - 1]
                L.kvo_multi_mp_sgd_update(w.size, K._ptr(_u16(outs[k])), mp_, K._ptr(w32),
                                          K._ptr(_u16(g)), 0, clip, momentum, float(lrs[k]),
                                          float(wds[k]), rescale, 1)
            else:
                L.kvo_multi_sgd_update(w.size, K._ptr(outs[k]), mp_, K._ptr(w), K._ptr(g), clip,
                                       momentum, float(lrs[k]), float(wds[k]), rescale, 1)

    def _op_preloaded_multi_sgd_update(self, i, o, p):
        self._preloaded(i, o, p, 2, False, False)

    def _op_preloaded_multi_sgd_mom_update(self, i, o, p):
        self._preloaded(i, o, p, 3, True, False)

    def _op_preloaded_multi_mp_sgd_update(self, i, o, p):
        self._preloaded(i, o, p, 3, False, True)

    def _op_preloaded_multi_mp_sgd_mom_update(self, i, o, p):
        self._preloaded(i, o, p, 4, True, True)

    def _op_multi_sgd_update(self, i, o, p):
        self._multi_sgd(i, o, p, 2, False, False, _tuple(p['lrs']), _tuple(p['wds']))

    def _op_multi_sgd_mom_update(self, i, o, p):
        self._multi_sgd(i, o, p, 3, True, False, _tuple(p['lrs']), _tuple(p['wds']))

    def _op_multi_mp_sgd_update(self, i, o, p):
        self._multi_sgd(i, o, p, 3, False, True, _tuple(p['lrs']), _tuple(p['wds']))

    def _op_multi_mp_sgd_mom_update(self, i, o, p):
        self._multi_sgd(i, o, p, 4, True, True, _tuple(p['lrs']), _tuple(p['wds']))

    def _op_adam_update(self, ins, outs, p):
        w, g, mean, var = ins
        c = self._adam_common(p)
        self.o.lib.kvo_adam_update(w.size, K._ptr(outs[0]), K._ptr(mean), K._ptr(var), K._ptr(w), K._ptr(g),
                                   c['clip'], self._s(p, 'rescale_grad', 1.0), c['beta1'], c['beta2'],
                                   self._s(p, 'lr', None), self._s(p, 'wd', 0.0), c['eps'], 1)

    def _adam_common(self, p):
        return dict(beta1=self._s(p, 'beta1', K.f32(0.9)), beta2=self._s(p, 'beta2', K.f32(0.999)),
                    eps=self._s(p, 'epsilon', K.f32(1e-8)), clip=self._clipv(p))

    def _op_adamw_update(self, ins, outs, p):
        w, g, mean, var, rescale = ins
        c = self._adam_common(p)
        if outs[0] is not w:
            raise NotImplementedError("oracle front: out must be the weight array")
        self.o.adamw_update(w, g, mean, var, float(rescale[0]), self._s(p, 'lr', None),
                            self._s(p, 'eta', None), wd=self._s(p, 'wd', 0.0), **c)

    def _op_mp_adamw_update(self, ins, outs, p):
        w16, g16, mean, var, w32, rescale = ins
        c = self._adam_common(p)
        self.o.mp_adamw_update(_u16(outs[0]), _u16(g16), mean, var, w32, 0, float(rescale[0]),
                               self._s(p, 'lr', None), self._s(p, 'eta', None),
                               wd=self._s(p, 'wd', 0.0), **c)

    def _multi_adamw(self, ins, outs, p, mp):
        n = int(p['num_weights'])
        stride = 5 if mp else 4
        rescale = float(ins[n * stride][0])
        c = self._adam_common(p)
        t = [ins[k * stride:(k + 1) * stride] for k in range(n)]
        for k in range(n):
            assert outs[k] is t[k][0], "oracle front: out must be the weight arrays"
        self.o.multi_adamw_update([_u16(x[0]) for x in t], [_u16(x[1]) for x in t],
                                  [x[2] for x in t], [x[3] for x in t], rescale, _tuple(p['lrs']),
                                  _tuple(p['wds']), _tuple(p['etas']),
                                  w32s=[x[4] for x in t] if mp else None, kind=0, **c)

    def _op_multi_adamw_update(self, i, o, p):
        self._multi_adamw(i, o, p, False)

    def _op_multi_mp_adamw_update(self, i, o, p):
        self._multi_adamw(i, o, p, True)

    def _lamb1_common(self, p):
        return dict(t=int(p['t']), beta1=self._s(p, 'beta1', K.f32(0.9)),
                    beta2=self._s(p, 'beta2', K.f32(0.999)), eps=self._s(p, 'epsilon', K.f32(1e-6)),
                    wd=self._s(p, 'wd', None), rescale=self._s(p, 'rescale_grad', 1.0),
                    clip=self._clipv(p), bias_correction=str(p.get('bias_correction', True)) == 'True')

    def _op_lamb_update_phase1(self, ins, outs, p):
        w, g, mean, var = ins
        outs[0][:] = self.o.lamb_phase1(w, g, mean, var, **self._lamb1_common(p))

    def _op_mp_lamb_update_phase1(self, ins, outs, p):
        w16, g16, mean, var, w32 = ins
        outs[0][:] = self.o.lamb_phase1(w32, None, mean, var, g16=_u16(g16), kind=0,
                                        **self._lamb1_common(p))

    def _bounds(self, p):
        return (self._s(p, 'lower_bound', None) if 'lower_bound' in p else None,
                self._s(p, 'upper_bound', None) if 'upper_bound' in p else None)

    def _op_lamb_update_phase2(self, ins, outs, p):
        w, g, r1, r2 = ins
        lb, ub = self._bounds(p)
        outs[0][:] = self.o.lamb_phase2(w, g, float(r1[0]), float(r2[0]), self._s(p, 'lr', None), lb, ub)

    def _op_mp_lamb_update_phase2(self, ins, outs, p):
        w16, g, r1, r2, w32 = ins
        lb, ub = self._bounds(p)
        _u16(outs[0])[:] = self.o.lamb_phase2(w32, g, float(r1[0]), float(r2[0]),
                                              self._s(p, 'lr', None), lb, ub, out16_kind=0)

    def _multi_lamb(self, ins, outs, p, mp):
        n = int(p['num_tensors'])
        stride = 5 if mp else 4
        t = [ins[k * stride:(k + 1) * stride] for k in range(n)]
        for k in range(n):
            assert outs[k] is t[k][0], "oracle front: out must be the weight arrays"
        lb, ub = self._bounds(p)
        self.o.multi_lamb_update([_u16(x[0]) for x in t], [_u16(x[1]) for x in t],
                                 [x[2] for x in t], [x[3] for x in t],
                                 [int(s) for s in p['step_count']], _tuple(p['learning_rates']),
                                 _tuple(p['wds']), beta1=self._s(p, 'beta1', K.f32(0.9)),
                                 beta2=self._s(p, 'beta2', K.f32(0.999)),
                                 eps=self._s(p, 'epsilon', K.f32(1e-6)),
                                 rescale=self._s(p, 'rescale_grad', 1.0), lower_bound=lb,
                                 upper_bound=ub, clip=self._clipv(p),
                                 bias_correction=str(p.get('bias_correction', True)) == 'True',
                                 w32s=[x[4] for x in t] if mp else None, kind=0)

    def _op_multi_lamb_update(self, i, o, p):
        self._multi_lamb(i, o, p, False)

    def _op_multi_mp_lamb_update(self, i, o, p):
        self._multi_lamb(i, o, p, True)


# ---------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------
SHAPES = [(7,), (3, 5), (1,), (257,), (64, 33), (4099,)]


def _rng(case):
    return np.random.default_rng(abs(hash(case)) % (2 ** 31) if False else
                                 int.from_bytes(case.encode(), 'little') % (2 ** 31))


def _f(rng, shape, lo=-1.0, hi=1.0):
    return rng.uniform(lo, hi, shape).astype(np.float32)


def _h(rng, shape, lo=-1.0, hi=1.0):
    return rng.uniform(lo, hi, shape).astype(np.float16)


def case_sum_sq_f32(b, rng):
    xs = [_f(rng, s, 0, 10) for s in SHAPES]
    out = np.zeros(len(xs), np.float32)
    b.invoke('multi_sum_sq', xs, [out], num_arrays=len(xs))
    return {'out': out}


def case_sum_sq_f16(b, rng):
    xs = [_h(rng, s, 0, 10) for s in SHAPES]
    out = np.zeros(len(xs), np.float32)
    b.invoke('multi_sum_sq', xs, [out], num_arrays=len(xs))
    return {'out': out}


def case_lars(b, rng):
    n = 11
    lrs, wds = _f(rng, n, 0.001, 0.011), _f(rng, n, 1e-4, 1.1e-3)
    wsq, gsq = _f(rng, n, 0, 100), _f(rng, n, 0, 10)
    wsq[2] = 0
    gsq[4] = 0
    out = np.zeros(n, np.float32)
    b.invoke('multi_lars', [lrs, wsq, gsq, wds], [out], eta=0.37, eps=1.3e-05, rescale_grad=77.3)
    out2 = np.zeros(n, np.float32)
    b.invoke('multi_lars', [lrs, wsq, gsq, wds], [out2], eta=0.001, eps=0)
    return {'out': out, 'out_default_rescale': out2}


def _preloaded(b, rng, mom, mp, clip):
    n = len(SHAPES)
    mk = _h if mp else _f
    ws, gs = [mk(rng, s, -100, 100) for s in SHAPES], [mk(rng, s, -100, 100) for s in SHAPES]
    moms = [_f(rng, s) for s in SHAPES] if mom else None
    w32 = [w.astype(np.float32) for w in ws] if mp else None
    lrs, wds = _f(rng, n, 0.001, 0.011), _f(rng, n, 1e-4, 1.1e-3)
    ins = []
    for k in range(n):
        ins += [ws[k], gs[k]] + ([moms[k]] if mom else []) + ([w32[k]] if mp else [])
    ins += [lrs, wds]
    name = 'preloaded_multi_%ssgd_%supdate' % ('mp_' if mp else '', 'mom_' if mom else '')
    kw = dict(num_weights=n, rescale_grad=0.95)
    if mom:
        kw['momentum'] = 0.9
    if clip:
        kw['clip_gradient'] = 2.5
    b.invoke(name, ins, ws, **kw)
    out = {'w%d' % k: ws[k] for k in range(n)}
    if mom:
        out.update({'m%d' % k: moms[k] for k in range(n)})
    if mp:
        out.update({'w32_%d' % k: w32[k] for k in range(n)})
    return out


def case_preloaded_sgd(b, rng):
    return _preloaded(b, rng, False, False, False)


def case_preloaded_sgd_mom_clip(b, rng):
    return _preloaded(b, rng, True, False, True)


def case_preloaded_mp_sgd(b, rng):
    return _preloaded(b, rng, False, True, True)


def case_preloaded_mp_sgd_mom(b, rng):
    return _preloaded(b, rng, True, True, False)


def _adamw_single(b, rng, mp, clip, rescale):
    s = (64, 33)
    w, g = (_h if mp else _f)(rng, s), (_h if mp else _f)(rng, s, -3, 3)
    mean, var = _f(rng, s, -0.1, 0.1), _f(rng, s, 0, 0.1)
    rs = np.array([rescale], np.float32)
    kw = dict(lr=0.003, eta=0.7, beta1=0.9, beta2=0.98, epsilon=1e-06, wd=0.013)
    if clip:
        kw['clip_gradient'] = 0.5
    out = {}
    for step in range(2):
        if mp:
            if step == 0:
                w32 = w.astype(np.float32)
            b.invoke('_mp_adamw_update', [w, g, mean, var, w32, rs], [w], **kw)
        else:
            b.invoke('_adamw_update', [w, g, mean, var, rs], [w], **kw)
    out.update(w=w, mean=mean, var=var, g_after=g)
    if mp:
        out['w32'] = w32
    return out


def case_adamw(b, rng):
    return _adamw_single(b, rng, False, False, 1.0 / 64)


def case_adamw_clip(b, rng):
    return _adamw_single(b, rng, False, True, 0.37)


def case_adamw_skip(b, rng):
    r = _adamw_single(b, rng, False, False, float('inf'))
    r.update({'zero_' + k: v for k, v in _adamw_single(b, rng, False, False, 0.0).items()})
    return r


def case_mp_adamw(b, rng):
    return _adamw_single(b, rng, True, True, 0.37)


def _multi_adamw(b, rng, mp, clip):
    n = len(SHAPES)
    mk = _h if mp else _f
    ws, gs = [mk(rng, s) for s in SHAPES], [mk(rng, s, -3, 3) for s in SHAPES]
    means, vars_ = [_f(rng, s, -0.1, 0.1) for s in SHAPES], [_f(rng, s, 0, 0.1) for s in SHAPES]
    w32 = [w.astype(np.float32) for w in ws] if mp else None
    rs = np.array([0.37], np.float32)
    lrs = [0.001 * (k + 1) for k in range(n)]
    wds = [0.01 * (k % 3) for k in range(n)]
    etas = [1.0 - 0.1 * k for k in range(n)]
    ins = []
    for k in range(n):
        ins += [ws[k], gs[k], means[k], vars_[k]] + ([w32[k]] if mp else [])
    ins.append(rs)
    kw = dict(lrs=lrs, wds=wds, etas=etas, beta1=0.9, beta2=0.98, epsilon=1e-06, num_weights=n)
    if clip:
        kw['clip_gradient'] = 0.5
    name = '_multi_mp_adamw_update' if mp else '_multi_adamw_update'
    for _ in range(2):
        b.invoke(name, ins, ws, **kw)
    out = {}
    for k in range(n):
        out.update({'w%d' % k: ws[k], 'mean%d' % k: means[k], 'var%d' % k: vars_[k]})
        if mp:
            out['w32_%d' % k] = w32[k]
    return out


def case_multi_adamw(b, rng):
    return _multi_adamw(b, rng, False, False)


def case_multi_adamw_clip(b, rng):
    return _multi_adamw(b, rng, False, True)


def case_multi_mp_adamw(b, rng):
    return _multi_adamw(b, rng, True, True)


def _lamb_phases(b, rng, mp, clip, bias, bounds):
    s = (64, 33)
    w, g = (_h if mp else _f)(rng, s), (_h if mp else _f)(rng, s, -3, 3)
    mean, var = _f(rng, s, -0.1, 0.1), _f(rng, s, 0, 0.1)
    w32 = w.astype(np.float32) if mp else None
    gout = np.zeros(s, np.float32)
    kw = dict(beta1=0.9, beta2=0.98, epsilon=1e-06, t=3, bias_correction=bias, wd=0.013,
              rescale_grad=0.37)
    if clip:
        kw['clip_gradient'] = 0.5
    if mp:
        b.invoke('mp_lamb_update_phase1', [w, g, mean, var, w32], [gout], **kw)
    else:
        b.invoke('lamb_update_phase1', [w, g, mean, var], [gout], **kw)
    # r1, r2 are inputs of phase 2 (norms computed by the caller): fixed values here
    r1, r2 = np.array([7.25], np.float32), np.array([3.5], np.float32)
    kw2 = dict(lr=0.003)
    if bounds:
        kw2.update(lower_bound=0.5, upper_bound=6.0)
    if mp:
        b.invoke('mp_lamb_update_phase2', [w, gout, r1, r2, w32], [w], **kw2)
    else:
        b.invoke('lamb_update_phase2', [w, gout, r1, r2], [w], **kw2)
    out = dict(w=w, g=gout, mean=mean, var=var)
    if mp:
        out['w32'] = w32
    # zero-norm branch
    z = np.array([0.0], np.float32)
    w2 = w.copy()
    if mp:
        b.invoke('mp_lamb_update_phase2', [w2, gout, z, r2, w32], [w2], **kw2)
    else:
        b.invoke('lamb_update_phase2', [w2, gout, z, r2], [w2], lr=0.003)
    out['w_zero_r1'] = w2
    return out


def case_lamb_phases(b, rng):
    return _lamb_phases(b, rng, False, False, True, False)


def case_lamb_phases_clip_nobias_bounds(b, rng):
    return _lamb_phases(b, rng, False, True, False, True)


def case_mp_lamb_phases(b, rng):
    return _lamb_phases(b, rng, True, True, True, True)


def _multi_lamb(b, rng, mp, clip, bias, bounds):
    n = len(SHAPES)
    mk = _h if mp else _f
    ws, gs = [mk(rng, s) for s in SHAPES], [mk(rng, s, -3, 3) for s in SHAPES]
    means, vars_ = [_f(rng, s, -0.1, 0.1) for s in SHAPES], [_f(rng, s, 0, 0.1) for s in SHAPES]
    w32 = [w.astype(np.float32) for w in ws] if mp else None
    ws[2][...] = 0     # zero weight norm -> trust ratio 1
    if mp:
        w32[2][...] = 0
    ins = []
    for k in range(n):
        ins += [ws[k], gs[k], means[k], vars_[k]] + ([w32[k]] if mp else [])
    kw = dict(learning_rates=[0.001 * (k + 1) for k in range(n)],
              wds=[0.01 * (k % 3) for k in range(n)], beta1=0.9, beta2=0.98, epsilon=1e-06,
              rescale_grad=0.37, bias_correction=bias, num_tensors=n,
              step_count=[k + 1 for k in range(n)])
    if clip:
        kw['clip_gradient'] = 0.5
    if bounds:
        kw.update(lower_bound=0.5, upper_bound=6.0)
    name = '_multi_mp_lamb_update' if mp else '_multi_lamb_update'
    b.invoke(name, ins, ws, **kw)
    out = {}
    for k in range(n):
        out.update({'w%d' % k: ws[k], 'mean%d' % k: means[k], 'var%d' % k: vars_[k]})
        if mp:
            out['w32_%d' % k] = w32[k]
    return out


def case_multi_lamb(b, rng):
    return _multi_lamb(b, rng, False, False, True, False)


def case_multi_lamb_clip_nobias_bounds(b, rng):
    return _multi_lamb(b, rng, False, True, False, True)


def case_multi_mp_lamb(b, rng):
    return _multi_lamb(b, rng, True, True, True, True)


CASES = {k[5:]: v for k, v in list(globals().items()) if k.startswith('case_')}

# results that depend on the ORDER of a floating-point reduction (sum of squares): other
# implementations match these within a tolerance, not bit for bit (see tests/test_ops_gpu.py)
REDUCTION_CASES = {'sum_sq_f32', 'sum_sq_f16', 'multi_lamb', 'multi_lamb_clip_nobias_bounds',
                   'multi_mp_lamb'}


class _RefBackend(object):
    def __init__(self, ref):
        self.ref = ref

    def invoke(self, op, inputs, outputs, **params):
        self.ref.op_invoke(op, inputs, outputs, **params)


def run_case(case, oracle=None, ref=None, backend=None):
    if backend is None:
        backend = _RefBackend(ref) if ref is not None else OracleOps(oracle)
    out = CASES[case](backend, _rng(case))
    return {k: np.ascontiguousarray(v).copy() for k, v in out.items()}


def main():
    ref = K.ref()
    assert ref is not None and ref.has_ops(), "build oracle/_ref first (make -C oracle ref)"
    blob = {}
    for case in sorted(CASES):
        for k, v in run_case(case, ref=ref).items():
            blob[case + "/" + k] = v
    path = os.path.join(os.path.dirname(_HERE), "tests", "golden", "multi_tensor_ops.npz")
    np.savez_compressed(path, **blob)
    print("wrote", path, len(blob), "arrays", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

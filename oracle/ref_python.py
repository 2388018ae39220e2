"""TEST INFRASTRUCTURE ONLY -- runs the reference's OWN Python optimizer front-end
(/root/reference/python/mxnet/optimizer/optimizer.py and lr_scheduler.py, loaded from where they
lie, unmodified) on top of the reference's OWN compiled operator code (oracle/_ref/libmxref.so,
`Ref.op_invoke`: the real dmlc::Parameter parser + FCompute<cpu> of each optimizer operator).

libmxnet.so is not buildable here, so `import mxnet` is not possible; what the optimizer module needs
from the rest of the package is small and is supplied by stand-ins:

  * ``mxnet.ndarray``   a numpy-backed ``NDArray`` (dtype / shape / stype / context / astype / slices
                        / the few arithmetic forms Test uses) and one function per optimizer
                        operator that forwards its arguments to ``Ref.op_invoke`` -- parameters
                        stringified with ``str`` exactly as the generated front-end does
                        (python/mxnet/_ctypes/ndarray.py:106 ``c_str_array([str(s) for s in vals])``);
  * ``mxnet.base`` / ``mxnet.util`` / ``mxnet.random`` / ``mxnet.numpy``   the names imported from them.

Everything that decides WHICH operator runs with WHICH numbers -- update counts, num_update, the
scheduler call, lr / wd multipliers by index or name, the default wd_mult of non-weights, Adam's
bias-corrected step size in python double, SGD's aggregation into multi_* calls, mixed precision
states, LARS's layer split, Updater's state handling -- is the reference's code, untouched.

Used by tests/test_reference_python.py to pin (a) kvoracle.LocalKVStoreModel and (b) the mirror
under tests/compat/ to it, and by oracle/gen_golden.py to write tests/golden/updater_trajectories.npz
(the reference Python cannot travel to the GPU box; the fixture does).
"""
import contextlib
import importlib.util
import os
import sys
import types

import numpy as np

import kvoracle as K

_TREE = K.reference_tree()
REF_PY = os.path.join(_TREE, "python", "mxnet") if _TREE else None


def available():
    r = K.ref()
    return REF_PY is not None and os.path.isfile(os.path.join(REF_PY, "optimizer", "optimizer.py")) and \
        r is not None and r.has_ops()


class Context(object):
    def __init__(self, device_id=0, device_type='cpu'):
        self.device_id, self.device_type = device_id, device_type

    def __eq__(self, other):
        return (self.device_id, self.device_type) == (other.device_id, other.device_type)

    def __hash__(self):
        return hash((self.device_id, self.device_type))


class NDArray(object):
    """numpy-backed stand-in for mx.nd.NDArray: a buffer the operators update in place"""

    def __init__(self, data, ctx=None):
        self.a = data if isinstance(data, np.ndarray) else np.asarray(data)
        self.context = ctx or Context()

    stype = 'default'
    dtype = property(lambda self: self.a.dtype.type)
    shape = property(lambda self: self.a.shape)
    size = property(lambda self: self.a.size)

    def astype(self, dtype, copy=True):
        return NDArray(self.a.astype(np.dtype(dtype)), self.context)

    def asnumpy(self):
        return self.a.copy()

    def as_in_context(self, ctx):
        self.context = ctx
        return self

    def copy(self):
        return NDArray(self.a.copy(), self.context)

    def __len__(self):
        return len(self.a)

    def __getitem__(self, key):
        return NDArray(self.a[key], self.context)          # slices share the buffer, as mx.nd slices do

    def __setitem__(self, key, value):
        self.a[key] = value.a if isinstance(value, NDArray) else value

    def __mul__(self, scalar):
        # NDArray * python scalar -> _mul_scalar(scalar=str(scalar)): the scalar goes through dmlc::stof
        LOG.append(('_mul_scalar', {'scalar': str(scalar)}))
        s = np.float32(_stof(repr(float(scalar))))
        return NDArray((self.a * s).astype(self.a.dtype), self.context)

    def __iadd__(self, other):
        self.a += other.a
        return self

    def __getstate__(self):
        return {'a': self.a, 'ctx': (self.context.device_id, self.context.device_type)}

    def __setstate__(self, st):
        self.a, self.context = st['a'], Context(*st['ctx'])


def zeros(shape, ctx=None, dtype=None, stype=None, **_):
    assert stype in (None, 'default')
    return NDArray(np.zeros(shape, np.float32 if dtype is None else np.dtype(dtype)), ctx)


def array(source, ctx=None, dtype=None):
    return NDArray(np.array(source, np.float32 if dtype is None else np.dtype(dtype)), ctx)


def cast(data, dtype, out=None):
    """Cast: float32 -> float16 goes through mshadow's half_t constructor (round to nearest even)"""
    res = K.get_oracle().to_half(data.a, 1).view(np.float16).reshape(data.a.shape) \
        if (np.dtype(dtype) == np.float16 and data.a.dtype == np.float32) else data.a.astype(np.dtype(dtype))
    if out is None:
        return NDArray(res, data.context)
    out.a[...] = res
    return out


LOG = []          # (operator, {parameter: string}) of every call, in order -- compared between front-ends

# what runs the operators and parses scalar parameters: the reference's own code (oracle/_ref) unless
# use_oracle_ops() switched to the plain-C restatement (golden_ops.OracleOps, kvoracle.dmlc_stof)
_OPS = {}


def use_oracle_ops(on=True):
    _OPS.clear()
    if on:
        import golden_ops
        _OPS.update(invoke=golden_ops.OracleOps().invoke, stof=K.dmlc_stof)


def _op_invoke(*args, **params):
    return (_OPS.get('invoke') or K.ref().op_invoke)(*args, **params)


def _stof(text):
    return (_OPS.get('stof') or K.ref().dmlc_stof)(text)


def _flat(x):
    out = []
    for v in x:
        out.extend(_flat(v) if isinstance(v, (list, tuple)) else [v])
    return out


def _invoke(name, args, out, kwargs, new_out=None):
    views = {}

    def view(a):                 # an array both read and written is one and the same view
        return views.setdefault(id(a), a.a.reshape(-1))
    ins = [view(a) for a in _flat(args)]
    params = {k: v for k, v in kwargs.items()}
    LOG.append((name, {k: str(v) for k, v in params.items()}))
    if out is None:
        out = new_out(ins, params)
    outs = _flat([out])
    _op_invoke(name, ins, [view(o) for o in outs], **params)
    return out


def _update_op(name, internal=None):
    def op(*args, **kwargs):
        out = kwargs.pop('out')
        kwargs.pop('name', None)
        return _invoke(internal or name, args, out, kwargs)
    op.__name__ = name
    return op


def multi_sum_sq(*arrays, **kwargs):
    return _invoke('multi_sum_sq', arrays, kwargs.pop('out', None), kwargs,
                   lambda ins, p: NDArray(np.zeros(len(ins), np.float32), arrays[0].context))


def multi_lars(lrs, w_sum_sq, g_sum_sq, wds, **kwargs):
    return _invoke('multi_lars', (lrs, w_sum_sq, g_sum_sq, wds), kwargs.pop('out', None), kwargs,
                   lambda ins, p: NDArray(np.zeros_like(ins[0]), lrs.context))


def lamb_phase1(name):
    def op(*args, **kwargs):
        return _invoke(name, args, kwargs.pop('out', None), kwargs,
                       lambda ins, p: NDArray(np.zeros(args[0].shape, np.float32), args[0].context))
    return op


def multi_lamb_update(weights, grads, mean, var, step_count, lrs, wds, out=None, num_tensors=0, **kwargs):
    """python/mxnet/ndarray/contrib.py:609-644: flatten (w, g, mean, var) per tensor, num_tensors =
    len(weights), call _multi_lamb_update with learning_rates / wds / step_count"""
    if not num_tensors:
        num_tensors = len(weights)
    temp = _flat(zip(weights, grads, mean, var))
    return _invoke('_multi_lamb_update', temp, out, dict(num_tensors=num_tensors, learning_rates=lrs,
                                                          wds=wds, step_count=step_count, **kwargs))


def multi_mp_lamb_update(weights, grads, mean, var, weights32, step_count, lrs, wds, out=None,
                         num_tensors=0, **kwargs):
    """python/mxnet/ndarray/contrib.py:646-684"""
    if not num_tensors:
        num_tensors = len(weights)
    temp = _flat(zip(weights, grads, mean, var, weights32))
    return _invoke('_multi_mp_lamb_update', temp, out, dict(num_tensors=num_tensors, learning_rates=lrs,
                                                             wds=wds, step_count=step_count, **kwargs))


_UPDATE_OPS = ['sgd_update', 'sgd_mom_update', 'mp_sgd_update', 'mp_sgd_mom_update', 'multi_sgd_update',
               'multi_sgd_mom_update', 'multi_mp_sgd_update', 'multi_mp_sgd_mom_update', 'adam_update',
               'preloaded_multi_sgd_update', 'preloaded_multi_sgd_mom_update',
               'preloaded_multi_mp_sgd_update', 'preloaded_multi_mp_sgd_mom_update',
               'lamb_update_phase2', 'mp_lamb_update_phase2']
# imported by optimizer.py but belonging to optimizers outside the KVStore path's scope
_UNUSED = ['clip', 'sqrt', 'maximum', 'abs', 'multiply', 'norm', 'rmsprop_update', 'rmspropalex_update',
           'square', 'ftrl_update', 'ftml_update', 'signsgd_update', 'signum_update', 'nag_mom_update',
           'mp_nag_mom_update']


def op_table():
    """name -> callable for every operator / helper the front-end uses"""
    t = {n: _update_op(n) for n in _UPDATE_OPS}
    t.update(NDArray=NDArray, zeros=zeros, array=array, cast=cast, multi_sum_sq=multi_sum_sq,
             multi_lars=multi_lars, lamb_update_phase1=lamb_phase1('lamb_update_phase1'),
             mp_lamb_update_phase1=lamb_phase1('mp_lamb_update_phase1'))
    return t


def _unused(name):
    def f(*a, **k):
        raise NotImplementedError("%s is outside the harness" % name)
    return f


def _stub_modules():
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m
    nd = mod('mxnet.ndarray', **op_table())
    for n in _UNUSED:
        setattr(nd, n, _unused(n))
    nd.contrib = mod('mxnet.ndarray.contrib', multi_lamb_update=multi_lamb_update,
                     multi_mp_lamb_update=multi_mp_lamb_update)
    nd.sparse = mod('mxnet.ndarray.sparse')
    root = mod('mxnet')
    root.__path__ = []
    pkg = mod('mxnet.optimizer')
    pkg.__path__ = [os.path.join(REF_PY, 'optimizer')]
    mods = {
        'mxnet': root, 'mxnet.optimizer': pkg, 'mxnet.ndarray': nd, 'mxnet.ndarray.contrib': nd.contrib,
        'mxnet.ndarray.sparse': nd.sparse,
        'mxnet.base': mod('mxnet.base', py_str=lambda b: b.decode('utf-8')),
        'mxnet.random': mod('mxnet.random', normal=_unused('normal')),
        'mxnet.util': mod('mxnet.util', is_np_array=lambda: False),
        'mxnet.numpy': mod('mxnet.numpy', ndarray=type('ndarray', (), {})),
    }
    root.ndarray, root.optimizer = nd, pkg
    return mods


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


@contextlib.contextmanager
def reference_python():
    """with reference_python() as (opt, sched): opt = the reference's optimizer module, sched = its
    lr_scheduler module. The stand-in `mxnet.*` entries live in sys.modules only inside the block
    (Updater.__call__ imports ..numpy lazily), so nothing else in the process ever sees them."""
    assert available(), "needs the reference tree (kvoracle.reference_tree) and oracle/_ref/libmxref.so"
    saved = {k: v for k, v in sys.modules.items() if k == 'mxnet' or k.startswith('mxnet.')}
    for k in saved:
        del sys.modules[k]
    sys.modules.update(_stub_modules())
    try:
        sched = _load('mxnet.lr_scheduler', os.path.join(REF_PY, 'lr_scheduler.py'))
        opt = _load('mxnet.optimizer.optimizer', os.path.join(REF_PY, 'optimizer', 'optimizer.py'))
        yield opt, sched
    finally:
        for k in [k for k in sys.modules if k == 'mxnet' or k.startswith('mxnet.')]:
            del sys.modules[k]
        sys.modules.update(saved)

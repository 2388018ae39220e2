"""CPU-only checks of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/b200kv_c_api.h declares, fails loudly without a GPU (no CPU fallback), and its host-only
pieces (chunk planner, plugin registry, front-end bookkeeping) behave."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope="module")
def mx():
    import anand_mxnet_b200 as mx
    return mx


def test_library_exports_every_declared_symbol(mx):
    hdr = open(os.path.join(ROOT, "include", "b200kv_c_api.h")).read()
    names = set(re.findall(r"B200KV_DLL\s+[\w\s\*]+?\b((?:MX|NN|B200KV)\w+)\s*\(", hdr))
    assert len(names) > 70, len(names)
    # the KVStore entry points of the reference's C API that python/mxnet/kvstore/kvstore.py binds
    for required in ("MXKVStoreCreate", "MXKVStoreFree", "MXKVStoreInit", "MXKVStoreInitEx",
                     "MXKVStorePush", "MXKVStorePushEx", "MXKVStorePullWithSparse",
                     "MXKVStorePullWithSparseEx", "MXKVStorePushPull", "MXKVStorePushPullEx",
                     "MXKVStorePullRowSparse", "MXKVStorePullRowSparseEx", "MXKVStoreSetUpdaterEx",
                     "MXKVStoreSetGradientCompression", "MXKVStoreGetType", "MXKVStoreGetRank",
                     "MXKVStoreGetGroupSize", "MXKVStoreIsWorkerNode", "MXKVStoreBarrier",
                     "MXKVStoreSendCommmandToServers", "MXGetLastError"):
        assert required in names
    lib = ctypes.CDLL(os.path.join(ROOT, "anand_mxnet_b200", "libb200kv.so"))
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
def test_fails_loudly_without_gpu(mx):
    with pytest.raises(mx.MXNetError, match="no CPU fallback"):
        mx.kv.create('device')
    with pytest.raises(mx.MXNetError, match="needs a CUDA device"):
        mx.nd.zeros((2, 2))


def test_error_convention(mx):
    lib = mx.base._LIB
    h = ctypes.c_void_p()
    assert lib.NNGetOpHandle(b"Convolution", ctypes.byref(h)) == -1
    assert b"not registered" in lib.MXGetLastError()
    assert lib.NNGetOpHandle(b"sgd_mom_update", ctypes.byref(h)) == 0
    v = ctypes.c_int()
    assert lib.MXGetVersion(ctypes.byref(v)) == 0 and v.value == 10600
    for fn in (lib.MXKVStoreIsWorkerNode, lib.MXKVStoreIsServerNode, lib.MXKVStoreIsSchedulerNode):
        assert fn(ctypes.byref(v)) == 0
    assert lib.MXKVStoreIsWorkerNode(ctypes.byref(v)) == 0 and v.value == 1


def test_chunk_planner(mx):
    """Host-only planner: every element of every key lands in exactly one chunk of <= 4096
    elements; stripes of 32768 elements rotate over the devices; balance within one stripe/key."""
    from bench import resnet50_shapes, bert_base_shapes
    lib = mx.base._LIB
    for shapes in (resnet50_shapes(), bert_base_shapes(), [(3,), (1,), (4097,), (32768 * 3 + 5,)]):
        sizes = [int(np.prod(s)) for s in shapes]
        arr = (ctypes.c_uint64 * len(sizes))(*sizes)
        for ndev in (1, 2, 4, 8):
            counts = (ctypes.c_uint64 * ndev)()
            elems = (ctypes.c_uint64 * ndev)()
            assert lib.B200KVTestPlanChunks(arr, len(sizes), ndev, counts, elems) == 0
            assert sum(elems) == sum(sizes)
            if sum(sizes) > 64 * 32768 * ndev:
                share = sum(sizes) / ndev
                assert max(elems) - min(elems) <= 0.05 * share, (ndev, list(elems))


def test_registry_and_teststore(mx):
    # python/mxnet/kvstore/base.py:221-245,441-455: registry first, native factory otherwise
    @mx.kv.KVStoreBase.register
    class MyStore(mx.kv.KVStoreBase):
        pass
    assert isinstance(mx.kv.create('MyStore'), MyStore)
    assert mx.kv.create('teststore').type == 'teststore'
    assert mx.kv.TestStore.is_capable('optimizer') is False
    assert mx.kv.KVStore.is_capable('optimizer') is True
    with pytest.raises(TypeError):
        mx.kv.create(3)


def test_optimizer_bookkeeping(mx):
    """the hyper-parameter record kv.set_optimizer takes: per-parameter lr / wd multipliers with the
    reference's lookup order (optimizer.py:432-509), no device work involved."""
    opt = mx.optimizer.SGD(learning_rate=0.1, wd=0.01, param_idx2name={0: 'fc_weight', 1: 'fc_bias'})
    opt.set_lr_mult({'fc_bias': 2.0})
    assert opt.multipliers(0) == (1.0, 1.0)
    assert opt.multipliers(1) == (2.0, 0.0)            # biases get wd_mult 0 by name
    opt.set_wd_mult({1: 0.5})                            # an index entry beats the name rule
    assert opt.multipliers(1) == (2.0, 0.5)

    class P(object):
        lr_mult, wd_mult = 3.0, 4.0
    opt.param_dict = {0: P()}                            # a Parameter object beats both tables
    assert opt.multipliers(0) == (3.0, 4.0)
    adam = mx.optimizer.create('adam', learning_rate=3e-4)
    assert adam.lr == 3e-4 and adam.kind == 'adam' and adam.beta2 == 0.999
    assert adam.op_params()['epsilon'] == 1e-8 and mx.optimizer.fused_kind(adam) == 'adam'
    with pytest.raises(ValueError):
        mx.optimizer.create('lars')                      # no fused kernel: callback route only
    with pytest.raises(TypeError):
        mx.optimizer.get_updater(opt)                    # a record carries no update rule


def test_optimizer_record_rules(mx):
    """the rest of the record's contract: defaults, scheduler handling, objects of the reference's
    classes (tests/compat mirror) read as records, pickling without Parameter objects"""
    import pickle
    from compat import mxnet_optimizer as mxopt

    class Sched(object):
        base_lr = 0.5

        def __call__(self, num_update):
            return self.base_lr / (1 + num_update)
    sgd = mx.optimizer.SGD(lr_scheduler=Sched(), momentum=0.9)
    assert sgd.lr is None and sgd.learning_rate == 0.5          # the scheduler supplies the rate
    sgd.num_update = 4
    assert sgd.learning_rate == 0.1
    with pytest.raises(UserWarning):
        sgd.set_learning_rate(0.3)                              # optimizer.py:356-365
    s2 = Sched()
    explicit = mx.optimizer.SGD(learning_rate=0.2, lr_scheduler=s2)
    assert s2.base_lr == 0.2 and explicit.lr == 0.2             # an explicit rate wins (optimizer.py:117-123)
    with pytest.raises(TypeError):
        mx.optimizer.SGD(beta1=0.9)                              # not an SGD parameter
    p = mx.optimizer.Adam(clip_gradient=None, wd=0.01).op_params()
    assert p['clip_gradient'] == 0.0 and p['wd'] == 0.01 and p['lazy_update'] is True
    assert set(mx.optimizer.Test().op_params()) == {'learning_rate', 'wd', 'rescale_grad', 'clip_gradient',
                                                    'multi_precision', 'begin_num_update'}
    # an object of the reference's SGD class is recognised by class name + attributes ...
    ref_sgd = mxopt.SGD(learning_rate=0.05, momentum=0.8, wd=1e-3, param_idx2name={0: 'a_weight', 1: 'a_bias'})
    assert mx.optimizer.fused_kind(ref_sgd) == 'sgd'
    rec = mx.optimizer.record_of(ref_sgd)
    assert rec.kind == 'sgd' and rec.momentum == 0.8 and rec.multipliers(1) == (1.0, 0.0)
    assert rec.op_params()['learning_rate'] == 0.05
    # ... one of another class is not (callback route), and get_updater wraps its own update rule
    lars = mxopt.LARS(learning_rate=0.1)
    assert mx.optimizer.fused_kind(lars) is None
    upd = mx.optimizer.get_updater(lars)
    assert upd.optimizer is lars and upd.states == {}
    # Parameter objects do not travel with a pickled record (optimizer.py:512-519)

    class P(object):
        lr_mult, wd_mult = 2.0, 3.0
    adam = mx.optimizer.Adam(param_dict={7: P()})
    assert adam.multipliers(7) == (2.0, 3.0)
    back = pickle.loads(pickle.dumps(adam))
    assert back.param_dict == {} and back.kind == 'adam' and back.beta1 == 0.9
    # the callback updater's pickle: {index: state}, or (states, optimizer)
    upd.states = {3: None}
    assert pickle.loads(upd.get_states()) == {3: None}
    st, opt = pickle.loads(upd.get_states(dump_optimizer=True))
    assert st == {3: None} and type(opt).__name__ == 'LARS'


# ---------------------------------------------------------------- drop-in boundary: signatures
# headers of the reference's source tree, read only while its results are recorded (oracle/refrecord.py)
_REF_HEADERS = [("include/mxnet/c_api.h", "MXNET_DLL"), ("3rdparty/tvm/nnvm/include/nnvm/c_api.h", "NNVM_DLL")]
_BASE = {'int', 'char', 'void', 'float', 'double', 'size_t', 'bool', 'uint32_t', 'int64_t', 'uint64_t', 'unsigned',
         'const', 'int32_t', 'uint8_t'}


def _c_declarations(path, macro):
    """{function: (return type tokens, [parameter type tokens])} and {typedef: tokens} of a C header;
    parameter names, comments, whitespace and DEFAULT(...) default arguments dropped"""
    import re
    txt = open(path).read()
    txt = re.sub(r'/\*.*?\*/', ' ', txt, flags=re.S)
    txt = re.sub(r'//[^\n]*', ' ', txt)
    txt = re.sub(r'DEFAULT\([^)]*\)', ' ', txt)
    typedefs = {m.group(2): re.findall(r'\w+|\*', m.group(1))
                for m in re.finditer(r'typedef\s+([\w\s\*]+?)\s*\b(\w+)\s*;', txt)}

    def split(a):
        parts, depth, cur = [], 0, ''
        for ch in a:
            depth += (ch == '(') - (ch == ')')
            if ch == ',' and depth == 0:
                parts.append(cur)
                cur = ''
            else:
                cur += ch
        return parts + [cur]

    def param(p):
        if '(' in p:                          # function-pointer parameter: compare its text without names
            return [re.sub(r'\s+', '', re.sub(r'\b\w+\s*(?=[,)])', '', p))]
        toks = re.findall(r'\w+|\*|\[\]', p)
        if toks[-1] == '[]':
            toks = toks[:-2] + ['*']          # T name[]  ==  T* name
        elif len(toks) >= 2 and toks[-1] != '*' and toks[-1] not in _BASE and toks[-1] not in typedefs \
                and not toks[-1][0].isupper():
            toks = toks[:-1]                  # trailing identifier = the parameter's name
        return toks
    # function-type typedefs (callbacks): "typedef void (Name)(params);" / "typedef void (*Name)(params);"
    for m in re.finditer(r'typedef\s+([\w\s\*]+?)\(\s*(\*?)\s*(\w+)\s*\)\s*\(([^;]*?)\)\s*;', txt, flags=re.S):
        typedefs[m.group(3)] = ['fn' + m.group(2)] + re.findall(r'\w+|\*', m.group(1)) + \
            ['('] + [x for a in split(m.group(4)) for x in param(a.strip()) + [',']] + [')']
    fns = {}
    for m in re.finditer(macro + r'\s+([\w\s\*]+?)\b(\w+)\s*\(([^;{]*?)\)\s*;', txt, flags=re.S):
        args = m.group(3).strip()
        fns[m.group(2)] = (re.findall(r'\w+|\*', m.group(1)),
                           [] if args in ('', 'void') else [param(a.strip()) for a in split(args)])
    return fns, typedefs


def _resolve(toks, typedefs):
    out = []
    for t in toks:
        t = {'mx_uint': 'uint32_t', 'mx_float': 'float', 'unsigned': 'uint32_t'}.get(t, t)
        seen = set()
        while t in typedefs and t not in seen and len(typedefs[t]) <= 3:
            seen.add(t)
            sub = [x for x in typedefs[t]]
            if len(sub) == 1:
                t = sub[0]
                continue
            out.extend(_resolve(sub[:-1], typedefs))
            t = sub[-1]
        out.append(t)
    return out


def test_signatures_match_reference_headers():
    """every MX* / NN* function include/b200kv_c_api.h declares has, type for type, the signature the
    reference declares in include/mxnet/c_api.h (or nnvm/c_api.h): return type, parameter count, every
    parameter's type after resolving the handle typedefs -- so a binding written against the
    reference's header binds libb200kv.so unchanged"""
    import refrecord as R
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    mine, my_td = _c_declarations(os.path.join(root, "include", "b200kv_c_api.h"), "B200KV_DLL")
    names = sorted(n for n in mine if not n.startswith("B200KV"))     # B200KV*: extensions, no counterpart
    callbacks = ("MXKVStoreUpdater", "MXKVStoreStrUpdater", "MXKVStoreServerController", "EngineAsyncFunc",
                 "EngineSyncFunc", "EngineFuncParamDeleter")

    def signatures(fns, td):
        """function -> digest of (resolved return type, resolved parameter types)"""
        out = {n: R.digest_json([_resolve(ret, td), [_resolve(a, td) for a in params]])
               for n, (ret, params) in fns.items()}
        for cb in callbacks:                   # the callback types those functions take
            out[cb] = R.digest_json([td[cb][0], _resolve(td[cb][1:], {k: v for k, v in td.items() if k != cb})])
        return out

    def reference(_):
        ref, ref_td = {}, {}
        for path, macro in _REF_HEADERS:
            f, t = _c_declarations(os.path.join(R.tree(), path), macro)
            ref.update(f)
            ref_td.update(t)
        return signatures(ref, ref_td)
    want = R.reference("test_abi::signatures", reference)
    got = signatures(mine, my_td)
    for name in names:
        assert name in want, "%s is not a function of the reference's C API" % name
        assert got[name] == want[name], "%s: return or parameter types differ from the reference's %s" % (
            name, mine[name])
    assert len(names) >= 60
    for cb in callbacks:
        assert my_td[cb][0].startswith('fn') and got[cb] == want[cb], "callback type %s differs: %s" % (
            cb, my_td[cb])


def test_python_kvstore_surface_matches_reference():
    """boundary B1: every method / property of the reference's python KVStore and KVStoreBase classes
    (python/mxnet/kvstore/{kvstore,base}.py, parsed, not imported) exists on this package's classes
    with the same parameter names, defaults and decorators"""
    import ast

    def methods(path, cls):
        out = {}
        for node in ast.parse(open(path).read()).body:
            if isinstance(node, ast.ClassDef) and node.name == cls:
                for f in node.body:
                    if isinstance(f, ast.FunctionDef):
                        out[f.name] = ([a.arg for a in f.args.args], [ast.unparse(d) for d in f.args.defaults],
                                       [ast.unparse(d) for d in f.decorator_list])
        return out
    import refrecord as R
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = (("kvstore.py", "KVStore"), ("base.py", "KVStoreBase"))
    # the reference's methods: name -> digest of (parameter names, defaults, decorators)
    want = R.reference("test_abi::python_kvstore_surface", lambda _: {
        cls: {n: R.digest_json(sig) for n, sig in methods(os.path.join(R.tree(), "python/mxnet/kvstore", fname), cls).items()}
        for fname, cls in files})
    total = 0
    for fname, cls in files:
        mine = methods(os.path.join(root, "anand_mxnet_b200", "kvstore", fname), cls)
        assert len(want[cls]) >= 10
        for name, sig in want[cls].items():
            assert name in mine, "%s.%s is missing" % (cls, name)
            assert R.digest_json(list(mine[name])) == sig, \
                "%s.%s: parameters, defaults or decorators differ from the reference's: %s" % (cls, name, mine[name])
            total += 1
    assert total >= 25


def test_key_value_marshalling_vs_reference(mx):
    """kvstore/base.py:_ctype_key_value here is a one-pass rewrite of the reference's recursive helper
    (python/mxnet/kvstore/base.py:33-65). The reference's function -- and the ctypes helpers it uses
    from python/mxnet/base.py -- are compiled from their source text at run time (ast; nothing is
    imported, libmxnet is not needed) and both are fed the same keys / values: same C key array, same
    handle order, same str-key flag, same refusals. What the reference's function returned is stored
    by oracle/refrecord.py, handles as their position in the list of arrays fed to it."""
    import ast
    import ctypes
    from array import array
    import refrecord as R
    from anand_mxnet_b200.base import _LIB
    from anand_mxnet_b200.kvstore.base import _ctype_key_value as mine
    from anand_mxnet_b200.ndarray import NDArray

    def functions(path, names):
        found = {}
        for n in ast.walk(ast.parse(open(path).read())):
            if isinstance(n, ast.FunctionDef) and n.name in names and n.col_offset <= 4:
                if n.name not in found or n.lineno > found[n.name].lineno:
                    found[n.name] = n            # python-2 / python-3 twins: the later one is python 3's
        assert sorted(found) == sorted(names), (path, names)
        return ast.Module(body=sorted(found.values(), key=lambda n: n.lineno), type_ignores=[])

    def reference_helper():
        ns = {'ctypes': ctypes, 'array': array, 'NDArray': NDArray, 'string_types': (str,),
              'py_str': lambda b: b.decode()}
        exec(compile(functions(os.path.join(R.tree(), "python/mxnet/base.py"),
                               ['c_str', 'c_str_array', 'c_array', 'c_array_buf', 'c_handle_array']),
                     "reference base.py", "exec"), ns)
        exec(compile(functions(os.path.join(R.tree(), "python/mxnet/kvstore/base.py"), ['_ctype_key_value']),
                     "reference kvstore/base.py", "exec"), ns)
        return ns['_ctype_key_value']

    def nd():
        h = ctypes.c_void_p()
        assert _LIB.MXNDArrayCreateNone(ctypes.byref(h)) == 0        # an empty handle: no device needed
        return NDArray(h)
    a = [nd() for _ in range(12)]
    pos = {x.handle.value: i for i, x in enumerate(a)}

    def flat(res):
        keys, handles, use_str = res
        ks = [k.decode() if isinstance(k, bytes) else int(k) for k in keys]
        hs = [h if isinstance(h, int) else ctypes.cast(h, ctypes.c_void_p).value for h in handles]
        return [ks, [pos[h] for h in hs], bool(use_str)]
    cases = [
        (3, a[0]), ('w', a[0]), (3, [a[0], a[1], a[2]]), ('w', (a[0], a[1])),
        ([1, 2, 3], [a[0], a[1], a[2]]), (['a', 'b'], [a[0], a[1]]), ((5, 4), (a[0], a[1])),
        ([1, 2], [[a[0], a[1]], [a[2], a[3]]]), (['x', 'y'], [[a[0]], [a[1], a[2], a[3]]]),
        ([7, 7, 8], [a[0], a[1], a[2]]),                                  # duplicate keys = several devices
        ([1, 2, 3], [a[0], [a[1], a[2]], a[3]]),                          # mixed nesting
        ([9, 3, 5], [[a[0], a[1]], a[2], [a[3]]]),
        ([], []), ([4], [[]]),
        (list(range(157)), [[a[i % 12], a[(i + 1) % 12]] for i in range(157)]),
    ]
    # and what the reference refuses
    refused = [([1, 'a'], [a[0], a[1]]), ([1, 2], [a[0]]), (1.5, a[0]), ([1.5], [a[0]]),
               (['a', 2], [[a[0]], [a[1]]])]

    def run(fn):
        def refuses(keys, vals):
            try:
                fn(keys, vals)
            except AssertionError:
                return True
            return False
        return [flat(fn(keys, vals)) for keys, vals in cases], [refuses(k, v) for k, v in refused]
    want = R.reference("test_abi::ctype_key_value", lambda _: run(reference_helper()))
    got = run(mine)
    for i, (case, g, w) in enumerate(zip(cases, got[0], want[0])):
        assert g == w, "case %d, keys %r: got %r, the reference returned %r" % (i, case[0], g, w)
    assert want[1] == [True] * len(refused) and got[1] == want[1]

"""TEST INFRASTRUCTURE ONLY -- numpy front-end of the CPU oracle (oracle/kvoracle.c) and of the
reference harness (oracle/_ref/libmxref.so, built from the reference's own headers).

Importers allowed: tests/, __graft_entry__.smoke(), bench.py's cpu_baseline / --impl reference legs.
The product package (anand_mxnet_b200) never imports this module.

Two objects are exported:
  * ``oracle``  -- the plain-C restatement (always available; built on demand with gcc)
  * ``ref()``   -- the reference harness or ``None`` when oracle/_ref/libmxref.so is absent

plus a pure-numpy restatement of the host orchestration the reference performs around the
arithmetic (key grouping, update counts, lr/wd multipliers, Adam bias correction), each citing the
reference file:line it follows.
"""
import ctypes
import math
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_F = ctypes.c_float
_P = ctypes.c_void_p
_SZ = ctypes.c_size_t
_I = ctypes.c_int


def build(ref=True):
    """Compile oracle/libkvoracle.so (and oracle/_ref/libmxref.so when /root/reference exists)."""
    subprocess.run(["make", "-s", "-C", _HERE, "oracle"], check=True)
    if ref and os.path.isdir("/root/reference/src/kvstore"):
        subprocess.run(["make", "-s", "-C", _HERE, "ref"], check=True)


def reference_tree():
    """The reference's source tree: $B200KV_REFERENCE_TREE, else the tree oracle/_ref/libmxref.so was
    built from (`make ref` records it); None when neither names a tree that exists here."""
    t = os.environ.get("B200KV_REFERENCE_TREE")
    if not t:
        try:
            with open(os.path.join(_HERE, "_ref", "reference_tree")) as f:
                t = f.read().strip()
        except OSError:
            return None
    return t if os.path.isdir(os.path.join(t, "src", "kvstore")) else None


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr_array(arrs):
    return (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])


class Oracle(object):
    """numpy API over oracle/libkvoracle.so (the plain-C restatement)."""

    def __init__(self):
        path = os.path.join(_HERE, "libkvoracle.so")
        src = os.path.join(_HERE, "kvoracle.c")
        if (not os.path.exists(path)) or os.path.getmtime(path) < os.path.getmtime(src):
            build(ref=False)
        self.lib = ctypes.CDLL(path)
        L = self.lib
        L.kvo_half_to_float.restype = _F
        L.kvo_half_to_float.argtypes = [ctypes.c_uint16, _I]
        L.kvo_float_to_half.restype = ctypes.c_uint16
        L.kvo_float_to_half.argtypes = [_F, _I]
        L.kvo_unique_i64.restype = _SZ
        L.kvo_rsp_reduce.restype = _SZ
        L.kvo_reduce_local.argtypes = [_P, _I, _SZ, _P, _I]
        L.kvo_reduce_device.argtypes = [_P, _I, _SZ, _P, _I]
        L.kvo_sgd_update.argtypes = [_SZ, _P, _P, _P, _F, _F, _F, _F, _I]
        L.kvo_sgd_mom_update.argtypes = [_SZ, _P, _P, _P, _P, _F, _F, _F, _F, _F, _I]
        L.kvo_multi_sgd_update.argtypes = [_SZ, _P, _P, _P, _P, _F, _F, _F, _F, _F, _I]
        L.kvo_adam_update.argtypes = [_SZ, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _F, _F, _I]
        L.kvo_test_update.argtypes = [_SZ, _P, _P, _P, _F, _I]
        L.kvo_mp_sgd_update.argtypes = [_SZ, _P, _P, _P, _I, _F, _F, _F, _F, _I]
        L.kvo_mp_sgd_mom_update.argtypes = [_SZ, _P, _P, _P, _P, _I, _F, _F, _F, _F, _F, _I]
        L.kvo_multi_mp_sgd_update.argtypes = [_SZ, _P, _P, _P, _P, _I, _F, _F, _F, _F, _F, _I]
        L.kvo_unique_i64.argtypes = [_P, _SZ]
        L.kvo_rsp_reduce.argtypes = [_I, _P, _P, _P, _SZ, _P, _P]
        L.kvo_sparse_retain.argtypes = [_P, _SZ, _P, _SZ, _P, _SZ, _I, _P, _P]
        L.kvo_sgd_rsp_update.argtypes = [_SZ, _SZ, _P, _P, _P, _F, _F, _F, _F]
        L.kvo_sgd_mom_rsp_update.argtypes = [_SZ, _SZ, _P, _P, _P, _P, _F, _F, _F, _F, _F]
        L.kvo_adam_rsp_update.argtypes = [_SZ, _SZ, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _F, _F]
        L.kvo_quantize_2bit.argtypes = [_SZ, _P, _P, _P, _F]
        L.kvo_dequantize_2bit.argtypes = [_SZ, _P, _P, _F]
        L.kvo_sgd_std_rsp_update.argtypes = [_SZ, _SZ, _P, _P, _P, _SZ, _F, _F, _F, _F]
        L.kvo_sgd_mom_std_rsp_update.argtypes = [_SZ, _SZ, _P, _P, _P, _P, _SZ, _F, _F, _F, _F, _F]
        L.kvo_adam_std_rsp_update.argtypes = [_SZ, _SZ, _P, _P, _P, _P, _P, _SZ] + [_F] * 7
        L.kvo_sum_sq.restype = _F
        L.kvo_sum_sq.argtypes = [_P, _SZ, _I]
        L.kvo_multi_lars.argtypes = [_SZ, _P, _P, _P, _P, _P, _F, _F, _F]
        L.kvo_adamw_update.argtypes = [_SZ, _P, _P, _P, _P, _P] + [_F] * 8
        L.kvo_mp_adamw_update.argtypes = [_SZ, _P, _P, _P, _P, _P, _I] + [_F] * 8
        L.kvo_multi_adamw_update.argtypes = [_SZ, _P, _P, _P, _P, _I, _P, _P] + [_F] * 8
        L.kvo_lamb_phase1.argtypes = [_SZ, _P, _P, _P, _P, _P, _P, _I] + [_F] * 8 + [_I]
        L.kvo_lamb_phase2.argtypes = [_SZ, _P, _P, _I, _P, _P] + [_F] * 5
        L.kvo_multi_lamb_step1.argtypes = [_SZ, _P, _P, _P, _P, _P, _P, _I] + [_F] * 6 + [_I, _I]
        L.kvo_multi_lamb_step2.argtypes = [_SZ, _P, _P, _I, _P] + [_F] * 5

    # ---- standard (non-lazy) updates, row_sparse gradient over a dense (rows, row_len) weight ----
    def sgd_std_rsp_update(self, w, gidx, gval, lr, wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.kvo_sgd_std_rsp_update(w.shape[0], w[0].size, _ptr(w), _ptr(gidx), _ptr(gval),
                                        gidx.size, self._clip(clip), lr, wd, rescale)
        return w

    def sgd_mom_std_rsp_update(self, w, mom, gidx, gval, lr, momentum, wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.kvo_sgd_mom_std_rsp_update(w.shape[0], w[0].size, _ptr(w), _ptr(mom), _ptr(gidx),
                                            _ptr(gval), gidx.size, self._clip(clip), momentum, lr,
                                            wd, rescale)
        return w

    def adam_std_rsp_update(self, w, mean, var, gidx, gval, lr, beta1=0.9, beta2=0.999, eps=1e-8,
                            wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.kvo_adam_std_rsp_update(w.shape[0], w[0].size, _ptr(w), _ptr(mean), _ptr(var),
                                         _ptr(gidx), _ptr(gval), gidx.size, self._clip(clip), beta1,
                                         beta2, lr, wd, eps, rescale)
        return w

    # ---- multi-tensor optimizer operators (SURVEY 8f-f1); arrays are updated in place ----------
    @staticmethod
    def _kind(a):
        """-1 fp32, 0 fp16 (numpy float16 or uint16 bit patterns are both accepted as fp16)"""
        return -1 if a.dtype == np.float32 else 0

    def multi_sum_sq(self, arrays, kind=None):
        out = np.empty(len(arrays), dtype=np.float32)
        for i, a in enumerate(arrays):
            a = np.ascontiguousarray(a)
            out[i] = self.lib.kvo_sum_sq(_ptr(a), a.size, self._kind(a) if kind is None else kind)
        return out

    def multi_lars(self, lrs, w_sum_sq, g_sum_sq, wds, eta, eps, rescale_grad=1.0):
        lrs, w_sum_sq, g_sum_sq, wds = _f32(lrs), _f32(w_sum_sq), _f32(g_sum_sq), _f32(wds)
        out = np.empty_like(lrs)
        self.lib.kvo_multi_lars(lrs.size, _ptr(out), _ptr(lrs), _ptr(w_sum_sq), _ptr(g_sum_sq),
                                _ptr(wds), eta, eps, rescale_grad)
        return out

    def adamw_update(self, w, g, mean, var, rescale, lr, eta, beta1=0.9, beta2=0.999, eps=1e-8,
                     wd=0.0, clip=None):
        """_adamw_update; returns False (nothing touched) when rescale is 0 / inf / nan
        (adamw-inl.h:449-461 PrepareInputBlobs). NOTE: g is overwritten with the scaled gradient."""
        if not np.isfinite(np.float32(rescale)) or np.float32(rescale) == 0:
            return False
        self.lib.kvo_adamw_update(w.size, _ptr(w), _ptr(mean), _ptr(var), _ptr(w), _ptr(g),
                                  rescale, self._clip(clip), beta1, beta2, eta, lr, wd, eps)
        return True

    def mp_adamw_update(self, w16, g16, mean, var, w32, kind, rescale, lr, eta, beta1=0.9,
                        beta2=0.999, eps=1e-8, wd=0.0, clip=None):
        if not np.isfinite(np.float32(rescale)) or np.float32(rescale) == 0:
            return False
        self.lib.kvo_mp_adamw_update(w32.size, _ptr(w16), _ptr(mean), _ptr(var), _ptr(w32),
                                     _ptr(g16), kind, rescale, self._clip(clip), beta1, beta2, eta,
                                     lr, wd, eps)
        return True

    def multi_adamw_update(self, ws, gs, means, vars_, rescale, lrs, wds, etas, beta1=0.9,
                           beta2=0.999, eps=1e-8, clip=None, w32s=None, kind=0):
        """_multi_adamw_update (w32s None) / _multi_mp_adamw_update (ws, gs 16-bit patterns)"""
        if not np.isfinite(np.float32(rescale)) or np.float32(rescale) == 0:
            return False
        for k in range(len(ws)):
            if w32s is None:
                self.lib.kvo_multi_adamw_update(ws[k].size, _ptr(ws[k]), _ptr(gs[k]), None, None, 0,
                                                _ptr(means[k]), _ptr(vars_[k]), rescale,
                                                self._clip(clip), beta1, beta2, f32(etas[k]),
                                                f32(lrs[k]), f32(wds[k]), eps)
            else:
                self.lib.kvo_multi_adamw_update(ws[k].size, _ptr(w32s[k]), None, _ptr(ws[k]),
                                                _ptr(gs[k]), kind, _ptr(means[k]), _ptr(vars_[k]),
                                                rescale, self._clip(clip), beta1, beta2,
                                                f32(etas[k]), f32(lrs[k]), f32(wds[k]), eps)
        return True

    @staticmethod
    def beta_pow(beta, t):
        """DType(std::pow(param.beta, param.t)), optimizer_op-inl.h:1660-1661: float beta, int t ->
        double pow -> float"""
        return float(np.float32(math.pow(float(np.float32(beta)), int(t))))

    def lamb_phase1(self, w, g, mean, var, t, beta1=0.9, beta2=0.999, eps=1e-6, wd=0.0,
                    rescale=1.0, clip=None, bias_correction=True, g16=None, kind=0):
        """lamb_update_phase1 (g16 None) / mp_lamb_update_phase1 (w = fp32 master, g16 patterns)"""
        out = np.empty(w.shape, dtype=np.float32)
        self.lib.kvo_lamb_phase1(w.size, _ptr(out), _ptr(mean), _ptr(var), _ptr(w),
                                 _ptr(g) if g16 is None else None,
                                 None if g16 is None else _ptr(g16), kind, self._clip(clip),
                                 rescale, beta1, self.beta_pow(beta1, t), beta2,
                                 self.beta_pow(beta2, t), wd, eps, int(bool(bias_correction)))
        return out

    def lamb_phase2(self, w, g, r1, r2, lr, lower_bound=None, upper_bound=None, out16_kind=None):
        """lamb_update_phase2 -> new fp32 weight; with out16_kind: mp variant -> 16-bit patterns
        (w is then the fp32 master copy, which the reference leaves unchanged)"""
        lb = -1.0 if lower_bound is None else lower_bound
        ub = -1.0 if upper_bound is None else upper_bound
        if out16_kind is None:
            out = np.empty(w.shape, dtype=np.float32)
            self.lib.kvo_lamb_phase2(w.size, _ptr(out), None, 0, _ptr(w), _ptr(g), r1, r2, lr, lb, ub)
        else:
            out = np.empty(w.shape, dtype=np.uint16)
            self.lib.kvo_lamb_phase2(w.size, None, _ptr(out), out16_kind, _ptr(w), _ptr(g), r1, r2,
                                     lr, lb, ub)
        return out

    def multi_lamb_update(self, ws, gs, means, vars_, step_count, lrs, wds, beta1=0.9, beta2=0.999,
                          eps=1e-6, rescale=1.0, lower_bound=None, upper_bound=None, clip=None,
                          bias_correction=True, w32s=None, kind=0):
        """_multi_lamb_update / _multi_mp_lamb_update (multi_lamb-inl.h:268-338 orchestration:
        sum_sq(weights) -> step1 -> sum_sq(temp_g) -> step2); returns (r1_sumsq, r2_sumsq)"""
        lb = -1.0 if lower_bound is None else lower_bound
        ub = -1.0 if upper_bound is None else upper_bound
        n = len(ws)
        # MultiSumSqRun over the WEIGHT inputs (the 16-bit weights in the mp variant)
        r1 = np.array([self.lib.kvo_sum_sq(_ptr(ws[k]), ws[k].size, -1 if w32s is None else kind)
                       for k in range(n)], dtype=np.float32)
        temp = [np.empty(ws[k].size, dtype=np.float32) for k in range(n)]
        for k in range(n):
            master = ws[k] if w32s is None else w32s[k]
            self.lib.kvo_multi_lamb_step1(master.size, _ptr(temp[k]), _ptr(means[k]), _ptr(vars_[k]),
                                          _ptr(master), _ptr(gs[k]) if w32s is None else None,
                                          None if w32s is None else _ptr(gs[k]), kind,
                                          self._clip(clip), rescale, beta1, beta2, eps, f32(wds[k]),
                                          int(step_count[k]), int(bool(bias_correction)))
        r2 = np.array([self.lib.kvo_sum_sq(_ptr(temp[k]), temp[k].size, -1) for k in range(n)],
                      dtype=np.float32)
        for k in range(n):
            master = ws[k] if w32s is None else w32s[k]
            self.lib.kvo_multi_lamb_step2(master.size, _ptr(master),
                                          None if w32s is None else _ptr(ws[k]), kind, _ptr(temp[k]),
                                          float(r1[k]), float(r2[k]), f32(lrs[k]), lb, ub)
        return r1, r2

    # ---- dense reduce -------------------------------------------------------------------
    def reduce(self, srcs, order="local", nthreads=1):
        """Sum a list of equal-shape fp32 arrays in the reference's association order."""
        srcs = [_f32(s).ravel() for s in srcs]
        out = np.empty_like(srcs[0])
        fn = self.lib.kvo_reduce_local if order == "local" else self.lib.kvo_reduce_device
        fn(_ptr_array(srcs), len(srcs), srcs[0].size, _ptr(out), nthreads)
        return out

    # ---- optimizers (in place on w / states, returns w) ----------------------------------
    @staticmethod
    def _clip(c):
        return -1.0 if (c is None or c is False) else float(c)

    def sgd_update(self, w, g, lr, wd=0.0, rescale=1.0, clip=None, nthreads=1):
        self.lib.kvo_sgd_update(w.size, _ptr(w), _ptr(w), _ptr(g), self._clip(clip), lr, wd,
                                rescale, nthreads)
        return w

    def sgd_mom_update(self, w, g, mom, lr, momentum, wd=0.0, rescale=1.0, clip=None, nthreads=1):
        self.lib.kvo_sgd_mom_update(w.size, _ptr(w), _ptr(mom), _ptr(w), _ptr(g), self._clip(clip),
                                    momentum, lr, wd, rescale, nthreads)
        return w

    def multi_sgd_update(self, w, g, mom, lr, momentum=0.0, wd=0.0, rescale=1.0, clip=None,
                         nthreads=1):
        self.lib.kvo_multi_sgd_update(w.size, _ptr(w), _ptr(mom) if mom is not None else None,
                                      _ptr(w), _ptr(g), self._clip(clip), momentum, lr, wd,
                                      rescale, nthreads)
        return w

    def adam_update(self, w, g, mean, var, lr, beta1=0.9, beta2=0.999, eps=1e-8, wd=0.0,
                    rescale=1.0, clip=None, nthreads=1):
        self.lib.kvo_adam_update(w.size, _ptr(w), _ptr(mean), _ptr(var), _ptr(w), _ptr(g),
                                 self._clip(clip), rescale, beta1, beta2, lr, wd, eps, nthreads)
        return w

    def test_update(self, w, g, rescale=1.0, nthreads=1):
        self.lib.kvo_test_update(w.size, _ptr(w), _ptr(w), _ptr(g), rescale, nthreads)
        return w

    # ---- 16-bit -----------------------------------------------------------------------
    def to_half(self, a, kind):
        """fp32 -> uint16 bit patterns (kind 0 = fp16, 1 = bf16), round-to-nearest-even."""
        a = _f32(a)
        f = self.lib.kvo_float_to_half
        return np.array([f(float(x), kind) for x in a.ravel()], dtype=np.uint16).reshape(a.shape) \
            if a.size < 4096 else self._to_half_np(a, kind)

    @staticmethod
    def _to_half_np(a, kind):
        if kind == 0:
            return a.astype(np.float16).view(np.uint16)
        x = a.view(np.uint32).astype(np.uint64)
        x = x + 0x7fff + ((x >> 16) & 1)
        return (x >> 16).astype(np.uint16)

    @staticmethod
    def from_half(h, kind):
        h = np.ascontiguousarray(h, dtype=np.uint16)
        if kind == 0:
            return h.view(np.float16).astype(np.float32)
        return (h.astype(np.uint32) << 16).view(np.float32)

    def mp_sgd_update(self, w16, w32, g16, kind, lr, wd=0.0, rescale=1.0, clip=None, nthreads=1):
        self.lib.kvo_mp_sgd_update(w32.size, _ptr(w16), _ptr(w32), _ptr(g16), kind,
                                   self._clip(clip), lr, wd, rescale, nthreads)
        return w16

    def multi_mp_sgd_update(self, w16, w32, g16, mom, kind, lr, momentum=0.0, wd=0.0, rescale=1.0,
                            clip=None, nthreads=1):
        self.lib.kvo_multi_mp_sgd_update(w32.size, _ptr(w16),
                                         _ptr(mom) if mom is not None else None, _ptr(w32),
                                         _ptr(g16), kind, self._clip(clip), momentum, lr, wd,
                                         rescale, nthreads)
        return w16

    # ---- row_sparse -------------------------------------------------------------------
    def unique(self, ids):
        ids = np.ascontiguousarray(ids, dtype=np.int64).ravel().copy()
        n = self.lib.kvo_unique_i64(_ptr(ids), ids.size)
        return ids[:n]

    def rsp_reduce(self, idxs, vals):
        """idxs: list of int64 [nnr_s]; vals: list of fp32 [nnr_s, row_len] -> (idx, val)."""
        idxs = [np.ascontiguousarray(i, dtype=np.int64) for i in idxs]
        vals = _rows2d(idxs, vals)
        row_len = vals[0].shape[1]
        total = sum(len(i) for i in idxs)
        out_idx = np.empty(max(total, 1), dtype=np.int64)
        out_val = np.empty((max(total, 1), row_len), dtype=np.float32)
        nrows = (ctypes.c_size_t * len(idxs))(*[len(i) for i in idxs])
        nnr = self.lib.kvo_rsp_reduce(len(idxs), _ptr_array(idxs), nrows, _ptr_array(vals),
                                      row_len, _ptr(out_idx), _ptr(out_val))
        return out_idx[:nnr].copy(), out_val[:nnr].copy()

    def sparse_retain(self, src_idx, src_val, ids, src_dense_rows=False):
        src_idx = np.ascontiguousarray(src_idx, dtype=np.int64)
        src_val = _f32(src_val)
        src_val = src_val.reshape(src_val.shape[0], int(np.prod(src_val.shape[1:])))
        ids = np.ascontiguousarray(ids, dtype=np.int64).ravel()
        out_idx = np.empty(ids.size, dtype=np.int64)
        out_val = np.empty((ids.size, src_val.shape[1]), dtype=np.float32)
        self.lib.kvo_sparse_retain(_ptr(src_idx), src_idx.size, _ptr(src_val), src_val.shape[1],
                                   _ptr(ids), ids.size, int(bool(src_dense_rows)), _ptr(out_idx),
                                   _ptr(out_val))
        return out_idx, out_val

    def sgd_rsp_update(self, w, gidx, gval, lr, wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.kvo_sgd_rsp_update(gidx.size, w.shape[1], _ptr(w), _ptr(gidx), _ptr(gval),
                                    self._clip(clip), lr, wd, rescale)
        return w

    def sgd_mom_rsp_update(self, w, mom, gidx, gval, lr, momentum, wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.kvo_sgd_mom_rsp_update(gidx.size, w.shape[1], _ptr(w), _ptr(mom), _ptr(gidx),
                                        _ptr(gval), self._clip(clip), momentum, lr, wd, rescale)
        return w

    def adam_rsp_update(self, w, mean, var, gidx, gval, lr, beta1=0.9, beta2=0.999, eps=1e-8,
                        wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.kvo_adam_rsp_update(gidx.size, w.shape[1], _ptr(w), _ptr(mean), _ptr(var),
                                     _ptr(gidx), _ptr(gval), self._clip(clip), beta1, beta2, lr,
                                     wd, eps, rescale)
        return w

    # ---- 2-bit ------------------------------------------------------------------------
    def quantize_2bit(self, grad, residual, threshold):
        grad = _f32(grad).ravel()
        comp = np.zeros((grad.size + 15) // 16, dtype=np.uint32)
        self.lib.kvo_quantize_2bit(grad.size, _ptr(comp), _ptr(grad), _ptr(residual), threshold)
        return comp

    def dequantize_2bit(self, comp, n, threshold):
        out = np.empty(n, dtype=np.float32)
        self.lib.kvo_dequantize_2bit(n, _ptr(out), _ptr(comp), threshold)
        return out


def _rows2d(idxs, vals):
    """fp32 [nnr_s, row_len] views of the sources' rows; an empty source takes the others' row_len"""
    vals = [_f32(v) for v in vals]
    row_len = 1
    for i, v in zip(idxs, vals):
        if v.ndim >= 2:
            row_len = int(np.prod(v.shape[1:]))
            break
        if len(i):
            row_len = v.size // len(i)
            break
    return [v.reshape(len(i), row_len) for i, v in zip(idxs, vals)]


class Ref(object):
    """numpy API over oracle/_ref/libmxref.so (the reference's own code, see ref_harness.cc)."""

    def __init__(self, path):
        self.lib = ctypes.CDLL(path)
        L = self.lib
        L.mxref_reduce_sum_cpu.argtypes = [_P, _I, _SZ]
        L.mxref_reduce_sum_cpu_impl.argtypes = [_P, _I, _SZ, _I, _SZ]
        L.mxref_sgd_update.argtypes = [_SZ, _P, _P, _P, _F, _F, _F, _F, _I]
        L.mxref_sgd_mom_update.argtypes = [_SZ, _P, _P, _P, _P, _F, _F, _F, _F, _F, _I]
        L.mxref_mp_sgd_update_f16.argtypes = [_SZ, _P, _P, _P, _P, _F, _F, _F, _F, _I]
        L.mxref_mp_sgd_mom_update_f16.argtypes = [_SZ, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _I]
        L.mxref_multi_sgd_update.argtypes = [_I, _P, _P, _P, _P, _P, _P, _P, _F, _F, _F, _I]
        L.mxref_multi_mp_sgd_update_f16.argtypes = [_I, _P, _P, _P, _P, _P, _P, _P, _P, _F, _F, _F,
                                                    _I]
        L.mxref_adam_update.argtypes = [_SZ, _P, _P, _P, _P, _P, _F, _F, _F, _F, _F, _F, _F, _I]
        L.mxref_sgd_rsp_update.argtypes = [_SZ, ctypes.c_int64, _P, _P, _P, _P, _F, _F, _F, _F, _I]
        L.mxref_sgd_mom_rsp_update.argtypes = [_SZ, ctypes.c_int64, _P, _P, _P, _P, _P, _F, _F, _F,
                                               _F, _F, _I]
        L.mxref_adam_rsp_update.argtypes = [_SZ, ctypes.c_int64, _P, _P, _P, _P, _P, _P, _F, _F, _F,
                                            _F, _F, _F, _F, _I]
        L.mxref_quantize_2bit.argtypes = [_SZ, _P, _P, _P, _F, _F]
        L.mxref_dequantize_2bit.argtypes = [_SZ, _P, _P, _F, _F]
        L.mxref_dmlc_stof.restype = _F
        L.mxref_dmlc_stof.argtypes = [ctypes.c_char_p]

    @staticmethod
    def _clip(c):
        return -1.0 if (c is None or c is False) else float(c)

    _DT = {np.dtype(np.float32): 0, np.dtype(np.float64): 1, np.dtype(np.float16): 2,
           np.dtype(np.uint8): 3, np.dtype(np.int32): 4, np.dtype(np.int8): 5, np.dtype(np.int64): 6}

    def op_invoke(self, op, inputs, outputs, **params):
        """Run the reference's own FCompute<cpu> of `op` (oracle/ref_ops.cc). inputs / outputs are
        C-contiguous numpy arrays (outputs are written in place; pass the same array as input and
        output for in-place updates, as `out=weight` does). Parameters are stringified the way the
        generated Python front-end does (python/mxnet/ndarray/register.py: str(value))."""
        for a in list(inputs) + list(outputs):
            assert a.flags['C_CONTIGUOUS']
        ni, no = len(inputs), len(outputs)
        ip = (ctypes.c_void_p * ni)(*[a.ctypes.data for a in inputs])
        idt = (ctypes.c_int * ni)(*[self._DT[a.dtype] for a in inputs])
        isz = (ctypes.c_int64 * ni)(*[a.size for a in inputs])
        op_ = (ctypes.c_void_p * no)(*[a.ctypes.data for a in outputs])
        odt = (ctypes.c_int * no)(*[self._DT[a.dtype] for a in outputs])
        osz = (ctypes.c_int64 * no)(*[a.size for a in outputs])
        keys = [k.encode() for k in params]
        vals = [str(v).encode() for v in params.values()]
        ck = (ctypes.c_char_p * len(keys))(*keys)
        cv = (ctypes.c_char_p * len(vals))(*vals)
        err = ctypes.create_string_buffer(2048)
        rc = self.lib.mxref_op_invoke(op.encode(), ni, ip, idt, isz, no, op_, odt, osz, len(keys),
                                      ck, cv, err, 2048)
        if rc != 0:
            raise RuntimeError(err.value.decode(errors='replace'))

    def sgd_std_rsp_update(self, w, gidx, gval, lr, wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        f = self.lib.mxref_sgd_std_rsp_update
        f.argtypes = [ctypes.c_int64, ctypes.c_int64, _P, _P, _P, ctypes.c_int64, _F, _F, _F, _F]
        f(w.shape[0], w[0].size, _ptr(w), _ptr(gidx), _ptr(gval), gidx.size, self._clip(clip), lr, wd,
          rescale)
        return w

    def sgd_mom_std_rsp_update(self, w, mom, gidx, gval, lr, momentum, wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        f = self.lib.mxref_sgd_mom_std_rsp_update
        f.argtypes = [ctypes.c_int64, ctypes.c_int64, _P, _P, _P, _P, ctypes.c_int64, _F, _F, _F, _F, _F]
        f(w.shape[0], w[0].size, _ptr(w), _ptr(mom), _ptr(gidx), _ptr(gval), gidx.size,
          self._clip(clip), momentum, lr, wd, rescale)
        return w

    def adam_std_rsp_update(self, w, mean, var, gidx, gval, lr, beta1=0.9, beta2=0.999, eps=1e-8,
                            wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        f = self.lib.mxref_adam_std_rsp_update
        f.argtypes = [ctypes.c_int64, ctypes.c_int64, _P, _P, _P, _P, _P, ctypes.c_int64] + [_F] * 7
        f(w.shape[0], w[0].size, _ptr(w), _ptr(mean), _ptr(var), _ptr(gidx), _ptr(gval), gidx.size,
          self._clip(clip), beta1, beta2, lr, wd, eps, rescale)
        return w

    def ndarray_save(self, a, ctx=(1, 0), idx=None):
        """bytes of NDArray::Save for a dense array `a` (or a row_sparse one: a = stored rows, idx =
        their ids, shape0 = table height via a.shape0 attribute of the call) -- see ref_ops.cc"""
        raise NotImplementedError

    def ndarray_save_bytes(self, shape, data, ctx=(1, 0), idx=None):
        data = np.ascontiguousarray(data)
        shp = (ctypes.c_int64 * len(shape))(*shape)
        f = self.lib.mxref_ndarray_save
        f.restype = ctypes.c_size_t
        f.argtypes = [_I, _P, _I, _I, _I, _P, ctypes.c_size_t, ctypes.c_int64, _P, _P, ctypes.c_size_t]
        nnr = -1 if idx is None else len(idx)
        ip = None
        if idx is not None:
            idx = np.ascontiguousarray(idx, dtype=np.int64)
            ip = _ptr(idx)
        cap = 256 + data.nbytes + (0 if idx is None else idx.nbytes)
        out = ctypes.create_string_buffer(cap)
        n = f(len(shape), shp, ctx[0], ctx[1], self._DT[data.dtype], _ptr(data), data.nbytes, nnr, ip,
              out, cap)
        assert n <= cap
        return out.raw[:n]

    def has_ops(self):
        return hasattr(self.lib, 'mxref_op_invoke')

    def dmlc_stof(self, s):
        """the reference's own dmlc::stof"""
        return float(self.lib.mxref_dmlc_stof(s.encode()))

    def reduce(self, srcs, nthreads=1, bigarray_bound=1000 * 1000):
        """CommCPU 'local' reduce; the result lands in a copy of srcs[0] (reference sums in place)."""
        bufs = [_f32(s).ravel().copy() for s in srcs]
        if nthreads <= 1:
            self.lib.mxref_reduce_sum_cpu(_ptr_array(bufs), len(bufs), bufs[0].size)
        else:
            self.lib.mxref_reduce_sum_cpu_impl(_ptr_array(bufs), len(bufs), bufs[0].size, nthreads,
                                               bigarray_bound)
        return bufs[0]

    def reduce_inplace(self, bufs, nthreads, bigarray_bound=1000 * 1000):
        self.lib.mxref_reduce_sum_cpu_impl(_ptr_array(bufs), len(bufs), bufs[0].size, nthreads,
                                           bigarray_bound)

    def sgd_update(self, w, g, lr, wd=0.0, rescale=1.0, clip=None, nthreads=1):
        self.lib.mxref_sgd_update(w.size, _ptr(w), _ptr(w), _ptr(g), self._clip(clip), lr, wd,
                                  rescale, nthreads)
        return w

    def sgd_mom_update(self, w, g, mom, lr, momentum, wd=0.0, rescale=1.0, clip=None, nthreads=1):
        self.lib.mxref_sgd_mom_update(w.size, _ptr(w), _ptr(mom), _ptr(w), _ptr(g),
                                      self._clip(clip), momentum, lr, wd, rescale, nthreads)
        return w

    def multi_sgd_update(self, ws, gs, moms, lrs, wds, momentum=0.0, rescale=1.0, clip=None,
                         nthreads=1):
        n = len(ws)
        sizes = (ctypes.c_size_t * n)(*[w.size for w in ws])
        lrs_c = (ctypes.c_float * n)(*lrs)
        wds_c = (ctypes.c_float * n)(*wds)
        self.lib.mxref_multi_sgd_update(n, sizes, _ptr_array(ws), _ptr_array(gs),
                                        _ptr_array(moms) if moms is not None else None,
                                        _ptr_array(ws), lrs_c, wds_c, self._clip(clip), rescale,
                                        momentum, nthreads)
        return ws

    def multi_mp_sgd_update_f16(self, w16s, w32s, g16s, moms, lrs, wds, momentum=0.0, rescale=1.0,
                                clip=None, nthreads=1):
        n = len(w16s)
        sizes = (ctypes.c_size_t * n)(*[w.size for w in w16s])
        lrs_c = (ctypes.c_float * n)(*lrs)
        wds_c = (ctypes.c_float * n)(*wds)
        self.lib.mxref_multi_mp_sgd_update_f16(n, sizes, _ptr_array(w16s), _ptr_array(g16s),
                                               _ptr_array(moms) if moms is not None else None,
                                               _ptr_array(w32s), _ptr_array(w16s), lrs_c, wds_c,
                                               self._clip(clip), rescale, momentum, nthreads)
        return w16s

    def mp_sgd_update_f16(self, w16, w32, g16, lr, wd=0.0, rescale=1.0, clip=None, nthreads=1):
        self.lib.mxref_mp_sgd_update_f16(w16.size, _ptr(w16), _ptr(w16), _ptr(g16), _ptr(w32),
                                         self._clip(clip), lr, wd, rescale, nthreads)
        return w16

    def mp_sgd_mom_update_f16(self, w16, w32, g16, mom, lr, momentum, wd=0.0, rescale=1.0,
                              clip=None, nthreads=1):
        self.lib.mxref_mp_sgd_mom_update_f16(w16.size, _ptr(w16), _ptr(mom), _ptr(w16), _ptr(g16),
                                             _ptr(w32), self._clip(clip), momentum, lr, wd,
                                             rescale, nthreads)
        return w16

    def adam_update(self, w, g, mean, var, lr, beta1=0.9, beta2=0.999, eps=1e-8, wd=0.0,
                    rescale=1.0, clip=None, nthreads=1):
        self.lib.mxref_adam_update(w.size, _ptr(w), _ptr(mean), _ptr(var), _ptr(w), _ptr(g),
                                   self._clip(clip), rescale, beta1, beta2, lr, wd, eps, nthreads)
        return w

    def sgd_rsp_update(self, w, gidx, gval, lr, wd=0.0, rescale=1.0, clip=None, nthreads=1):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.mxref_sgd_rsp_update(gidx.size, w.shape[1], _ptr(w), _ptr(w), _ptr(gidx),
                                      _ptr(gval), self._clip(clip), lr, wd, rescale, nthreads)
        return w

    def sgd_mom_rsp_update(self, w, mom, gidx, gval, lr, momentum, wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.mxref_sgd_mom_rsp_update(gidx.size, w.shape[1], _ptr(w), _ptr(mom), _ptr(w),
                                          _ptr(gidx), _ptr(gval), self._clip(clip), momentum, lr,
                                          wd, rescale, 1)
        return w

    def adam_rsp_update(self, w, mean, var, gidx, gval, lr, beta1=0.9, beta2=0.999, eps=1e-8,
                        wd=0.0, rescale=1.0, clip=None):
        gidx = np.ascontiguousarray(gidx, dtype=np.int64)
        self.lib.mxref_adam_rsp_update(gidx.size, w.shape[1], _ptr(w), _ptr(mean), _ptr(var),
                                       _ptr(w), _ptr(gidx), _ptr(gval), self._clip(clip), beta1,
                                       beta2, lr, wd, eps, rescale, 1)
        return w

    def quantize_2bit(self, grad, residual, threshold):
        grad = _f32(grad).ravel()
        comp = np.zeros((grad.size + 15) // 16, dtype=np.float32)
        self.lib.mxref_quantize_2bit(grad.size, _ptr(comp), _ptr(grad), _ptr(residual),
                                     -1 * threshold, threshold)
        return comp.view(np.uint32)

    def dequantize_2bit(self, comp, n, threshold):
        out = np.empty(n, dtype=np.float32)
        comp = np.ascontiguousarray(comp).view(np.float32)
        self.lib.mxref_dequantize_2bit(n, _ptr(out), _ptr(comp), -1 * threshold, threshold)
        return out

    # ---- row_sparse reduce / retain / unique: the reference's own code (oracle/ref_sparse.cc) ----
    def has_sparse(self):
        return hasattr(self.lib, 'mxref_rsp_reduce')

    def rsp_reduce(self, idxs, vals, nthreads=1):
        """ElementwiseSumRsp (ndarray_function.cc:155-176); same signature as Oracle.rsp_reduce"""
        idxs = [np.ascontiguousarray(i, dtype=np.int64) for i in idxs]
        vals = _rows2d(idxs, vals)
        row_len = vals[0].shape[1]
        total = sum(len(i) for i in idxs)
        out_idx = np.empty(max(total, 1), dtype=np.int64)
        out_val = np.empty((max(total, 1), row_len), dtype=np.float32)
        nnr = (ctypes.c_int64 * len(idxs))(*[len(i) for i in idxs])
        f = self.lib.mxref_rsp_reduce
        f.restype = ctypes.c_int64
        f.argtypes = [_I, _P, _P, _P, ctypes.c_int64, _P, _P, _I]
        n = f(len(idxs), _ptr_array(idxs), nnr, _ptr_array(vals), row_len, _ptr(out_idx), _ptr(out_val),
              nthreads)
        return out_idx[:n].copy(), out_val[:n].copy()

    def sparse_retain(self, src_idx, src_val, ids, src_dense_rows=False, row_block=False, nthreads=1):
        """SparseRetainOpForwardRspImpl's kernels (sparse_retain-inl.h:121-262)"""
        src_idx = np.ascontiguousarray(src_idx, dtype=np.int64)
        src_val = _f32(src_val)
        src_val = src_val.reshape(src_val.shape[0], int(np.prod(src_val.shape[1:])))
        ids = np.ascontiguousarray(ids, dtype=np.int64).ravel()
        out_idx = np.empty(ids.size, dtype=np.int64)
        out_val = np.empty((ids.size, src_val.shape[1]), dtype=np.float32)
        f = self.lib.mxref_sparse_retain
        f.restype = None
        f.argtypes = [_P, ctypes.c_int64, _P, ctypes.c_int64, _P, ctypes.c_int64, _I, _I, _P, _P, _I]
        f(_ptr(src_idx), src_idx.size, _ptr(src_val), src_val.shape[1], _ptr(ids), ids.size,
          int(bool(src_dense_rows)), int(bool(row_block)), _ptr(out_idx), _ptr(out_val), nthreads)
        return out_idx, out_val

    def group_positions(self, keys):
        """the reference's own KVStoreLocal::GroupKVPairs (kvstore_local.h:377-407) compiled against
        this toolchain's libstdc++: (uniq keys, positions per key in the order it hands them on)"""
        keys = np.ascontiguousarray(keys, dtype=np.int32)
        n = keys.size
        uniq, counts, pos = (np.zeros(max(n, 1), np.int32) for _ in range(3))
        f = self.lib.mxref_group_kv_pairs
        f.restype = ctypes.c_int64
        f.argtypes = [ctypes.c_int64, _P, _P, _P, _P]
        g = f(n, _ptr(keys), _ptr(uniq), _ptr(counts), _ptr(pos))
        out, p = [], 0
        for c in counts[:g]:
            out.append([int(x) for x in pos[p:p + c]])
            p += c
        return [int(k) for k in uniq[:g]], out

    def unique(self, ids):
        """UniqueImpl<cpu> (kvstore_utils.cc:31-44)"""
        ids = np.ascontiguousarray(ids, dtype=np.int64).ravel().copy()
        f = self.lib.mxref_unique
        f.restype = ctypes.c_int64
        f.argtypes = [_P, ctypes.c_int64]
        n = f(_ptr(ids), ids.size)
        return ids[:n]


_oracle = None
_ref = False


def get_oracle():
    global _oracle
    if _oracle is None:
        _oracle = Oracle()
    return _oracle


def ref():
    """The reference harness, or None when oracle/_ref/libmxref.so has not been built."""
    global _ref
    if _ref is False:
        path = os.path.join(_HERE, "_ref", "libmxref.so")
        _ref = Ref(path) if os.path.exists(path) else None
    return _ref


# ------------------------------------------------------------------------------------------
# Host orchestration restated in numpy/python (not header-callable in the reference)
# ------------------------------------------------------------------------------------------

def f32(x):
    """Python double -> nearest float32 -> python float: how TUPLE op parameters (lrs, wds of the
    multi_* ops) arrive -- str(tuple) parsed by std::istream >> float (include/mxnet/tuple.h),
    which is correctly rounded."""
    return float(np.float32(x))


def dmlc_stof(s):
    """dmlc::stof == ParseFloat<float> (3rdparty/dmlc-core/include/dmlc/strtonum.h:99-254) restated
    with numpy float32 arithmetic: float(int part) + float(double(frac digits)/double(10^k)), then
    scaled by powers of ten IN FLOAT. Not a correctly rounded conversion -- and it is what every
    SCALAR op parameter (lr, wd, rescale_grad, momentum, clip_gradient, beta1, ...) goes through."""
    F = np.float32
    p = s.strip()
    sign = 1.0
    if p[:1] in '+-':
        sign = -1.0 if p[0] == '-' else 1.0
        p = p[1:]
    low = p.lower()
    if low in ('inf', 'infinity'):
        return float(F(sign * np.inf))
    if low.startswith('nan'):
        return float('nan')
    i = 0
    predec = 0
    while i < len(p) and p[i].isdigit():
        predec = predec * 10 + int(p[i])
        i += 1
    value = F(predec)
    if i < len(p) and p[i] == '.':
        i += 1
        val2, pow10, cnt = 0, 1, 0
        while i < len(p) and p[i].isdigit():
            if cnt < 19:
                val2 = val2 * 10 + int(p[i])
                pow10 *= 10
            cnt += 1
            i += 1
        value = F(value + F(float(val2) / float(pow10)))
    if i < len(p) and p[i] in 'eE':
        i += 1
        frac = False
        if i < len(p) and p[i] in '+-':
            frac = p[i] == '-'
            i += 1
        expon = 0
        while i < len(p) and p[i].isdigit():
            expon = expon * 10 + int(p[i])
            i += 1
        scale = F(1.0)
        while expon >= 8:
            scale = F(scale * F(1e8))
            expon -= 8
        while expon > 0:
            scale = F(scale * F(10.0))
            expon -= 1
        value = F(value / scale) if frac else F(value * scale)
    assert i == len(p) or p[i:] in ('f', 'F'), "cannot parse %r" % s
    return float(F(sign) * value)


def scalar_param(v):
    """python float -> str() -> dmlc::stof: the value a scalar operator parameter really takes."""
    return dmlc_stof(repr(float(v)))


def _libstdcxx_sort_by_key(idx):
    """std::sort(idx.begin(), idx.end(), by .first) as libstdc++ implements it (bits/stl_algo.h:
    introsort -- median-of-three pivot moved to the front, unguarded Hoare partition, ranges of at
    most 16 left for one final insertion sort). NOT stable: pairs with equal keys leave it in an
    order that depends on these very steps, which is why it is restated step by step. `idx` is a
    list of (key, position); sorted in place. The heap-sort fallback (recursion deeper than
    2*log2(n)) is not restated: no key pattern of a kvstore call reaches it."""
    def less(a, b):
        return a[0] < b[0]

    def move_median_to_first(res, a, b, c):
        if less(idx[a], idx[b]):
            pick = b if less(idx[b], idx[c]) else (c if less(idx[a], idx[c]) else a)
        else:
            pick = a if less(idx[a], idx[c]) else (c if less(idx[b], idx[c]) else b)
        idx[res], idx[pick] = idx[pick], idx[res]

    def partition(first, last, pivot):
        while True:
            while less(idx[first], idx[pivot]):
                first += 1
            last -= 1
            while less(idx[pivot], idx[last]):
                last -= 1
            if not first < last:
                return first
            idx[first], idx[last] = idx[last], idx[first]
            first += 1

    def introsort_loop(first, last, depth):
        while last - first > 16:
            if depth == 0:
                raise NotImplementedError("heap-sort fallback of std::sort")
            depth -= 1
            move_median_to_first(first, first + 1, first + (last - first) // 2, last - 1)
            cut = partition(first + 1, last, first)
            introsort_loop(cut, last, depth)
            last = cut

    def linear_insert(last):            # __unguarded_linear_insert
        val = idx[last]
        nxt = last - 1
        while less(val, idx[nxt]):
            idx[last] = idx[nxt]
            last = nxt
            nxt -= 1
        idx[last] = val

    def insertion_sort(first, last):
        for i in range(first + 1, last):
            if less(idx[i], idx[first]):
                val = idx[i]
                idx[first + 1:i + 1] = idx[first:i]
                idx[first] = val
            else:
                linear_insert(i)
    n = len(idx)
    if n == 0:
        return
    introsort_loop(0, n, 2 * (n.bit_length() - 1))
    if n > 16:
        insertion_sort(0, 16)
        for i in range(16, n):
            linear_insert(i)
    else:
        insertion_sort(0, n)


def group_positions(keys, order='call'):
    """KVStoreLocal::GroupKVPairs, src/kvstore/kvstore_local.h:377-407, on the positions of a call's
    (key, value) pairs: returns (uniq_keys ascending, [positions of each key's values]).

    order='call' : values of a key in the order the call lists them (a stable sort by key) -- what
        the product does, and what the reference does whenever a call has at most 16 pairs, i.e. for
        every per-parameter call of gluon.Trainer / Module (one key x its devices) and for the
        reference's own unit tests.
    order='reference': the reference sorts the pairs with std::sort, which is not stable; in a call
        with MORE than 16 pairs (e.g. a list of 10 keys x 4 devices) the values of a key reach the
        reduce in the order libstdc++'s introsort happens to leave them -- restated step by step in
        _libstdcxx_sort_by_key and pinned to the reference's own function compiled against
        libstdc++ (Ref.group_positions)."""
    idx = [(int(k), i) for i, k in enumerate(keys)]
    if order == 'call':
        idx.sort(key=lambda p: p[0])       # python's sort is stable
    elif order == 'reference':
        _libstdcxx_sort_by_key(idx)
    else:
        raise ValueError(order)
    uniq, grouped = [], []
    for k, i in idx:
        if not uniq or k != uniq[-1]:
            uniq.append(k)
            grouped.append([i])
        else:
            grouped[-1].append(i)
    return uniq, grouped


def group_kv_pairs(keys, values, order='call'):
    """group_positions applied to the values: (uniq_keys ascending, grouped values)"""
    uniq, pos = group_positions(keys, order)
    return uniq, [[values[i] for i in g] for g in pos]


def adam_lr(lr, beta1, beta2, t):
    """python/mxnet/optimizer/optimizer.py:1617-1620: bias-corrected step size in python double."""
    coef1 = 1. - beta1 ** t
    coef2 = 1. - beta2 ** t
    return lr * math.sqrt(coef2) / coef1


class LocalKVStoreModel(object):
    """numpy model of kvstore('local') with an optional fused optimizer: the end-to-end checker.

    Follows KVStoreLocal::PushImpl/PullImpl (src/kvstore/kvstore_local.h:208-261): push = reduce the
    per-device values of a key (CommCPU association, comm.h:357-392, or 'device' left fold), then
    either run the updater on (merged, stored) or replace the stored value by the merged one; pull =
    copy of the stored value. The optimizer step follows python/mxnet/optimizer/optimizer.py
    (SGD._update_impl :603-659 -> multi_sgd[_mom]_update for dense; Adam.update :1610-1629).
    """

    def __init__(self, order="local"):
        self.order = order
        self.store = {}
        self.opt = None
        self.state = {}
        self.count = {}
        self.o = get_oracle()

    def init(self, key, value):
        assert key not in self.store, "duplicate init of key %s" % key
        self.store[key] = _f32(value).copy()

    def set_optimizer(self, kind, lr=0.01, momentum=0.0, wd=0.0, rescale_grad=1.0,
                      clip_gradient=None, beta1=0.9, beta2=0.999, epsilon=1e-8, lr_mult=None,
                      wd_mult=None):
        self.opt = dict(kind=kind, lr=lr, momentum=momentum, wd=wd, rescale=rescale_grad,
                        clip=clip_gradient, beta1=beta1, beta2=beta2, eps=epsilon,
                        lr_mult=lr_mult or {}, wd_mult=wd_mult or {})

    def push(self, key, values):
        values = values if isinstance(values, (list, tuple)) else [values]
        shape = self.store[key].shape
        merged = self.o.reduce(values, self.order).reshape(shape)
        if self.opt is None:
            self.store[key] = merged
            return
        p = self.opt
        w = self.store[key]
        self.count[key] = self.count.get(key, 0) + 1
        lr = p['lr'] * p['lr_mult'].get(key, 1.0)
        wd = p['wd'] * p['wd_mult'].get(key, 1.0)
        clip = p['clip'] if p['clip'] else None  # optimizer.py:623-624 passes clip only if truthy
        sp = scalar_param
        if p['kind'] == 'sgd':
            # multi_sgd[_mom]_update: lrs/wds are tuple parameters (nearest float32), the rest are
            # scalar parameters (dmlc::stof); momentum is only passed when > 0 (optimizer.py:618-621)
            mom = None
            if p['momentum'] != 0.0:
                mom = self.state.setdefault(key, np.zeros_like(w))
            self.o.multi_sgd_update(w.reshape(-1), merged.reshape(-1),
                                    mom.reshape(-1) if mom is not None else None, f32(lr),
                                    sp(p['momentum']) if p['momentum'] > 0 else 0.0, f32(wd),
                                    sp(p['rescale']), sp(clip) if clip else None)
        elif p['kind'] == 'adam':
            # adam_update: every hyper-parameter is a scalar parameter
            m, v = self.state.setdefault(key, (np.zeros_like(w), np.zeros_like(w)))
            lr_t = adam_lr(lr, p['beta1'], p['beta2'], self.count[key])
            self.o.adam_update(w.reshape(-1), merged.reshape(-1), m.reshape(-1), v.reshape(-1),
                               sp(lr_t), sp(p['beta1']), sp(p['beta2']), sp(p['eps']), sp(wd),
                               sp(p['rescale']), sp(clip) if clip else None)
        elif p['kind'] == 'test':
            # grad * rescale_grad -> _mul_scalar(scalar=str(rescale_grad))
            self.o.test_update(w.reshape(-1), merged.reshape(-1), sp(p['rescale']))
        else:
            raise ValueError(p['kind'])

    def pull(self, key):
        return self.store[key].copy()

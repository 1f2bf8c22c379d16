"""daccord_b200 -- B200-native engine for daccord's per-window local de Bruijn consensus path.

Python here is plumbing only (ctypes over the C ABI in include/daccord_b200.h); the product is the
CUDA library daccord_b200/_build/libdaccord_b200.so.  There is no CPU fallback: importing the engine
without the built library, or running it without a GPU, raises.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_build", "libdaccord_b200.so")

SLICE_DT = np.dtype([("gpos", "<u4"), ("len", "<u2"), ("flags", "<u2")])
WINDOW_DT = np.dtype([("slice_begin", "<u4"), ("slice_cnt", "<u2"), ("reserved", "<u2"), ("aread", "<u4"), ("astart", "<u4")])
RESULT_DT = np.dtype([("status", "u1"), ("k", "u1"), ("ff", "i1"), ("clen", "u1"), ("err", "<u4"), ("nops", "<u2"),
                      ("ncand", "<u2"), ("elength", "<i4")])
SEGMENT_DT = np.dtype([("aread", "<u4"), ("first", "<u4"), ("last", "<u4"), ("reserved", "<u4"), ("len", "<u8"), ("off", "<u8")])
CONS_STRIDE, OPS_STRIDE = 64, 128
WIN_SKIPPED, WIN_OK, WIN_FAILED = 0, 1, 2


class Params(C.Structure):
    """dcu_params: -w, -k, -m, --min/maxfilterfreq, -e and the error profile (reference src/daccord.cpp:1282-1305)."""
    _fields_ = [("w", C.c_uint32), ("k_lo", C.c_uint32), ("k_hi", C.c_uint32), ("min_cov", C.c_uint32),
                ("min_ff", C.c_int32), ("max_ff", C.c_int32), ("max_err", C.c_uint64),
                ("p_i", C.c_double), ("p_d", C.c_double), ("est_cor", C.c_double)]

    @staticmethod
    def default(**kw):
        p = Params(w=40, k_lo=8, k_hi=8, min_cov=3, min_ff=0, max_ff=2, max_err=2**64 - 1, p_i=0.09, p_d=0.045, est_cor=0.85)
        for k, v in kw.items():
            setattr(p, k, v)
        return p


class DcuError(RuntimeError):
    pass


_lib = None


def load_library():
    """dlopen the CUDA library; raises if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DcuError("CUDA library %s not built: run `python -m daccord_b200.build` (nvcc, sm_100a)" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        lib.dcu_strerror.restype = C.c_char_p
        lib.dcu_last_error.restype = C.c_char_p
        lib.dcu_get_tables.restype = C.c_int64
        _lib = lib
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Engine:
    """One dcu_ctx (one GPU).  Mirrors the C ABI one to one."""

    def __init__(self, params=None, device=0):
        self.lib = load_library()
        self.params = params or Params.default()
        self.ctx = C.c_void_p()
        self._ck(self.lib.dcu_create(C.byref(self.params), C.c_int(device), C.byref(self.ctx)))
        self.nwin = 0

    def _ck(self, rc, allow=()):
        if rc != 0 and rc not in allow:
            msg = self.lib.dcu_strerror(rc).decode()
            if self.ctx:
                msg += ": " + self.lib.dcu_last_error(self.ctx).decode()
            raise DcuError(msg)
        return rc

    def close(self):
        if self.ctx:
            self.lib.dcu_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_reads(self, packed):
        packed = np.ascontiguousarray(packed, np.uint8)
        self._ck(self.lib.dcu_set_reads(self.ctx, _p(packed), C.c_uint64(packed.size)))

    def set_reads_device(self, dptr, nbytes):
        self._ck(self.lib.dcu_set_reads_device(self.ctx, C.c_void_p(dptr), C.c_uint64(nbytes)))

    def share_reads(self, owner):
        """use the read database of another Engine on the same device (several batches in flight: one Engine per batch)"""
        self._ck(self.lib.dcu_share_reads(self.ctx, owner.ctx))

    def upload(self, win, sl):
        assert win.dtype == WINDOW_DT and sl.dtype == SLICE_DT
        self.nwin = len(win)
        self._ck(self.lib.dcu_upload(self.ctx, _p(win), C.c_uint64(len(win)), _p(sl), C.c_uint64(len(sl))))

    def pile(self, ovl, trace, tspace, read_boff, read_len, advance=10, maxalign=2**64 - 1):
        """trace reconstruction + window / slice extraction on the GPU; the batch stays resident (then launch / download)"""
        nw, ns = C.c_uint64(0), C.c_uint64(0)
        self._ck(self.lib.dcu_pile(self.ctx, _p(ovl), C.c_uint64(len(ovl)), _p(trace), C.c_uint64(len(trace)), C.c_int32(tspace), _p(read_boff), _p(read_len),
                                   C.c_uint64(len(read_len)), C.c_uint32(advance), C.c_uint64(maxalign), C.byref(nw), C.byref(ns)))
        self.nwin, self.nsl = nw.value, ns.value
        return nw.value, ns.value

    def get_windows(self, with_slices=False):
        win = np.zeros(self.nwin, WINDOW_DT)
        sl = np.zeros(self.nsl, SLICE_DT) if with_slices else None
        self._ck(self.lib.dcu_get_windows(self.ctx, _p(win), _p(sl)))
        return (win, sl) if with_slices else win

    def launch(self):
        ms = C.c_float(0)
        self._ck(self.lib.dcu_launch(self.ctx, C.byref(ms)))
        return ms.value

    def download(self, out=None):
        res, cons, ops = out if out is not None else alloc_out(self.nwin)
        self._ck(self.lib.dcu_download(self.ctx, _p(res), _p(cons), _p(ops)))
        return res, cons, ops

    def run(self, win, sl, out=None):
        """host buffers in, host buffers out (the call a user of the library makes)"""
        res, cons, ops = out if out is not None else alloc_out(len(win))
        self._ck(self.lib.dcu_run(self.ctx, _p(win), C.c_uint64(len(win)), _p(sl), C.c_uint64(len(sl)), _p(res), _p(cons), _p(ops)))
        return res, cons, ops

    def vote(self, producefull=False, minlen=0, read_boff=None, read_len=None, chars_out=None):
        """pile vote of the resident results on the GPU; returns (segments, chars) -- see dcu_vote in include/daccord_b200.h.
        chars_out: optional uint8 buffer (e.g. pinned host memory) the corrected bases are copied into when it is large enough"""
        ns, nc = C.c_uint64(0), C.c_uint64(0)
        nreads = 0 if read_len is None else len(read_len)
        self._ck(self.lib.dcu_vote(self.ctx, C.c_int(1 if producefull else 0), C.c_uint64(minlen), _p(read_boff), _p(read_len), C.c_uint64(nreads), C.byref(ns), C.byref(nc)))
        seg = np.zeros(ns.value, SEGMENT_DT)
        chars = chars_out[:nc.value] if (chars_out is not None and len(chars_out) >= nc.value) else np.zeros(nc.value, np.uint8)
        self._ck(self.lib.dcu_get_corrected(self.ctx, _p(seg), _p(chars)))
        return seg, chars

    def stats(self):
        a, b = C.c_uint64(0), C.c_uint64(0)
        self._ck(self.lib.dcu_last_stats(self.ctx, C.byref(a), C.byref(b)))
        c, d = C.c_uint64(0), C.c_uint64(0); e, f = C.c_uint32(0), C.c_uint32(0)
        self._ck(self.lib.dcu_last_stats2(self.ctx, C.byref(c), C.byref(d), C.byref(e), C.byref(f)))
        return {"launches": a.value, "hard_windows": b.value, "second_pass_windows": c.value, "lost_windows": d.value, "smem_warps": e.value, "smem_bytes_per_warp": f.value}

    def tables(self, which):
        """table `which` (0 DPn, 1 DPsq, 2 VSq, 3 suplo/suphi pairs, 4 klim, 5 NP/MS/KLIMN) as read back from device memory"""
        n = self.lib.dcu_get_tables(self.ctx, C.c_int(which), None, C.c_int64(0))
        if n < 0:
            raise DcuError("dcu_get_tables: " + self.lib.dcu_last_error(self.ctx).decode())
        out = np.zeros(n, np.float64)
        self.lib.dcu_get_tables(self.ctx, C.c_int(which), _p(out), C.c_int64(n))
        return out


def alloc_out(nwin):
    return (np.zeros(nwin, RESULT_DT), np.zeros(nwin * CONS_STRIDE, np.uint8), np.zeros(nwin * OPS_STRIDE, np.uint8))

"""ctypes binding of libgarlic_b200.so (include/garlic_b200.h) and a thin Python mirror of the
reference's hot-path call sequence (garlic-main.cpp:216-406).

There is no CPU fallback: importing works anywhere (so the symbol table can be checked without a GPU),
but creating a ``GarlicGPU`` fails loudly unless the CUDA library loads and a device is present.
"""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgarlic_b200.so")
MISSING = -9999.0
GL_TYPES = {"GQ": 0, "GL": 1, "PL": 2, "ERROR": -1}

EXPORTS = [
    "garlic_gpu_create", "garlic_gpu_destroy", "garlic_gpu_last_error", "garlic_gpu_launch_count",
    "garlic_gpu_stream", "garlic_gpu_sync", "garlic_gpu_host_alloc", "garlic_gpu_host_free", "garlic_gpu_set_shape", "garlic_gpu_put_alleles",
    "garlic_gpu_first_allele_keys_dev", "garlic_gpu_code_alleles", "garlic_gpu_put_tped_text", "garlic_gpu_set_phased", "garlic_gpu_put_packed",
    "garlic_gpu_put_packed_dev", "garlic_gpu_count_packed", "garlic_gpu_counts_dev", "garlic_gpu_get_counts",
    "garlic_gpu_get_one_allele", "garlic_gpu_put_gl", "garlic_gpu_put_gl_dev", "garlic_gpu_filter",
    "garlic_gpu_set_tables", "garlic_gpu_set_lut", "garlic_gpu_get_lut", "garlic_gpu_get_hom_freq",
    "garlic_gpu_ld_band", "garlic_gpu_set_wlod", "garlic_gpu_window_slots", "garlic_gpu_windows",
    "garlic_gpu_windows_dev", "garlic_gpu_windows_gather", "garlic_gpu_comm_id", "garlic_gpu_comm_init",
    "garlic_gpu_call_roh", "garlic_gpu_last_stats", "garlic_gpu_n_kept", "garlic_gpu_get_kept_index",
    "garlic_gpu_get_genotypes", "garlic_gpu_get_piece_bounds", "garlic_gpu_set_prune", "garlic_gpu_kde", "garlic_gpu_put_tgls_text", "garlic_gpu_get_gl",
    "garlic_gpu_put_bed", "garlic_gpu_put_bed_dev", "garlic_gpu_put_vcf_text",
]


class RohRec(C.Structure):
    _fields_ = [("ind", C.c_int32), ("chr", C.c_int32), ("start_idx", C.c_int32), ("stop_idx", C.c_int32)]


_LIB = None


def load_library():
    """Load libgarlic_b200.so (must have been built by garlic_b200/build.py). Raises if absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libgarlic_b200.so is not built (run `python garlic_b200/build.py`); "
                           "garlic_b200 has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    L.garlic_gpu_last_error.restype = C.c_char_p
    L.garlic_gpu_launch_count.restype = C.c_uint64
    L.garlic_gpu_stream.restype = C.c_void_p
    L.garlic_gpu_host_alloc.restype = C.c_void_p
    L.garlic_gpu_host_alloc.argtypes = [C.c_size_t]
    L.garlic_gpu_host_free.argtypes = [C.c_void_p]
    L.garlic_gpu_first_allele_keys_dev.restype = C.c_void_p
    L.garlic_gpu_counts_dev.restype = C.c_void_p
    L.garlic_gpu_window_slots.restype = C.c_int64
    L.garlic_gpu_n_kept.restype = C.c_int64
    for name in EXPORTS:
        getattr(L, name)
    _LIB = L
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class GarlicError(RuntimeError):
    pass


class GarlicGPU:
    """One handle = one GPU (garlic_gpu_t)."""

    def __init__(self, device=0):
        self.lib = load_library()
        self.h = C.c_void_p()
        rc = self.lib.garlic_gpu_create(C.c_int(device), C.byref(self.h))
        if rc != 0 or not self.h:
            raise GarlicError("garlic_gpu_create failed (rc=%d): no usable CUDA device; there is no CPU fallback" % rc)

    def host_array(self, n, dtype):
        """numpy array in page-locked host memory (garlic_gpu_host_alloc); freed with the handle."""
        dt = np.dtype(dtype)
        ptr = self.lib.garlic_gpu_host_alloc(C.c_size_t(max(1, n) * dt.itemsize))
        if not ptr:
            return np.empty(n, dt)
        self._pinned = getattr(self, "_pinned", [])
        self._pinned.append(ptr)
        buf = (C.c_char * (max(1, n) * dt.itemsize)).from_address(ptr)
        return np.frombuffer(buf, dtype=dt, count=n)

    def close(self):
        for ptr in getattr(self, "_pinned", []):
            self.lib.garlic_gpu_host_free(C.c_void_p(ptr))
        self._pinned = []
        self._freq_buf = self._keep_buf = self._win_buf = None
        if self.h:
            self.lib.garlic_gpu_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise GarlicError(self.lib.garlic_gpu_last_error(self.h).decode())

    # ---------------------------------------------------------------- ingest
    def set_shape(self, n_ind, n_loci, chr_offsets, pos, ind_offset=0):
        co = np.ascontiguousarray(chr_offsets, np.int64)
        po = np.ascontiguousarray(pos, np.int32)
        self.n_ind, self.L0, self.n_chr = int(n_ind), int(n_loci), len(co) - 1
        self._ck(self.lib.garlic_gpu_set_shape(self.h, C.c_int(n_ind), C.c_int(ind_offset), C.c_int64(n_loci),
                                               C.c_int(self.n_chr), _p(co), _p(po)))

    def put_alleles(self, alleles, snp0=0, missing="0"):
        a = np.ascontiguousarray(alleles, np.uint8)
        self._ck(self.lib.garlic_gpu_put_alleles(self.h, _p(a), C.c_int64(snp0), C.c_int(a.shape[0]),
                                                 C.c_char(missing.encode())))

    def put_tped_text(self, text: bytes, line_off, snp0=0, missing="0"):
        """K0: raw tped line tails → alleles on the device; returns the non-blank character count per line."""
        off = np.ascontiguousarray(line_off, np.int64)
        n = len(off) - 1
        nb = np.empty(n, np.int32)
        buf = np.frombuffer(text, np.uint8)
        self._ck(self.lib.garlic_gpu_put_tped_text(self.h, _p(buf), _p(off), C.c_int64(snp0), C.c_int(n),
                                                   C.c_char(missing.encode()), _p(nb)))
        return nb

    def put_vcf_text(self, text: bytes, line_off, snp0=0):
        """VCF sample columns (the text after FORMAT's tab per record, vcf.sample_text) → allele index bytes on the device
        (255 = missing).  Returns per record (sample columns, largest allele index or -1, first malformed column or -1)."""
        off = np.ascontiguousarray(line_off, np.int64)
        n = len(off) - 1
        nc, mx, bad = np.empty(n, np.int32), np.empty(n, np.int32), np.empty(n, np.int32)
        buf = np.frombuffer(text, np.uint8) if len(text) else np.zeros(1, np.uint8)
        self._ck(self.lib.garlic_gpu_put_vcf_text(self.h, _p(buf), _p(off), C.c_int64(snp0), C.c_int(n), _p(nc), _p(mx),
                                                  _p(bad)))
        return nc, mx, bad

    def put_bed(self, rows, snp0=0):
        """rows: uint8[n_snp, ceil(N_total/4)] SNP-major .bed rows of the whole fileset (no magic bytes); this handle keeps
        its own individuals' columns and records the first-allele keys and counters (phase a)."""
        r = np.ascontiguousarray(rows, np.uint8)
        self._ck(self.lib.garlic_gpu_put_bed(self.h, _p(r), C.c_int64(r.shape[1]), C.c_int64(snp0), C.c_int(r.shape[0])))

    def put_bed_dev(self, ptr, stride, n_snp, snp0=0):
        self._ck(self.lib.garlic_gpu_put_bed_dev(self.h, C.c_void_p(ptr), C.c_int64(stride), C.c_int64(snp0), C.c_int(n_snp)))

    def code_alleles(self):
        self._ck(self.lib.garlic_gpu_code_alleles(self.h))

    def put_packed(self, rows):
        r = np.ascontiguousarray(rows, np.uint8)
        self._ck(self.lib.garlic_gpu_put_packed(self.h, _p(r), C.c_int64(r.shape[1])))

    def put_packed_dev(self, ptr, stride):
        self._ck(self.lib.garlic_gpu_put_packed_dev(self.h, C.c_void_p(ptr), C.c_int64(stride)))

    def count_packed(self, nalleles_corr=None, total_corr=None):
        a = None if nalleles_corr is None else np.ascontiguousarray(nalleles_corr, np.int32)
        t = None if total_corr is None else np.ascontiguousarray(total_corr, np.int32)
        self._ck(self.lib.garlic_gpu_count_packed(self.h, _p(a), _p(t)))

    def counts_dev(self):
        return self.lib.garlic_gpu_counts_dev(self.h)

    def first_allele_keys_dev(self):
        return self.lib.garlic_gpu_first_allele_keys_dev(self.h)

    def get_counts(self):
        out = [np.empty(self.L0, np.int32) for _ in range(4)]
        self._ck(self.lib.garlic_gpu_get_counts(self.h, *[_p(o) for o in out]))
        return out

    def get_one_allele(self, missing="0"):
        """missing: the value for a SNP without a present allele, a one-character str or an int (255 for VCF input)."""
        a = np.empty(self.L0, np.uint8)
        m = bytes([missing]) if isinstance(missing, int) else missing.encode()
        self._ck(self.lib.garlic_gpu_get_one_allele(self.h, _p(a), C.c_char(m)))
        return a

    def put_gl(self, values_ind_major, gl_type):
        v = np.ascontiguousarray(values_ind_major, np.float64)
        assert v.shape == (self.n_ind, self.L0)
        self._ck(self.lib.garlic_gpu_put_gl(self.h, _p(v), C.c_int(GL_TYPES[gl_type])))

    # ---------------------------------------------------------------- filter / tables
    def put_tgls_text(self, text: bytes, line_off, gl_type, snp0=0):
        """K0-GL: tgls value columns from raw text (what follows the 4th field of each line).  → tokens per line."""
        t = {"GQ": 0, "GL": 1, "PL": 2, None: -1}[gl_type] if not isinstance(gl_type, int) else gl_type
        off = np.ascontiguousarray(line_off, np.int64)
        n = len(off) - 1
        ntok = np.zeros(n, np.int32)
        buf = np.frombuffer(text, np.uint8)
        self._ck(self.lib.garlic_gpu_put_tgls_text(self.h, _p(buf), _p(off), C.c_int64(snp0), C.c_int(n), C.c_int(t), _p(ntok)))
        return ntok

    def get_gl(self):
        out = np.empty((self.n_ind, self.L0), np.float64)
        self._ck(self.lib.garlic_gpu_get_gl(self.h, _p(out)))
        return out

    def filter(self, oob=False, chr_param=None, freq_override=None, want_freq=True, want_keep=True, wait=True):
        """→ (freq float64[L0], keep bool[L0], L).  The two arrays are views of page-locked buffers owned by this object
        and are overwritten by the next filter() call (repeated runs then touch no fresh pages).  The library fills
        page-locked buffers behind the call; wait=False leaves it at that (they are complete once the next windows /
        call_roh / sync call has returned), wait=True synchronises before returning."""
        if getattr(self, "_freq_buf", None) is None or len(self._freq_buf) != self.L0:
            self._freq_buf = self.host_array(self.L0, np.float64)      # page-locked: no staging copy
            self._keep_buf = self.host_array(self.L0, np.uint8)
        freq = self._freq_buf if want_freq else None
        keep = self._keep_buf if want_keep else None
        n = C.c_int64(0)
        cp = None if chr_param is None else np.ascontiguousarray(chr_param, np.int32)
        fo = None if freq_override is None else np.ascontiguousarray(freq_override, np.float64)
        self._ck(self.lib.garlic_gpu_filter(self.h, C.c_int(int(oob)), _p(cp), _p(fo), _p(freq), _p(keep), C.byref(n)))
        if wait and (want_freq or want_keep):
            self.sync()
        self.L = n.value
        return freq, (keep.view(np.bool_) if keep is not None else None), n.value

    def set_tables(self, error, max_gap, centromeres, gpos=None):
        cen = np.ascontiguousarray(centromeres, np.int32).reshape(-1)
        g = None if gpos is None else np.ascontiguousarray(gpos, np.float64)
        self._ck(self.lib.garlic_gpu_set_tables(self.h, C.c_double(-1.0 if error is None else error), C.c_int(max_gap),
                                                _p(cen), _p(g)))

    def set_lut(self, lut):
        l = np.ascontiguousarray(lut, np.float64)
        assert l.shape == (self.L, 4)
        self._ck(self.lib.garlic_gpu_set_lut(self.h, _p(l)))

    def get_lut(self):
        l = np.empty((self.L, 4), np.float64)
        self._ck(self.lib.garlic_gpu_get_lut(self.h, _p(l)))
        return l

    def get_hom_freq(self):
        f = np.empty(self.L, np.float64)
        self._ck(self.lib.garlic_gpu_get_hom_freq(self.h, _p(f)))
        return f

    def get_genotypes(self, filtered=False):
        n = self.L if filtered else self.L0
        rows = np.empty((self.n_ind, (n + 3) // 4), np.uint8)
        self._ck(self.lib.garlic_gpu_get_genotypes(self.h, C.c_int(int(filtered)), _p(rows), C.c_int64(rows.shape[1])))
        return rows

    def get_kept_index(self):
        s = np.empty(self.L, np.int32)
        self._ck(self.lib.garlic_gpu_get_kept_index(self.h, _p(s)))
        return s

    # ---------------------------------------------------------------- weighted
    def set_phased(self, on=True):
        self._ck(self.lib.garlic_gpu_set_phased(self.h, C.c_int(int(on))))

    def set_wlod(self, mu, M):
        self._ck(self.lib.garlic_gpu_set_wlod(self.h, C.c_double(mu), C.c_int(M)))

    def ld_band(self, W, ld_individuals=None, want_ld=False):
        idx = None if ld_individuals is None else np.ascontiguousarray(ld_individuals, np.int32)
        out = np.empty((self.L, W), np.float64) if want_ld else None
        self._ck(self.lib.garlic_gpu_ld_band(self.h, C.c_int(W), _p(idx), C.c_int(0 if idx is None else len(idx)), _p(out)))
        return out

    # ---------------------------------------------------------------- windows / ROH
    def window_slots(self, step):
        return int(self.lib.garlic_gpu_window_slots(self.h, C.c_int(step)))

    def windows(self, W, step=1, weighted=False, individuals=None, exact=True, reuse=False):
        """reuse=True: the result is a view of a page-locked buffer owned by this object, overwritten by the next call."""
        idx = None if individuals is None else np.ascontiguousarray(individuals, np.int32)
        n = self.n_ind if idx is None else len(idx)
        shape = (n, self.window_slots(step))
        if reuse and shape[0] * shape[1] <= (1 << 23):
            # small results (the KDE's thinned windows) land in a page-locked buffer kept between calls: a fresh
            # pageable array costs more in page faults than the whole pass
            if getattr(self, "_win_buf", None) is None or self._win_buf.size < shape[0] * shape[1]:
                self._win_buf = self.host_array(max(shape[0] * shape[1], 1), np.float64)
            out = self._win_buf[:shape[0] * shape[1]].reshape(shape)
        else:
            out = np.empty(shape, np.float64)
        self._ck(self.lib.garlic_gpu_windows(self.h, C.c_int(W), C.c_int(step), C.c_int(int(weighted)), _p(idx),
                                             C.c_int(n), C.c_int(int(exact)), _p(out)))
        return out

    def windows_dev(self, W, step=1, weighted=False, individuals=None, exact=True):
        """→ (device pointer, n, slots): the window matrix left on the GPU."""
        idx = None if individuals is None else np.ascontiguousarray(individuals, np.int32)
        n = self.n_ind if idx is None else len(idx)
        ptr = C.c_void_p()
        self._ck(self.lib.garlic_gpu_windows_dev(self.h, C.c_int(W), C.c_int(step), C.c_int(int(weighted)), _p(idx),
                                                 C.c_int(n), C.c_int(int(exact)), C.byref(ptr)))
        return ptr.value, n, self.window_slots(step)

    def windows_gather(self, W, step, individuals, rows_per_rank, world, weighted=False, exact=False, want=True):
        """All ranks' thinned windows: float64[world*rows_per_rank, slots] (MISSING rows = padding).  want=False: this
        rank only contributes (returns None; the gathered matrix stays on its GPU)."""
        idx = np.ascontiguousarray(individuals, np.int32)
        slots = self.window_slots(step)
        key = (world * rows_per_rank, slots)
        if want and (getattr(self, "_gather_buf", None) is None or self._gather_buf.shape != key):
            self._gather_buf = self.host_array(key[0] * key[1], np.float64).reshape(key)
        self._ck(self.lib.garlic_gpu_windows_gather(self.h, C.c_int(W), C.c_int(step), C.c_int(int(weighted)), _p(idx),
                                                    C.c_int(len(idx)), C.c_int(rows_per_rank), C.c_int(int(exact)),
                                                    _p(self._gather_buf) if want else None))
        return self._gather_buf if want else None

    def kde(self, values=None, m=512):
        """computeKDE (garlic-kde.cpp:14-101) on the device, of `values` or — None — of the window matrix the last
        windows / windows_dev / windows_gather call left on the GPU.  → (x[m], y[m] normalised as the reference's
        .kde, n, bandwidth)."""
        v = None if values is None else np.ascontiguousarray(values, np.float64)
        x, y = np.empty(m, np.float64), np.empty(m, np.float64)
        n, h = C.c_int64(0), C.c_double(0)
        self._ck(self.lib.garlic_gpu_kde(self.h, _p(v), C.c_int64(0 if v is None else v.size), C.c_int(m), _p(x), _p(y),
                                         C.byref(n), C.byref(h)))
        y = y / (y.sum() * (x[1] - x[0]))                       # garlic-kde.cpp:86-95
        return x, y, n.value, h.value

    @staticmethod
    def comm_id():
        lib = load_library()
        buf = np.zeros(128, np.uint8)
        if lib.garlic_gpu_comm_id(_p(buf)) != 0:
            raise GarlicError("ncclGetUniqueId failed")
        return buf

    def comm_init(self, comm_id, rank, world):
        buf = np.ascontiguousarray(comm_id, np.uint8)
        self._ck(self.lib.garlic_gpu_comm_init(self.h, _p(buf), C.c_int(rank), C.c_int(world)))

    def call_roh(self, W, cutoff, overlap_frac, weighted=False, exact=False, cap=1 << 16, copy=True):
        """→ int32[n, 4] rows (ind, chr, start_idx, stop_idx), sorted by (ind, chr, start).  copy=False: a view of a
        buffer owned by this object, overwritten by the next call."""
        buf = getattr(self, "_roh_buf", None)
        if buf is None or len(buf) < cap:
            buf = self._roh_buf = np.empty((cap, 4), np.int32)
        while True:
            cnt = C.c_int64(0)
            self._ck(self.lib.garlic_gpu_call_roh(self.h, C.c_int(W), C.c_double(cutoff), C.c_double(overlap_frac),
                                                  C.c_int(int(weighted)), C.c_int(int(exact)), _p(buf),
                                                  C.c_int64(len(buf)), C.byref(cnt)))
            if cnt.value <= len(buf):
                break
            buf = self._roh_buf = np.empty((cnt.value + 1024, 4), np.int32)
        return buf[:cnt.value].copy() if copy else buf[:cnt.value]

    def last_stats(self):
        s = (C.c_double * 8)()
        self.lib.garlic_gpu_last_stats(self.h, s)
        return dict(items=s[0], units=s[1], ambiguous_pairs=s[2], kernel_ms=s[3], select_ms=s[4],
                    candidate_pairs=s[5], all_pairs=s[6], squeeze_ms=s[7])

    def set_prune(self, on=True):
        self._ck(self.lib.garlic_gpu_set_prune(self.h, C.c_int(int(on))))

    def piece_bounds(self, W):
        """uint32[n_pieces, n_ind]: the pruning bound's piece maxima (low / high int16, 1/64 LOD)."""
        n_pieces = (self.L + 255) // 256
        out = np.empty((n_pieces, self.n_ind), np.uint32)
        n = C.c_int64(0)
        self._ck(self.lib.garlic_gpu_get_piece_bounds(self.h, C.c_int(W), _p(out), C.c_int64(out.size), C.byref(n)))
        assert n.value == n_pieces
        return out

    def launch_count(self):
        return int(self.lib.garlic_gpu_launch_count(self.h))

    def stream(self):
        return self.lib.garlic_gpu_stream(self.h)

    def sync(self):
        self._ck(self.lib.garlic_gpu_sync(self.h))


def overlap_threshold(frac, W):
    """garlic-roh.cpp:422-424 clamp, as the integer the comparisons at :466/:477 reduce to."""
    t = frac * W
    t = t if t >= 1 else 1
    t = t if t <= W else W
    return int(math.ceil(t))

"""ctypes bindings of include/grlgpu.h (device parse phase) and include/grlbwt.h (host side).

There is no fallback: if the shared libraries are missing, or no CUDA device is usable, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

LIB_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib")
FLAG_SMALL_TABLE, FLAG_FORCE_SLOW_SCAN, FLAG_KEEP_DICT, FLAG_FORCE_UNCACHED, FLAG_SMALL_PILOT, FLAG_FORCE_DOUBLING = 1, 2, 4, 8, 16, 32
FLAG_FORCE_WALK, FLAG_FORCE_JUMP = 64, 128   # tests: grlgpu_invert takes the walk per string / pointer jumping regardless of the chains
CELL = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}


class GrlGpuError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"grlgpu status {status}: {msg}")
        self.status = status


class Stats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("n_syms", "n_strings", "longest_string", "min_sym", "max_sym", "max_sym_freq", "sep_sym")]


class Round(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("round", "n_in", "n_strings", "parse_len", "n_phrases", "dict_syms", "max_freq", "alphabet",
                                          "tot_phrases", "n_pre_runs", "algorithmic_bytes")] + \
               [(k, C.c_uint32) for k in ("cell_bytes_in", "cell_bytes_out", "sym_bytes", "done")] + \
               [(k, C.c_float) for k in ("device_ms", "text_pass_ms", "dict_ms", "rewrite_ms")]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Slice(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("rank_base", "tot_local", "pre_first", "n_pre_local", "exchange_bytes", "n_in_local", "parse_len_local")] + \
               [("sym_bytes", C.c_uint32), ("reserved", C.c_uint32)]


class Invert(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("n", "n_strings", "n_runs", "n_out")] + [(k, C.c_uint32) for k in ("path", "jump_rounds")] + \
               [(k, C.c_float) for k in ("device_ms", "lf_ms", "invert_ms")]


class FmInfo(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("n", "n_strings", "n_runs", "sigma", "sep")] + [("load_ms", C.c_float)]


class FmQuery(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("n_pat", "n_pat_syms", "n_occ")] + [(k, C.c_uint32) for k in ("path", "jump_rounds")] + \
               [(k, C.c_float) for k in ("device_ms", "search_ms", "locate_ms")]


class FmApprox(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("n_pat", "n_pat_syms", "n_hits", "n_occ", "n_lf")] + [(k, C.c_uint32) for k in ("path", "jump_rounds")] + \
               [(k, C.c_float) for k in ("device_ms", "search_ms", "locate_ms")]


class FmExtract(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("n_req", "n_cells")] + [(k, C.c_uint32) for k in ("path", "jump_rounds")] + \
               [(k, C.c_float) for k in ("device_ms", "extract_ms")]


class BwtResult(C.Structure):
    _fields_ = [("n_runs", C.c_uint64), ("sb", C.c_uint64), ("fb", C.c_uint64), ("syms", C.POINTER(C.c_uint64)),
                ("lens", C.POINTER(C.c_uint64)), ("n_rounds", C.c_uint64), ("h2d_ms", C.c_double), ("par_phase_ms", C.c_double),
                ("ind_phase_ms", C.c_double), ("device_ms", C.c_double), ("algorithmic_bytes", C.c_uint64), ("induced_on_device", C.c_uint64)]


_gpu = None
_host = None


def lib_gpu():
    global _gpu
    if _gpu is None:
        path = os.path.join(LIB_DIR, "libgrlgpu.so")
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: build it with `make -C grlbwt_b200` (or __graft_entry__.build()); there is no fallback path")
        L = C.CDLL(path)
        vp, u64 = C.c_void_p, C.c_uint64
        L.grlgpu_create.argtypes = [C.POINTER(vp), C.c_int, u64]
        L.grlgpu_destroy.argtypes = [vp]
        L.grlgpu_set_text.argtypes = [vp, vp, u64, C.c_int]
        L.grlgpu_set_text_device.argtypes = [vp, vp, u64, C.c_int]
        L.grlgpu_stats.argtypes = [vp, C.POINTER(Stats)]
        L.grlgpu_round.argtypes = [vp, C.POINTER(Round)]
        L.grlgpu_fetch_level.argtypes = [vp, vp, vp, vp, vp, vp]
        L.grlgpu_fetch_level_async.argtypes = [vp, vp, vp, vp, vp, vp]
        L.grlgpu_fetch_level32.argtypes = [vp, vp, vp, vp, vp, vp, C.c_int]
        L.grlgpu_fetch_wait.argtypes = [vp]
        L.grlgpu_level_checksum.argtypes = [vp, vp]
        L.grlgpu_fetch_parse.argtypes = [vp, vp]
        L.grlgpu_fetch_str_ptrs.argtypes = [vp, vp]
        L.grlgpu_fetch_dictionary.argtypes = [vp, vp, vp, vp, vp]
        L.grlgpu_strerror.restype = C.c_char_p
        L.grlgpu_strerror.argtypes = [C.c_int]
        L.grlgpu_last_error.restype = C.c_char_p
        L.grlgpu_last_error.argtypes = [vp]
        L.grlgpu_create_on_stream.argtypes = [C.POINTER(vp), C.c_int, u64, vp]
        L.grlgpu_profile_enable.argtypes = [vp, C.c_int]
        L.grlgpu_profile_reset.argtypes = [vp]
        L.grlgpu_launch_count.argtypes = [vp]
        L.grlgpu_launch_count.restype = u64
        L.grlgpu_profile_entry.argtypes = [vp, C.c_int, C.c_char_p, C.c_int, C.POINTER(u64), C.POINTER(C.c_double), C.POINTER(u64)]
        L.grlgpu_histogram.argtypes = [vp, vp]
        L.grlgpu_nccl_unique_id.argtypes = [vp]
        L.grlgpu_comm_create_nccl.argtypes = [C.POINTER(vp), vp, C.c_int, C.c_int, C.c_int]
        L.grlgpu_comm_create_ipc.argtypes = [C.POINTER(vp), C.c_char_p, C.c_int, C.c_int, C.c_int]
        L.grlgpu_can_peer.argtypes = [C.c_int, C.c_int]
        L.grlgpu_local_group_create.argtypes = [C.POINTER(vp), C.c_int]
        L.grlgpu_local_group_abort.argtypes = [vp]
        L.grlgpu_local_group_destroy.argtypes = [vp]
        L.grlgpu_comm_create_local.argtypes = [C.POINTER(vp), vp, C.c_int, C.c_int]
        L.grlgpu_comm_destroy.argtypes = [vp]
        L.grlgpu_comm_info.argtypes = [vp, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64), C.c_char_p, C.c_int]
        L.grlgpu_comm_times.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.grlgpu_set_peers.argtypes = [vp, vp, C.c_int]
        L.grlgpu_mg_stats.argtypes = [vp, vp, C.POINTER(Stats)]
        L.grlgpu_mg_round.argtypes = [vp, vp, C.POINTER(Round)]
        L.grlgpu_mg_slice_info.argtypes = [vp, C.POINTER(Slice)]
        L.grlgpu_mg_fetch_slice.argtypes = [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int]
        L.grlgpu_mg_slice_checksum.argtypes = [vp, vp]
        L.grlgpu_text_begin.argtypes = [vp, u64, C.c_int, u64]
        L.grlgpu_text_stage.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
        L.grlgpu_text_commit.argtypes = [vp, u64]
        L.grlgpu_text_end.argtypes = [vp]
        L.grlgpu_level_park.argtypes = [vp, C.c_int, vp]
        L.grlgpu_copy_to_host.argtypes = [C.c_int, vp, vp, u64]
        L.grlgpu_invert.argtypes = [vp, vp, u64, C.c_int, u64, vp, u64, C.POINTER(Invert)]
        L.grlgpu_fm_load.argtypes = [vp, vp, u64, C.POINTER(FmInfo)]
        L.grlgpu_fm_count.argtypes = [vp, vp, vp, u64, C.c_int, vp, C.POINTER(FmQuery)]
        L.grlgpu_fm_locate.argtypes = [vp, vp, vp, u64, C.c_int, vp, vp, vp, u64, C.POINTER(FmQuery)]
        L.grlgpu_fm_approx_count.argtypes = [vp, vp, vp, u64, C.c_int, C.c_uint32, vp, vp, vp, u64, C.POINTER(FmApprox)]
        L.grlgpu_fm_approx_locate.argtypes = [vp, vp, vp, u64, C.c_int, C.c_uint32, vp, vp, vp, vp, u64, C.POINTER(FmApprox)]
        L.grlgpu_fm_extract.argtypes = [vp, vp, vp, vp, u64, C.c_int, vp, vp, u64, C.POINTER(FmExtract)]
        L.grlgpu_fm_drop.argtypes = [vp]
        L.grlgpu_selftest_scan.argtypes = [vp, u64, vp, vp]
        L.grlgpu_selftest_sort.argtypes = [vp, vp, u64, C.c_int]
        L.grlgpu_selftest_compact.argtypes = [vp, vp, u64, vp, vp]
        L.grlgpu_selftest_ipc_rendezvous.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int]
        _gpu = L
    return _gpu


def lib_host():
    global _host
    if _host is None:
        lib_gpu()
        path = os.path.join(LIB_DIR, "libgrlbwt.so")
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: build it with `make -C grlbwt_b200`")
        L = C.CDLL(path)
        L.grlbwt_build.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(BwtResult)]
        L.grlbwt_free_result.argtypes = [C.POINTER(BwtResult)]
        L.grlbwt_build_file.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.grlbwt_last_error.restype = C.c_char_p
        L.grlbwt_build_mg.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(BwtResult)]
        L.grlbwt_build_to.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(BwtResult)]
        L.grlbwt_build_packed.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64),
                                          C.POINTER(BwtResult)]
        L.grlbwt_last_digests.argtypes = [C.c_void_p, C.c_uint64]
        L.grlbwt_last_digests.restype = C.c_uint64
        L.grlbwt_last_exchange_bytes.restype = C.c_uint64
        L.grlbwt_last_comm.restype = C.c_char_p
        _host = L
    return _host


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _carve(sizes, arena, offset):
    """[(count, dtype)] -> (arrays, end): fresh zeroed arrays (end None) without an arena, else views of `arena` placed from byte
    `offset` on at 16-byte boundaries, and the 16-byte aligned end of the last one"""
    if arena is None:
        return [np.zeros(n, dt) for n, dt in sizes], None
    arrs, off = [], int(offset)
    for n, dt in sizes:
        nb = n * np.dtype(dt).itemsize
        off = (off + 15) & ~15
        if off + nb > arena.size:
            raise GrlGpuError(-1, "fetch arena too small")
        arrs.append(arena[off:off + nb].view(dt))
        off += nb
    return arrs, (off + 15) & ~15


class GrlGpu:
    """One device context = the GPU parse strategy (mirrors the duck-typed strategy concept used by
    par_round, exact_par_phase.cpp:374-497: get_phrases / map / parse_text, fused into round())."""

    def __init__(self, device: int = 0, flags: int = 0, stream: int = 0):
        self._L = lib_gpu()
        self._h = C.c_void_p()
        self._check(self._L.grlgpu_create_on_stream(C.byref(self._h), device, flags, C.c_void_p(stream) if stream else None), ctx=False)
        self.last = None
        self._keep = None
        self._sym_bytes = 1
        self._round_started = False

    def _check(self, rc, ctx=True):
        if rc != 0:
            msg = self._L.grlgpu_strerror(rc).decode()
            if ctx and self._h:
                msg += " | " + self._L.grlgpu_last_error(self._h).decode()
            raise GrlGpuError(rc, msg)

    def set_text(self, text: np.ndarray):
        text = np.ascontiguousarray(text)
        if text.dtype not in (np.uint8, np.uint16, np.uint32, np.uint64):
            raise GrlGpuError(-1, "symbol width must be 1, 2, 4 or 8 bytes")
        self._keep = text
        self._sym_bytes, self._round_started, self.last = text.dtype.itemsize, False, None
        self._check(self._L.grlgpu_set_text(self._h, _ptr(text) if text.size else None, text.size, text.dtype.itemsize))

    def set_text_device(self, dev_ptr: int, n_syms: int, sym_bytes: int):
        self._keep, self._sym_bytes, self._round_started, self.last = None, sym_bytes, False, None
        self._check(self._L.grlgpu_set_text_device(self._h, C.c_void_p(dev_ptr), n_syms, sym_bytes))

    def stats(self) -> Stats:
        s = Stats()
        self._check(self._L.grlgpu_stats(self._h, C.byref(s)))
        return s

    def round(self) -> Round:
        r = Round()
        self._check(self._L.grlgpu_round(self._h, C.byref(r)))
        self.last = r
        self._round_started = True
        return r

    def level_checksum(self):
        """four order-insensitive sums over the last round's rules / hocc marks / preliminary BWT (see grlgpu.h)"""
        out = np.zeros(4, np.uint64)
        self._check(self._L.grlgpu_level_checksum(self._h, _ptr(out)))
        return [int(x) for x in out]

    def fetch_wait(self):
        self._check(self._L.grlgpu_fetch_wait(self._h))

    def fetch_level(self, arena: np.ndarray | None = None, widen: bool = True, async_: bool = False, offset: int = 0, narrow_len: bool = False):
        """-> dict(rule_l, rule_r, has_hocc, pre_sym, pre_len) as numpy arrays.
        arena: optional uint8 buffer (e.g. pinned host memory) the arrays are carved from, so the copies are
        direct DMA; widen=False keeps rule/pre_sym in the device's element width (sym_bytes) instead of u64;
        narrow_len: 32-bit run lengths (grlgpu_fetch_level32) whenever the round's n_in + parse_len < 2^32."""
        r = self.last
        st = np.uint32 if r.sym_bytes == 4 else np.uint64
        narrow = bool(narrow_len) and r.n_in + r.parse_len < (1 << 32)
        sizes = [(r.tot_phrases, st), (r.tot_phrases, st), (r.tot_phrases, np.uint8), (r.n_pre_runs, st), (r.n_pre_runs, np.uint32 if narrow else np.uint64)]
        (rl, rr, hh, ps, pl), end = _carve(sizes, arena, offset)
        if narrow:
            self._check(self._L.grlgpu_fetch_level32(self._h, _ptr(rl), _ptr(rr), _ptr(hh), _ptr(ps), _ptr(pl), int(async_)))
        else:
            fn = self._L.grlgpu_fetch_level_async if async_ else self._L.grlgpu_fetch_level
            self._check(fn(self._h, _ptr(rl), _ptr(rr), _ptr(hh), _ptr(ps), _ptr(pl)))
        if arena is not None:
            self.arena_end = end
        if widen and arena is None:
            rl, rr, ps = rl.astype(np.uint64), rr.astype(np.uint64), ps.astype(np.uint64)
        return {"rule_l": rl, "rule_r": rr, "has_hocc": hh, "pre_sym": ps, "pre_len": pl}

    def fetch_parse(self, arena: np.ndarray | None = None) -> np.ndarray:
        r = self.last
        if arena is None:
            out = np.zeros(r.parse_len, CELL[r.cell_bytes_out])
        else:
            out = arena[: r.parse_len * r.cell_bytes_out].view(CELL[r.cell_bytes_out])
        self._check(self._L.grlgpu_fetch_parse(self._h, _ptr(out)))
        return out

    def fetch_str_ptrs(self) -> np.ndarray:
        out = np.zeros(self.last.n_strings + 1, np.uint64)
        self._check(self._L.grlgpu_fetch_str_ptrs(self._h, _ptr(out)))
        return out

    def fetch_dictionary(self):
        r = self.last
        syms, lens = np.zeros(r.dict_syms, np.uint64), np.zeros(r.n_phrases, np.uint64)
        freqs, metas = np.zeros(r.n_phrases, np.uint64), np.zeros(r.n_phrases, np.uint64)
        self._check(self._L.grlgpu_fetch_dictionary(self._h, _ptr(syms), _ptr(lens), _ptr(freqs), _ptr(metas)))
        return syms, lens, freqs, metas

    # ---- multi-GPU rounds: every rank makes the same calls in the same order (include/grlgpu.h) ----
    def histogram(self) -> np.ndarray:
        h = np.zeros(256, np.uint64)
        self._check(self._L.grlgpu_histogram(self._h, _ptr(h)))
        return h

    def set_peers(self, devices):
        d = np.asarray(devices, np.int32)
        self._check(self._L.grlgpu_set_peers(self._h, _ptr(d), d.size))

    def mg_stats(self, comm) -> Stats:
        s = Stats()
        self._check(self._L.grlgpu_mg_stats(self._h, comm.handle, C.byref(s)))
        return s

    def mg_round(self, comm) -> Round:
        r = Round()
        self._check(self._L.grlgpu_mg_round(self._h, comm.handle, C.byref(r)))
        self.last = r
        self._round_started = True
        return r

    def mg_slice_info(self) -> Slice:
        s = Slice()
        self._check(self._L.grlgpu_mg_slice_info(self._h, C.byref(s)))
        return s

    def mg_slice_checksum(self):
        out = np.zeros(4, np.uint64)
        self._check(self._L.grlgpu_mg_slice_checksum(self._h, _ptr(out)))
        return [int(x) for x in out]

    def mg_fetch_slice(self, arena: np.ndarray | None = None, offset: int = 0, narrow_len: bool = False, async_: bool = False):
        """this rank's part of the last level -> dict of numpy arrays (carved from `arena`, e.g. pinned memory, when given)"""
        sl = self.mg_slice_info()
        st = np.uint32 if sl.sym_bytes == 4 else np.uint64
        sizes = [(sl.tot_local, st), (sl.tot_local, st), (sl.tot_local, np.uint8), (sl.n_pre_local, st), (sl.n_pre_local, np.uint32 if narrow_len else np.uint64)]
        (rl, rr, hh, ps, pl), end = _carve(sizes, arena, offset)
        if arena is not None:
            self.arena_end = end
        self._check(self._L.grlgpu_mg_fetch_slice(self._h, _ptr(rl), _ptr(rr), _ptr(hh), _ptr(ps), _ptr(pl), 4 if narrow_len else 8, int(async_)))
        return {"rule_l": rl, "rule_r": rr, "has_hocc": hh, "pre_sym": ps, "pre_len": pl, "rank_base": sl.rank_base, "pre_first": sl.pre_first}

    def fetch_parse_local(self, n_cells: int, arena: np.ndarray | None = None) -> np.ndarray:
        """multi-GPU: this rank's part of the current parse (parse_len_local cells of grlgpu_slice_t)"""
        r = self.last
        out = np.zeros(n_cells, CELL[r.cell_bytes_out]) if arena is None else arena[: n_cells * r.cell_bytes_out].view(CELL[r.cell_bytes_out])
        self._check(self._L.grlgpu_fetch_parse(self._h, _ptr(out)))
        return out

    def invert(self, image, cell_bytes: int = 1, n_seqs: int | None = None, out: np.ndarray | None = None):
        """invert_rl_bwt on this context (its text, levels and BWT are left as they are)"""
        raw, out = _invert_args(image, cell_bytes, n_seqs, out)
        info = Invert()
        rc = self._L.grlgpu_invert(self._h, _ptr(raw), raw.size, cell_bytes, (1 << 64) - 1 if n_seqs is None else int(n_seqs), _ptr(out), out.size, C.byref(info))
        d = {k: getattr(info, k) for k, _ in Invert._fields_}
        if rc != 0:
            err = GrlGpuError(rc, self._L.grlgpu_strerror(rc).decode() + " | " + self._L.grlgpu_last_error(self._h).decode())
            err.info = d
            raise err
        return out[: d["n_out"] * cell_bytes].view(CELL[cell_bytes]), d

    def _fm_call(self, rc, info):
        d = {k: getattr(info, k) for k, _ in type(info)._fields_}
        if rc != 0:
            err = GrlGpuError(rc, self._L.grlgpu_strerror(rc).decode() + " | " + self._L.grlgpu_last_error(self._h).decode())
            err.info = d
            raise err
        return d

    def fm_load(self, image):
        """Loads a .rl_bwt image (what parse_rl_bwt takes: a path, bytes or a uint8 array) as this context's FM-index, replacing the
        one loaded before; its text, levels and BWT are left as they are. -> dict of grlgpu_fm_t (n, n_strings, n_runs, sigma, sep)"""
        raw = _image_bytes(image)
        info = FmInfo()
        return self._fm_call(self._L.grlgpu_fm_load(self._h, _ptr(raw), raw.size, C.byref(info)), info)

    def fm_count(self, patterns):
        """Backward search of every pattern (see _fm_patterns for the forms accepted) -> (sp, ep, info): uint64 arrays, the rows
        [sp, ep) whose suffix starts with the pattern (sp = ep = 0 when it does not occur), and the dict of grlgpu_fm_query_t"""
        cells, off = _fm_patterns(patterns)
        n_pat = off.size - 1
        sp_ep = np.zeros(2 * max(n_pat, 1), np.uint64)
        info = FmQuery()
        d = self._fm_call(self._L.grlgpu_fm_count(self._h, _ptr(cells), _ptr(off), n_pat, cells.dtype.itemsize, _ptr(sp_ep), C.byref(info)), info)
        return sp_ep[0:2 * n_pat:2].copy(), sp_ep[1:2 * n_pat:2].copy(), d

    def fm_locate(self, patterns):
        """Every occurrence of every pattern -> (occ_off, str_id, str_pos, info): pattern q's occurrences are
        [occ_off[q], occ_off[q + 1]) of str_id (string k) and str_pos (offset p), in row order. The output is sized by a count call."""
        cells, off = _fm_patterns(patterns)
        n_pat = off.size - 1
        sp, ep, _ = self.fm_count((cells, off))
        n_occ = int((ep - sp).sum())
        occ_off = np.zeros(n_pat + 1, np.uint64)
        str_id, str_pos = np.zeros(max(n_occ, 1), np.uint32), np.zeros(max(n_occ, 1), np.uint32)
        info = FmQuery()
        d = self._fm_call(self._L.grlgpu_fm_locate(self._h, _ptr(cells), _ptr(off), n_pat, cells.dtype.itemsize, _ptr(occ_off), _ptr(str_id), _ptr(str_pos),
                                                   n_occ, C.byref(info)), info)
        return occ_off, str_id[:n_occ], str_pos[:n_occ], d

    def fm_approx_count(self, patterns, k: int):
        """Search with at most k <= 3 mismatches (substitutions) -> (hit_off, sp, ep, mm, info): pattern q's hits are
        [hit_off[q], hit_off[q + 1]) of the uint64 arrays sp, ep and the uint8 array mm; a hit is one distinct string Q within
        Hamming distance mm of the pattern that occurs, at the rows [sp, ep), listed by ascending sp. info is the dict of
        grlgpu_fm_approx_t (n_occ = the sum of ep - sp). The hits are written into a guessed capacity; when it is short, a second
        call writes them, and device_ms / search_ms are the sums of both calls."""
        cells, off, k = _fm_approx_args(patterns, k)
        n_pat = off.size - 1
        hit_off = np.zeros(n_pat + 1, np.uint64)
        cap, first = max(1024, 4 * n_pat), None
        while True:
            sp_ep, mm, info = np.zeros(2 * cap, np.uint64), np.zeros(cap, np.uint8), FmApprox()
            rc = self._L.grlgpu_fm_approx_count(self._h, _ptr(cells), _ptr(off), n_pat, cells.dtype.itemsize, k, _ptr(hit_off), _ptr(sp_ep), _ptr(mm), cap,
                                                C.byref(info))
            if first is not None or rc != -1 or info.n_hits <= cap:
                break
            first, cap = {f: getattr(info, f) for f, _ in FmApprox._fields_}, int(info.n_hits)
        d = self._fm_call(rc, info)
        if first:
            d["device_ms"] += first["device_ms"]
            d["search_ms"] += first["search_ms"]
        n = d["n_hits"]
        return hit_off, sp_ep[0:2 * n:2].copy(), sp_ep[1:2 * n:2].copy(), mm[:n].copy(), d

    def fm_approx_locate(self, patterns, k: int):
        """Every occurrence with at most k <= 3 mismatches -> (occ_off, str_id, str_pos, mm, info): pattern q's occurrences are
        [occ_off[q], occ_off[q + 1]) of str_id (string k), str_pos (offset p) and mm (mismatches d), in row order. The output is
        sized by a fm_approx_count call."""
        cells, off, k = _fm_approx_args(patterns, k)
        n_pat = off.size - 1
        n_occ = int(self.fm_approx_count((cells, off), k)[4]["n_occ"])
        occ_off = np.zeros(n_pat + 1, np.uint64)
        str_id, str_pos, mm = np.zeros(max(n_occ, 1), np.uint32), np.zeros(max(n_occ, 1), np.uint32), np.zeros(max(n_occ, 1), np.uint8)
        info = FmApprox()
        d = self._fm_call(self._L.grlgpu_fm_approx_locate(self._h, _ptr(cells), _ptr(off), n_pat, cells.dtype.itemsize, k, _ptr(occ_off), _ptr(str_id),
                                                          _ptr(str_pos), _ptr(mm), n_occ, C.byref(info)), info)
        return occ_off, str_id[:n_occ], str_pos[:n_occ], mm[:n_occ], d

    def fm_extract(self, str_id, start=0, length=None, cell_bytes: int = 1):
        """Substrings of the indexed strings (see _fm_requests for the forms accepted) -> (out_off, cells, info): request q is
        S_k[start .. min(start + length, |S_k|)) with k = str_id[q] (to the end of the string when length is None), the cells
        [out_off[q], out_off[q + 1]) of `cells`, whose dtype has cell_bytes bytes (each cell the symbol's low bytes), and the dict
        of grlgpu_fm_extract_t. The output is sized from the lengths when they are given and small, else by a first call without
        capacity; info then covers both calls: device_ms and extract_ms are their sums, jump_rounds those of the call that built
        the locate table."""
        ids, frm, ln = _fm_requests(str_id, start, length, cell_bytes)
        n_req = ids.size
        out_off = np.zeros(n_req + 1, np.uint64)
        info = FmExtract()
        cap = int(ln.sum(dtype=np.uint64)) if length is not None else None
        sizing = None
        if cap is None or cap > _FM_EXTRACT_DIRECT_CAP:
            rc = self._L.grlgpu_fm_extract(self._h, _ptr(ids), _ptr(frm), _ptr(ln), n_req, cell_bytes, _ptr(out_off), None, 0, C.byref(info))
            if rc != -1 or info.n_cells == 0:   # done (no cells), or an error other than the capacity
                return out_off, np.zeros(0, CELL[cell_bytes]), self._fm_call(rc, info)
            sizing = {k: getattr(info, k) for k, _ in FmExtract._fields_}
            cap = int(info.n_cells)
        cells = np.zeros(max(cap, 1), CELL[cell_bytes])
        d = self._fm_call(self._L.grlgpu_fm_extract(self._h, _ptr(ids), _ptr(frm), _ptr(ln), n_req, cell_bytes, _ptr(out_off), _ptr(cells), cap, C.byref(info)), info)
        if sizing:
            d["device_ms"] += sizing["device_ms"]
            d["extract_ms"] += sizing["extract_ms"]
            d["jump_rounds"] = max(d["jump_rounds"], sizing["jump_rounds"])
        n = d["n_cells"]
        return out_off, (cells[:n].copy() if n < cap // 2 else cells[:n]), d   # lengths past the strings: do not keep the whole allocation

    def fm_drop(self):
        """Frees this context's FM-index"""
        self._check(self._L.grlgpu_fm_drop(self._h))

    def profile_enable(self, on: bool = True):
        self._check(self._L.grlgpu_profile_enable(self._h, int(on)))

    def profile_reset(self):
        self._check(self._L.grlgpu_profile_reset(self._h))

    def launch_count(self) -> int:
        return int(self._L.grlgpu_launch_count(self._h))

    def profile(self):
        """-> {kernel name: (launches, total_ms, model_bytes)} measured with CUDA events on the launch stream"""
        out, i = {}, 0
        name = C.create_string_buffer(128)
        n, ms, by = C.c_uint64(), C.c_double(), C.c_uint64()
        while self._L.grlgpu_profile_entry(self._h, i, name, 128, C.byref(n), C.byref(ms), C.byref(by)) == 0:
            out[name.value.decode()] = (int(n.value), float(ms.value), int(by.value))
            i += 1
        return out

    def close(self):
        if self._h:
            self._L.grlgpu_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def build_bwt(text: np.ndarray, device: int = 0, n_threads: int = 1, verbose: bool = False):
    """Whole construction (device parse phase + host induction) -> (syms u64, lens u64, sb, fb, info dict)."""
    L = lib_host()
    text = np.ascontiguousarray(text)
    res = BwtResult()
    rc = L.grlbwt_build(_ptr(text), text.size, text.dtype.itemsize, device, n_threads, int(verbose), C.byref(res))
    if rc != 0:
        raise GrlGpuError(rc, L.grlbwt_last_error().decode())
    try:
        syms = np.ctypeslib.as_array(res.syms, shape=(res.n_runs,)).copy()
        lens = np.ctypeslib.as_array(res.lens, shape=(res.n_runs,)).copy()
        info = {k: getattr(res, k) for k in ("n_rounds", "h2d_ms", "par_phase_ms", "ind_phase_ms", "device_ms", "algorithmic_bytes", "induced_on_device")}
        return syms, lens, int(res.sb), int(res.fb), info
    finally:
        L.grlbwt_free_result(C.byref(res))


def build_bwt_to(text: np.ndarray, out_syms: np.ndarray, out_lens: np.ndarray, devices=(0,), n_threads: int = 1, comm: int = 0):
    """Whole construction with the run-length BWT delivered into caller-owned uint32 arrays (e.g. views of pinned memory that is
    reused from call to call). -> (n_runs, sb, fb, info)"""
    L = lib_host()
    text = np.ascontiguousarray(text)
    assert out_syms.dtype == np.uint32 and out_lens.dtype == np.uint32 and out_syms.flags.c_contiguous and out_lens.flags.c_contiguous
    dv = np.asarray(devices, np.int32)
    res = BwtResult()
    rc = L.grlbwt_build_to(_ptr(text), text.size, text.dtype.itemsize, _ptr(dv), dv.size, n_threads, comm, _ptr(out_syms), _ptr(out_lens),
                           min(out_syms.size, out_lens.size), C.byref(res))
    if rc != 0:
        raise GrlGpuError(rc, L.grlbwt_last_error().decode())
    info = {k: getattr(res, k) for k in ("n_rounds", "h2d_ms", "par_phase_ms", "ind_phase_ms", "device_ms", "algorithmic_bytes", "induced_on_device")}
    return int(res.n_runs), int(res.sb), int(res.fb), info


def build_bwt_packed(text: np.ndarray, out_image: np.ndarray, devices=(0,), n_threads: int = 1, comm: int = 0):
    """Whole construction with the run-length BWT delivered as the image of the .rl_bwt file ([sb u64][fb u64] + records of sb + fb
    bytes) in a caller-owned uint8 array; the records are packed on the device. -> (image_bytes, n_runs, sb, fb, info)"""
    L = lib_host()
    text = np.ascontiguousarray(text)
    assert out_image.dtype == np.uint8 and out_image.flags.c_contiguous
    dv = np.asarray(devices, np.int32)
    res = BwtResult()
    nb = C.c_uint64()
    rc = L.grlbwt_build_packed(_ptr(text), text.size, text.dtype.itemsize, _ptr(dv), dv.size, n_threads, comm, _ptr(out_image), out_image.size, C.byref(nb), C.byref(res))
    if rc != 0:
        raise GrlGpuError(rc, L.grlbwt_last_error().decode())
    info = {k: getattr(res, k) for k in ("n_rounds", "h2d_ms", "par_phase_ms", "ind_phase_ms", "device_ms", "algorithmic_bytes", "induced_on_device")}
    return int(nb.value), int(res.n_runs), int(res.sb), int(res.fb), info


def parse_rl_bwt(image) -> tuple:
    """The .rl_bwt format (reference include/bwt_io.h:377-382,448-490) as numpy arrays: `image` is a file path or the bytes /
    uint8 array of a file image (what build_bwt_packed fills). -> (syms uint64[r], lens uint64[r], sb, fb). Host-side helper."""
    raw = np.fromfile(image, np.uint8) if isinstance(image, (str, os.PathLike)) else np.frombuffer(image, np.uint8)
    if raw.size < 16:
        raise ValueError("truncated header")
    sb, fb = (int(x) for x in raw[:16].view(np.uint64))
    if not (1 <= sb <= 8 and 1 <= fb <= 8):
        raise ValueError(f"bad header widths sb={sb} fb={fb}")
    body = raw[16:]
    if body.size % (sb + fb):
        raise ValueError("truncated record at the end of the image")
    rec = body.reshape(-1, sb + fb)
    syms = np.zeros(rec.shape[0], np.uint64)
    lens = np.zeros(rec.shape[0], np.uint64)
    for i in range(sb):
        syms |= rec[:, i].astype(np.uint64) << np.uint64(8 * i)
    for i in range(fb):
        lens |= rec[:, sb + i].astype(np.uint64) << np.uint64(8 * i)
    return syms, lens, sb, fb


def _image_bytes(image) -> np.ndarray:
    """a .rl_bwt image as contiguous uint8: a path is read, bytes and arrays are viewed"""
    if isinstance(image, (str, os.PathLike)):
        return np.fromfile(image, np.uint8)
    return np.ascontiguousarray(np.frombuffer(image, np.uint8))


def _fm_patterns(patterns) -> tuple:
    """checks of the patterns of fm_count / fm_locate, before the library is called -> (cells, uint64 offsets). Accepted: a list
    of patterns (bytes, or 1-d arrays of one unsigned cell type), or a tuple (concatenated cells, offsets) with offsets[0] = 0.
    Every pattern has at least one cell."""
    if isinstance(patterns, tuple):
        if len(patterns) != 2:
            raise GrlGpuError(-1, "patterns: a pair (cells, offsets) is expected")
        cells, off = np.asarray(patterns[0]), np.asarray(patterns[1])
        if off.ndim != 1 or off.size == 0 or off.dtype.kind not in "iu":
            raise GrlGpuError(-1, "patterns: offsets must be a non-empty 1-d integer array")
        if off.dtype.kind == "i" and (off < 0).any():
            raise GrlGpuError(-1, "patterns: offsets must not be negative")
        off = off.astype(np.uint64)
    elif isinstance(patterns, list):
        parts = [np.frombuffer(p, np.uint8) if isinstance(p, (bytes, bytearray)) else np.asarray(p) for p in patterns]
        if any(p.ndim != 1 for p in parts):
            raise GrlGpuError(-1, "patterns: every pattern must be bytes or a 1-d array")
        kinds = {p.dtype for p in parts}
        if len(kinds) > 1:
            raise GrlGpuError(-1, "patterns: every pattern must have the same cell type")
        dt = kinds.pop() if kinds else np.dtype(np.uint8)
        cells = np.concatenate(parts).astype(dt, copy=False) if parts else np.zeros(0, dt)
        off = np.zeros(len(parts) + 1, np.uint64)
        off[1:] = np.cumsum([p.size for p in parts], dtype=np.uint64)
    else:
        raise GrlGpuError(-1, "patterns: a list of patterns or a pair (cells, offsets) is expected")
    if cells.ndim != 1 or cells.dtype not in [np.dtype(t) for t in CELL.values()]:
        raise GrlGpuError(-1, "patterns: cells must be a 1-d array of uint8, uint16, uint32 or uint64")
    if off[0] != 0 or int(off[-1]) > cells.size:
        raise GrlGpuError(-1, "patterns: offsets must start at 0 and end inside the cells")
    if (np.diff(off.astype(np.int64)) <= 0).any():
        raise GrlGpuError(-1, "patterns: every pattern must have at least one cell (offsets strictly increasing)")
    return np.ascontiguousarray(cells), np.ascontiguousarray(off)


def _fm_approx_args(patterns, k) -> tuple:
    """checks of fm_approx_count / fm_approx_locate, before the library is called -> (cells, uint64 offsets, k): the patterns as
    _fm_patterns takes them, k an integer from 0 to 3"""
    if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)) or not 0 <= int(k) <= 3:
        raise GrlGpuError(-1, "approximate search: k must be an integer from 0 to 3")
    cells, off = _fm_patterns(patterns)
    return cells, off, int(k)


_FM_EXTRACT_DIRECT_CAP = 1 << 26   # fm_extract: cells allocated up front from the given lengths; beyond, the library sizes the output
_U32_MAX = (1 << 32) - 1


def _fm_requests(str_id, start=0, length=None, cell_bytes=1) -> tuple:
    """checks of fm_extract's arguments, before the library is called -> three contiguous uint32 arrays (str_id, start, length).
    str_id is an integer or a 1-d integer array; start and length are integers or 1-d integer arrays of its size; length None means
    to the end of the string. Offsets are 32-bit on the device: a length beyond 32 bits is taken as 2^32 - 1 (still to the end), a
    start at or beyond 2^32 gives an empty substring."""
    if cell_bytes not in CELL:
        raise GrlGpuError(-1, "extract: cell_bytes must be 1, 2, 4 or 8")
    n_req = np.asarray(str_id).size if np.ndim(str_id) else 1
    cols = []
    for v, what in ((str_id, "str_id"), (start, "start"), (length, "length")):
        a = np.asarray(_U32_MAX if v is None else v)
        if a.size == 0:
            a = a.astype(np.uint64)
        if a.ndim > 1 or a.dtype.kind not in "iu":
            raise GrlGpuError(-1, f"extract: {what} must be an integer or a 1-d integer array")
        if a.dtype.kind == "i" and (a < 0).any():
            raise GrlGpuError(-1, f"extract: {what} must not be negative")
        a = a.astype(np.uint64)
        if a.ndim == 0:
            a = np.full(n_req, a, np.uint64)
        elif a.size != n_req:
            raise GrlGpuError(-1, f"extract: {what} has {a.size} entries for {n_req} requests")
        cols.append(a)
    ids, frm, ln = cols
    if (ids > _U32_MAX).any():
        raise GrlGpuError(-1, "extract: str_id must be below 2^32")
    far = frm > _U32_MAX
    return (np.ascontiguousarray(ids.astype(np.uint32)), np.ascontiguousarray(np.where(far, _U32_MAX, frm).astype(np.uint32)),
            np.ascontiguousarray(np.where(far, 0, np.minimum(ln, _U32_MAX)).astype(np.uint32)))


def _invert_args(image, cell_bytes, n_seqs, out):
    """checks of invert_rl_bwt's arguments, before the library is called -> (uint8 image, output buffer)"""
    if cell_bytes not in CELL:
        raise GrlGpuError(-1, "cell_bytes must be 1, 2, 4 or 8")
    if n_seqs is not None and int(n_seqs) < 0:
        raise GrlGpuError(-1, "n_seqs must be >= 0")
    if out is not None and (not isinstance(out, np.ndarray) or out.dtype != np.uint8 or out.ndim != 1 or not out.flags.c_contiguous or not out.flags.writeable):
        raise GrlGpuError(-1, "out must be a writable contiguous 1-d uint8 array")
    raw = np.fromfile(image, np.uint8) if isinstance(image, (str, os.PathLike)) else np.ascontiguousarray(np.frombuffer(image, np.uint8))
    if out is None:   # the BWT length n bounds the output; a malformed header is left to the library to report
        n = 0
        if raw.size >= 16:
            sb, fb = (int(x) for x in raw[:16].view(np.uint64))
            if 1 <= sb <= 8 and 1 <= fb <= 8:
                rec = raw[16:16 + (raw.size - 16) // (sb + fb) * (sb + fb)].reshape(-1, sb + fb)
                n = sum(int(rec[:, sb + i].sum(dtype=np.uint64)) << (8 * i) for i in range(fb))
        out = np.zeros(n * cell_bytes, np.uint8)
    return raw, out


def invert_rl_bwt(image, cell_bytes: int = 1, n_seqs: int | None = None, device: int = 0, flags: int = 0, out: np.ndarray | None = None):
    """Inverts a BCR BWT on the device (grlgpu_invert): `image` is what parse_rl_bwt takes (a path, bytes or a uint8 array).
    -> (the first min(n_seqs, N) strings, each followed by the separator, as cells of cell_bytes bytes; dict of grlgpu_invert_t).
    out: optional caller-owned uint8 buffer (e.g. pinned memory) the cells are written to; the result is a view of it.
    Errors of the call raise GrlGpuError, whose `info` holds the dict (n_out = cells needed when `out` is too small)."""
    raw, out = _invert_args(image, cell_bytes, n_seqs, out)
    with GrlGpu(device, flags) as ctx:
        return ctx.invert(raw, cell_bytes, n_seqs, out)


def build_bwt_file(inp: str, out: str, sym_bytes: int = 1, device: int = 0, n_threads: int = 1, verbose: bool = False):
    L = lib_host()
    rc = L.grlbwt_build_file(inp.encode(), out.encode(), sym_bytes, device, n_threads, int(verbose))
    if rc != 0:
        raise GrlGpuError(rc, L.grlbwt_last_error().decode())


def selftest_induce(levels, final_parse: np.ndarray, n_threads: int = 0):
    """levels: list of dicts with alphabet, tot, rule_l, rule_r (u64), has_hocc (u8), pre_sym, pre_len (u64). CPU only."""
    L = lib_host()
    n = len(levels)
    u64p, u8p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint8)
    keep = []

    def arr(key, dt, ptype):
        out = (ptype * n)()
        for i, lv in enumerate(levels):
            a = np.ascontiguousarray(lv[key], dt)
            if a.size == 0:
                a = np.zeros(1, dt)
            keep.append(a)
            out[i] = a.ctypes.data_as(ptype)
        return out

    alph = np.array([lv["alphabet"] for lv in levels], np.uint64)
    tot = np.array([lv["tot"] for lv in levels], np.uint64)
    npre = np.array([len(lv["pre_sym"]) for lv in levels], np.uint64)
    fp = np.ascontiguousarray(final_parse, np.uint64)
    res = BwtResult()
    L.grlbwt_selftest_induce.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.POINTER(u64p), C.POINTER(u64p), C.POINTER(u8p), C.c_void_p,
                                         C.POINTER(u64p), C.POINTER(u64p), C.c_void_p, C.c_uint64, C.c_int, C.POINTER(BwtResult)]
    rc = L.grlbwt_selftest_induce(n, _ptr(alph), _ptr(tot), arr("rule_l", np.uint64, u64p), arr("rule_r", np.uint64, u64p),
                                  arr("has_hocc", np.uint8, u8p), _ptr(npre), arr("pre_sym", np.uint64, u64p), arr("pre_len", np.uint64, u64p),
                                  _ptr(fp), fp.size, n_threads, C.byref(res))
    if rc != 0:
        raise RuntimeError(L.grlbwt_last_error().decode())
    try:
        return (np.ctypeslib.as_array(res.syms, shape=(res.n_runs,)).copy(), np.ctypeslib.as_array(res.lens, shape=(res.n_runs,)).copy())
    finally:
        L.grlbwt_free_result(C.byref(res))


def selftest_scan(a: np.ndarray):
    a = np.ascontiguousarray(a, np.uint32)
    out, tot = np.zeros(a.size, np.uint64), np.zeros(1, np.uint64)
    rc = lib_gpu().grlgpu_selftest_scan(_ptr(a), a.size, _ptr(out), _ptr(tot))
    if rc != 0:
        raise GrlGpuError(rc, lib_gpu().grlgpu_strerror(rc).decode())
    return out, int(tot[0])


def selftest_sort(keys: np.ndarray, vals: np.ndarray, n_bits: int):
    k, v = np.ascontiguousarray(keys, np.uint64).copy(), np.ascontiguousarray(vals, np.uint32).copy()
    rc = lib_gpu().grlgpu_selftest_sort(_ptr(k), _ptr(v), k.size, n_bits)
    if rc != 0:
        raise GrlGpuError(rc, lib_gpu().grlgpu_strerror(rc).decode())
    return k, v


def selftest_compact(bits: np.ndarray, prev_bits, n_bits: int):
    b = np.ascontiguousarray(bits, np.uint32)
    pb = None if prev_bits is None else np.ascontiguousarray(prev_bits, np.uint32)
    out, cnt = np.zeros(max(1, n_bits), np.uint64), np.zeros(1, np.uint64)
    rc = lib_gpu().grlgpu_selftest_compact(_ptr(b), _ptr(pb), n_bits, _ptr(out), _ptr(cnt))
    if rc != 0:
        raise GrlGpuError(rc, lib_gpu().grlgpu_strerror(rc).decode())
    return out[: int(cnt[0])]

"""ctypes front-end of the CPU oracle (TEST INFRASTRUCTURE ONLY).

Loads oracle/libwf_oracle.so (plain-C restatement of the reference algorithms, see wf_oracle.c) and, when
present, the reference pins under oracle/_ref/ (the reference's own wf/flatfat.hpp / wf/flatfat_gpu.hpp
compiled unmodified by oracle/Makefile). Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this module; windflow_b200/ never does.
"""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

TUPLE64 = np.dtype([("key", "<u8"), ("id", "<u8"), ("ivalue", "<i8"), ("fvalue", "<f8"), ("pad", "<u8", (4,))])
RES = np.dtype([("key", "<u8"), ("id", "<u8"), ("isum", "<i8"), ("fsum", "<f8")])
assert TUPLE64.itemsize == 64 and RES.itemsize == 32

SEED = 0x5EED5EED  # SURVEY.md section 8d
KEY_RR, KEY_UNIFORM, KEY_ZIPF = 0, 1, 2
MAP_NONE, MAP_ADD_SCALE = 0, 1
FILT_NONE, FILT_EVEN, FILT_MOD = 0, 1, 2

_u64, _i64, _f64, _u32, _i32, _u8 = C.c_uint64, C.c_int64, C.c_double, C.c_uint32, C.c_int32, C.c_uint8
_vp = C.c_void_p


def build(force=False):
    """Compile the oracle (and the reference pins when /root/reference exists)."""
    so = os.path.join(HERE, "libwf_oracle.so")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(os.path.join(HERE, "wf_oracle.c")):
        subprocess.check_call(["make", "-C", HERE, "-s", os.path.join(HERE, "libwf_oracle.so")])
    if os.path.isdir("/root/reference/wf"):
        subprocess.check_call(["make", "-C", HERE, "-s", "ref"])


def _p(a):
    return a.ctypes.data_as(_vp)


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(os.path.join(HERE, "libwf_oracle.so"))
        L.wfo_gen_tuple64.argtypes = [_u64, _u64, _u64, C.c_int, _u64, _vp, _vp, _vp]
        L.wfo_map.argtypes = [_vp, _vp, _u64, C.c_int, _i64, _f64]
        L.wfo_filter_mask.argtypes = [_vp, _u64, C.c_int, _i64, _vp]
        L.wfo_filter_mask.restype = _u64
        L.wfo_keyby_group.argtypes = [_vp, _u64, C.c_int, _vp, _vp, _vp]
        L.wfo_keyby_group.restype = _u64
        L.wfo_route.argtypes = [_vp, _u64, _u32, _vp]
        L.wfo_reduce_by_key.argtypes = [_vp, _vp, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp]
        L.wfo_reduce_by_key.restype = _u64
        L.wfo_ffat_gpu_create.argtypes = [_u64, _u64, _u64, C.c_int]
        L.wfo_ffat_gpu_create.restype = _vp
        L.wfo_ffat_gpu_destroy.argtypes = [_vp]
        L.wfo_ffat_gpu_process_batch.argtypes = [_vp, _vp, _u64, _u64, _vp, _vp, _u64]
        L.wfo_ffat_gpu_process_batch.restype = _u64
        L.wfo_ffat_gpu_window_linear.argtypes = [_vp, _u64, _u64, _vp]
        L.wfo_ffat_gpu_window_linear.restype = C.c_int
        L.wfo_ffat_tb_create.argtypes = [_u64, _u64, _u64, _u64]
        L.wfo_ffat_tb_create.restype = _vp
        L.wfo_ffat_tb_destroy.argtypes = [_vp]
        L.wfo_ffat_tb_ignored.argtypes = [_vp]
        L.wfo_ffat_tb_ignored.restype = _u64
        L.wfo_ffat_tb_process_batch.argtypes = [_vp, _vp, _vp, _u64, _u64, _vp, _vp, _u64]
        L.wfo_ffat_tb_process_batch.restype = _u64
        L.wfo_ffat_cpu_create.argtypes = [_u64, _u64]
        L.wfo_ffat_cpu_create.restype = _vp
        L.wfo_ffat_cpu_destroy.argtypes = [_vp]
        L.wfo_ffat_cpu_process.argtypes = [_vp, _vp, _u64, _u64, _vp, _vp, _u64]
        L.wfo_ffat_cpu_process.restype = _u64
        L.wfo_ffat_cpu_eos.argtypes = [_vp, _vp, _vp, _u64]
        L.wfo_ffat_cpu_eos.restype = _u64
        L.wfo_cpu_pipe_create.argtypes = [C.c_int, _i64, _f64, C.c_int, _i64, _u64, _u64, _u32, _u32]
        L.wfo_cpu_pipe_create.restype = _vp
        L.wfo_cpu_pipe_destroy.argtypes = [_vp]
        L.wfo_cpu_pipe_run.argtypes = [_vp, _vp, _vp, _u64, _u64, _vp]
        L.wfo_cpu_pipe_run.restype = _u64
        _lib = L
    return _lib


# ---------------------------------------------------------------------------------------------------
# synthetic stream (SURVEY 8d)
# ---------------------------------------------------------------------------------------------------
def zipf_cdf(nkeys, s=0.8):
    w = 1.0 / np.power(np.arange(1, nkeys + 1, dtype=np.float64), s)
    c = np.cumsum(w)
    c /= c[-1]
    c[-1] = 1.0
    return c


def gen_tuple64(start, n, key_mode=KEY_UNIFORM, nkeys=65536, seed=SEED, cdf=None):
    out = np.zeros(n, dtype=TUPLE64)
    ts = np.zeros(n, dtype=np.uint64)
    if key_mode == KEY_ZIPF and cdf is None:
        cdf = zipf_cdf(nkeys)
    lib().wfo_gen_tuple64(seed, start, n, key_mode, nkeys, _p(cdf) if cdf is not None else None, _p(out), _p(ts))
    return out, ts


# ---------------------------------------------------------------------------------------------------
# Map / Filter (column-wise)
# ---------------------------------------------------------------------------------------------------
def scan_keys(start, n, key_mode, nkeys, sel, ia=2, fa=1.0000001, seed=SEED):
    """Survivors (bench functors) of the keys marked in `sel` (uint8[nkeys]) among stream indices [start, start+n), in stream order:
    (key, index, mapped ivalue, mapped fvalue) arrays. For the check of the full-size bench configuration."""
    L = lib()
    L.wfo_scan_keys.argtypes = [_u64, _u64, _u64, C.c_int, _u64, _vp, _i64, _f64, _vp, _vp, _vp, _vp, _u64]
    L.wfo_scan_keys.restype = _u64
    sel = np.ascontiguousarray(sel, dtype=np.uint8)
    cap = max(1024, int(n * (int(sel.sum()) + 1) / max(1, nkeys)) * 2 + 1024)
    while True:
        ok, oi = np.zeros(cap, dtype=np.uint64), np.zeros(cap, dtype=np.uint64)
        ov, of = np.zeros(cap, dtype=np.int64), np.zeros(cap, dtype=np.float64)
        m = L.wfo_scan_keys(seed, start, n, key_mode, nkeys, _p(sel), ia, fa, _p(ok), _p(oi), _p(ov), _p(of), cap)
        if m <= cap:
            return ok[:m], oi[:m], ov[:m], of[:m]
        cap = int(m) + 1024


def map_cols(ival, fval, kind, ia=0, fa=1.0):
    ival = np.ascontiguousarray(ival, dtype=np.int64).copy()
    fval = None if fval is None else np.ascontiguousarray(fval, dtype=np.float64).copy()
    lib().wfo_map(_p(ival), _p(fval) if fval is not None else None, len(ival), kind, ia, fa)
    return ival, fval


def filter_mask(ival, kind, im=1):
    ival = np.ascontiguousarray(ival, dtype=np.int64)
    mask = np.zeros(len(ival), dtype=np.uint8)
    lib().wfo_filter_mask(_p(ival), len(ival), kind, im, _p(mask))
    return mask.astype(bool)


def map_filter_tuple64(tuples, ts, map_kind, ia, fa, filt_kind, im=1):
    """Map_GPU then Filter_GPU over a tuple64 batch: returns (survivor tuples, survivor ts, mask)."""
    t = tuples.copy()
    iv, fv = map_cols(t["ivalue"], t["fvalue"], map_kind, ia, fa)
    t["ivalue"], t["fvalue"] = iv, fv
    m = filter_mask(iv, filt_kind, im)
    return t[m], ts[m], m


# ---------------------------------------------------------------------------------------------------
# key grouping / routing / reduce
# ---------------------------------------------------------------------------------------------------
def keyby_group(keys, order):
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    n = len(keys)
    start = np.zeros(n, dtype=np.int32)
    mp = np.zeros(n, dtype=np.int32)
    dk = np.zeros(n, dtype=np.uint64)
    nk = lib().wfo_keyby_group(_p(keys), n, order, _p(start), _p(mp), _p(dk))
    return start[:nk], mp, dk[:nk]


def route(keys, num_dests):
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    d = np.zeros(len(keys), dtype=np.uint32)
    lib().wfo_route(_p(keys), len(keys), num_dests, _p(d))
    return d


def reduce_by_key(keys, ival, fval, ts):
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    ival = np.ascontiguousarray(ival, dtype=np.int64)
    fval = None if fval is None else np.ascontiguousarray(fval, dtype=np.float64)
    ts = np.ascontiguousarray(ts, dtype=np.uint64)
    n = len(keys)
    ok = np.zeros(n, dtype=np.uint64)
    oi = np.zeros(n, dtype=np.int64)
    of = np.zeros(n, dtype=np.float64)
    ot = np.zeros(n, dtype=np.uint64)
    sf = np.zeros(n, dtype=np.uint32)
    sl = np.zeros(n, dtype=np.uint32)
    nk = lib().wfo_reduce_by_key(_p(keys), _p(ival), _p(fval) if fval is not None else None, _p(ts), n,
                                 _p(ok), _p(oi), _p(of), _p(ot), _p(sf), _p(sl))
    return ok[:nk], oi[:nk], of[:nk], ot[:nk], sf[:nk], sl[:nk]


def reduce_tuple64(tuples, ts):
    """Reduce_GPU keyed over a tuple64 batch with the bench functor (field-wise +, keeps t1.key; fresh tuple
    otherwise). Single-occurrence keys pass through untouched (thrust::reduce_by_key never calls the functor)."""
    ok, oi, of, ot, sf, sl = reduce_by_key(tuples["key"], tuples["ivalue"], tuples["fvalue"], ts)
    out = np.zeros(len(ok), dtype=TUPLE64)
    out["key"], out["ivalue"], out["fvalue"] = ok, oi, of
    single = sl == 1
    out[single] = tuples[sf[single]]
    return out, ot


# ---------------------------------------------------------------------------------------------------
# FFAT
# ---------------------------------------------------------------------------------------------------
def lift_tuple64(tuples):
    r = np.zeros(len(tuples), dtype=RES)
    r["key"], r["isum"], r["fsum"] = tuples["key"], tuples["ivalue"], tuples["fvalue"]
    return r


class FfatGpuOracle:
    """Ffat_Windows_GPU, count-based (wf/ffat_replica_gpu.hpp:734-867 over wf/flatfat_gpu.hpp)."""

    def __init__(self, win, slide, nb, keep_history=False):
        self.win, self.slide, self.nb = win, slide, nb
        self.h = lib().wfo_ffat_gpu_create(win, slide, nb, int(keep_history))

    def process_batch(self, res, watermark):
        res = np.ascontiguousarray(res, dtype=RES)
        cap = max(1024, (len(res) // max(1, self.slide) + 2) * self.nb + self.nb)
        while True:
            out = np.zeros(cap, dtype=RES)
            ots = np.zeros(cap, dtype=np.uint64)
            # process_batch mutates state: probe size first on a generous buffer (cap is an upper bound:
            # at most one trigger per slide*nb appended results per key, each emitting nb results)
            n = lib().wfo_ffat_gpu_process_batch(self.h, _p(res), len(res), watermark, _p(out), _p(ots), cap)
            assert n <= cap, "oracle output capacity estimate too small"
            return out[:n], ots[:n]

    def window_linear(self, key, gwid):
        r = np.zeros(1, dtype=RES)
        ok = lib().wfo_ffat_gpu_window_linear(self.h, key, gwid, _p(r))
        return r[0] if ok else None

    def close(self):
        if self.h:
            lib().wfo_ffat_gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()


class FfatTbOracle:
    """Ffat_Windows_GPU, time-based (wf/ffat_replica_gpu.hpp:870-1047): win / slide / lateness in timestamp units."""

    def __init__(self, win, slide, lateness, nb):
        self.win, self.slide, self.lateness, self.nb = win, slide, lateness, nb
        self.h = lib().wfo_ffat_tb_create(win, slide, lateness, nb)

    def process_batch(self, res, ts, watermark):
        res = np.ascontiguousarray(res, dtype=RES)
        ts = np.ascontiguousarray(ts, dtype=np.uint64)
        cap = 1 << 16
        while True:
            out = np.zeros(cap, dtype=RES)
            ots = np.zeros(cap, dtype=np.uint64)
            n = lib().wfo_ffat_tb_process_batch(self.h, _p(res), _p(ts), len(res), watermark, _p(out), _p(ots), cap)
            assert n <= cap, "oracle output capacity estimate too small (state already advanced)"
            return out[:n], ots[:n]

    @property
    def ignored(self):
        return int(lib().wfo_ffat_tb_ignored(self.h))

    def close(self):
        if self.h:
            lib().wfo_ffat_tb_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()


class FfatCpuOracle:
    """CPU Ffat_Windows replica, count-based (wf/ffat_replica.hpp:215-278, :406-427 over wf/flatfat.hpp)."""

    def __init__(self, win, slide):
        self.win, self.slide = win, slide
        self.h = lib().wfo_ffat_cpu_create(win, slide)

    def process(self, res, watermark):
        res = np.ascontiguousarray(res, dtype=RES)
        cap = len(res) + 16
        out = np.zeros(cap, dtype=RES)
        ots = np.zeros(cap, dtype=np.uint64)
        n = lib().wfo_ffat_cpu_process(self.h, _p(res), len(res), watermark, _p(out), _p(ots), cap)
        return out[:n], ots[:n]

    def eos(self, cap=1 << 20):
        out = np.zeros(cap, dtype=RES)
        ots = np.zeros(cap, dtype=np.uint64)
        n = lib().wfo_ffat_cpu_eos(self.h, _p(out), _p(ots), cap)
        assert n <= cap
        return out[:n], ots[:n]

    def close(self):
        if self.h:
            lib().wfo_ffat_cpu_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()


class CpuPipe:
    """Reference CPU path Map -> Filter -> Ffat_Windows(CB) on one key shard (one replica == one thread).
    kind "port": the oracle's restatement (wf_oracle.c); kind "reference": the reference's own wf/flatfat.hpp under
    the restated replica loop (oracle/_ref/libwfref_flatfat.so)."""

    def __init__(self, kind, map_kind, ia, fa, filt_kind, im, win, slide, shard, nshards):
        self.kind = kind
        if kind == "reference":
            self.L = ref_cpu_lib()
            self.L.wfref_cpu_pipe_create.argtypes = [C.c_int, _i64, _f64, C.c_int, _i64, _u64, _u64, _u32, _u32]
            self.L.wfref_cpu_pipe_create.restype = _vp
            self.L.wfref_cpu_pipe_destroy.argtypes = [_vp]
            self.L.wfref_cpu_pipe_run.argtypes = [_vp, _vp, _vp, _u64, _u64, _vp]
            self.L.wfref_cpu_pipe_run.restype = _u64
            self._run, self._destroy = self.L.wfref_cpu_pipe_run, self.L.wfref_cpu_pipe_destroy
            self.h = self.L.wfref_cpu_pipe_create(map_kind, ia, fa, filt_kind, im, win, slide, shard, nshards)
        else:
            self.L = lib()
            self._run, self._destroy = self.L.wfo_cpu_pipe_run, self.L.wfo_cpu_pipe_destroy
            self.h = self.L.wfo_cpu_pipe_create(map_kind, ia, fa, filt_kind, im, win, slide, shard, nshards)
        self.checksum = C.c_int64(0)
        self.windows = 0

    def run(self, tuples, ts, batch):
        self.windows += self._run(self.h, _p(tuples), _p(ts), len(tuples), batch, C.byref(self.checksum))

    def close(self):
        if self.h:
            self._destroy(self.h)
            self.h = None


# ---------------------------------------------------------------------------------------------------
# reference pins (oracle/_ref)
# ---------------------------------------------------------------------------------------------------
_ref_cpu = None


def ref_cpu_lib():
    """The reference's own wf/flatfat.hpp (or None when oracle/_ref is absent)."""
    global _ref_cpu
    if _ref_cpu is None:
        so = os.path.join(HERE, "_ref", "libwfref_flatfat.so")
        if not os.path.exists(so):
            return None
        L = C.CDLL(so)
        L.wfref_ffat_cpu_create.argtypes = [_u64, _u64]
        L.wfref_ffat_cpu_create.restype = _vp
        L.wfref_ffat_cpu_destroy.argtypes = [_vp]
        L.wfref_ffat_cpu_process.argtypes = [_vp, _vp, _u64, _u64, _vp, _vp, _u64]
        L.wfref_ffat_cpu_process.restype = _u64
        L.wfref_ffat_cpu_eos.argtypes = [_vp, _vp, _vp, _u64]
        L.wfref_ffat_cpu_eos.restype = _u64
        L.wfref_fat_create.argtypes = [_u64, _u64]
        L.wfref_fat_create.restype = _vp
        L.wfref_fat_destroy.argtypes = [_vp]
        L.wfref_fat_insert.argtypes = [_vp, _vp, _u64]
        L.wfref_fat_remove.argtypes = [_vp, _u64]
        L.wfref_fat_result.argtypes = [_vp, _u64, _vp]
        _ref_cpu = L
    return _ref_cpu


class RefFfatCpu:
    """Reference wf::FlatFAT driven by the restated FFAT_Replica CB loop (oracle/ref_flatfat.cpp)."""

    def __init__(self, win, slide):
        self.L = ref_cpu_lib()
        self.h = self.L.wfref_ffat_cpu_create(win, slide)

    def process(self, res, watermark):
        res = np.ascontiguousarray(res, dtype=RES)
        cap = len(res) + 16
        out = np.zeros(cap, dtype=RES)
        ots = np.zeros(cap, dtype=np.uint64)
        n = self.L.wfref_ffat_cpu_process(self.h, _p(res), len(res), watermark, _p(out), _p(ots), cap)
        return out[:n], ots[:n]

    def eos(self, cap=1 << 20):
        out = np.zeros(cap, dtype=RES)
        ots = np.zeros(cap, dtype=np.uint64)
        n = self.L.wfref_ffat_cpu_eos(self.h, _p(out), _p(ots), cap)
        return out[:n], ots[:n]

    def close(self):
        if self.h:
            self.L.wfref_ffat_cpu_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()


_ref_gpu = None


def ref_gpu_lib():
    """The reference's own wf/flatfat_gpu.hpp for sm_100a (needs a GPU to run; None when absent)."""
    global _ref_gpu
    if _ref_gpu is None:
        so = os.path.join(HERE, "_ref", "libwfref_flatfat_gpu.so")
        if not os.path.exists(so):
            return None
        L = C.CDLL(so)
        L.wfref_ffat_gpu_create.argtypes = [_u64, _u64, _u64, _u64]
        L.wfref_ffat_gpu_create.restype = _vp
        L.wfref_ffat_gpu_destroy.argtypes = [_vp]
        L.wfref_ffat_gpu_process.argtypes = [_vp, _vp, _u64, _u64, _vp, _vp, _u64]
        L.wfref_ffat_gpu_process.restype = _u64
        _ref_gpu = L
    return _ref_gpu


def sort_results(res, ts=None):
    """Canonical order for comparing window results: (key, gwid)."""
    order = np.lexsort((res["id"], res["key"]))
    return (res[order], ts[order]) if ts is not None else res[order]


# ---------------------------------------------------------------------------------------------------
# golden records of the reference's outputs (tests/golden/ref/*.npz, written by tests/golden/make_ref_golden.py)
# ---------------------------------------------------------------------------------------------------
GOLDEN_SAMPLE = 1024  # floating-point sums stored per record: all of them up to this many rows, a seeded sample beyond


def digest(*cols):
    """SHA-256 of the columns' bytes: a golden record keeps it in place of outputs that are compared bit for bit."""
    h = hashlib.sha256()
    for c in cols:
        h.update(np.ascontiguousarray(c).tobytes())
    return h.hexdigest()


def _exact_cols(r, with_ts):
    cols = [r["key"].astype("<u8"), r["id"].astype("<u8"), r["isum"].astype("<i8")]
    return cols + [r["ts"].astype("<u8")] if with_ts else cols


def windows_record(res, prefix, with_ts=True):
    """Golden record of window results (fields key, id, isum, fsum[, ts]) in (key, id) order: the row count, a digest of
    the exact columns and the floating-point sums (a fixed sample of GOLDEN_SAMPLE rows beyond that size), as npz entries."""
    r = np.sort(res, order=["key", "id"])
    n = len(r)
    idx = np.arange(n) if n <= GOLDEN_SAMPLE else np.sort(np.random.default_rng(0).choice(n, GOLDEN_SAMPLE, replace=False))
    return {prefix + ".n": np.int64(n), prefix + ".digest": np.array(digest(*_exact_cols(r, with_ts))),
            prefix + ".idx": idx.astype("<u4"), prefix + ".fsum": r["fsum"][idx]}


def check_windows_record(got, golden, prefix, rtol, with_ts=True):
    """`got` equals the recorded windows: same count, same keys / window ids / integer sums (/ timestamps), floating-point
    sums within `rtol` of the recorded ones."""
    r = np.sort(got, order=["key", "id"])
    assert len(r) == int(golden[prefix + ".n"]), (len(r), int(golden[prefix + ".n"]))
    assert digest(*_exact_cols(r, with_ts)) == str(golden[prefix + ".digest"]), "keys, window ids, integer sums or timestamps differ"
    idx = golden[prefix + ".idx"]
    assert np.allclose(r["fsum"][idx], golden[prefix + ".fsum"], rtol=rtol, atol=0)


# ---------------------------------------------------------------------------------------------------
# keyed-stateful Map / Filter (wf/map_gpu.hpp:80-102 Stateful_MAPGPU_Kernel, wf/filter_gpu.hpp:91-117): func(tuple, state)
# in per-key arrival order; functors of tests/graph_tests_gpu/graph_common_gpu.hpp:221-231, :256-265 and
# tests/merge_tests_gpu/merge_common_gpu_kb.hpp:153-168 (kind 2: on the key's parity). `state` maps key -> counter and
# persists across calls. Pure-Python loops: small cases only.
# ---------------------------------------------------------------------------------------------------
def stateful_map(tuples, field, state, map_kind=1):
    out = tuples.copy()
    for i in range(len(out)):
        k = int(out["key"][i])
        c = state.get(k, 0)
        c = c - 1 if (map_kind == 2 and (k & 1)) else c + 1
        state[k] = c
        out[field][i] += c
    return out


def stateful_filter(tuples, ts, field, state, filt_kind=0, mod=1):
    out = tuples.copy()
    keep = np.zeros(len(out), dtype=bool)
    for i in range(len(out)):
        k = int(out["key"][i])
        c = state.get(k, 0) + 1
        state[k] = c
        out[field][i] += c
        v = int(out[field][i])
        keep[i] = True if filt_kind == 0 else ((v & 1) == 0 if filt_kind == 1 else (v % mod) == 0)
    return out[keep], (ts[keep] if ts is not None else None), keep

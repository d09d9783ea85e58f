"""Count-based Ffat_Windows_GPU at real key counts, against a plain numpy reference of keyed count-based windows.

wfb_ffat_create picks the update path from max_keys: bits = ceil(log2(max_keys)), bucket_shift = max(0, bits - 10). Up to
65 536 keys (1 << shift <= 64) the segment is partitioned into 1024 buckets of min(64, 1 << shift) consecutive slots and
k_ffat_update_buckets (k_ffat_update_stream with WFB_UPDATE=stream) folds every bucket in chunks of 2304 items; above that, or
with WFB_UPDATE=lanes, a full radix sort feeds k_ffat_update_lanes (one thread per key) and k_ffat_update (one warp per key
with more than light_max items in the call). Lazy FlatFAT levels (the update writes only the leaves, the levels are built when
a group is evaluated) are chosen on the bucket path when the on-chip tree fits and the rebuild pays. A fired group waits for
the deferred window pass unless its key completes more panes later in the call than the spare ring leaves hold; it is then
evaluated inside the update kernel. Every case id names the path the create-time rule, restated in `_path`, selects for it.

Bars: keys, window ids, integer sums and result timestamps bit-exact; floating-point sums within 1e-6 relative; no duplicate
(key, id); no error flag. `cb_windows_reference` is independent of the oracle's FlatFAT restatement; the CPU test below pins it
to that oracle, which the recorded outputs of the reference (tests/golden/ref/) pin in turn."""
import math
from functools import lru_cache

import numpy as np
import pytest

gpu = pytest.mark.gpu
FP_RTOL = 1e-6
BATCH = 65536           # tuples per batch
CALL = 8                # batches per call (one stream segment)
BK_CHUNK = 2304         # items per chunk of k_ffat_update_buckets (BK_THREADS * BK_IT)
RES = np.dtype([("key", "<u8"), ("id", "<u8"), ("isum", "<i8"), ("fsum", "<f8")])


# ---------------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------------
def cb_windows_reference(keys, ivalue, fvalue, batch_sizes, watermarks, win, slide, nb):
    """Every window a keyed count-based operator (withCBWindows(win, slide), nb windows per fired group) emits over a
    stream whose items arrive in order, cut into batches of `batch_sizes` with the given watermarks.

    A key's items are ranked in arrival order. With B = (nb - 1) * slide + win, group g of a key with c items fires when
    B + g * slide * nb <= c and emits the windows g * nb + i, i in [0, nb); window `id` covers ranks [id * slide, id * slide + win)
    and carries the watermark of the batch that held the key's item of rank B + g * slide * nb - 1. Sums are differences of
    per-key prefix sums: int64 (exact) and extended precision. Returns (results in (key, id) order, their timestamps)."""
    keys = np.asarray(keys)
    n = len(keys)
    B = (nb - 1) * slide + win
    per_group = slide * nb
    if n == 0:
        return np.zeros(0, RES), np.zeros(0, np.uint64)
    order = np.argsort(keys, kind="stable")          # arrival order inside every key
    sk = keys[order]
    first = np.empty(n, bool)
    first[0] = True
    np.not_equal(sk[1:], sk[:-1], out=first[1:])
    start = np.flatnonzero(first)                    # first sorted index of every key
    cnt = np.diff(np.append(start, n))
    ci = np.zeros(n + 1, np.int64)
    np.cumsum(np.asarray(ivalue, np.int64)[order], out=ci[1:])
    cf = np.zeros(n + 1, np.longdouble)
    np.cumsum(np.asarray(fvalue, np.float64)[order].astype(np.longdouble), out=cf[1:])
    groups = np.where(cnt >= B, 1 + (cnt - B) // per_group, 0)
    ng = int(groups.sum())
    gk = np.repeat(np.arange(len(cnt)), groups)      # key (index) of every fired group
    g = np.arange(ng) - np.repeat(np.cumsum(groups) - groups, groups)
    trig_pos = order[start[gk] + B + g * per_group - 1]  # arrival position of the item that fires the group
    bi = np.searchsorted(np.cumsum(batch_sizes), trig_pos, side="right")
    gts = np.asarray(watermarks, np.uint64)[bi]
    wk = np.repeat(gk, nb)
    wid = np.repeat(g, nb) * nb + np.tile(np.arange(nb), ng)
    lo = start[wk] + wid * slide
    hi = lo + win
    out = np.zeros(ng * nb, RES)
    out["key"] = sk[start][wk]
    out["id"] = wid
    out["isum"] = ci[hi] - ci[lo]
    out["fsum"] = (cf[hi] - cf[lo]).astype(np.float64)
    return out, np.repeat(gts, nb)


REF_CASES = [  # win, slide, nb, nkeys, batch sizes (None: 40 batches of 97)
    (10, 3, 2, 5, None),                                  # pane = 1
    (7, 3, 4, 3, None),                                   # pane = 1, odd geometry
    (8, 24, 2, 4, None),                                  # slide > win
    (16, 16, 1, 2, None),                                 # tumbling
    (16, 4, 1, 6, None),                                  # Nb = 1
    (256, 4, 65, 3, [1000] * 8),                          # Nb = 65 (the bench's tree shape)
    (64, 16, 5, 40, [0, 1, 5, 0, 300, 1, 2, 1023, 0, 77, 4096, 3, 0, 0, 9, 2000, 1500]),  # ragged and empty batches
    (32, 8, 2, 1, [777] * 7),                             # a single key
    (4096, 64, 65, 2, [4096] * 6),                        # B = 8192
    (64, 16, 5, 300, [2048] * 40),                        # many keys
]


@pytest.mark.parametrize("case", REF_CASES, ids=[f"w{c[0]}_s{c[1]}_nb{c[2]}_k{c[3]}" for c in REF_CASES])
def test_reference_matches_oracle(oracle, case):
    """cb_windows_reference == the oracle's Ffat_Windows_GPU restatement (FfatGpuOracle), batch by batch."""
    O = oracle
    win, slide, nb, nkeys, sizes = case
    sizes = sizes or [97] * 40
    n = sum(sizes)
    rng = np.random.default_rng(win * 1000 + nkeys)
    keys = rng.integers(0, nkeys, n).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)  # scattered 64-bit keys
    iv = rng.integers(-1000, 65536, n)
    fv = rng.random(n)
    wms = 1000 + 7 * np.arange(len(sizes))
    go = O.FfatGpuOracle(win, slide, nb)
    exp, ets, off = [], [], 0
    for sz, wm in zip(sizes, wms):
        r = np.zeros(sz, O.RES)
        r["key"], r["isum"], r["fsum"] = keys[off:off + sz], iv[off:off + sz], fv[off:off + sz]
        e, et = go.process_batch(r, int(wm))
        exp.append(e); ets.append(et)
        off += sz
    e, et = O.sort_results(np.concatenate(exp), np.concatenate(ets))
    got, gts = cb_windows_reference(keys, iv, fv, sizes, wms, win, slide, nb)
    assert len(got) == len(e) > 0, (len(got), len(e))
    assert np.array_equal(got["key"], e["key"]) and np.array_equal(got["id"], e["id"])
    assert np.array_equal(got["isum"], e["isum"]) and np.array_equal(gts, et)
    assert np.allclose(got["fsum"], e["fsum"], rtol=1e-9, atol=0)


# ---------------------------------------------------------------------------------------------------------------------
# the create-time rule (wfb_ffat_create), restated to name the path every case drives
# ---------------------------------------------------------------------------------------------------------------------
def _path(win, slide, nb, max_keys, rb=32, env=None):
    env = env or {}
    pane = math.gcd(win, slide)
    B = (nb - 1) * slide + win
    bp = B // pane
    n, lg = 1, 0
    while n < bp + min(bp, 32):
        n, lg = n * 2, lg + 1
    bits = max(0, (max_keys - 1).bit_length())
    shift = max(0, bits - 10)
    buckets = env.get("WFB_UPDATE") != "lanes" and (1 << shift) <= 64
    fits = buckets and 2 * n * rb <= 32 << 10
    pays = n <= 2 * max(1, lg) * (slide // pane) * nb
    lazy = fits and (env["WFB_LAZY_TREE"] != "0" if "WFB_LAZY_TREE" in env else pays)
    kernel = ("stream" if env.get("WFB_UPDATE") == "stream" else "buckets") if buckets else "lanes"
    return dict(pane=pane, B=B, n_leaves=n, defer_items=(n - bp + 1) * pane, kpb=min(64, 1 << shift) if buckets else 0,
                lazy=lazy, kernel=kernel,
                name=(f"{min(64, 1 << shift)}perbucket_" if buckets else "") + ("lazy" if lazy else "eager") + "_" + kernel)


# ---------------------------------------------------------------------------------------------------------------------
# streams, feeding, comparison
# ---------------------------------------------------------------------------------------------------------------------
def _scatter(idx):
    """Key index -> scattered 64-bit key (a bijection of 64-bit words)."""
    return np.asarray(idx, np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(0x632BE59BD9B4E019)


class Stream:
    """A keyed stream: key index per item (dense key = index; hash-table key = table[index]), values, batches, calls."""

    def __init__(self, kidx, nkeys, seed, dense=True, calls=None, table=None):
        rng = np.random.default_rng(seed)
        n = len(kidx)
        self.kidx, self.nkeys, self.dense = kidx, nkeys, dense
        self.iv = rng.integers(0, 1 << 16, n)
        self.fv = rng.random(n)
        self.table = None if dense else (table if table is not None else _scatter(np.arange(nkeys)))
        assert dense or not (self.table == np.uint64(0xffffffffffffffff)).any()  # (the key table's empty marker)
        # calls: list of batch-size lists (default: CALL batches of BATCH)
        if calls is None:
            sizes = [BATCH] * (n // BATCH) + ([n % BATCH] if n % BATCH else [])
            calls = [sizes[i:i + CALL] for i in range(0, len(sizes), CALL)]
        assert sum(map(sum, calls)) == n
        self.calls = calls
        self.sizes = [s for c in calls for s in c]
        self.wms = 1000 + 3 * np.arange(len(self.sizes), dtype=np.uint64)
        self._ref = {}

    def keys(self, lo=0, hi=None):
        k = self.kidx[lo:hi]
        return k.astype(np.uint64) if self.dense else self.table[k]

    def reference(self, win, slide, nb):
        if (win, slide, nb) not in self._ref:
            self._ref[(win, slide, nb)] = cb_windows_reference(self.kidx, self.iv, self.fv, self.sizes, self.wms, win, slide, nb)
        return self._ref[(win, slide, nb)]


def _records(ops, prog, st, lo, hi):
    dt = ops.TUPLE_DTYPE[prog]
    r = np.zeros(hi - lo, dt)
    r["key"] = st.keys(lo, hi)
    if prog == ops.PROG_WFWIN24:
        r["value"] = st.iv[lo:hi]
    elif prog == ops.PROG_LIFTED32:
        r["isum"], r["fsum"] = st.iv[lo:hi], st.fv[lo:hi]
    else:
        r["ivalue"], r["fvalue"] = st.iv[lo:hi], st.fv[lo:hi]
    return r


def _fetch(ff, out, out_ts, n_out):
    n = int(n_out.item())
    rb = ff.res_dtype.itemsize
    return out[:n * rb].cpu().numpy().view(ff.res_dtype).copy(), out_ts[:n].cpu().numpy().view(np.uint64).copy()


def run_handle(ops, ff, st, prog):
    """Feeds the stream call by call (batches laid out back to back in one buffer, i.e. at their tile positions); a pipelined
    handle hands results over one call late, then by flush. Returns (results, timestamps)."""
    import torch
    cap_items = max(map(sum, st.calls))
    cap = ff.max_results(cap_items)
    out = torch.empty(cap * ff.res_dtype.itemsize, dtype=torch.uint8, device="cuda")
    out_ts = torch.empty(cap, dtype=torch.int64, device="cuda")
    n_out = torch.zeros(1, dtype=torch.int32, device="cuda")
    tb = ops.TUPLE_DTYPE[prog].itemsize
    got, gts, pos, b = [], [], 0, 0
    for call in st.calls:
        m = sum(call)
        dev = ops.to_device(_records(ops, prog, st, pos, pos + m))
        batches, o = [], 0
        for sz in call:
            batches.append(ops.DeviceBatch(dev[o * tb:(o + sz) * tb], None, sz, int(st.wms[b])))
            o += sz; b += 1
        ff.process(batches, out=out, out_ts=out_ts, n_out=n_out)
        r, t = _fetch(ff, out, out_ts, n_out)
        got.append(r); gts.append(t)
        pos += m
    if ff.pipelined:
        for _ in range(2):
            ff.flush(out=out, out_ts=out_ts, n_out=n_out)
            r, t = _fetch(ff, out, out_ts, n_out)
            got.append(r); gts.append(t)
        assert len(got[-1]) == 0
    return np.concatenate(got), np.concatenate(gts)


def key_index(st, keys):
    """Result keys -> key indices of the stream (asserts every key is one of the stream's)."""
    keys = np.asarray(keys, np.uint64)
    if st.dense:
        assert (keys < st.nkeys).all()
        return keys.astype(np.int64)
    perm = np.argsort(st.table)
    srt = st.table[perm]
    p = np.minimum(np.searchsorted(srt, keys), len(srt) - 1)
    assert np.array_equal(srt[p], keys), "a result carries a key the stream never had"
    return perm[p].astype(np.int64)


def check_windows(st, got, gts, exp, ets, value_field="isum", fsum=True, only=None):
    """got == exp: same (key, id) set without duplicates, same integer sums and timestamps, fsum within FP_RTOL.
    `only`: compare only the expected windows of these key indices (keys that own a slot)."""
    gi = key_index(st, got["key"])
    gid = got["id"].astype(np.int64)
    assert gid.max(initial=0) < 1 << 40
    gc = (gi << 40) | gid
    o = np.argsort(gc, kind="stable")
    gc, got, gts = gc[o], got[o], gts[o]
    assert not (gc[1:] == gc[:-1]).any(), "duplicate (key, id)"
    ek = exp["key"].astype(np.int64)
    if only is not None:
        sel = np.isin(ek, only)
        exp, ets, ek = exp[sel], ets[sel], ek[sel]
    ec = (ek << 40) | exp["id"].astype(np.int64)
    assert len(gc) == len(ec), (len(gc), len(ec))
    assert np.array_equal(gc, ec), "keys or window ids differ"
    assert np.array_equal(got[value_field], exp["isum"]), "integer sums differ"
    assert np.array_equal(gts, ets), "result timestamps differ"
    if fsum:
        assert np.allclose(got["fsum"], exp["fsum"], rtol=FP_RTOL, atol=0)


def run_and_check(ops, st, geom, max_keys, prog=None, pipelined=False):
    prog = ops.PROG_TUPLE64 if prog is None else prog
    win, slide, nb = geom
    exp, ets = st.reference(win, slide, nb)
    assert len(exp) > 0
    ff = ops.FfatWindowsGPU(prog, win, slide, nb, max_keys=max_keys, dense_keys=st.dense, pipelined=pipelined)
    try:
        got, gts = run_handle(ops, ff, st, prog)
        nk, err = ff.stats()
    finally:
        ff.close()
    assert err == 0, err
    if not st.dense:
        assert nk == len(np.unique(st.kidx))
    w24 = prog == ops.PROG_WFWIN24
    check_windows(st, got, gts, exp, ets, value_field="value" if w24 else "isum", fsum=not w24)
    return got, gts


# key distributions over `nkeys` key indices
def _keys(O, dist, nkeys, n, seed):
    rng = np.random.default_rng(seed)
    dt = np.uint16 if nkeys <= 1 << 16 else np.uint32
    if dist == "uniform":
        return rng.integers(0, nkeys, n).astype(dt)
    if dist == "rr":
        return (np.arange(n) % nkeys).astype(dt)
    if dist == "zipf":
        return np.minimum(np.searchsorted(O.zipf_cdf(nkeys), rng.random(n), side="right"), nkeys - 1).astype(dt)
    if dist == "hot":  # key 0: half of every call; keys 1..63 (its bucket): 1/16; the other keys: the rest
        u = rng.random(n)
        k = np.where(u < 0.5, 0, np.where(u < 0.5 + 1 / 16, 1 + rng.integers(0, 63, n), 64 + rng.integers(0, nkeys - 64, n)))
        return k.astype(dt)
    raise ValueError(dist)


def _items(geom, nkeys, dist):
    """Stream length: about 1.5 groups past the first trigger per key on average (uniform / round-robin)."""
    win, slide, nb = geom
    B = (nb - 1) * slide + win
    per_key = B + (3 * slide * nb) // 2 + 8
    if dist == "hot":
        return 4 * 2 * CALL * BATCH
    n = nkeys * per_key
    return max(n, 4 * BATCH)


@lru_cache(maxsize=1)
def _matrix_stream(O, dist, nkeys, geom, dense):
    n = _items(geom, nkeys, dist)
    calls = None
    if dist == "hot":  # calls of 16 batches: key 0 brings ~227 chunks of 2304 items to bucket 0 in every call
        calls = [[BATCH] * (2 * CALL)] * (n // (2 * CALL * BATCH))
    return Stream(_keys(O, dist, nkeys, n, seed=nkeys + sum(geom)), nkeys, seed=7, dense=dense, calls=calls)


# ---------------------------------------------------------------------------------------------------------------------
# 2-4: the bucket path, the lanes path on the same streams, the streaming kernel, forced lazy / eager levels
# ---------------------------------------------------------------------------------------------------------------------
G_LAZY, G_EAGER, G_PANE1, G_GAPS, G_BENCH = (64, 16, 5), (16, 4, 1), (10, 3, 2), (8, 24, 2), (256, 4, 65)
MATRIX = []  # (max_keys, geom, dist, dense, prog, pipelined, env); cases of one stream are adjacent (the stream is cached)
for mk, geoms in [(1024, [(G_LAZY, "uniform"), (G_EAGER, "zipf")]), (1500, [(G_PANE1, "uniform"), (G_LAZY, "rr")]),
                  (4096, [(G_EAGER, "uniform"), (G_GAPS, "zipf")]), (39999, [(G_LAZY, "uniform"), (G_PANE1, "rr")])]:
    for geom, dist in geoms:
        for dense in (True, False):
            MATRIX.append((mk, geom, dist, dense, "TUPLE64", False, {}))
for geom, extra in [(G_LAZY, [{"WFB_LAZY_TREE": "0"}, {"WFB_LAZY_TREE": "1"}]), (G_EAGER, []), (G_PANE1, []), (G_GAPS, []),
                    (G_BENCH, [{"WFB_LAZY_TREE": "0"}, {"WFB_LAZY_TREE": "1"}])]:
    for env in [{}, {"WFB_UPDATE": "lanes"}, {"WFB_UPDATE": "stream"}] + extra:
        MATRIX.append((65536, geom, "uniform", True, "TUPLE64", False, env))
    if geom == G_LAZY:
        MATRIX.append((65536, geom, "uniform", True, "TUPLE64", True, {}))
        MATRIX.append((65536, geom, "uniform", True, "WFWIN24", False, {}))
for geom, dist in [(G_LAZY, "zipf"), (G_EAGER, "rr"), (G_GAPS, "zipf")]:
    MATRIX.append((65536, geom, dist, False, "TUPLE64", False, {}))
for geom in (G_LAZY, G_PANE1):
    for env in [{}, {"WFB_UPDATE": "lanes"}]:
        MATRIX.append((65536, geom, "hot", True, "TUPLE64", False, env))


def _matrix_id(c):
    mk, geom, dist, dense, prog, pipelined, env = c
    p = _path(*geom, mk, rb=24 if prog == "WFWIN24" else 32, env=env)
    extra = "_inkernel_eval_chunked" if dist == "hot" else ""
    return (f"k{mk}_w{geom[0]}s{geom[1]}nb{geom[2]}_{p['name']}_{dist}{extra}_{'dense' if dense else 'hash'}"
            + ("_pipelined" if pipelined else "") + ("" if prog == "TUPLE64" else "_" + prog)
            + "".join(f"_{k}={v}" for k, v in env.items() if k != "WFB_UPDATE"))


@gpu
@pytest.mark.parametrize("case", MATRIX, ids=[_matrix_id(c) for c in MATRIX])
def test_keys_matrix(wfb, oracle, monkeypatch, case):
    """Window parity at 1024 (one key per bucket), 1500 (2), 4096 (4), 39 999 (64, partial last bucket) and 65 536 keys (64),
    dense and hash-table keys, over the five geometries of the create-time rule; the 65 536-key streams again with the lanes
    path, the streaming kernel and forced lazy / eager levels. 'hot': key 0 takes half of every call, so bucket 0 is folded in
    hundreds of chunks and key 0's groups are evaluated inside the update kernel."""
    ops = wfb
    mk, geom, dist, dense, prog, pipelined, env = case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    st = _matrix_stream(oracle, dist, mk, geom, dense)
    run_and_check(ops, st, geom, mk, prog=getattr(ops, "PROG_" + prog), pipelined=pipelined)


CHUNK_EDGES = [(geom, items, spread) for geom in (G_LAZY, (128, 64, 2)) for items in (BK_CHUNK, BK_CHUNK + 1, 2 * BK_CHUNK)
               for spread in (64, 1)]


@gpu
@pytest.mark.parametrize("case", CHUNK_EDGES, ids=[f"w{g[0]}s{g[1]}nb{g[2]}_{_path(*g, 65536)['name']}_bucket{n}items_{s}keys"
                                                   for g, n, s in CHUNK_EDGES])
def test_chunk_edges(wfb, case):
    """One call in which bucket 5 (keys 320..383, 64 keys per bucket) receives exactly 2304 (one full chunk), 2305 (a chunk and
    one item) or 4608 items (two chunks), over its 64 keys or over key 320 alone, after a call that brings bucket 5's keys
    close to their first trigger and before a call of uniform keys."""
    ops = wfb
    geom, items, spread = case
    rng = np.random.default_rng(items + spread)
    nk = 65536
    B = _path(*geom, nk)["B"]
    before = np.concatenate([rng.integers(0, nk, CALL * BATCH), np.repeat(np.arange(320, 384), B - 20)])  # bucket 5's keys near B
    before = before[rng.permutation(len(before))]
    mine = 320 + (rng.integers(0, 64, items) if spread == 64 else np.zeros(items, np.int64))
    others = rng.integers(0, nk - 64, 2 * BATCH)
    others = np.where(others >= 320, others + 64, others)            # every key but bucket 5's
    edge = np.concatenate([mine, others])[rng.permutation(items + len(others))]
    after = rng.integers(0, nk, CALL * BATCH)
    kidx = np.concatenate([before, edge, after]).astype(np.uint16)
    calls = [[len(before)], [len(edge)], [BATCH] * CALL]
    st = Stream(kidx, nk, seed=3, calls=calls)
    exp, ets = st.reference(*geom)
    assert len(_fired_in_call(st, exp, ets, 1) & set(range(320, 384))) >= min(spread, 32)  # bucket 5 fires groups in that call
    run_and_check(ops, st, geom, nk)


@gpu
def test_key_shard_replicas_32_keys_per_bucket(wfb):
    """PROG_LIFTED32 replicas of two key shards (32 768 keys each: 32 keys per bucket, lazy levels), fed their keys' lifted
    records in place (k_slots_inplace): together they produce the windows of one operator over the whole stream."""
    import torch
    ops = wfb
    nk, shards, geom = 65536, 2, G_LAZY
    n = _items(geom, nk, "uniform")
    per_call = CALL * BATCH
    st = Stream(_keys(None, "uniform", nk, n, 5), nk, seed=9, calls=[[min(per_call, n - o)] for o in range(0, n, per_call)])
    exp, ets = st.reference(*geom)
    reps = []
    for r in range(shards):
        ff = ops.FfatWindowsGPU(ops.PROG_LIFTED32, *geom, max_keys=nk // shards, dense_keys=True)
        ff.set_key_shard(shards, r)
        reps.append(ff)
    got, gts, pos = [], [], 0
    for b, call in enumerate(st.calls):
        m = call[0]
        rec = _records(ops, ops.PROG_LIFTED32, st, pos, pos + m)
        for r, ff in enumerate(reps):
            mine = rec[rec["key"] % shards == r]
            out, out_ts, n_out = ff.process([ops.DeviceBatch.from_host(mine, None, int(st.wms[b]))])
            torch.cuda.synchronize()
            g_, t_ = _fetch(ff, out, out_ts, n_out)
            got.append(g_); gts.append(t_)
        pos += m
    for ff in reps:
        assert ff.stats()[1] == 0
        ff.close()
    check_windows(st, np.concatenate(got), np.concatenate(gts), exp, ets)


# ---------------------------------------------------------------------------------------------------------------------
# 3. more than 65 536 keys: full sort, k_ffat_update_lanes (light keys), k_ffat_update (heavy keys)
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("geom,dense", [(G_PANE1, True), (G_EAGER, False)],
                         ids=[f"k65537_{_path(*G_PANE1, 65537)['name']}_uniform_dense", f"k65537_{_path(*G_EAGER, 65537)['name']}_uniform_hash"])
def test_65537_keys_lanes_path(wfb, geom, dense):
    """65 537 keys (bucket shift 7): the full-sort path with one thread per light key."""
    st = Stream(_keys(None, "uniform", 65537, _items(geom, 65537, "uniform"), 11), 65537, seed=12, dense=dense)
    run_and_check(wfb, st, geom, 65537)


@lru_cache(maxsize=1)
def _zipf_1m(O):
    nk = 1 << 20
    return Stream(_keys(O, "zipf", nk, 24 * CALL * BATCH, 13), nk, seed=14)


@gpu
@pytest.mark.parametrize("geom", [G_LAZY, G_PANE1], ids=lambda g: f"w{g[0]}s{g[1]}nb{g[2]}_{_path(*g, 1 << 20)['name']}_heavy")
@pytest.mark.parametrize("pipelined", [False, True], ids=["direct", "pipelined"])
def test_1m_zipf_keys(wfb, oracle, geom, pipelined):
    """2^20 Zipf keys (BASELINE config 3's key space): the hottest keys take the heavy-key kernel, the tail the lanes kernel."""
    run_and_check(wfb, _zipf_1m(oracle), geom, 1 << 20, pipelined=pipelined)


def _edge_stream(nk, specials, seed, per_key=3):
    """One call per entry of `specials` ({key: items}): every key of the entry gets exactly that many items, every key named in
    no entry gets 1..per_key items, in random order. Keys named in some entry appear in no other call."""
    rng = np.random.default_rng(seed)
    named = sorted({k for sp in specials for k in sp})
    calls, parts = [], []
    for sp in specials:
        bg = np.repeat(np.arange(nk), rng.integers(1, per_key + 1, nk))
        bg = bg[~np.isin(bg, named)]
        bg = np.concatenate([bg] + [np.full(m, k) for k, m in sp.items()])
        parts.append(bg[rng.permutation(len(bg))])
        calls.append([BATCH] * (len(bg) // BATCH) + ([len(bg) % BATCH] if len(bg) % BATCH else []))
    dt = np.uint16 if nk <= 1 << 16 else np.uint32
    return Stream(np.concatenate(parts).astype(dt), nk, seed=seed + 1, calls=calls)


def _fired_in_call(st, exp, ets, call):
    """Key indices with a group fired by an item of call `call`."""
    b0 = sum(len(c) for c in st.calls[:call])
    sel = np.isin(ets, st.wms[b0:b0 + len(st.calls[call])])
    return set(np.unique(exp["key"][sel]).tolist())


LIGHT_HEAVY = {100: 255, 200: 256, 300: 257, 400: 1000}


@gpu
@pytest.mark.parametrize("light_max", [None, "0", "1"], ids=["light_max256_lanes_and_heavy", "light_max0_all_heavy", "light_max1"])
def test_light_heavy_edge(wfb, monkeypatch, light_max):
    """65 537 keys (lanes path), pane 1 (10, 3, 2): in one call keys get exactly 255, 256, 257 and 1000 items next to keys with
    1-3 items: 255 and 256 are light (k_ffat_update_lanes), 257 and 1000 heavy (k_ffat_update). Key 500 ends that call with
    exactly B items and starts a later call with them. WFB_LIGHT_MAX=0 puts every key on the heavy list, =1 nearly every key."""
    if light_max is not None:
        monkeypatch.setenv("WFB_LIGHT_MAX", light_max)
    nk, geom = 65537, G_PANE1
    B = _path(*geom, nk)["B"]
    st = _edge_stream(nk, [{}, {**LIGHT_HEAVY, 500: B}, {}, {500: 40}, {}], seed=21)
    exp, ets = st.reference(*geom)
    assert set(LIGHT_HEAVY) <= _fired_in_call(st, exp, ets, 1) and 500 in _fired_in_call(st, exp, ets, 3)
    run_and_check(wfb, st, geom, nk)


@gpu
@pytest.mark.parametrize("light_max", [None, "0"], ids=["lanes_and_heavy", "light_max0_all_heavy"])
def test_defer_edge(wfb, monkeypatch, light_max):
    """(16, 4, 1) on the lanes path: pane 4, 8 ring leaves for the 4 panes a group reads, defer_items = 20. Keys new in the call
    with 35 / 36 items (light: k_ffat_update_lanes) and 299 / 300 items (heavy: k_ffat_update) each have a group after which
    exactly 19 items of the key follow in the call (evaluated later) or exactly 20 (evaluated at once, in the update kernel)."""
    if light_max is not None:
        monkeypatch.setenv("WFB_LIGHT_MAX", light_max)
    nk, geom = 65537, G_EAGER
    p = _path(*geom, nk)
    assert p["kernel"] == "lanes" and p["defer_items"] == 20
    B, D, per_group = p["B"], p["defer_items"], geom[1] * geom[2]
    special = {1000: B + D - 1, 1001: B + D, 2000: 299, 2001: 300}
    assert (299 - (D - 1) - B) % per_group == 0 and (300 - D - B) % per_group == 0  # a trigger D - 1 / D items before the end
    st = _edge_stream(nk, [{}, special, {}], seed=51, per_key=2)
    run_and_check(wfb, st, geom, nk)


# ---------------------------------------------------------------------------------------------------------------------
# 5. hash-table keys
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_hash_65536_new_keys_in_one_call(wfb):
    """65 536 distinct scattered 64-bit keys (0 and 2^64 - 2 among them) all inserted in the first call, where every key occurs
    8 times, in 8 different tiles: max_keys = 65 536 exactly, 64 keys per bucket, eager levels (16, 4, 1)."""
    nk = 65536
    table = _scatter(np.arange(nk))
    table[0], table[1] = 0, np.uint64((1 << 64) - 2)
    assert len(np.unique(table)) == nk
    rng = np.random.default_rng(61)
    kidx = np.concatenate([rng.permutation(np.tile(np.arange(nk), 8)) for _ in range(12)]).astype(np.uint16)
    st = Stream(kidx, nk, seed=62, dense=False, table=table)
    run_and_check(wfb, st, G_EAGER, nk)


def _unmix64(h):
    """Inverse of the key table's hash mix64 (xorshift-33 and odd multipliers are bijections of 64-bit words)."""
    M = (1 << 64) - 1
    h ^= h >> 33
    h = (h * pow(0xc4ceb9fe1a85ec53, -1, 1 << 64)) & M
    h ^= h >> 33
    h = (h * pow(0xff51afd7ed558ccd, -1, 1 << 64)) & M
    h ^= h >> 33
    return h


def _mix64(x):
    M = (1 << 64) - 1
    x ^= x >> 33; x = (x * 0xff51afd7ed558ccd) & M; x ^= x >> 33; x = (x * 0xc4ceb9fe1a85ec53) & M; x ^= x >> 33
    return x


@gpu
def test_hash_probe_chains(wfb):
    """4096 keys in 128 groups of 32 whose hashes share the low 13 bits (the table mask of max_keys = 4096): every insert
    and lookup walks a probe chain of up to 32 entries, and neighbouring chains run into each other."""
    nk, mask = 4096, 8191
    rng = np.random.default_rng(71)
    homes = rng.choice(mask + 1, 128, replace=False)
    keys = []
    for i, h0 in enumerate(homes):
        for j in range(32):
            k = _unmix64((int(rng.integers(0, 1 << 50)) << 13) | int(h0))
            assert _mix64(k) & mask == h0 and k != (1 << 64) - 1
            keys.append(k)
    table = np.array(keys, np.uint64)
    assert len(np.unique(table)) == nk
    n = nk * 400
    st = Stream(rng.integers(0, nk, n).astype(np.uint16), nk, seed=72, dense=False, table=table)
    run_and_check(wfb, st, G_LAZY, nk)


@gpu
def test_hash_one_key_over_capacity(wfb):
    """max_keys + 1 distinct keys: the table-full flag is raised, at most max_keys keys appear in the results, and every key
    that does has exactly its reference windows (a key owns a slot for all of its items or for none)."""
    import torch
    ops = wfb
    nk = 4096
    rng = np.random.default_rng(81)
    st = Stream(rng.integers(0, nk + 1, (nk + 1) * 300).astype(np.uint16), nk + 1, seed=82, dense=False)
    exp, ets = st.reference(*G_LAZY)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, *G_LAZY, max_keys=nk, dense_keys=False)
    got, gts = run_handle(ops, ff, st, ops.PROG_TUPLE64)
    nk_got, err = ff.stats()
    ff.close()
    assert err & 1
    owners = np.unique(key_index(st, got["key"]))
    assert 0 < len(owners) <= nk and nk_got >= nk
    assert len(owners) >= nk - 1  # the keys that got no slot bring no results; all others fire windows here
    check_windows(st, got, gts, exp, ets, only=owners)


# ---------------------------------------------------------------------------------------------------------------------
# 6. time-based windows with many keys (their count-based back end consumes the popped panes through the bucket path)
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("nkeys,mode,dense,nb", [(5000, "jitter", False, 2), (65536, "mono", True, 1)],
                         ids=["k5000_8perbucket_hash_jitter", "k65536_64perbucket_dense_mono"])
def test_time_based_many_keys(wfb, oracle, nkeys, mode, dense, nb):
    """Time-based windows (60, 20) over round-robin keys, one item per key every 3 time units: 5000 hash-table keys with
    out-of-order timestamps and 65 536 dense keys (every key fires at every slide boundary: Nb = 1 keeps one boundary's
    results within the oracle's per-batch output)."""
    import torch
    O, ops = oracle, wfb
    win, slide, lateness = 60, 20, 0
    per_key = 100
    n = nkeys * per_key
    rng = np.random.default_rng(nkeys)
    t = np.zeros(n, ops.TUPLE64)
    t["key"] = np.arange(n) % nkeys
    t["ivalue"] = rng.integers(0, 1 << 16, n)
    t["fvalue"] = rng.random(n)
    ts = (np.arange(n) // nkeys) * 3                   # every key: one item per 3 time units
    if mode == "jitter":
        ts = ts + rng.integers(-4, 5, n)
    ts = np.maximum(ts, 0).astype(np.uint64)
    batch = max(1024, nkeys // 4)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=nkeys, dense_keys=dense, win_type=1, lateness=lateness)
    tb = O.FfatTbOracle(win, slide, lateness, nb)
    got, gts, exp, ets = [], [], [], []
    for b in range(0, n, batch):
        tb_, tsb = t[b:b + batch], ts[b:b + batch]
        wm = int(tsb.min()) if mode == "jitter" else int(tsb[0])
        r, rt = tb.process_batch(O.lift_tuple64(tb_), tsb, wm)
        exp.append(r); ets.append(rt)
        out, out_ts, n_out = ff.process([ops.DeviceBatch.from_host(tb_, tsb, watermark=wm)])
        torch.cuda.synchronize()
        g_, gt_ = ff.results_to_host(out, out_ts, n_out)
        got.append(g_); gts.append(gt_)
    g, gt = O.sort_results(np.concatenate(got), np.concatenate(gts))
    e, et = O.sort_results(np.concatenate(exp), np.concatenate(ets))
    assert len(g) == len(e) > nkeys, (len(g), len(e))
    assert np.array_equal(g["key"], e["key"]) and np.array_equal(g["id"], e["id"])
    assert np.array_equal(gt, et) and np.array_equal(g["isum"], e["isum"])
    assert np.allclose(g["fsum"], e["fsum"], rtol=FP_RTOL, atol=0)
    nk, err = ff.stats()
    assert err == 0
    ff.close()

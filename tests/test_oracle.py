"""CPU tests (-m "not gpu"): the oracle against the golden vectors generated from the reference's own
wf/flatfat.hpp (tests/golden/*.npz, tests/golden/ref/flatfat_cpu.npz), and its own internal consistency
(tree order vs linear fold, GPU-operator semantics vs CPU-operator windows)."""
import glob
import os

import numpy as np
import pytest

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))


def _stream(O, rng, n, nkeys):
    r = np.zeros(n, dtype=O.RES)
    r["key"] = rng.integers(0, nkeys, n)
    r["isum"] = rng.integers(-1000, 1000, n)
    r["fsum"] = rng.random(n)
    return r


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_cpu_ffat_matches_reference_golden(oracle, path):
    O = oracle
    g = np.load(path)
    win, slide, batch = int(g["win"]), int(g["slide"]), int(g["batch"])
    res = np.zeros(len(g["key"]), dtype=O.RES)
    res["key"], res["isum"], res["fsum"] = g["key"], g["isum"], g["fsum"]
    oc = O.FfatCpuOracle(win, slide)
    outs, tss = [], []
    for b in range(0, len(res), batch):
        o, t = oc.process(res[b:b + batch], b)
        outs.append(o); tss.append(t)
    out = np.concatenate(outs); ts = np.concatenate(tss)
    assert len(out) == len(g["out_key"]) > 0
    assert np.array_equal(out["key"], g["out_key"]) and np.array_equal(out["id"], g["out_id"])
    assert np.array_equal(out["isum"], g["out_isum"])
    assert np.array_equal(out["fsum"], g["out_fsum"])  # same tree, same association: bit-exact
    assert np.array_equal(ts, g["out_ts"])
    eo, _ = oc.eos()
    eo = O.sort_results(eo)
    assert np.array_equal(eo["key"], g["eos_key"]) and np.array_equal(eo["id"], g["eos_id"])
    assert np.array_equal(eo["isum"], g["eos_isum"]) and np.array_equal(eo["fsum"], g["eos_fsum"])


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
@pytest.mark.parametrize("nb", [1, 3])
def test_gpu_operator_oracle_matches_reference_golden(oracle, path, nb):
    """Ffat_Windows_GPU semantics (groups of Nb, no EOS flush): every emitted window equals the reference window
    with the same (key, gwid); the emitted set is exactly the windows whose group trigger was reached."""
    O = oracle
    g = np.load(path)
    win, slide, batch = int(g["win"]), int(g["slide"]), int(g["batch"])
    res = np.zeros(len(g["key"]), dtype=O.RES)
    res["key"], res["isum"], res["fsum"] = g["key"], g["isum"], g["fsum"]
    go = O.FfatGpuOracle(win, slide, nb, keep_history=True)
    outs = []
    for b in range(0, len(res), batch):
        o, t = go.process_batch(res[b:b + batch], b)
        assert (t == b).all()
        outs.append(o)
    out = np.concatenate(outs)
    ref = {(int(k), int(i)): (int(s), float(f)) for k, i, s, f in zip(g["out_key"], g["out_id"], g["out_isum"], g["out_fsum"])}
    assert len(out) > 0
    for r in out:
        s, f = ref[(int(r["key"]), int(r["id"]))]
        assert r["isum"] == s
        assert abs(r["fsum"] - f) <= 1e-9 * max(1.0, abs(f))
        lin = go.window_linear(int(r["key"]), int(r["id"]))
        assert lin is not None and lin["isum"] == r["isum"]
    # expected count: per key, groups fired = c < B ? 0 : 1 + (c - B) // (S*Nb)
    B = (nb - 1) * slide + win
    exp = 0
    for k in np.unique(res["key"]):
        c = int((res["key"] == k).sum())
        exp += 0 if c < B else (1 + (c - B) // (slide * nb)) * nb
    assert len(out) == exp


LIVE_CASES = [(4, 2, 3), (8, 8, 1), (10, 3, 5), (7, 7, 2), (5, 1, 4), (32, 8, 6), (256, 64, 3)]  # win, slide, nkeys


def live_streams(O):
    """The streams of test_cpu_ffat_matches_live_reference, one per LIVE_CASES entry, all drawn from one seeded generator."""
    rng = np.random.default_rng(7)
    for (W, S, nk) in LIVE_CASES:
        yield W, S, nk, _stream(O, rng, max(6000, W * nk * 6), nk)


def ffat_cpu_record(O, ffat, r):
    """Digests of what a CPU FlatFAT operator emits on stream r in batches of 257 (windows, their timestamps, the windows
    flushed at end of stream) and the per-batch window counts."""
    outs, tss, counts = [], [], []
    for b in range(0, len(r), 257):
        o, ot = ffat.process(r[b:b + 257], b)
        outs.append(o); tss.append(ot); counts.append(len(o))
    eo, _ = ffat.eos()
    return {"out": O.digest(np.concatenate(outs)), "ts": O.digest(np.concatenate(tss)), "eos": O.digest(O.sort_results(eo)),
            "counts": np.array(counts, dtype=np.int64)}


def test_cpu_ffat_matches_live_reference(oracle):
    """The oracle's CPU FlatFAT operator equals, bit for bit, the reference's own wf/flatfat.hpp under the restated replica
    loop (oracle/_ref/libwfref_flatfat.so), whose outputs on these streams are stored in tests/golden/ref/flatfat_cpu.npz."""
    O = oracle
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref", "flatfat_cpu.npz"))
    for W, S, nk, r in live_streams(O):
        t = f"{W}_{S}_{nk}"
        assert O.digest(r) == str(g[t + ".input"]), "the seeded input stream changed: the recorded outputs no longer apply"
        got = ffat_cpu_record(O, O.FfatCpuOracle(W, S), r)
        assert np.array_equal(got["counts"], g[t + ".counts"])
        for k in ("out", "ts", "eos"):
            assert got[k] == str(g[t + "." + k]), (t, k)


def test_stream_generator(oracle):
    O = oracle
    t, ts = O.gen_tuple64(1000, 4096, O.KEY_UNIFORM, 65536)
    assert np.array_equal(ts, np.arange(1000, 1000 + 4096, dtype=np.uint64))
    assert np.array_equal(t["id"], ts)
    assert (t["ivalue"] >= 0).all() and (t["ivalue"] <= 0xFFFF).all()
    assert (t["fvalue"] >= 0).all() and (t["fvalue"] < 1).all()
    assert (t["key"] < 65536).all() and len(np.unique(t["key"])) > 3000
    t2, _ = O.gen_tuple64(1000, 4096, O.KEY_RR, 100)
    assert np.array_equal(t2["key"], np.arange(1000, 1000 + 4096) % 100)
    assert np.array_equal(t2["ivalue"], t["ivalue"])
    t3, _ = O.gen_tuple64(0, 20000, O.KEY_ZIPF, 1000)
    c = np.bincount(t3["key"].astype(np.int64), minlength=1000)
    assert c[0] > c[10] > c[500]


def test_map_filter_columns(oracle):
    O = oracle
    t, ts = O.gen_tuple64(0, 5000, O.KEY_UNIFORM, 64)
    surv, sts, m = O.map_filter_tuple64(t, ts, O.MAP_ADD_SCALE, 2, 1.0000001, O.FILT_EVEN)
    exp_iv = t["ivalue"] + 2
    assert np.array_equal(m, (exp_iv & 1) == 0)
    assert np.array_equal(surv["ivalue"], exp_iv[m]) and np.array_equal(sts, ts[m])
    assert np.allclose(surv["fvalue"], (t["fvalue"] * 1.0000001)[m], rtol=0, atol=0)
    assert np.array_equal(surv["id"], t["id"][m])  # stable: arrival order kept
    _, _, m3 = O.map_filter_tuple64(t, ts, O.MAP_NONE, 0, 1.0, O.FILT_MOD, 3)
    assert np.array_equal(m3, t["ivalue"] % 3 == 0)
    neg = np.array([-4, -3, -2, -1, 0, 1, 2, 3], dtype=np.int64)
    assert np.array_equal(O.filter_mask(neg, O.FILT_MOD, 2), [True, False, True, False, True, False, True, False])


def test_keyby_group_and_route(oracle):
    O = oracle
    rng = np.random.default_rng(3)
    keys = rng.integers(0, 37, 1000).astype(np.uint64)
    for order in (0, 1):
        start, mp, dk = O.keyby_group(keys, order)
        assert len(dk) == len(np.unique(keys))
        if order == 1:
            assert np.array_equal(dk, np.unique(keys))
        else:
            _, first = np.unique(keys, return_index=True)
            assert np.array_equal(dk, keys[np.sort(first)])
        seen = np.zeros(len(keys), dtype=bool)
        for k, s in zip(dk, start):
            idx = int(s); prev = -1
            assert idx == int(np.nonzero(keys == k)[0][0])
            while idx != -1:
                assert keys[idx] == k and idx > prev and not seen[idx]
                seen[idx] = True; prev = idx; idx = int(mp[idx])
        assert seen.all()
    assert np.array_equal(O.route(keys, 8), keys % 8)
    assert len(O.keyby_group(np.zeros(0, dtype=np.uint64), 1)[2]) == 0


def test_reduce_by_key(oracle):
    O = oracle
    t, ts = O.gen_tuple64(0, 3000, O.KEY_UNIFORM, 50)
    t["key"][7] = 999  # a key seen once passes through untouched
    out, ot = O.reduce_tuple64(t, ts)
    uk = np.unique(t["key"])
    assert np.array_equal(out["key"], uk)
    for r, tts in zip(out, ot):
        sel = t["key"] == r["key"]
        assert r["ivalue"] == t["ivalue"][sel].sum()
        assert abs(r["fvalue"] - t["fvalue"][sel].sum()) < 1e-9
        assert tts == ts[sel].max()
        if sel.sum() == 1:
            assert r["id"] == t["id"][sel][0]
        else:
            assert r["id"] == 0


def test_tb_oracle_matches_the_window_definition():
    """Time-based restatement (process_batch_tb / PendingPanes_Queue): on a stream whose keys appear in every batch, window
    gwid of key k is the fold of the key's tuples with ts in [gwid*slide, gwid*slide + win), consecutive gwids from 0, and
    the result timestamp is the watermark of the batch that fired it."""
    from oracle import oracle as O
    for win, slide, nb, lateness in [(40, 10, 3, 0), (30, 45, 2, 0), (64, 16, 1, 32)]:
        nkeys, n, B = 5, 6000, 500
        t, _ = O.gen_tuple64(0, n, O.KEY_RR, nkeys)
        ts = np.arange(n, dtype=np.uint64)
        res = O.lift_tuple64(t)
        tb = O.FfatTbOracle(win, slide, lateness, nb)
        outs = []
        for b in range(0, n, B):
            o, ots = tb.process_batch(res[b:b + B], ts[b:b + B], int(ts[b]))
            assert np.all(ots == int(ts[b]))
            outs.append(o)
        out = np.concatenate(outs)
        assert len(out) > 0 and tb.ignored == 0
        for r in out:
            k, g = int(r["key"]), int(r["id"])
            m = (t["key"] == k) & (ts >= g * slide) & (ts < g * slide + win)
            assert r["isum"] == t["ivalue"][m].sum()
            assert abs(r["fsum"] - t["fvalue"][m].sum()) <= 1e-9 * max(1.0, abs(r["fsum"]))
        for k in range(nkeys):
            ids = np.sort(out["id"][out["key"] == k])
            assert np.array_equal(ids, np.arange(len(ids)))


def _tb_model(batches, win, slide, lateness, nb):
    """Second, independent restatement of Ffat_Replica_GPU::process_batch_tb / process_wins_tb (wf/ffat_replica_gpu.hpp:870-1047)
    with plain Python containers: per key a dict pane -> (isum, fsum) of pending panes, the id of the first pending pane, the
    triggering pane and the list of panes already handed to the FlatFAT (windows are folds over that list). Pure model: no ring,
    no tree."""
    from math import gcd
    pane_len = gcd(win, slide)
    wp, sp = win // pane_len, slide // pane_len
    bp, group = (nb - 1) * sp + wp, sp * nb
    keys = {}
    out = []
    for res, ts, wm in batches:
        first_incomplete = (wm - lateness) // pane_len if wm >= lateness else 0
        present = []
        parts = {}
        for r, t in zip(res, ts):  # arrival order inside a (key, pane)
            k, p = int(r["key"]), int(t) // pane_len
            if k not in parts:
                parts[k] = {}
                present.append(k)
            a = parts[k].get(p)
            parts[k][p] = (int(r["isum"]), float(r["fsum"])) if a is None else (a[0] + int(r["isum"]), a[1] + float(r["fsum"]))
        for k in sorted(present):
            st = keys.setdefault(k, {"first": 0, "pend": {}, "end": 0, "trig": bp - 1, "done": False, "fed": [], "gwid": 0})
            for p in sorted(parts[k], reverse=True):  # the reference walks them newest first
                if p < st["first"]:
                    continue  # pane already consumed: dropped
                if p < st["end"]:
                    a = st["pend"].get(p, (0, 0.0))
                    st["pend"][p] = (a[0] + parts[k][p][0], a[1] + parts[k][p][1])
                else:
                    st["pend"][p] = parts[k][p]
            newest = max(parts[k])
            if newest >= st["end"]:
                st["end"] = newest + 1
            while st["trig"] < first_incomplete:
                need = group if st["done"] else bp
                for p in range(st["first"], st["first"] + need):
                    st["fed"].append(st["pend"].pop(p, (0, 0.0)))  # a missing pane is an empty pane
                st["first"] += need
                st["end"] = max(st["end"], st["first"])
                st["done"] = True
                for i in range(nb):
                    g = st["gwid"] + i
                    panes = st["fed"][g * sp:g * sp + wp]
                    isum, fsum = 0, 0.0
                    for a in panes:
                        isum += a[0]; fsum += a[1]
                    out.append((k, g, isum, fsum, wm))
                st["gwid"] += nb
                st["trig"] += group
    return out


@pytest.mark.parametrize("cfg", [(40, 10, 0, 3), (64, 16, 100, 2), (30, 45, 0, 2), (96, 32, 64, 4)])
def test_tb_oracle_vs_independent_model(cfg):
    """The C restatement of the time-based path against a second restatement with Python containers, on streams with
    out-of-order timestamps, idle periods and tuples far behind the watermark."""
    from oracle import oracle as O
    win, slide, lateness, nb = cfg
    rng = np.random.default_rng(7)
    nkeys, n, B = 6, 9000, 750
    t, _ = O.gen_tuple64(3, n, O.KEY_RR, nkeys)
    ts = np.arange(n, dtype=np.int64) * 2 + rng.integers(-30, 31, n) + (np.arange(n) // 1500) * 400
    late = rng.random(n) < 0.02
    ts = np.maximum(np.where(late, ts - rng.integers(300, 2500, n), ts), 0).astype(np.uint64)
    res = O.lift_tuple64(t)
    tb = O.FfatTbOracle(win, slide, lateness, nb)
    got, batches = [], []
    for b in range(0, n, B):
        wm = int(ts[b:b + B].min())
        r, rt = tb.process_batch(res[b:b + B], ts[b:b + B], wm)
        assert np.all(rt == wm)
        got.extend((int(x["key"]), int(x["id"]), int(x["isum"]), float(x["fsum"]), wm) for x in r)
        batches.append((res[b:b + B], ts[b:b + B], wm))
    exp = _tb_model(batches, win, slide, lateness, nb)
    assert len(got) == len(exp) > 0
    got.sort(key=lambda x: (x[0], x[1])); exp.sort(key=lambda x: (x[0], x[1]))
    for a, e in zip(got, exp):
        assert a[0] == e[0] and a[1] == e[1] and a[2] == e[2] and a[4] == e[4], (a, e)
        assert abs(a[3] - e[3]) <= 1e-9 * max(1.0, abs(e[3]))

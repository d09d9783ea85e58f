"""The oracle and the CUDA path against what the UNMODIFIED reference computed on the same inputs.

oracle/_ref/ref_pipeline_{cpu,gpu} are the reference's own wf/windflow.hpp / wf/windflow_gpu.hpp (PipeGraph, MultiPipe, emitters,
collectors, Map/Filter/Ffat_Windows and their *_GPU versions) compiled from the reference sources by oracle/Makefile over this
repository's FastFlow-compatible runtime (include/ff/) and driven by oracle/ref_pipeline.cu on the bench schema. Their outputs
on the inputs below are stored under tests/golden/ref/ (tests/golden/make_ref_golden.py), so the tests need no reference build.

  CPU:  reference CPU pipeline Source -> Map -> Filter -> Ffat_Windows(CB), 4 replicas  ==  the oracle's restatement
  GPU:  reference GPU pipeline Source -> Map_GPU -> Filter_GPU -> Ffat_Windows_GPU, count-based AND time-based
        ==  the oracle's restatement  ==  libwfb200's kernels (through the C ABI)
        reference Map_GPU -> Filter_GPU and Reduce_GPU == oracle == kernels
This is what pins the oracle's trigger loops (count-based groups, time-based panes / watermarks / lateness, reduce, compaction),
not only the FlatFAT they share: SURVEY.md 8c.
"""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref")
CPU_CASES = [(7, 64, 16), (100, 1024, 32), (5, 10, 3)]                                          # nkeys, win, slide
CB_CASES = [(13, 64, 16, 2, 2048), (5, 1024, 32, 9, 4096), (64, 4096, 64, 65, 65536), (3, 10, 3, 4, 1000)]  # nkeys, win, slide, nb, batch
TB_CASES = [("monotone", 7, 4000, 1000, 3, 0), ("ooo", 11, 3000, 500, 4, 400), ("gaps", 5, 2000, 2000, 2, 0),
            ("ooo", 4, 900, 300, 5, 0)]                                                          # kind, nkeys, win, slide, nb, lateness
MF_BATCH, MF_N, MF_KEYS = 4096, 4096 * 6 + 123, 300
TB_BATCH, TB_N = 2048, 2048 * 14 + 700
RES_TS = np.dtype([("key", "<u8"), ("id", "<u8"), ("isum", "<i8"), ("fsum", "<f8"), ("ts", "<u8")])


def batch_watermarks(ts, batch):
    """The watermark every tuple carries in these tests: the last timestamp before its batch (0 for the first batch). The
    reference's shipper refuses a watermark above the highest timestamp already emitted (wf/source_shipper.hpp), so a batch
    cannot carry its own first timestamp; a batch's watermark is the minimum over its tuples (wf/batch_gpu_t.hpp:204-210)."""
    wm = np.zeros(len(ts), dtype=np.uint64)
    for b in range(batch, len(ts), batch):
        wm[b:b + batch] = ts[:b].max()
    return wm


def mf_digest(tuples, ts):
    """Digest of the Map -> Filter output columns in stream order (the golden record of ref_pipeline_gpu gpu_mf)."""
    from oracle import oracle as O
    return O.digest(tuples["key"].astype("<u8"), tuples["id"].astype("<u8"), tuples["ivalue"].astype("<i8"),
                    tuples["fvalue"].astype("<f8"), np.asarray(ts).astype("<u8"))


def tag(case):
    return "_".join(str(x) for x in case)


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def cpu_stream(O, nkeys):
    return O.gen_tuple64(0, 200_000, O.KEY_UNIFORM, nkeys)


def cb_stream(O, nkeys, win, batch):
    n = batch * 12 + batch // 3  # a ragged last batch too
    if win == 4096:
        n = batch * 20
    tuples, ts = O.gen_tuple64(0, n, O.KEY_UNIFORM, nkeys)
    return tuples, ts, batch_watermarks(ts, batch)


def with_ts(res, ts):
    out = np.zeros(len(res), dtype=RES_TS)
    for f in ("key", "id", "isum", "fsum"):
        out[f] = res[f]
    out["ts"] = ts
    return out


# ---- CPU: the reference's Map -> Filter -> Ffat_Windows pipeline == the oracle's restatement -------------------------------------
@pytest.mark.parametrize("nkeys,win,slide", CPU_CASES)
def test_reference_cpu_pipeline_matches_oracle(oracle, nkeys, win, slide):
    """Reference run: ref_pipeline_cpu cpu_cb, par=4 (1 source + 4 map/filter + 4 ffat + 1 sink: cfg 1 of BASELINE.json), det=1,
    watermarks every 4096 tuples."""
    O = oracle
    tuples, ts = cpu_stream(O, nkeys)
    surv, sts, _ = O.map_filter_tuple64(tuples, ts, 1, 2, 1.0000001, 1)
    cpu = O.FfatCpuOracle(win, slide)
    r, rt = cpu.process(O.lift_tuple64(surv), 0)
    r2, rt2 = cpu.eos()   # the CPU operator flushes the partial windows at end of stream (wf/ffat_replica.hpp:406-427)
    exp = with_ts(np.concatenate([r, r2]), np.concatenate([rt, rt2]))
    g = golden("cpu_pipeline")
    assert int(g[tag((nkeys, win, slide)) + ".n"]) > 0
    # (the CPU operator's result timestamps depend on replica interleaving: not compared)
    O.check_windows_record(exp, g, tag((nkeys, win, slide)), rtol=1e-9, with_ts=False)


# ---- GPU: reference GPU operators == oracle == libwfb200 ----------------------------------------------------------------------------
def _ours_cb(wfb, tuples, ts, wm, batch, win, slide, nb, nkeys):
    import torch
    ops = wfb
    f = ops.functors(map_kind=1, iadd=2, fscale=1.0000001, filt_kind=1)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=max(64, nkeys))
    res, rts = [], []
    for i in range(0, len(tuples), batch):
        b = ops.DeviceBatch.from_host(tuples[i:i + batch], ts[i:i + batch], watermark=int(wm[i]))
        out, out_ts, n_out = ff.process([b], pre=f)
        torch.cuda.synchronize()
        r, t = ff.results_to_host(out, out_ts, n_out)
        res.append(r); rts.append(t)
    return with_ts(np.concatenate(res), np.concatenate(rts))


def _oracle_cb(O, tuples, ts, wm, batch, win, slide, nb):
    go = O.FfatGpuOracle(win, slide, nb)
    res, rts = [], []
    for i in range(0, len(tuples), batch):
        surv, sts, _ = O.map_filter_tuple64(tuples[i:i + batch], ts[i:i + batch], 1, 2, 1.0000001, 1)
        r, t = go.process_batch(O.lift_tuple64(surv), int(wm[i]))
        res.append(r); rts.append(t)
    return with_ts(np.concatenate(res), np.concatenate(rts))


@pytest.mark.gpu
@pytest.mark.parametrize("nkeys,win,slide,nb,batch", CB_CASES)
def test_reference_gpu_cb_pipeline_matches_oracle_and_kernels(oracle, wfb, nkeys, win, slide, nb, batch):
    O = oracle
    tuples, ts, wm = cb_stream(O, nkeys, win, batch)
    g, t = golden("gpu_cb"), tag((nkeys, win, slide, nb, batch))
    assert int(g[t + ".n"]) > 0
    exp = _oracle_cb(O, tuples, ts, wm, batch, win, slide, nb)
    O.check_windows_record(exp, g, t, rtol=1e-9)         # oracle == reference (same tree association: tight)
    got = _ours_cb(wfb, tuples, ts, wm, batch, win, slide, nb, nkeys)
    O.check_windows_record(got, g, t, rtol=1e-6)         # kernels == reference (pane-then-tree association: north_star's 1e-6)


def _tb_stream(O, n, nkeys, kind, seed=3):
    tuples, ts = O.gen_tuple64(0, n, O.KEY_UNIFORM, nkeys)
    rng = np.random.default_rng(seed)
    if kind == "monotone":
        ts = np.cumsum(rng.integers(1, 40, size=n)).astype(np.uint64)
    elif kind == "ooo":       # out of order inside a bounded horizon
        base = np.cumsum(rng.integers(1, 40, size=n)).astype(np.int64)
        ts = np.maximum(0, base - rng.integers(0, 300, size=n)).astype(np.uint64)
    else:                      # idle gaps: the watermark jumps over many panes
        gaps = rng.integers(1, 20, size=n)
        gaps[rng.integers(0, n, size=8)] = 20000
        ts = np.cumsum(gaps).astype(np.uint64)
    return tuples, ts


@pytest.mark.gpu
@pytest.mark.parametrize("kind,nkeys,win,slide,nb,lateness", TB_CASES)
def test_reference_gpu_tb_pipeline_matches_oracle_and_kernels(oracle, wfb, kind, nkeys, win, slide, nb, lateness):
    """Time-based windows: the reference's own Ffat_Replica_GPU::process_batch_tb / process_wins_tb / PendingPanes_Queue."""
    import torch
    O, ops = oracle, wfb
    batch, n = TB_BATCH, TB_N
    tuples, ts = _tb_stream(O, n, nkeys, kind)
    wm = batch_watermarks(ts, batch)
    to = O.FfatTbOracle(win, slide, lateness, nb)
    f = ops.functors(map_kind=1, iadd=2, fscale=1.0000001, filt_kind=1)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=64, win_type=1, lateness=lateness)
    exp_r, exp_t, got_r, got_t = [], [], [], []
    for i in range(0, n, batch):
        surv, sts, _ = O.map_filter_tuple64(tuples[i:i + batch], ts[i:i + batch], 1, 2, 1.0000001, 1)
        r, t = to.process_batch(O.lift_tuple64(surv), sts, int(wm[i]))
        exp_r.append(r); exp_t.append(t)
        b = ops.DeviceBatch.from_host(tuples[i:i + batch], ts[i:i + batch], watermark=int(wm[i]))
        out, out_ts, n_out = ff.process([b], pre=f)
        torch.cuda.synchronize()
        r, t = ff.results_to_host(out, out_ts, n_out)
        got_r.append(r); got_t.append(t)
    exp = with_ts(np.concatenate(exp_r), np.concatenate(exp_t))
    got = with_ts(np.concatenate(got_r), np.concatenate(got_t))
    g, t = golden("gpu_tb"), tag((kind, nkeys, win, slide, nb, lateness))
    assert int(g[t + ".n"]) > 0
    O.check_windows_record(exp, g, t, rtol=1e-6)    # the oracle's restatement == the reference (pins SURVEY.md row a10)
    O.check_windows_record(got, g, t, rtol=1e-6)    # kernels == the reference


@pytest.mark.gpu
def test_reference_gpu_map_filter_and_reduce_match_oracle_and_kernels(oracle, wfb):
    import torch
    O, ops = oracle, wfb
    batch, n, nkeys = MF_BATCH, MF_N, MF_KEYS
    tuples, ts = O.gen_tuple64(0, n, O.KEY_UNIFORM, nkeys)
    g = golden("gpu_mf_red")
    # Map_GPU -> Filter_GPU: the stream of survivors, in order (one source, one replica each)
    surv, sts, _ = O.map_filter_tuple64(tuples, ts, 1, 2, 1.0000001, 1)
    assert len(surv) == int(g["mf.n"])
    assert mf_digest(surv, sts) == str(g["mf.digest"])   # key, id, ivalue, fvalue and ts of every survivor, bit for bit
    eng = ops.Engine(ops.PROG_TUPLE64)
    f = ops.functors(map_kind=1, iadd=2, fscale=1.0000001, filt_kind=1)
    got = []
    for i in range(0, n, batch):
        b = ops.DeviceBatch.from_host(tuples[i:i + batch], ts[i:i + batch])
        o, k = eng.map_filter(b, f)
        torch.cuda.synchronize()
        got.append(ops.to_host(o.tuples, O.TUPLE64, int(k.item())))
    got = np.concatenate(got)
    assert got.tobytes() == np.ascontiguousarray(surv).tobytes()
    # Reduce_GPU keyed: one item per distinct key and batch, ascending key
    exp = []
    for i in range(0, n, batch):
        r, rt = O.reduce_tuple64(tuples[i:i + batch], ts[i:i + batch])
        exp.append(r)
    exp = np.concatenate(exp)
    assert len(exp) == int(g["red.n"])
    assert O.digest(exp["key"].astype("<u8"), exp["ivalue"].astype("<i8")) == str(g["red.digest"])
    assert np.allclose(g["red.fvalue"], exp["fvalue"], rtol=1e-9)

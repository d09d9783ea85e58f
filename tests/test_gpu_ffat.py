"""GPU parity tests (-m gpu): Ffat_Windows_GPU (count-based) through the C ABI against the oracle, the golden
vectors generated from the reference's wf/flatfat.hpp, and the outputs of the reference's own wf/flatfat_gpu.hpp on a B200.
Bit-exact on keys, window ids, integer aggregates and result timestamps; floating-point aggregates within 1e-6
relative (the pane/tree association differs from the reference's)."""
import glob
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
FP_RTOL = 1e-6
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))


def _run_gpu(ops, ff, batches, pre=None, group=1):
    """Feeds the batches `group` at a time; a pipelined handle hands results over one call late (+ flush at the end)."""
    import torch
    got, gts = [], []
    for i in range(0, len(batches), group):
        out, out_ts, n_out = ff.process(batches[i:i + group], pre=pre)
        torch.cuda.synchronize()
        r, t = ff.results_to_host(out, out_ts, n_out)
        if ff.pipelined and i == 0:
            assert len(r) == 0
        got.append(r); gts.append(t)
    if ff.pipelined:
        out, out_ts, n_out = ff.flush(device=batches[0].tuples.device)
        torch.cuda.synchronize()
        r, t = ff.results_to_host(out, out_ts, n_out)
        got.append(r); gts.append(t)
        out, out_ts, n_out = ff.flush(device=batches[0].tuples.device)  # nothing left
        torch.cuda.synchronize()
        assert int(n_out.item()) == 0
    return np.concatenate(got), np.concatenate(gts)


def _check(O, got, gts, exp, ets, res_is32=True):
    g, gt = O.sort_results(got, gts)
    e, et = O.sort_results(exp, ets)
    assert len(g) == len(e), (len(g), len(e))
    assert np.array_equal(g["key"], e["key"]) and np.array_equal(g["id"], e["id"])
    assert np.array_equal(gt, et)
    if res_is32:
        assert np.array_equal(g["isum"], e["isum"])
        assert np.allclose(g["fsum"], e["fsum"], rtol=FP_RTOL, atol=0)
    else:
        assert np.array_equal(g["value"], e["isum"])


CASES = [  # win, slide, nb, nkeys, n, batch, group(batches per call), dense
    (4, 2, 1, 3, 3000, 257, 1, False),
    (4, 2, 3, 3, 3000, 257, 2, True),
    (10, 3, 2, 5, 5000, 100, 3, False),      # pane = 1
    (16, 16, 1, 2, 2000, 64, 1, False),      # tumbling
    (8, 24, 2, 4, 4000, 500, 2, False),      # hopping with gaps (slide > win)
    (64, 16, 5, 7, 20000, 333, 4, True),
    (1024, 32, 1, 4, 30000, 1000, 8, False),
    (4096, 64, 65, 3, 60000, 4096, 5, True),  # cfg-4 geometry (B = 8192), few keys
    (4096, 64, 1, 2, 30000, 4096, 3, False),
    (32, 8, 2, 1, 5000, 777, 1, False),      # single key (non-keyed shape)
    (32, 8, 2, 600, 60000, 5000, 4, False),  # many keys, few items each
]


@pytest.mark.parametrize("pipelined", [False, True], ids=["direct", "pipelined"])
@pytest.mark.parametrize("case", CASES, ids=[f"w{c[0]}_s{c[1]}_nb{c[2]}_k{c[3]}" for c in CASES])
def test_ffat_cb_vs_oracle(wfb, oracle, case, pipelined):
    O, ops = oracle, wfb
    win, slide, nb, nkeys, n, batch, group, dense = case
    t, ts = O.gen_tuple64(0, n, O.KEY_UNIFORM, nkeys)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=max(nkeys, 8), dense_keys=dense, pipelined=pipelined)
    go = O.FfatGpuOracle(win, slide, nb)
    batches, exp, ets = [], [], []
    for b in range(0, n, batch):
        batches.append(ops.DeviceBatch.from_host(t[b:b + batch], ts[b:b + batch]))
        r, rt = go.process_batch(O.lift_tuple64(t[b:b + batch]), int(ts[b]))
        exp.append(r); ets.append(rt)
    got, gts = _run_gpu(ops, ff, batches, group=group)
    _check(O, got, gts, np.concatenate(exp), np.concatenate(ets))
    nk, err = ff.stats()
    assert err == 0
    if not dense:
        assert nk == len(np.unique(t["key"]))


def test_ffat_fused_map_filter(wfb, oracle):
    """Map_GPU -> Filter_GPU -> Ffat_Windows_GPU fused in one pass == the three operators applied in turn."""
    O, ops = oracle, wfb
    win, slide, nb, nkeys, n, batch = 64, 16, 2, 50, 100000, 8192
    t, ts = O.gen_tuple64(0, n, O.KEY_UNIFORM, nkeys)
    f = ops.functors(map_kind=1, iadd=2, fscale=1.0000001, filt_kind=1)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=64)
    go = O.FfatGpuOracle(win, slide, nb)
    batches, exp, ets = [], [], []
    for b in range(0, n, batch):
        batches.append(ops.DeviceBatch.from_host(t[b:b + batch], ts[b:b + batch]))
        surv, sts, _ = O.map_filter_tuple64(t[b:b + batch], ts[b:b + batch], 1, 2, 1.0000001, 1)
        r, rt = go.process_batch(O.lift_tuple64(surv), int(ts[b]))
        exp.append(r); ets.append(rt)
    got, gts = _run_gpu(ops, ff, batches, pre=f, group=5)
    _check(O, got, gts, np.concatenate(exp), np.concatenate(ets))
    # unfused: Filter_GPU output batches fed to a second FFAT handle give the same windows
    eng = ops.Engine(ops.PROG_TUPLE64)
    ff2 = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=64)
    import torch
    filtered = []
    for b in batches:
        out, n_out = eng.map_filter(b, f)
        out.n = int(n_out.item())
        filtered.append(out)
    got2, gts2 = _run_gpu(ops, ff2, filtered, group=3)
    _check(O, got2, gts2, np.concatenate(exp), np.concatenate(ets))


def test_ffat_ragged_and_empty_batches(wfb, oracle):
    import torch
    O, ops = oracle, wfb
    win, slide, nb, nkeys = 16, 4, 2, 6
    rng = np.random.default_rng(11)
    sizes = [0, 1, 5, 0, 300, 1, 2, 1023, 0, 77, 4096, 3, 0, 0, 9]
    t, ts = O.gen_tuple64(0, sum(sizes), O.KEY_UNIFORM, nkeys)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=8, pipelined=True)
    go = O.FfatGpuOracle(win, slide, nb)
    batches, exp, ets, off = [], [], [], 0
    for k, sz in enumerate(sizes):
        wm = 1000 + k
        if sz:
            batches.append(ops.DeviceBatch.from_host(t[off:off + sz], ts[off:off + sz], watermark=wm))
        else:
            batches.append(ops.DeviceBatch(torch.empty(0, dtype=torch.uint8, device="cuda"),
                                           torch.empty(0, dtype=torch.int64, device="cuda"), 0, wm))
        r, rt = go.process_batch(O.lift_tuple64(t[off:off + sz]), wm)
        exp.append(r); ets.append(rt)
        off += sz
    got, gts = _run_gpu(ops, ff, batches, group=4)
    _check(O, got, gts, np.concatenate(exp), np.concatenate(ets))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
@pytest.mark.parametrize("nb", [1, 4])
def test_ffat_cb_vs_reference_golden(wfb, oracle, path, nb):
    """Windows must equal the ones the reference's own wf/flatfat.hpp produced (tests/golden/make_golden.py)."""
    O, ops = oracle, wfb
    g = np.load(path)
    win, slide, batch = int(g["win"]), int(g["slide"]), int(g["batch"])
    n = len(g["key"])
    t = np.zeros(n, dtype=ops.TUPLE64)
    t["key"], t["ivalue"], t["fvalue"] = g["key"], g["isum"], g["fsum"]
    ts = np.arange(n, dtype=np.uint64)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=16)
    batches = [ops.DeviceBatch.from_host(t[b:b + batch], ts[b:b + batch], watermark=b) for b in range(0, n, batch)]
    got, gts = _run_gpu(ops, ff, batches, group=3)
    ref = {(int(k), int(i)): (int(s), float(f)) for k, i, s, f in zip(g["out_key"], g["out_id"], g["out_isum"], g["out_fsum"])}
    B = (nb - 1) * slide + win
    expn = 0
    for k in np.unique(g["key"]):
        c = int((g["key"] == k).sum())
        expn += 0 if c < B else (1 + (c - B) // (slide * nb)) * nb
    assert len(got) == expn > 0
    assert len({(int(r["key"]), int(r["id"])) for r in got}) == len(got)
    for r in got:
        s, f = ref[(int(r["key"]), int(r["id"]))]
        assert r["isum"] == s
        assert abs(r["fsum"] - f) <= FP_RTOL * abs(f)


def test_ffat_wfwin24_reference_functors(wfb, oracle):
    """The reference's win test functors: lift value, comb + (win_common_gpu.hpp:295-314), source value = i per key
    (win_common_gpu.hpp:100-116): closed form sum of window g = sum_{j=g*S+1}^{g*S+W} j."""
    O, ops = oracle, wfb
    win, slide, nb, nkeys, per_key = 20, 5, 3, 4, 500
    t = np.zeros(per_key * nkeys, dtype=ops.WFWIN24)
    i = np.repeat(np.arange(1, per_key + 1), nkeys)
    t["key"] = np.tile(np.arange(nkeys), per_key)
    t["value"] = i
    ts = np.arange(len(t), dtype=np.uint64) * 7
    ff = ops.FfatWindowsGPU(ops.PROG_WFWIN24, win, slide, nb, max_keys=8)
    batches = [ops.DeviceBatch.from_host(t[b:b + 150], ts[b:b + 150]) for b in range(0, len(t), 150)]
    got, gts = _run_gpu(ops, ff, batches, group=2)
    B = (nb - 1) * slide + win
    groups = 1 + (per_key - B) // (slide * nb)
    assert len(got) == groups * nb * nkeys
    for r in got:
        g = int(r["id"])
        a, b = g * slide + 1, g * slide + win
        assert r["value"] == (a + b) * win // 2
    res = np.zeros(len(t), dtype=O.RES)
    res["key"], res["isum"] = t["key"], t["value"]
    go = O.FfatGpuOracle(win, slide, nb)
    exp, ets = [], []
    for b in range(0, len(t), 150):
        r, rt = go.process_batch(res[b:b + 150], int(ts[b]))
        exp.append(r); ets.append(rt)
    _check(O, got, gts, np.concatenate(exp), np.concatenate(ets), res_is32=False)


REF_GPU_GEOMS = [(64, 16, 5), (4096, 64, 1), (4096, 64, 65), (16, 4, 5)]  # win, slide, nb
REF_GPU_STEP = 1000


def ref_gpu_stream(O, geom):
    """The stream of test_reference_flatfat_gpu_on_this_box: one key, power-of-two B, fed in chunks of REF_GPU_STEP."""
    win, slide, nb = geom
    B = (nb - 1) * slide + win
    assert B & (B - 1) == 0
    n = B * 3 + 1234
    rng = np.random.default_rng(5)
    res = np.zeros(n, dtype=O.RES)
    res["key"] = 42
    res["isum"] = rng.integers(-1000, 1000, n)
    res["fsum"] = rng.random(n)
    return res


@pytest.mark.parametrize("geom", REF_GPU_GEOMS)
def test_reference_flatfat_gpu_on_this_box(wfb, oracle, geom):
    """The reference's own FlatFAT_GPU (wf/flatfat_gpu.hpp compiled for sm_100a into oracle/_ref, run on a B200; its outputs
    on this stream are stored in tests/golden/ref/flatfat_gpu.npz): pins the oracle's restatement of K12-K14 bit for bit,
    and through it our kernels, against the reference itself (power-of-two B)."""
    import torch
    O, ops = oracle, wfb
    win, slide, nb = geom
    res = ref_gpu_stream(O, geom)
    n = len(res)
    g, tag = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref", "flatfat_gpu.npz")), "_".join(map(str, geom))
    assert O.digest(res) == str(g[tag + ".input"]), "the seeded input stream changed: the recorded outputs no longer apply"
    go = O.FfatGpuOracle(win, slide, nb)
    t = np.zeros(n, dtype=ops.TUPLE64)
    t["key"], t["ivalue"], t["fvalue"] = res["key"], res["isum"], res["fsum"]
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, win, slide, nb, max_keys=4)
    step = REF_GPU_STEP
    exp, exp_ts, counts = [], [], []
    for b in range(0, n, step):
        chunk = res[b:b + step]
        e, et = go.process_batch(chunk, b)
        exp.append(e); exp_ts.append(et); counts.append(len(e))
        o, o_ts, n_out = ff.process([ops.DeviceBatch.from_host(t[b:b + step], np.arange(b, b + len(chunk), dtype=np.uint64), watermark=b)])
        torch.cuda.synchronize()
        r, rt = ff.results_to_host(o, o_ts, n_out)
        k = len(e)
        assert len(r) == k
        if k:
            rs, rts = O.sort_results(r, rt)
            assert np.array_equal(rs["id"], e["id"]) and np.array_equal(rs["isum"], e["isum"])
            assert np.allclose(rs["fsum"], e["fsum"], rtol=FP_RTOL, atol=0)
            assert np.array_equal(rts, et)
    # oracle == reference kernels, bit for bit (same tree order): per-chunk counts, windows and their timestamps
    assert np.array_equal(np.array(counts, dtype=np.int64), g[tag + ".counts"])
    assert O.digest(np.concatenate(exp)) == str(g[tag + ".out"])
    assert O.digest(np.concatenate(exp_ts)) == str(g[tag + ".ts"])


def test_ffat_capacity_error_flag(wfb, oracle):
    O, ops = oracle, wfb
    t, ts = O.gen_tuple64(0, 5000, O.KEY_UNIFORM, 100)
    ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, 8, 4, 1, max_keys=10)
    ff.process([ops.DeviceBatch.from_host(t, ts)])
    nk, err = ff.stats()
    assert err & 1


def test_ffat_full_size_property(wfb, oracle):
    """BASELINE config 4 geometry at full key count (win 4096, slide 64, 65536 keys, round-robin keys, value = per-key
    sequence number): every window sum has a closed form, and window ids per key are consecutive from 0."""
    import torch
    O, ops = oracle, wfb
    win, slide, nb, nkeys = 4096, 64, 1, 65536
    per_key = win + 3 * slide  # 4 windows per key
    ff = ops.FfatWindowsGPU(ops.PROG_WFWIN24, win, slide, nb, max_keys=nkeys, dense_keys=True)
    batch = 65536 * 8
    total = per_key * nkeys
    outs, outts = [], []
    keys = torch.arange(nkeys, dtype=torch.int64, device="cuda")
    for start in range(0, total, batch * 8):
        bs = []
        for b0 in range(start, min(total, start + batch * 8), batch):
            m = min(batch, total - b0)
            idx = torch.arange(b0, b0 + m, dtype=torch.int64, device="cuda")
            rec = torch.stack([idx % nkeys, torch.zeros_like(idx), idx // nkeys + 1], dim=1).contiguous()
            bs.append(ops.DeviceBatch(rec.view(torch.uint8).reshape(-1), None, m, watermark=b0))
        out, out_ts, n_out = ff.process(bs)
        torch.cuda.synchronize()
        r, rt = ff.results_to_host(out, out_ts, n_out)
        outs.append(r); outts.append(rt)
    got = np.concatenate(outs)
    assert len(got) == 4 * nkeys
    g = got["id"].astype(np.int64)
    a, b = g * slide + 1, g * slide + win
    assert np.array_equal(got["value"], (a + b) * win // 2)
    srt = O.sort_results(got)
    assert np.array_equal(srt["key"], np.repeat(np.arange(nkeys), 4))
    assert np.array_equal(srt["id"], np.tile(np.arange(4), nkeys))
    assert ff.stats()[1] == 0


@pytest.mark.parametrize("shards", [2, 3, 8])
def test_ffat_key_shard_replicas(wfb, oracle, shards):
    """`shards` replicas, each owning the keys with key % shards == r on compact slots (wfb_ffat_set_key_shard) and fed
    its keys' tuples in arrival order, together produce the windows of one operator over the whole stream; the in-place
    path of the lifted-record program is used when the chunks sit at their tile positions."""
    import torch
    O, ops = oracle, wfb
    win, slide, nb, nkeys, n, batch = 64, 16, 3, 50, 80000, 5000
    t, ts = O.gen_tuple64(0, n, O.KEY_UNIFORM, nkeys)
    go = O.FfatGpuOracle(win, slide, nb)
    reps = []
    for r in range(shards):
        ff = ops.FfatWindowsGPU(ops.PROG_LIFTED32, win, slide, nb, max_keys=(nkeys + shards - 1) // shards, dense_keys=True)
        ff.set_key_shard(shards, r)
        reps.append(ff)
    got, gts, exp, ets = [], [], [], []
    for b in range(0, n, batch):
        tb, tsb = t[b:b + batch], ts[b:b + batch]
        r_, rt_ = go.process_batch(O.lift_tuple64(tb), int(ts[b]))
        exp.append(r_); ets.append(rt_)
        lifted = O.lift_tuple64(tb)
        for r, ff in enumerate(reps):
            mine = lifted[lifted["key"] % shards == r]
            # two chunks laid out at their tile positions in one buffer (what the multi-GPU receive side does)
            h = len(mine) // 2
            off2 = ((h + 255) // 256) * 256
            buf = torch.zeros((off2 + len(mine) - h) * 32, dtype=torch.uint8, device="cuda")
            buf[:h * 32] = torch.from_numpy(mine[:h].view(np.uint8).copy()).cuda()
            buf[off2 * 32:(off2 + len(mine) - h) * 32] = torch.from_numpy(mine[h:].view(np.uint8).copy()).cuda()
            chunks = [ops.DeviceBatch(buf[:h * 32], None, h, int(ts[b])), ops.DeviceBatch(buf[off2 * 32:], None, len(mine) - h, int(ts[b]))]
            out, out_ts, n_out = ff.process(chunks)
            torch.cuda.synchronize()
            g_, gt_ = ff.results_to_host(out, out_ts, n_out)
            got.append(g_); gts.append(gt_)
    _check(O, np.concatenate(got), np.concatenate(gts), np.concatenate(exp), np.concatenate(ets))
    for ff in reps:
        assert ff.stats()[1] == 0
    # a key of another shard is a capacity error, not a silent drop
    bad = O.lift_tuple64(t[:10]); bad["key"] = 1
    reps[0].process([ops.DeviceBatch.from_host(bad, None, 0)])
    torch.cuda.synchronize()
    assert reps[0].stats()[1] & 1

#!/usr/bin/env python
"""bench.py -- tuples/sec of the Map_GPU -> Filter_GPU -> Ffat_Windows_GPU (count-based) pipeline on N B200s.

    python bench.py --gpus N --steps K --warmup W                 (our arm; one process per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K --warmup W   (the reference's CPU path on the host cores)

Workload (BASELINE.json north_star / SURVEY.md 8d): 64-byte tuples of the seeded synthetic stream, batch 65536,
65536 uniform keys, map (ivalue += 2, fvalue *= 1.0000001) -> filter ((ivalue & 1) == 0) -> count-based sliding
windows win 4096 / slide 64, Nb 65, lift {isum, fsum}, comb +. A *step* is one stream segment of `--batches-per-step`
consecutive batches handed to the operator in one call (the operator coalesces queued batches; one launch sequence
per segment). Every step reads a DIFFERENT segment of the stream, resident in HBM (no segment is replayed inside the
timed region; each is larger than L2). The window state is primed (untimed): every key is past its first trigger and
the keys' trigger phases are spread evenly over the trigger period, so every timed step fires the same expected number
of windows (keys / 65 groups of 65) whatever K and N are.

One JSON line is printed by rank 0 (see the contract in the task statement): value = whole-job tuples/s with inputs
resident in HBM; e2e = the same through the public call with HOST (pinned) buffers, host<->device copies inside the
timed region; roofline = the whole pipeline against the measured HBM peak with SURVEY 8d's bytes per tuple (+ the
per-kernel table); cpu_baseline = the reference's own CPU pipeline timed on this box's cores on a bounded sample;
gpu_reference = the reference's own GPU operators (unmodified headers compiled for sm_100a) on this box; facade = the
same pipeline driven through the builder API (include/wf/windflow_gpu.hpp) for K queued batches per call; check =
window results of a sample of keys at this exact configuration against an independent reconstruction of their history.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 65536
TUPLE_BYTES = 64
NKEYS = 65536
WIN, SLIDE = 4096, 64
MAP = dict(map_kind=1, iadd=2, fscale=1.0000001)
FILT = dict(filt_kind=1, mod=1)
SIGMA = 0.5  # selectivity of (ivalue & 1) == 0 on the synthetic stream
CHECK_STEPS = 2
PHASE_STEPS = 8
CHECK_KEYS = 48

# algorithmic bytes per input tuple (SURVEY.md 8d / DESIGN.md section 4)
METRIC = "tuples/sec, Map_GPU->Filter_GPU->Ffat_Windows_GPU (CB win 4096 slide 64) pipeline"
PIPELINE_BYTES_PER_TUPLE = 123.3        # SURVEY.md 8d: read I + sigma*(3R + (O+12R)/S), I=72 R=32 O=40 S=64
KERNEL_BYTES_PER_TUPLE = {              # compulsory traffic of each phase of one call, per input tuple
    "tile_pass (map, filter, lift, key->slot)": 64 + SIGMA * (32 + 4),      # read tuple; write sigma * (lifted result + slot)
    "partition (per-tile counts -> offsets -> scatter)": SIGMA * (4 + 8),    # read sigma slots; write sigma (slot, position) pairs
    "window update + queries": SIGMA * (8 + 32 + (32 + 8 + 7 * 64 + 8 * 32) / 64 + (40 + 12 * 32) / 64),  # pairs + records; per pane: state, leaf, path; windows
}
REF_CPU = os.path.join(ROOT, "oracle", "_ref", "ref_pipeline_cpu")
REF_GPU = os.path.join(ROOT, "oracle", "_ref", "ref_pipeline_gpu")
FACADE_APP = os.path.join(ROOT, "windflow_b200", "apps", "pipeline_bench.bin")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram bytes per launch of the kernels from the committed ncu captures (profiles/traffic.json), or {}."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return {}
    return {}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML DURING the timed region (a 2 ms poll in a thread)."""

    def __init__(self, index=0):
        self.index, self.samples, self.reasons, self.max_mhz, self.ok = index, [], set(), None, False
        self._stop = threading.Event()
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _poll(self):
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")]}
        self._stop.set()
        self.t.join(timeout=1)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own CPU pipeline (Source -> Map -> Filter -> Ffat_Windows, PipeGraph) on the host cores
# ----------------------------------------------------------------------------------------------------------
def cpu_reference_sample(target_seconds, nb):
    """One bounded sample of the bench workload through the UNMODIFIED reference (oracle/_ref/ref_pipeline_cpu: wf/windflow.hpp
    compiled from /root/reference over include/ff/): Source -> Map(par) -> Filter(par) -> Ffat_Windows(par, keyby) -> Sink,
    65536 uniform keys, win 4096 / slide 64. Returns (tuples/s, threads, kind, description)."""
    cores = host_cores()
    if os.path.exists(REF_CPU):
        par = max(1, (cores - 2) // 2)  # 1 source + par (map+filter chained) + par ffat + 1 sink threads = the cores we may use
        n = 1 << 21
        # calibrate on one pass over 2 Mi tuples, then size the sample for the time budget
        def run(reps):
            p = subprocess.run([REF_CPU, "cpu_cb", f"gen={n}", f"keys={NKEYS}", f"win={WIN}", f"slide={SLIDE}", f"par={par}", f"reps={reps}"],
                               capture_output=True, text=True, timeout=900)
            if p.returncode != 0:
                raise RuntimeError("ref_pipeline_cpu failed: " + p.stderr[-500:])
            return json.loads(p.stdout.strip().splitlines()[-1])
        r = run(1)
        reps = int(max(1, min(64, target_seconds / max(r["seconds"], 1e-3))))
        if reps > 1:
            r = run(reps)
        desc = (f"the reference's own PipeGraph (wf/windflow.hpp unmodified, FastFlow API from include/ff/): Source(1) -> Map({par}) -> Filter({par}) -> "
                f"Ffat_Windows({par}, keyby, CB {WIN}/{SLIDE}) -> Sink(1), {r['threads']} threads on {cores} usable cores; first {r['tuples']} tuples of the "
                f"stream, {NKEYS} uniform keys: the per-tuple FlatFAT inserts are paid, no window has fired yet (a key needs {WIN} tuples: "
                f"{WIN * NKEYS * 2} tuples of this stream, hours at this rate); {r['seconds']:.1f} s")
        return r["tuples_per_s"], r["threads"], "reference", desc
    # the reference was not compiled here: the oracle's restatement, one key shard per Python thread (ctypes releases the GIL)
    from oracle import oracle as O
    threads = max(1, cores)
    kpt = max(1, NKEYS // threads)
    n_buf = 1 << 18
    bufs = [O.gen_tuple64(s * n_buf, n_buf, O.KEY_UNIFORM, kpt) for s in range(threads)]
    pipes = [O.CpuPipe("port", 1, 2, 1.0000001, 1, 1, WIN, SLIDE, 0, 1) for _ in range(threads)]

    def run_all(reps):
        def work(p, buf):
            for _ in range(reps):
                p.run(buf[0], buf[1], BATCH)
        th = [threading.Thread(target=work, args=(p, b)) for p, b in zip(pipes, bufs)]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        return time.perf_counter() - t0
    dt1 = run_all(1)
    reps = max(1, int(target_seconds / max(dt1, 1e-3)))
    dt = run_all(reps)
    for p in pipes:
        p.close()
    return reps * n_buf * threads / dt, threads, "port", (f"oracle port of map.hpp/filter.hpp/ffat_replica.hpp/flatfat.hpp, {threads} threads x {kpt} keys "
                                                         f"({threads * kpt} keys in all), pre-routed streams, {reps} x {n_buf} tuples per thread")


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step = 60.0 / max(1, args.steps + args.warmup)
    vals, desc, threads, kind = [], "", 0, "reference"
    for i in range(args.warmup + args.steps):
        tps, threads, kind, desc = cpu_reference_sample(max(2.0, min(10.0, per_step)), args.nb)
        if i >= args.warmup:
            vals.append(tps)
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": v,
        "unit": "tuples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * BATCH * args.batches_per_step / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "i64+f64", "data": "synthetic",
        "config": {"workload": "map_filter_ffat_cb", "batch": BATCH, "tuple_bytes": TUPLE_BYTES, "keys": NKEYS, "key_dist": "uniform",
                   "win": WIN, "slide": SLIDE, "wins_per_batch": args.nb, "map": "ivalue+=2,fvalue*=1.0000001", "filter": "(ivalue&1)==0",
                   "selectivity": SIGMA,
                   "note": "the reference's CPU Map->Filter->Ffat_Windows pipeline on this box's host cores; every step is a bounded sample of "
                           "the same stream (wins_per_batch is a GPU-operator parameter: the CPU operator emits every window on its own); "
                           "values of the steps: " + ", ".join(f"{x / 1e6:.2f}M" for x in vals)},
        "cpu_baseline": {"value": v, "unit": "tuples/s", "cores": threads, "kind": kind, "sample": desc},
        "e2e": {"value": v, "unit": "tuples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
# the stream the GPU arm feeds: every segment is logged so that the check can rebuild the history of a few keys
# ----------------------------------------------------------------------------------------------------------
def stagger_rounds(world):
    """Untimed priming rounds that spread the keys' trigger phases: round r feeds one pane (64 surviving tuples) to the keys
    < NKEYS (r+1)/65, so key k ends up 65 - floor(65 k / NKEYS) panes ahead -- uniformly spread over the period of 65 panes."""
    rounds = []
    for r in range(65):
        nk = max(1, NKEYS * (r + 1) // 65)
        n = int(np.ceil(SLIDE / SIGMA * nk / (BATCH * world))) * BATCH  # per rank, whole batches
        rounds.append((nk, n))
    return rounds


def expected_windows_for_keys(hist, keys, O, nb):
    """Independent reconstruction: `hist` = the segments fed so far in global stream order, each (start, n, nkeys_gen, first_wm,
    tag). Returns {key: (ivals, fvals, wms)} of the key's surviving tuples in arrival order (wm = watermark of the tuple's batch)."""
    sel = np.zeros(NKEYS, dtype=np.uint8)
    sel[keys] = 1
    acc = {int(k): ([], [], []) for k in keys}
    for (start, n, nk, wm0, _tag) in hist:
        s = sel[:nk] if nk < NKEYS else sel
        k, idx, iv, fv = O.scan_keys(start, n, O.KEY_UNIFORM, nk, np.ascontiguousarray(s))
        wm = wm0 + ((idx - start) // BATCH) * BATCH
        for key in np.unique(k):
            m = k == key
            a = acc[int(key)]
            a[0].append(iv[m]); a[1].append(fv[m]); a[2].append(wm[m])
    return {k: (np.concatenate(v[0]) if v[0] else np.zeros(0, np.int64), np.concatenate(v[1]) if v[1] else np.zeros(0),
                np.concatenate(v[2]) if v[2] else np.zeros(0, np.uint64)) for k, v in acc.items()}


def check_results(hist, n_before, got, keys, O, nb, check_ts):
    """got: structured results (key, id, isum, fsum, ts) the operator produced for `keys` in the check steps. Expected: the groups
    whose triggering tuple (count B + g*slide*nb) arrived in the check steps (tuples after the first n_before[key] ones)."""
    B = (nb - 1) * SLIDE + WIN
    per = SLIDE * nb
    full = expected_windows_for_keys(hist, keys, O, nb)
    compared, bad = 0, []
    for key in keys:
        iv, fv, wm = full[int(key)]
        c0, c1 = n_before[int(key)], len(iv)
        g_lo = 0 if c0 < B else (c0 - B) // per + 1          # first group whose trigger count is > c0
        exp = []
        g = g_lo
        while B + g * per <= c1:
            trig = B + g * per                                # 1-based count of the triggering tuple
            for j in range(nb):
                w = g * nb + j
                a, b = w * SLIDE, w * SLIDE + WIN
                exp.append((w, int(iv[a:b].sum()), float(np.sum(fv[a:b])), int(wm[trig - 1])))
            g += 1
        mine = got[got["key"] == key]
        mine = mine[np.argsort(mine["id"])]
        if len(mine) != len(exp):
            bad.append(f"key {key}: {len(mine)} windows, expected {len(exp)}")
            continue
        for r, e in zip(mine, exp):
            ok = int(r["id"]) == e[0] and int(r["isum"]) == e[1] and abs(float(r["fsum"]) - e[2]) <= 1e-6 * abs(e[2]) and (not check_ts or int(r["ts"]) == e[3])
            if not ok:
                bad.append(f"key {key} window {e[0]}: got {(int(r['id']), int(r['isum']), float(r['fsum']), int(r['ts']))} expected {e}")
                break
        compared += len(exp)
    return compared, bad


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from windflow_b200 import build, ops, multigpu

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- windflow_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    build.build()

    bps = args.batches_per_step
    seg_tuples = bps * BATCH
    nb = args.nb
    B = (nb - 1) * SLIDE + WIN
    f = ops.functors(**MAP, **FILT)
    pipelined = args.pipeline
    e2e_steps = max(2, min(args.steps, args.e2e_steps))
    do_check = not args.no_check

    # ---- the stream: global step t covers world * seg_tuples consecutive indices, rank r owns [(t*world + r) * seg_tuples, +seg_tuples) ----
    hist = []          # every segment fed to the operator, global stream order: (start, n, nkeys of the generator, first watermark, tag)

    def gen_segment(start, n, nkeys=NKEYS):
        b = ops.gen_tuple64(start, n, ops.KEY_UNIFORM, nkeys)
        b.watermark = start
        seg = ops.Segment([ops.DeviceBatch(b.tuples[i * BATCH * 64:(i + 1) * BATCH * 64], b.ts[i * BATCH:(i + 1) * BATCH], BATCH, watermark=start + i * BATCH)
                           for i in range(n // BATCH)])
        ops._cbatches(seg)  # the C descriptors of the segment's batches, built now (a C++ replica fills them in a microsecond; ctypes needs ~0.2 ms)
        return b, seg

    def log(step_index, n, nkeys, tag, base=0):
        for r in range(world):
            start = base + (step_index * world + r) * n
            hist.append((start, n, nkeys, start, tag))

    if world == 1 and not args.mg_path:
        ff = ops.FfatWindowsGPU(ops.PROG_TUPLE64, WIN, SLIDE, nb, max_keys=NKEYS, dense_keys=True, pipelined=pipelined)
        pipe = None
    elif world == 1:  # profiling aid: the N>1 step (source pass -> exchange buffers -> update on records) with one rank, no NCCL
        pipe = multigpu.KeyShardedPipelineC(ops, f, WIN, SLIDE, nb, NKEYS, 0, 1, dev)
        ff = pipe.ff
    else:
        if args.py_exchange or args.sync_exchange:  # the torch.distributed version of the step (windflow_b200/multigpu.py)
            pipe = multigpu.KeyShardedPipeline(ops, f, WIN, SLIDE, nb, NKEYS, rank, world, dev, pipelined=not args.sync_exchange)
        else:                                        # the whole step under the C ABI (wfb_mg_step: NCCL send/recv groups issued from C)
            pipe = multigpu.KeyShardedPipelineC(ops, f, WIN, SLIDE, nb, NKEYS, rank, world, dev)
        ff = pipe.ff
    cap = ff.max_results(seg_tuples * (4 if pipe is not None else 1))  # (a flush of the multi-GPU pipeline delivers three steps at once)
    out = torch.empty(cap * 32, dtype=torch.uint8, device=dev)
    out_ts = torch.empty(cap, dtype=torch.int64, device=dev)
    n_out = torch.zeros(1, dtype=torch.int32, device=dev)

    def feed(whole, batches):
        if pipe is None:
            ff.process(batches, pre=f, out=out, out_ts=out_ts, n_out=n_out)
        else:
            pipe.step(batches, whole.watermark, out, out_ts, n_out)

    # ---- prime the window state (untimed setup): every key past its first trigger, phases spread over the period -------------------
    STAG_BASE = 1 << 44   # the stagger rounds draw from a far-away part of the index space (their own, logged, segments)
    t_step = 0            # global step counter of the main stream
    prime = int(np.ceil(B * NKEYS / SIGMA / (seg_tuples * world))) + 2
    if args.prime_steps >= 0:
        prime = args.prime_steps  # profiling runs only: the timed steps are then NOT steady state
    scratch = None
    for i in range(prime):
        scratch = gen_segment(multigpu.owner_span(t_step, rank, world, seg_tuples)[0], seg_tuples)
        feed(*scratch); log(t_step, seg_tuples, NKEYS, "prime"); t_step += 1
    stag_off = 0
    if args.prime_steps < 0:
        for (nk, n) in stagger_rounds(world):
            start = STAG_BASE + stag_off + rank * n
            scratch = gen_segment(start, n, nk)
            feed(*scratch)
            for r in range(world):
                s = STAG_BASE + stag_off + r * n
                hist.append((s, n, nk, s, "stagger"))
            stag_off += world * n
    torch.cuda.synchronize()
    del scratch

    # ---- the segments of the measured part, resident in HBM before the clock starts (each one read once) ------------------------------
    n_main = args.warmup + args.steps + PHASE_STEPS + e2e_steps + (CHECK_STEPS if do_check else 0)
    ring = min(n_main, max(4, args.ring))
    segs = [gen_segment(multigpu.owner_span(t_step + i, rank, world, seg_tuples)[0], seg_tuples) for i in range(ring)]
    replay = n_main > ring  # (only with --steps beyond the ring: segments then repeat, with their original indices)
    torch.cuda.synchronize()

    t0_main = t_step
    cur = {"j": 0}

    def log_main(jj, tag):  # the jj-th step of the measured part reads segs[jj % ring], generated for global step t0_main + jj % ring
        log(t0_main + (jj % ring), seg_tuples, NKEYS, tag)

    def step(tag="main"):   # next step of the measured part
        jj = cur["j"]
        feed(*segs[jj % ring])
        log_main(jj, tag)
        cur["j"] = jj + 1

    def launches_now():
        return ff.launches + (pipe.eng.launches if pipe is not None else 0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step("warmup")
    torch.cuda.synchronize()

    # ---- timed region: K steps, device-resident inputs ------------------------------------------------------------
    launches0 = launches_now()
    sampler = ClockSampler(local)
    torch.cuda.synchronize()
    results0 = ff.results_total()   # device-side counter of the handle: no per-step read-back, no extra kernels in the timed loop
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    host_t0 = time.perf_counter()
    for _ in range(args.steps):
        step("timed")
    host_ms = (time.perf_counter() - host_t0) * 1e3 / args.steps  # host time to ISSUE a step (must stay below the device time of a step)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    launches = launches_now() - launches0
    last_step = ff.results_to_host(out, out_ts, n_out) if args.dump_outputs else None  # (read after the clock stopped)
    results1 = ff.results_total()
    # per-phase device times (CUDA events inside the call) on PHASE_STEPS further steps, outside the timed region: the event records cost ~10 us per step
    for _ in range(2):
        step("phases")   # (re-fill the queue after the read-back above before the event-timed steps)
    ff.timing(True)
    for _ in range(PHASE_STEPS):
        step("phases")
    torch.cuda.synchronize()
    ing_ms, sort_ms, upd_ms, tot_ms, calls = ff.timing(False)
    err = ff.stats()[1]
    if err:
        raise SystemExit(f"bench.py: device error flags {err}")
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    wins = torch.tensor([float(results1 - results0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(wins, op=dist.ReduceOp.SUM)
    ms_max = float(t_ms.item())
    value = world * args.steps * seg_tuples / (ms_max * 1e-3)
    windows_timed = int(wins.item())
    windows_expected = args.steps * world * seg_tuples * SIGMA / SLIDE  # steady state: one window per slide surviving tuples of a key

    # ---- e2e: the same call with HOST (pinned) buffers, copies inside the timed region ------------------------------
    e2e = run_e2e(torch, ops, feed, segs, ring, cur["j"], seg_tuples, bps, dev, e2e_steps, world, out, n_out)
    for s_ in range(e2e_steps):
        log_main(cur["j"] + s_, "e2e")
    cur["j"] += e2e_steps

    # ---- check: two more steps, the results of a sample of keys against an independent reconstruction of their history ---------------------
    check = None
    if do_check and not replay:
        check = run_check(torch, dist, ops, ff, pipe, step, hist, out, out_ts, n_out, nb, rank, world, dev, pipelined or (pipe is not None and not args.sync_exchange))
    if pipe is not None:
        pipe.flush(out, out_ts, n_out)
        torch.cuda.synchronize()
    if last_step is not None:
        if world > 1:
            gathered = [None] * world if rank == 0 else None
            dist.gather_object(last_step, gathered, dst=0)
            if rank == 0:
                last_step = (np.concatenate([g[0] for g in gathered]), np.concatenate([g[1] for g in gathered]))
        if rank == 0:
            dump_outputs(args.dump_outputs, *last_step)
    if rank == 0:
        peak, peak_src = measured_peaks()
        traffic = ncu_traffic()
        calls = max(1, calls)
        phases = [("tile_pass (map, filter, lift, key->slot)", ing_ms / calls), ("partition (per-tile counts -> offsets -> scatter)", sort_ms / calls),
                  ("window update + queries", upd_ms / calls)]
        kernels = []
        for name, avg_ms in phases:
            bpt = KERNEL_BYTES_PER_TUPLE[name]
            ach = bpt * seg_tuples / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
            kernels.append({"phase": name, "avg_us": avg_ms * 1e3, "algorithmic_bytes": bpt * seg_tuples, "ncu_dram_bytes": traffic.get(name),
                            "achieved_gbs": ach, "frac": ach / peak})
        pipe_gbs = value / world * PIPELINE_BYTES_PER_TUPLE / 1e9
        cpu_tps, cpu_threads, cpu_kind, cpu_desc = cpu_reference_sample(args.cpu_seconds, nb)
        line = {
            "metric": METRIC,
            "value": value, "unit": "tuples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "host_issue_ms_per_step": host_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i64+f64", "data": "synthetic",
            "config": {"workload": "map_filter_ffat_cb", "batch": BATCH, "tuple_bytes": TUPLE_BYTES,
                       "batches_per_step": bps, "tuples_per_step_per_gpu": seg_tuples, "keys": NKEYS, "keys_per_gpu": NKEYS // world,
                       "key_dist": "uniform", "win": WIN, "slide": SLIDE, "wins_per_batch": nb,
                       "map": "ivalue+=2,fvalue*=1.0000001", "filter": "(ivalue&1)==0", "selectivity": SIGMA,
                       "l2": f"inputs larger than L2 and read once: {ring} distinct segments x {seg_tuples * 64 / 1e6:.0f} MB resident in HBM" + (" (replayed: more steps than --ring)" if replay else ""),
                       "state_primed_steps": prime, "phase_stagger_rounds": 65 if args.prime_steps < 0 else 0,
                       "windows_in_timed_region": windows_timed, "windows_expected_steady_state": windows_expected,
                       "pipelined": args.pipeline if world == 1 else (not args.sync_exchange),
                       "parallelism": f"keyby{world}" + ("" if world == 1 else (" (torch.distributed step: Map->Filter->lift + partition by key % N | NCCL all-to-all of 32-B results | Ffat on the key shard)"
                                                                                  if (args.py_exchange or args.sync_exchange) else
                                                                                  " (wfb_mg_step: Map->Filter->lift + ONE partition by (destination, bucket) at the source | 32-B results pushed over NVLink "
                                                                                  "(copy engine; NCCL when cudaIpc is unavailable) | run concatenation + window update on the key shard)"))},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "e2e": e2e,
            "roofline": {"bound": "hbm", "kernel": "whole pipeline (one call = tile pass + partition + window update + window queries), SURVEY 8d bytes per tuple",
                         "achieved": pipe_gbs, "peak": peak, "unit": "GB/s", "frac": pipe_gbs / peak,
                         "traffic": traffic.get("pipeline_dram_bytes_per_call"), "peak_source": peak_src,
                         "bytes_per_tuple": PIPELINE_BYTES_PER_TUPLE, "avg_launch_ms": tot_ms / calls,
                         "kernels": kernels if world == 1 else None,
                         "note": None if world == 1 else "per GPU; the per-kernel table is on the N=1 line (at N>1 the timed handle is the destination side)"},
            "cpu_baseline": {"value": cpu_tps, "unit": "tuples/s", "cores": cpu_threads, "kind": cpu_kind, "sample": cpu_desc},
            "check": check,
        }
        if world == 1 and not args.no_extras:
            line["gpu_reference"] = gpu_reference_sample(nb)
            line["facade"] = facade_sweep(nb)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, res, ts):
    """The window results the last timed step handed back (all ranks), in (key, window id) order, as DIR/window_<field>.npy in
    float64 (exact: keys, ids, integer sums and timestamps stay below 2^53). Beyond DUMP_MAX_BYTES a fixed, seeded sample of
    rows is written. The inputs depend only on the arguments, so two builds can be compared file by file."""
    order = np.lexsort((res["id"], res["key"]))
    cols = {"key": res["key"][order], "id": res["id"][order], "isum": res["isum"][order], "fsum": res["fsum"][order], "ts": ts[order]}
    rows = DUMP_MAX_BYTES // (8 * len(cols))
    if len(order) > rows:
        keep = np.sort(np.random.default_rng(0).choice(len(order), rows, replace=False))
        cols = {k: v[keep] for k, v in cols.items()}
    os.makedirs(path, exist_ok=True)
    for k, v in cols.items():
        np.save(os.path.join(path, f"window_{k}.npy"), v.astype(np.float64))


def run_check(torch, dist, ops, ff, pipe, step, hist, out, out_ts, n_out, nb, rank, world, dev, delayed):
    """CHECK_STEPS more steps; the windows of CHECK_KEYS sampled keys produced in them are compared (key, window id, integer sum exact,
    floating-point sum within 1e-6, result timestamp at N = 1) with sums over the keys' own tuples, rebuilt from the stream generator
    for the WHOLE history (priming, stagger, warm-up, timed, e2e and check steps). All ranks call this."""
    from oracle import oracle as O
    res_dt = np.dtype([("key", "<u8"), ("id", "<u8"), ("isum", "<i8"), ("fsum", "<f8"), ("ts", "<u8")])
    rng = np.random.default_rng(12345)
    keys = np.unique(np.concatenate([[0, 1, NKEYS - 1, NKEYS // 2], rng.integers(0, NKEYS, CHECK_KEYS)])).astype(np.int64)
    torch.cuda.synchronize()
    if delayed:  # results arrive one call late: drain what is pending first, so that the check steps' results are exactly the ones collected
        if pipe is not None:
            pipe.flush(out, out_ts, n_out)
        else:
            ff.flush(out, out_ts, n_out)
        torch.cuda.synchronize()
    n_hist = len(hist)
    got = []

    def collect():
        torch.cuda.synchronize()
        r, t = ff.results_to_host(out, out_ts, n_out)
        g = np.zeros(len(r), dtype=res_dt)
        for fld in ("key", "id", "isum", "fsum"):
            g[fld] = r[fld]
        g["ts"] = t
        got.append(g[np.isin(g["key"], keys)])
    for _ in range(CHECK_STEPS):
        step("check")
        collect()
    if delayed:
        if pipe is not None:
            pipe.flush(out, out_ts, n_out)
        else:
            ff.flush(out, out_ts, n_out)
        collect()
    mine = np.concatenate(got) if got else np.zeros(0, dtype=res_dt)
    if world > 1:
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(mine, gathered, dst=0)
        if rank != 0:
            return None
        mine = np.concatenate(gathered)
    # history before the check steps -> tuples each sampled key had then; whole history -> the expected windows
    before = expected_windows_for_keys(hist[:n_hist], keys, O, nb)
    n_before = {int(k): len(before[int(k)][0]) for k in keys}
    compared, bad = check_results(hist, n_before, mine, keys, O, nb, check_ts=(world == 1 and pipe is None))
    if bad:
        raise SystemExit("bench.py --check FAILED: " + "; ".join(bad[:5]))
    return {"passed": True, "keys_sampled": int(len(keys)), "windows_compared": int(compared), "steps": CHECK_STEPS,
            "history_segments": len(hist), "fsum_rtol": 1e-6, "timestamps_compared": world == 1 and pipe is None,
            "how": "sums over each sampled key's own surviving tuples (arrival ranks [64 w, 64 w + 4096)), rebuilt from the stream generator over the whole history"}


def gpu_reference_sample(nb):
    """The reference's own GPU operators on this box: oracle/_ref/ref_pipeline_gpu = wf/windflow_gpu.hpp (Map_GPU -> Filter_GPU ->
    Ffat_Windows_GPU, unmodified, nvcc -arch sm_100a) inside the reference's PipeGraph, on a bounded sample of the bench stream."""
    if not os.path.exists(REF_GPU):
        return {"unavailable": "oracle/_ref/ref_pipeline_gpu was not built (needs /root/reference at build time)"}
    out = {}
    try:
        for tag, keys, n in (("bench_config_65536_keys", NKEYS, 1 << 20), ("64_keys", 64, 1 << 22)):
            p = subprocess.run([REF_GPU, "gpu_cb", f"gen={n}", f"keys={keys}", f"batch={BATCH}", f"win={WIN}", f"slide={SLIDE}", f"nb={nb}"],
                               capture_output=True, text=True, timeout=300)
            if p.returncode != 0:
                out[tag] = {"error": p.stderr[-300:]}
                continue
            r = json.loads(p.stdout.strip().splitlines()[-1])
            out[tag] = {"value": r["tuples_per_s"], "unit": "tuples/s", "tuples": r["tuples"], "seconds": r["seconds"], "threads": r["threads"]}
        out["what"] = ("the reference's Map_GPU -> Filter_GPU -> Ffat_Windows_GPU (wf/*.hpp unmodified, Thrust + its own kernels, sm_100a) in its own "
                       "PipeGraph on this GPU; CPU source pushing tuple by tuple, batch 65536; the window operator loops over the distinct keys of "
                       "every batch on the host (wf/ffat_replica_gpu.hpp:783-827)")
    except Exception as e:  # pragma: no cover
        out["error"] = repr(e)
    return out


def facade_sweep(nb):
    """The same pipeline through the builder API (windflow_b200/apps/pipeline_bench.cu over include/wf/windflow_gpu.hpp): replicas on
    threads, queues between them, the window replica taking up to K queued batches per call."""
    if not os.path.exists(FACADE_APP):
        return {"unavailable": "windflow_b200/apps/pipeline_bench.bin not built"}
    rows = []
    for k, timed, style in ((1, 2048, "fluent"), (4, 8192, "fluent"), (16, 16384, "fluent"), (64, 24576, "fluent"), (128, 32768, "fluent"), (128, 32768, "statements")):
        try:
            p = subprocess.run([FACADE_APP, str(k), str(timed), str(NKEYS), str(nb), "512", "2", style], capture_output=True, text=True, timeout=300)
            if p.returncode != 0:
                rows.append({"max_batches_per_call": k, "style": style, "error": (p.stdout + p.stderr)[-300:]})
                continue
            r = json.loads(p.stdout.strip().splitlines()[-1])
            rows.append({"max_batches_per_call": k, "style": style, "value": r["tuples_per_s"], "unit": "tuples/s", "tuples": r["tuples"], "threads": r["threads"],
                         "windows": r["windows"]})
        except Exception as e:  # pragma: no cover
            rows.append({"max_batches_per_call": k, "style": style, "error": repr(e)})
    return {"api": "facade", "what": "SourceGPU (ring of batches in HBM) -> Map_GPU -> Filter_GPU -> Ffat_Windows_GPU -> Sink built with the builders and "
                                     "MultiPipe; Map and Filter are fused into the window operator's ingest pass -- style fluent: one chain expression, the functor types reach the "
                                     "program (inlined); style statements: one chain call per statement, fused through device function pointers; wall clock over the timed "
                                     "batches after priming",
            "rows": rows}


def _parse_cpulist(text):
    """'0-3,8,10-11' -> [0, 1, 2, 3, 8, 10, 11]"""
    cpus = []
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.extend(range(int(lo), int(hi or lo) + 1))
    return cpus


class numa_local:
    """While active, the calling thread runs on the CPUs of the NUMA node the GPU hangs off, so that host buffers allocated (and pinned)
    inside land in that node's memory: with 8 ranks on one box, pinned staging buffers on the far socket halve the H2D rate. Best effort:
    without the sysfs files, or without permission, nothing changes. The previous affinity is restored on exit (the CPU legs use all cores)."""

    def __init__(self, torch, index):
        self.cpus, self.prev = None, None
        try:
            p = torch.cuda.get_device_properties(index)
            bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
            node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
            if node >= 0:
                cpus = set(_parse_cpulist(open(f"/sys/devices/system/node/node{node}/cpulist").read())) & os.sched_getaffinity(0)
                self.cpus = cpus or None
                self.node = node
        except Exception:
            self.cpus = None

    def __enter__(self):
        if self.cpus:
            try:
                self.prev = os.sched_getaffinity(0)
                os.sched_setaffinity(0, self.cpus)
            except Exception:
                self.prev = None
        return self

    def __exit__(self, *exc):
        if self.prev is not None:
            try:
                os.sched_setaffinity(0, self.prev)
            except Exception:
                pass
        return False


def run_e2e(torch, ops, feed, segs, ring, j0, seg_tuples, bps, dev, steps, world, out, n_out):
    """Same operator call(s), inputs start in pinned host memory every step; result count + results come back."""
    import torch.distributed as dist
    nbuf = 2
    res_cap = out.numel() // 32
    with numa_local(torch, dev.index if dev.index is not None else 0) as nl:  # pinned staging buffers in the memory of the GPU's own NUMA node
        host_t = [torch.empty(seg_tuples * 64, dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
        host_ts = [torch.empty(seg_tuples, dtype=torch.int64).pin_memory() for _ in range(nbuf)]
        host_n = torch.zeros(1, dtype=torch.int32).pin_memory()
        host_res = torch.empty(res_cap * 32, dtype=torch.uint8).pin_memory()
        for t in host_t + host_ts + [host_res]:
            t.zero_()  # first touch while the thread sits on that node
    dev_t = [torch.empty(seg_tuples * 64, dtype=torch.uint8, device=dev) for _ in range(nbuf)]
    dev_ts = [torch.empty(seg_tuples, dtype=torch.int64, device=dev) for _ in range(nbuf)]
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream()
    ready = [torch.cuda.Event() for _ in range(nbuf)]
    freed = [torch.cuda.Event() for _ in range(nbuf)]

    def stage(k, s):  # the host side of the source: the step's segment sits in pinned host memory (copied out untimed)
        whole = segs[(j0 + s) % ring][0]
        host_t[k].copy_(whole.tuples); host_ts[k].copy_(whole.ts)
        return whole.watermark

    def h2d(k):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[k])
            dev_t[k].copy_(host_t[k], non_blocking=True)
            dev_ts[k].copy_(host_ts[k], non_blocking=True)
            ready[k].record(copy_stream)

    def compute(k, wm):
        main.wait_event(ready[k])
        whole = ops.DeviceBatch(dev_t[k], dev_ts[k], seg_tuples, wm)
        batches = [ops.DeviceBatch(dev_t[k][i * BATCH * 64:(i + 1) * BATCH * 64], dev_ts[k][i * BATCH:(i + 1) * BATCH], BATCH,
                                   watermark=wm + i * BATCH) for i in range(bps)]
        feed(whole, batches)
        freed[k].record(main)
        host_n.copy_(n_out, non_blocking=True)

    # the steps' segments are staged in host memory two at a time; the staging copy (device -> pinned) of step s+2 is NOT part of the
    # stream's work and happens while the clock is stopped -- so the timed region is split per pair of steps
    d2h_bytes, total_ms = 0, 0.0
    for k in range(nbuf):
        freed[k].record(main)
    s = 0
    while s < steps:
        pair = min(nbuf, steps - s)
        wms = [stage(k, s + k) for k in range(pair)]
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        h2d(0)
        for k in range(pair):
            if k + 1 < pair:
                h2d(k + 1)
            compute(k, wms[k])
            main.synchronize()                       # the caller reads the step's result count ...
            nres = int(host_n.item())
            if nres:                                  # ... and the window results themselves
                host_res[:nres * 32].copy_(out[:nres * 32], non_blocking=True)
                d2h_bytes += nres * 32
            d2h_bytes += 4
        e1.record()
        torch.cuda.synchronize()
        total_ms += e0.elapsed_time(e1)
        s += pair
    t_ms = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    val = world * steps * seg_tuples / (float(t_ms.item()) * 1e-3)
    return {"value": val, "unit": "tuples/s", "h2d_bytes_per_step": seg_tuples * 72, "d2h_bytes_per_step": d2h_bytes // steps,
            "steps": steps, "note": "pinned host segment -> H2D (double-buffered on a copy stream) -> the operator call(s) "
                                    "-> D2H of the result count and the window results; timed in pairs of steps (the clock stops while the next "
                                    "pair of segments is staged in host memory)",
            "host_buffers_numa_node": getattr(nl, "node", None) if nl.cpus else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=65)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batches-per-step", type=int, default=128, help="queued batches the replica hands to the operator per call (one stream segment)")
    ap.add_argument("--ring", type=int, default=96, help="distinct segments resident in HBM (more steps than this replay them)")
    ap.add_argument("--nb", type=int, default=65, help="withNumWinPerBatch")
    ap.add_argument("--e2e-steps", type=int, default=12)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--pipeline", action="store_true", help="WFB_FFAT_PIPELINED handle: results one call late, partition+update overlap the next ingest")
    ap.add_argument("--sync-exchange", action="store_true", help="N > 1: exchange and window update of a step right after its source pass (no overlap with the next step)")
    ap.add_argument("--mg-path", action="store_true", help="N = 1 only, profiling aid: run the N>1 step (wfb_mg_step) with a single rank")
    ap.add_argument("--py-exchange", action="store_true", help="N > 1: drive the exchange from Python (torch.distributed) instead of wfb_mg_step")
    ap.add_argument("--prime-steps", type=int, default=-1, help="override state priming (ncu runs); default: steady state")
    ap.add_argument("--no-check", action="store_true", help="skip the result check of the sampled keys")
    ap.add_argument("--no-extras", action="store_true", help="skip the gpu_reference and facade legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the window results of the last timed step to DIR/window_<field>.npy")
    args = ap.parse_args()
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

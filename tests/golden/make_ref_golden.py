"""Generates tests/golden/ref/*.npz: what the reference's own code, built into oracle/_ref/ by oracle/Makefile, computes
on the inputs of the tests that compare with it. The tests then compare with these records and need no reference build.

    python tests/golden/make_ref_golden.py cpu [DIR]   # cpu_pipeline.npz, flatfat_cpu.npz
    python tests/golden/make_ref_golden.py gpu [DIR]   # on a B200: gpu_cb.npz, gpu_tb.npz, gpu_mf_red.npz, flatfat_gpu.npz

DIR defaults to tests/golden/ref. Outputs the tests compare bit for bit are recorded as SHA-256 digests; floating-point
window sums compared within a tolerance are stored (a fixed sample of oracle.GOLDEN_SAMPLE rows beyond that size).
"""
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from oracle import oracle as O  # noqa: E402
import test_reference_live as T  # noqa: E402

REF_CPU = os.path.join(ROOT, "oracle", "_ref", "ref_pipeline_cpu")
REF_GPU = os.path.join(ROOT, "oracle", "_ref", "ref_pipeline_gpu")
TUP_TS = np.dtype([("key", "<u8"), ("id", "<u8"), ("ivalue", "<i8"), ("fvalue", "<f8"), ("pad", "<u8", (4,)), ("ts", "<u8")])


def run_ref(exe, mode, tuples, ts, wm, dtype=T.RES_TS, **kw):
    """One run of ref_pipeline_{cpu,gpu}: the stream goes in through a file, the results come back through another."""
    with tempfile.TemporaryDirectory() as d:
        inp, out = os.path.join(d, "in.bin"), os.path.join(d, "out.bin")
        with open(inp, "wb") as f:
            f.write(np.uint64(len(tuples)).tobytes())
            f.write(np.ascontiguousarray(tuples).tobytes()); f.write(np.ascontiguousarray(ts, dtype=np.uint64).tobytes())
            f.write(np.ascontiguousarray(wm, dtype=np.uint64).tobytes())
        p = subprocess.run([exe, mode, f"in={inp}", f"out={out}"] + [f"{k}={v}" for k, v in kw.items()], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        info = json.loads(p.stdout.strip().splitlines()[-1])
        raw = open(out, "rb").read()
    m = int(np.frombuffer(raw[:8], dtype=np.uint64)[0])
    res = np.frombuffer(raw[8:], dtype=dtype, count=m).copy()
    assert info["results"] == m and m > 0
    return res, info


def cpu(out_dir):
    import test_oracle
    rec = {}
    for nkeys, win, slide in T.CPU_CASES:
        tuples, ts = T.cpu_stream(O, nkeys)
        ref, info = run_ref(REF_CPU, "cpu_cb", tuples, ts, T.batch_watermarks(ts, 4096), keys=nkeys, win=win, slide=slide, par=4, det=1)
        assert info["threads"] >= 10  # 1 source + 4 map/filter + 4 ffat + 1 sink (cfg 1 of BASELINE.json)
        rec.update(O.windows_record(ref, T.tag((nkeys, win, slide)), with_ts=False))
    np.savez_compressed(os.path.join(out_dir, "cpu_pipeline.npz"), **rec)
    rec = {}
    for W, S, nk, r in test_oracle.live_streams(O):
        t = f"{W}_{S}_{nk}"
        rec[t + ".input"] = np.array(O.digest(r))
        for k, v in test_oracle.ffat_cpu_record(O, O.RefFfatCpu(W, S), r).items():
            rec[t + "." + k] = np.array(v)
    np.savez_compressed(os.path.join(out_dir, "flatfat_cpu.npz"), **rec)


def gpu(out_dir):
    import test_gpu_ffat
    from windflow_b200 import ops
    rec = {}
    for nkeys, win, slide, nb, batch in T.CB_CASES:
        tuples, ts, wm = T.cb_stream(O, nkeys, win, batch)
        ref, _ = run_ref(REF_GPU, "gpu_cb", tuples, ts, wm, keys=nkeys, win=win, slide=slide, nb=nb, batch=batch)
        rec.update(O.windows_record(ref, T.tag((nkeys, win, slide, nb, batch))))
    np.savez_compressed(os.path.join(out_dir, "gpu_cb.npz"), **rec)
    rec = {}
    for kind, nkeys, win, slide, nb, lateness in T.TB_CASES:
        tuples, ts = T._tb_stream(O, T.TB_N, nkeys, kind)
        ref, _ = run_ref(REF_GPU, "gpu_tb", tuples, ts, T.batch_watermarks(ts, T.TB_BATCH), keys=nkeys, win=win, slide=slide, nb=nb,
                         batch=T.TB_BATCH, lateness=lateness)
        rec.update(O.windows_record(ref, T.tag((kind, nkeys, win, slide, nb, lateness))))
    np.savez_compressed(os.path.join(out_dir, "gpu_tb.npz"), **rec)
    tuples, ts = O.gen_tuple64(0, T.MF_N, O.KEY_UNIFORM, T.MF_KEYS)
    wm = T.batch_watermarks(ts, T.MF_BATCH)
    mf, _ = run_ref(REF_GPU, "gpu_mf", tuples, ts, wm, dtype=TUP_TS, batch=T.MF_BATCH)
    red, _ = run_ref(REF_GPU, "gpu_red", tuples, ts, wm, dtype=TUP_TS, batch=T.MF_BATCH)
    np.savez_compressed(os.path.join(out_dir, "gpu_mf_red.npz"), **{
        "mf.n": np.int64(len(mf)), "mf.digest": np.array(T.mf_digest(mf, mf["ts"])),
        "red.n": np.int64(len(red)), "red.digest": np.array(O.digest(red["key"].astype("<u8"), red["ivalue"].astype("<i8"))),
        "red.fvalue": red["fvalue"].copy()})
    L = O.ref_gpu_lib()
    assert L is not None, "oracle/_ref/libwfref_flatfat_gpu.so missing: run make -C oracle"
    rec = {}
    for geom in test_gpu_ffat.REF_GPU_GEOMS:
        win, slide, nb = geom
        res = test_gpu_ffat.ref_gpu_stream(O, geom)
        h = L.wfref_ffat_gpu_create(win, slide, nb, 42)
        outs, tss, counts = [], [], []
        for b in range(0, len(res), test_gpu_ffat.REF_GPU_STEP):
            chunk = res[b:b + test_gpu_ffat.REF_GPU_STEP]
            d = ops.to_device(chunk)
            cap = (len(chunk) // slide + 2) * nb + nb
            out = np.zeros(cap, dtype=O.RES); ots = np.zeros(cap, dtype=np.uint64)
            k = L.wfref_ffat_gpu_process(h, C.c_void_p(d.data_ptr()), len(chunk), b, out.ctypes.data_as(C.c_void_p),
                                         ots.ctypes.data_as(C.c_void_p), cap)
            outs.append(out[:k]); tss.append(ots[:k]); counts.append(k)
        L.wfref_ffat_gpu_destroy(h)
        t = "_".join(map(str, geom))
        rec.update({t + ".input": np.array(O.digest(res)), t + ".counts": np.array(counts, dtype=np.int64),
                    t + ".out": np.array(O.digest(np.concatenate(outs))), t + ".ts": np.array(O.digest(np.concatenate(tss)))})
    np.savez_compressed(os.path.join(out_dir, "flatfat_gpu.npz"), **rec)


if __name__ == "__main__":
    which = sys.argv[1]
    out_dir = sys.argv[2] if len(sys.argv) > 2 else os.path.join(HERE, "ref")
    os.makedirs(out_dir, exist_ok=True)
    {"cpu": cpu, "gpu": gpu}[which](out_dir)
    for f in sorted(os.listdir(out_dir)):
        print(f, os.path.getsize(os.path.join(out_dir, f)), "bytes")

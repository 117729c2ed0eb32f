"""GPU-box parity + timing sweep (run under gpurun).

For every case: render with the unmodified reference build (oracle/_ref) and
with libmprb on the same packed tape, fingerprint both (tools/parity.py),
report every mismatching field, time both, and write
  gpurun_out/check.jsonl          one JSON line per case
  gpurun_out/golden/<case>.json   reference fingerprint summary (hashes, counts)
  gpurun_out/golden/<case>.npz    full reference arrays for the small cases
"""
import argparse
import json
import sys
import time
import traceback
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import oracle  # noqa: E402
import parity  # noqa: E402
from mpr_b200 import capi  # noqa: E402

CASES = [
    # model, dim, size
    ("hello_world", 2, 256),
    ("prospero", 2, 256),
    ("prospero", 2, 1024),
    ("involute_gear_2d", 2, 512),
    ("hello_world", 3, 128),
    ("bear", 3, 128),
    ("bear", 3, 256),
    ("architecture", 3, 256),
    ("involute_gear_3d", 3, 256),
    ("prospero", 2, 4096),
    ("involute_gear_2d", 2, 4096),
    ("bear", 3, 1024),
    ("architecture", 3, 1024),
    ("hello_world", 2, 1024),
    ("architecture", 3, 2048),
    ("involute_gear_3d", 3, 2048),
    ("bear", 3, 2048),
    # BASELINE.json configs 3 and 4 at the reference's table sizes (render_2d_table.cpp:50, render_3d_table.cpp:51)
    ("involute_gear_2d", 2, 256),
    ("involute_gear_2d", 2, 1024),
    ("involute_gear_2d", 2, 2048),
    ("involute_gear_2d", 2, 3072),
    ("bear", 3, 1536),
    ("prospero", 2, 2048),
    ("prospero", 2, 512),
    ("prospero", 2, 3072),
    ("bear", 3, 512),
    # the frames tests/test_gpu_parity.py::test_matches_live_reference_build checks
    ("architecture", 3, 512),
    ("involute_gear_3d", 3, 512),
]

SUBTAPES = 6400000   # the reference arm is built with -DBIG_SERVER


def timeit(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.mean(ts)), float(np.std(ts)), float(np.min(ts))


def run_case(model, dim, size, args, out_dir):
    rec = {"case": f"{model}_{dim}d_{size}", "model": model, "dim": dim, "size": size}
    cells = parity.load_tape(model)

    # ---- reference build ---------------------------------------------------------
    ref_fp = None
    if oracle.ref_available() and not args.no_ref:
        ref = oracle.RefGpu(size)
        render_ref = (lambda: ref.render2D(cells)) if dim == 2 else (lambda: ref.render3D(cells))
        render_ref()
        ref_fp = parity.fingerprint(ref, dim)
        rec["ref_tape_index"] = ref.tape_index()
        rec["ref_ms"] = timeit(render_ref, args.warmup, args.iters)
        summary = parity.summarize(ref_fp)
        (out_dir / "golden").mkdir(parents=True, exist_ok=True)
        (out_dir / "golden" / f"{rec['case']}.json").write_text(json.dumps(summary, indent=1) + "\n")
        if size <= 256:
            np.savez_compressed(out_dir / "golden" / f"{rec['case']}.npz",
                                **{k: v for k, v in ref_fp.items() if isinstance(v, np.ndarray)})
        ref.close()
        del ref

    # ---- libmprb ---------------------------------------------------------------------
    ctx = capi.Context(size, num_subtapes=SUBTAPES)
    tape = capi.Tape(cells)
    render_mine = (lambda: ctx.render2D(tape)) if dim == 2 else (lambda: ctx.render3D(tape))
    render_mine()
    mine_fp = parity.fingerprint(ctx, dim)
    st = ctx.stats()
    rec["stats"] = st.asdict()
    rec["mine_summary"] = {k: v for k, v in parity.summarize(mine_fp).items() if k in ("image", "normals")}
    render_mine()
    render_mine()          # settle managed pages back on the device before timing kernels
    ctx.set_timing(True)
    render_mine()
    rec["kernel_ms"] = [round(x, 4) for x in ctx.stats().kernel_ms[: ctx.stats().n_launches]]
    ctx.set_timing(False)
    rec["mine_ms"] = timeit(render_mine, args.warmup, args.iters)
    rec["mine_gpu_ms"] = ctx.stats().gpu_ms

    if ref_fp is not None:
        bad = parity.compare(ref_fp, mine_fp)
        rec["vs_ref"] = bad if bad else "EXACT"
        if "image" in bad:
            d = np.argwhere(ref_fp["image"] != mine_fp["image"])[:5]
            rec["image_diff_at"] = [[int(y), int(x), int(ref_fp["image"][y, x]), int(mine_fp["image"][y, x])] for y, x in d]
        if "normals" in bad:
            d = np.argwhere(ref_fp["normals"] != mine_fp["normals"])[:5]
            rec["normals_diff_at"] = [[int(y), int(x), hex(int(ref_fp["normals"][y, x])), hex(int(mine_fp["normals"][y, x]))] for y, x in d]
        for k in list(bad):
            if k.startswith("active") and ref_fp[k].shape != mine_fp[k].shape:
                a, b = set(ref_fp[k].tolist()), set(mine_fp[k].tolist())
                rec[k + "_only_ref"] = sorted(a - b)[:8]
                rec[k + "_only_mine"] = sorted(b - a)[:8]

    # ---- CPU oracle (small cases only) -------------------------------------------------
    if size <= 256 and not args.no_cpu:
        o = oracle.CpuOracle(size, SUBTAPES)
        t0 = time.perf_counter()
        (o.render2D if dim == 2 else o.render3D)(cells)
        rec["cpu_oracle_ms"] = (time.perf_counter() - t0) * 1e3
        cpu_fp = parity.fingerprint(o, dim)
        bad = parity.compare(cpu_fp, mine_fp, normals_lsb=1)
        rec["vs_cpu"] = bad if bad else "EXACT"
        o.close()
    tape.close()
    ctx.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="")
    ap.add_argument("--max-size", type=int, default=4096)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--no-ref", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--out", default=str(ROOT / "gpurun_out"))
    args = ap.parse_args()
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)
    want = set(args.cases.split(",")) if args.cases else None
    with open(out_dir / "check.jsonl", "a") as log:
        for model, dim, size in CASES:
            name = f"{model}_{dim}d_{size}"
            if size > args.max_size or (want and name not in want):
                continue
            try:
                rec = run_case(model, dim, size, args, out_dir)
            except Exception as e:  # keep going: one call should tell us as much as possible
                rec = {"case": name, "error": repr(e), "trace": traceback.format_exc()[-1500:]}
            line = json.dumps(rec)
            log.write(line + "\n")
            log.flush()
            brief = {k: rec.get(k) for k in ("case", "vs_ref", "vs_cpu", "ref_ms", "mine_ms", "mine_gpu_ms", "error")}
            print(json.dumps(brief), flush=True)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Benchmark of the hot path: ms/frame of the tile-recursive renderer on the reference's
own benchmark models (BASELINE.json: "ms/frame at 256-4096 on prospero 2D + bear 3D;
eval_tiles_i HBM GB/s vs peak").

A *step* renders one frame of every workload in --workload (default: the two headline
configurations of BASELINE.json's north_star, prospero 2D 4096x4096 and bear 3D 1024^3);
`value` is the mean ms per frame.  The protocol follows the reference's table drivers
(benchmark/render_2d_table.cpp, render_3d_table.cpp, stats.cpp): context built outside the
timed region, identity view in 2D, T(3,2)=0.3 perspective in 3D, frame time includes the
final device synchronisation.

  python bench.py [--gpus N] [--steps K] [--warmup W]          this repository's CUDA path
  python bench.py --impl reference ...                         the UNMODIFIED reference CUDA
                                                               renderer (oracle/_ref), same workload
  python bench.py ... --dump-outputs DIR                       also write what the last timed frame computed
Both arms also time the CPU restatement (oracle/) on the host cores as `cpu_baseline`.
Under torchrun (N > 1) every rank renders a band of 64-px tile rows and the bands are
exchanged with one NCCL all-gather per frame.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "ms/frame (prospero 2D + bear 3D)"
SUBTAPES = 6400000          # arena chunks: the reference's BIG_SERVER setting, both arms
PEAKS = ROOT / "MEASURED_PEAKS.json"
HBM_FALLBACK_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback


# The reference's table protocol (benchmark/render_2d_table.cpp:50, render_3d_table.cpp:51, run_benchmarks.sh:24-56):
# every size of the 2D table on prospero, every size of the 3D table on bear that its arena can hold
# (bear 2048^3 overflows the reference's subtape arena and is nondeterministic there).
SWEEP = ",".join([f"prospero_2d_{s}" for s in (256, 512, 1024, 2048, 3072, 4096)] +
                 [f"bear_3d_{s}" for s in (256, 512, 1024, 1536)])


def parse_workloads(spec: str):
    out = []
    if spec == "sweep":
        spec = SWEEP
    for w in spec.split(","):
        model, dim, size = w.rsplit("_", 2)
        out.append((model, int(dim[0]), int(size)))
    return out


def load_tape(model: str) -> np.ndarray:
    return np.fromfile(ROOT / "tests" / "golden" / "tapes" / f"{model}.u64", dtype="<u8")


class ClockSampler:
    """nvidia-smi samples while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_baseline(workloads, budget_s: float = 45.0) -> dict:
    """Two CPU arms on the host cores, each on a bounded sample of the same workload:
      * `value`: libfive's CPU renderer as the reference drivers call it (Heightmap::render,
        libfive/src/render/discrete/heightmap.cpp:195-318) - libfive itself cannot be built here (Eigen, Boost,
        libpng absent), so this is the stand-in the unchanged reference drivers link
        (mpr_b200/shim/src/heightmap_render.cpp: interval region recursion + point samples, no tape
        shortening) behind oracle/heightmap_cabi.cpp, fed the expression rebuilt from the packed tape;
      * `gpu_algorithm_port`: oracle/mpr_oracle.c, the tile-recursive GPU algorithm on OpenMP threads."""
    import oracle
    threads = oracle.oracle_lib().mpro_max_threads()
    out = {"unit": "ms/frame", "cores": threads, "kind": "port"}
    # (a) libfive-algorithm stand-in, at a resolution it finishes in seconds, scaled to the workload's
    t_total, frames, sample = 0.0, 0, []
    for model, dim, size in workloads:
        if t_total > budget_s:
            break
        cpu_size = min(size, 1024 if dim == 2 else 256)
        try:
            dt = oracle.heightmap_cpu_ms(load_tape(model), dim, cpu_size, threads)
        except Exception as e:          # the stand-in is optional test infrastructure
            sample.append(f"{model}: unavailable ({e})")
            continue
        scale = (size / cpu_size) ** 2              # a heightmap renderer's work follows the visible surface: ~ size^2
        t_total += dt * scale * 1e-3
        frames += 1
        sample.append(f"{model}_{dim}d: {dt:.1f} ms measured at {cpu_size}, x{scale:.0f} -> {dt * scale:.0f} ms at {size}")
    if frames:
        out.update({"value": t_total * 1e3 / frames,
                    "sample": "libfive-algorithm CPU stand-in (not libfive: unbuildable here), one frame of each workload "
                              "at a bounded size, scaled by (size ratio)^2 (" + "; ".join(sample) + ")"})
    # (b) the GPU algorithm restated on the CPU (oracle/mpr_oracle.c), full size
    t_total, frames, sample = 0.0, 0, []
    for model, dim, size in workloads:
        if t_total > budget_s:
            break
        o = oracle.CpuOracle(size, SUBTAPES)
        cells = load_tape(model)
        t0 = time.perf_counter()
        (o.render2D if dim == 2 else o.render3D)(cells, threads=threads)
        dt = time.perf_counter() - t0
        o.close()
        t_total += dt
        frames += 1
        sample.append(f"{model}_{dim}d_{size}: {dt * 1e3:.1f} ms")
    port = {"value": t_total * 1e3 / max(frames, 1), "unit": "ms/frame", "cores": threads,
            "sample": "one frame of each workload, oracle/mpr_oracle.c with OpenMP over tiles (" + "; ".join(sample) + ")"}
    out["gpu_algorithm_port"] = port
    if "value" not in out:
        out.update({"value": port["value"], "sample": port["sample"]})
    return out


def golden_digest(case: str):
    """sha of the reference build's image / normals for this case (tests/golden/ref, minted from oracle/_ref)."""
    f = ROOT / "tests" / "golden" / "ref" / f"{case}.json"
    if not f.exists():
        return None
    d = json.loads(f.read_text())
    return {k: d[k]["sha"] for k in ("image", "normals") if k in d}


def digest(a: np.ndarray) -> str:
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:32]


DUMP_BUDGET = 60 << 20      # bytes of array data --dump-outputs writes, all files together (< 64 MB with headers)


def dump_outputs(out_dir: str, jobs, holder: str):
    """--dump-outputs: the image (and in 3D the normals) that job[holder] - a context of either arm - holds
    for every workload, as <out_dir>/<model>_<dim>d_<size>_<image|normals>.npy in float64, which holds the
    int32 depth and 0 / 1 images and the packed uint32 normals exactly.  An array larger than its equal share
    of DUMP_BUDGET is written as a fixed sample instead: the elements at the flat indices
    np.random.default_rng(0) draws (without replacement, increasing), the same in every run."""
    arrays = {}
    for j in jobs:
        case = f"{j['model']}_{j['dim']}d_{j['size']}"
        arrays[f"{case}_image"] = np.array(j[holder].image())
        if j["dim"] == 3:
            arrays[f"{case}_normals"] = np.array(j[holder].normals())
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    share = DUMP_BUDGET // 8 // len(arrays)
    for name, a in arrays.items():
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(out / f"{name}.npy", a.astype(np.float64))


# Launch order inside one frame (mpr_b200/csrc/api.cu: render()).
def kernel_names(dim: int, n_launches: int):
    """The float pass is one launch, or two (work items on compacted tapes, then the rest)."""
    head = ["eval_tiles", "rank_tiles", "upsample_filled"] * (3 if dim == 3 else 2)
    tail = ["normals"] if dim == 3 else []
    return head + ["eval_voxels"] * max(n_launches - len(head) - len(tail), 1) + tail


def algorithmic_bytes(st, kernel: str) -> float:
    """Bytes a kernel must move per frame by the per-tile formulas of SURVEY.md section 8(d)
    (tape counted once per tile evaluation).  st = mprb_frame_stats of that frame."""
    if kernel == "eval_tiles":
        b = 0.0
        for l in range(3):
            # TileNode 12 + values 24 (+4 image) + 8*(F+1) read, 4 written; pushes re-read the tape
            # and write 8 bytes per kept cell (clauses, header, end cell, chunk links) + tile.tape
            b += st.i_tiles[l] * (12 + 24 + 4 + 8 + 4) + 8.0 * st.i_cells[l]
            b += 8.0 * st.p_cells[l] + 8.0 * st.p_kept[l] + 4.0 * st.p_tiles[l]
        return b
    if kernel == "eval_voxels":
        return st.f_tiles * (12 + 768 + 8 + 256) + 8.0 * st.f_cells
    if kernel == "normals":
        return st.n_pixels * (36 + 4 + 8 + 4) + 8.0 * st.n_cells
    return 0.0


OUT = sys.stdout          # where the JSON line goes (the real stdout, also after divert_stdout)
_DIVERTED = None


def divert_stdout(path):
    """Everything written to file descriptor 1 from here on (Python, NCCL, torch) lands in `path`;
    OUT keeps the real stdout."""
    global OUT, _DIVERTED
    sys.stdout.flush()
    OUT = os.fdopen(os.dup(1), "w")
    fd = os.open(path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
    os.dup2(fd, 1)
    os.close(fd)
    _DIVERTED = [path, 0]


def drain_diverted():
    """Copies what has been diverted since the last call to stderr; returns those lines."""
    if _DIVERTED is None:
        return []
    import ctypes
    sys.stdout.flush()
    ctypes.CDLL(None).fflush(None)            # NCCL writes through C stdio
    with open(_DIVERTED[0], errors="replace") as f:
        f.seek(_DIVERTED[1])
        text = f.read()
        _DIVERTED[1] = f.tell()
    if text:
        sys.stderr.write(text)
        sys.stderr.flush()
    return [l.strip() for l in text.splitlines()]


def run_mine(args, workloads):
    import torch
    import torch.distributed as dist
    from mpr_b200 import capi, sharding

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL reports its communicator (rank / nranks) at INFO level, on stdout.  File descriptor 1 is
        # pointed at a per-rank log for the whole run and the one JSON line goes to the real stdout
        # (OUT) at the end; rank 0 copies the log to stderr and the communicator lines into the JSON line
        # ("nccl") once the group is up.
        os.environ["NCCL_DEBUG"] = os.environ.get("MPRB_NCCL_DEBUG", "INFO")    # whatever the box's default is
        os.environ["NCCL_DEBUG_SUBSYS"] = os.environ.get("MPRB_NCCL_DEBUG_SUBSYS", "INIT")
        os.environ.pop("NCCL_DEBUG_FILE", None)
        divert_stdout(f"/tmp/mprb_stdout_{os.getpid()}_rank{rank}.log")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    class DevArray:   # wraps a raw device pointer for torch.as_tensor
        def __init__(self, ptr, n, typestr):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}

    jobs = []
    for model, dim, size in workloads:
        shard = sharding.diagonal_tiles if SHARD == "diag" else sharding.cyclic_rows
        ctx = capi.Context(size, device=local, num_subtapes=SUBTAPES, **shard(size, world, rank))
        cells_pinned = torch.from_numpy(load_tape(model).view(np.int64).copy()).pin_memory()
        cells = cells_pinned.numpy().view(np.uint64)
        tape = capi.Tape(cells)
        out_img = torch.empty((size, size), dtype=torch.int32).pin_memory()
        out_nrm = torch.empty((size, size), dtype=torch.int32).pin_memory() if dim == 3 else None
        job = dict(model=model, dim=dim, size=size, ctx=ctx, tape=tape, cells=cells, keep=cells_pinned,
                   out_img=out_img, out_nrm=out_nrm)
        if world > 1:
            # End-to-end frames land in ONE page-locked host frame shared by the ranks' processes (a shared-memory
            # file every rank maps and registers with CUDA): each GPU stores the blocks it owns over its own
            # PCIe link (mprb_ctx_publish) and nobody gathers the frame on a device first.
            n_int = size * size * (2 if dim == 3 else 1)
            path = [f"/dev/shm/mprb_bench_{os.getpid()}_{len(jobs)}" if rank == 0 else None]
            dist.broadcast_object_list(path, src=0)
            if rank == 0:
                with open(path[0], "wb") as f:
                    f.truncate(n_int * 4)
            dist.barrier()
            shared = torch.from_file(path[0], shared=True, size=n_int, dtype=torch.int32)
            err = torch.cuda.cudart().cudaHostRegister(shared.data_ptr(), n_int * 4, 3)     # portable | mapped
            if int(err) != 0:
                raise SystemExit(f"cudaHostRegister of the shared host frame failed: {err}")
            dist.barrier()
            if rank == 0:
                os.unlink(path[0])
            job["shared"] = shared
            job["out_img"] = shared[: size * size].view(size, size)
            job["out_nrm"] = shared[size * size:].view(size, size) if dim == 3 else None
            ptr, nbytes = ctx.device_image()
            job["dev_img"] = torch.as_tensor(DevArray(ptr, size * size, "<i4"), device=f"cuda:{local}").view(size, size)
            if dim == 3:
                ptr, nbytes = ctx.device_normals()
                job["dev_nrm"] = torch.as_tensor(DevArray(ptr, size * size, "<i4"), device=f"cuda:{local}").view(size, size)
            if SHARD == "diag":
                # a 2D frame is 0/1 and depth < size: they cross NVLink as uint8 / int16 (normals stay 32 bit)
                job["exchange"] = sharding.NativeExchange(ctx, dim, world, f"cuda:{local}")
        jobs.append(job)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}")   # > 126 MB L2
    nccl_info = None
    if world > 1:
        dist.barrier()                        # first collective: the communicator exists after this
        torch.cuda.synchronize()
        if rank == 0:
            lines = [l for l in drain_diverted() if "nranks" in l or "NCCL version" in l]
            lines = sorted(set(lines))[:8]
            nccl_info = {"world_size": dist.get_world_size(), "backend": dist.get_backend(), "log_lines": lines}

    def gather(job):
        """One all-gather of the band(s); returns device ms (0 on one GPU)."""
        if world == 1:
            return 0.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if SHARD == "diag":
            # tile-cyclic: depth and normals blocks travel in ONE all-gather; every rank ends up with the full frame
            job["exchange"].gather()
        else:
            # interleaved tile rows -> one all-gather per image
            job["dev_img"].copy_(sharding.all_gather_cyclic(job["dev_img"], job["size"]))
            if job["dim"] == 3:
                job["dev_nrm"].copy_(sharding.all_gather_cyclic(job["dev_nrm"], job["size"]))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def frame_device(job):
        ctx = job["ctx"]
        t0 = time.perf_counter()
        (ctx.render2D if job["dim"] == 2 else ctx.render3D)(job["tape"])      # returns after the device finished
        job["wall_ms"] = job.get("wall_ms", 0.0) + (time.perf_counter() - t0) * 1e3
        ms = ctx.stats().gpu_ms
        g = gather(job)
        job["gather_ms"] = job.get("gather_ms", 0.0) + g
        job["gather_n"] = job.get("gather_n", 0) + 1
        return ms + g

    def frame_e2e(job):
        ctx = job["ctx"]
        t0 = time.perf_counter()
        if world == 1:
            if job["dim"] == 2:
                ctx.render2D_host(job["cells"], job["out_img"].numpy())
            else:
                ctx.render3D_host(job["cells"], job["out_img"].numpy(), job["out_nrm"].numpy().view(np.uint32))
        else:
            if job["dim"] == 2:
                ctx.render2D_host(job["cells"], None)
                ctx.publish(2, job["out_img"].data_ptr())
            else:
                ctx.render3D_host(job["cells"], None, None)
                ctx.publish(3, job["out_img"].data_ptr(), job["out_nrm"].data_ptr())
        return (time.perf_counter() - t0) * 1e3

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(fn):
        flush.zero_()             # evict L2 between steps (outside every timed window)
        barrier()
        return [fn(j) for j in jobs]

    for _ in range(args.warmup):
        step(frame_device)
    for j in jobs:                                  # the first exchange includes NCCL's lazy setup
        j["gather_ms"], j["gather_n"], j["wall_ms"] = 0.0, 0, 0.0
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    barrier()
    t_wall0 = time.perf_counter()
    dev = np.array([step(frame_device) for _ in range(args.steps)])      # [K, n_jobs] device ms
    barrier()
    t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:     # the last timed frame (after the exchange when N > 1)
        dump_outputs(args.dump_outputs, jobs, "ctx")
    launches = sum(j["ctx"].stats().n_launches for j in jobs)
    dev_digest = {}
    if world > 1 and rank == 0:     # what the NCCL exchange left on rank 0's device after the last timed frame
        for j in jobs:
            d = {"image": digest(j["dev_img"].cpu().numpy())}
            if j["dim"] == 3:
                d["normals"] = digest(j["dev_nrm"].cpu().numpy().view(np.uint32))
            dev_digest[f"{j['model']}_{j['dim']}d_{j['size']}"] = d
        for j in jobs:              # the end-to-end frames must fill the host frame themselves
            j["shared"].zero_()
    barrier()
    for _ in range(min(args.warmup, 3)):
        step(frame_e2e)
    e2e = np.array([step(frame_e2e) for _ in range(args.steps)])         # [K, n_jobs] wall ms
    barrier()
    clk = clocks.stop() if rank == 0 else None

    # Every timed frame left its result in place: compare what rank 0 holds (after the exchange when N > 1)
    # with the reference build's own output for the case (tests/golden/ref/*.json, minted from oracle/_ref).
    verified, unverified, mismatched = [], [], []
    if rank == 0:
        for j in jobs:
            case = f"{j['model']}_{j['dim']}d_{j['size']}"
            want = golden_digest(case)
            if want is None:
                unverified.append(case)
                continue
            got = {"image": digest(j["out_img"].numpy())}
            if j["dim"] == 3:
                got["normals"] = digest(j["out_nrm"].numpy().view(np.uint32))
            ok = all(got[k] == want[k] for k in got)
            if case in dev_digest:
                ok = ok and all(dev_digest[case][k] == want[k] for k in got)
            (verified if ok else mismatched).append(case)

    # BASELINE.json config 4 ("bear 3D heightmap + normals + SSAO"): mpr::Effects::drawSSAO / drawShaded on the
    # last 3D frame, host clock around the synchronised calls (the reference's GUI times them the same way,
    # gui/main.cpp:372-391).  Not part of `value`.
    effects_ms = {}
    if rank == 0:
        for j in jobs:
            if j["dim"] != 3 or world > 1:
                continue
            fx = capi.Effects()
            for name, fn in (("ssao", fx.drawSSAO), ("shaded", fx.drawShaded)):
                fn(j["ctx"])
                t0 = time.perf_counter()
                for _ in range(10):
                    fn(j["ctx"])
                effects_ms[f"{j['model']}_{j['dim']}d_{j['size']}_{name}"] = (time.perf_counter() - t0) * 100.0
            lit = int((j["out_img"].numpy() != 0).sum())
            effects_ms[f"{j['model']}_{j['dim']}d_{j['size']}_ssao_algorithmic_bytes"] = lit * (64 * 4 + 12) + j["size"] ** 2 * 8
            fx.close()

    # per-kernel timing + counters on separate frames (events between launches perturb nothing
    # in the timed loops above)
    per_kernel, bytes_by_kernel, frames_k = {}, {}, 3
    stats_one = {}
    for j in jobs:
        ctx = j["ctx"]
        ctx.set_timing(True)
        for _ in range(frames_k):
            flush.zero_()
            torch.cuda.synchronize()
            (ctx.render2D if j["dim"] == 2 else ctx.render3D)(j["tape"])
            st = ctx.stats()
            names = kernel_names(j["dim"], st.n_launches)
            for name, ms in zip(names, list(st.kernel_ms)[: st.n_launches]):
                per_kernel[name] = per_kernel.get(name, 0.0) + ms / frames_k
            for name in set(names):
                bytes_by_kernel[name] = bytes_by_kernel.get(name, 0.0) + algorithmic_bytes(st, name) / frames_k
        ctx.set_timing(False)
        st = ctx.stats()
        stats_one[f"{j['model']}_{j['dim']}d_{j['size']}"] = {
            "n_active": list(st.n_active), "tape_index": st.tape_index, "interval_tiles": list(st.i_tiles),
            "interval_cells": list(st.i_cells), "float_tiles": st.f_tiles, "float_cells": st.f_cells,
            "float_items": st.f_items, "push_tiles": list(st.p_tiles), "push_cells_logical": list(st.p_kept),
            "push_cells_written": st.p_written}

    # max over ranks, step by step
    if world > 1:
        t = torch.tensor(np.concatenate([dev.sum(1), e2e.sum(1)]), device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = t.cpu().numpy()
        dev_step, e2e_step = t[: args.steps], t[args.steps:]
    else:
        dev_step, e2e_step = dev.sum(1), e2e.sum(1)

    if rank == 0:
        n_frames = len(jobs)
        peak = json.loads(PEAKS.read_text())["hbm_gbs"] if PEAKS.exists() else HBM_FALLBACK_GBS
        peak_src = "MEASURED_PEAKS.json hbm_gbs (copy, burst)" if PEAKS.exists() else "B200_PROFILING.md fallback"
        dom = max((k for k in per_kernel if bytes_by_kernel.get(k, 0) > 0), key=lambda k: per_kernel[k])

        def roof(k):
            ach = bytes_by_kernel[k] / (per_kernel[k] * 1e-3) / 1e9 if per_kernel[k] > 0 else 0.0
            out = {"kernel": "k_" + k, "bound": "hbm", "achieved": round(ach, 2), "peak": peak, "unit": "GB/s",
                   "frac": round(ach / peak, 5), "traffic": None, "peak_source": peak_src,
                   "algorithmic_bytes_per_step": int(bytes_by_kernel[k]), "kernel_ms_per_step": round(per_kernel[k], 4)}
            out.update(ncu_capture("k_" + k))
            return out

        h2d = sum(j["cells"].nbytes + (64 if j["dim"] == 3 else 36) for j in jobs)
        d2h = sum(j["size"] ** 2 * 4 * (2 if j["dim"] == 3 else 1) for j in jobs)
        line = {
            "metric": METRIC, "value": float(dev_step.mean() / n_frames), "unit": "ms/frame",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": float(dev_step.mean()), "higher_is_better": False, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "the reference's benchmark models as packed tapes (tests/golden/tapes)",
            "config": {"workload": "+".join(f"{j['model']}_{j['dim']}d_{j['size']}" for j in jobs),
                       "frames_per_step": n_frames, "view": "2D identity, 3D T(3,2)=0.3 (reference table drivers)",
                       "parallelism": (f"tile-cyclic 64x64-px screen columns x{world}, 1 NCCL all-gather per frame" if SHARD == "diag"
                                       else f"interleaved 64-px tile rows x{world}, 1 NCCL all-gather per image") if world > 1 else "1 GPU",
                       "num_subtapes": SUBTAPES, "l2": "flushed between steps (256 MiB memset, untimed)",
                       "timing": "value: CUDA events on the render stream per frame (+ all-gather events), max over ranks; "
                                 "wall_ms_per_frame: host clock around the same synchronised call (benchmark/stats.cpp protocol)",
                       "wall_ms_per_frame": {f"{j['model']}_{j['dim']}d_{j['size']}": j["wall_ms"] / args.steps for j in jobs},
                       "ms_per_frame": {f"{j['model']}_{j['dim']}d_{j['size']}": float(dev[:, i].mean()) for i, j in enumerate(jobs)},
                       "e2e_ms_per_frame": {f"{j['model']}_{j['dim']}d_{j['size']}": float(e2e[:, i].mean()) for i, j in enumerate(jobs)},
                       "e2e_protocol": ("host tape in, host frame out through mprb_render*_host (pinned buffers), wall clock" if world == 1 else
                                        "host tape in on every rank; each rank stores the blocks it owns into ONE page-locked host frame "
                                        "shared by the ranks (mprb_ctx_publish over its own PCIe link, no device-side gather); wall clock, max over ranks"),
                       "exchange_ms_per_frame_rank0": {f"{j['model']}_{j['dim']}d_{j['size']}": round(j.get("gather_ms", 0.0) / max(j.get("gather_n", 1), 1), 4) for j in jobs},
                       "wall_ms_per_step_incl_flush": t_wall * 1e3 / args.steps,
                       "frame_stats": stats_one, "effects_ms": effects_ms},
            "clocks": clk,
            "e2e": {"value": float(e2e_step.mean() / n_frames), "unit": "ms/frame", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches),
            "nccl": nccl_info,
            "frames_verified": (not mismatched) and bool(verified),
            "frames_verified_detail": {"equal_to_reference_build": verified, "no_fixture": unverified, "MISMATCH": mismatched},
            "kernel_ms_per_step": {k: round(v, 4) for k, v in per_kernel.items()},
            "roofline": roof(dom),
            "roofline_eval_tiles": roof("eval_tiles"),
        }
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(workloads)
        drain_diverted()
        print(json.dumps(line), file=OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and mismatched:
        raise SystemExit(f"frames differ from the reference build: {mismatched}")


def run_reference(args, workloads):
    """The unmodified reference CUDA renderer (single GPU, default stream, managed memory), timed with the
    same two clocks and the same host buffers as the other arm."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import oracle
    if not oracle.ref_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libmpr_ref.so missing (build needs /root/reference)"}))
        return
    import torch
    torch.cuda.set_device(0)
    jobs = []
    for model, dim, size in workloads:
        ref = oracle.RefGpu(size)
        cells = load_tape(model)
        out_img = torch.empty((size, size), dtype=torch.int32).pin_memory()
        out_nrm = torch.empty((size, size), dtype=torch.int32).pin_memory() if dim == 3 else None
        jobs.append(dict(model=model, dim=dim, size=size, ref=ref, cells=cells, out_img=out_img, out_nrm=out_nrm,
                         img=out_img.numpy(), nrm=out_nrm.numpy().view(np.uint32) if dim == 3 else None, wall_ms=0.0))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")   # > 126 MB L2, as in the other arm

    def frame(job):
        # Device time: CUDA events on the legacy default stream, which is where the reference launches
        # (it has no stream of its own) - the second event lands after its final cudaDeviceSynchronize.
        # Host wall clock around the same call = the reference's own protocol (benchmark/stats.cpp).
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        (job["ref"].render2D if job["dim"] == 2 else job["ref"].render3D)(job["cells"])     # Tape cached after frame 1
        e1.record()
        job["wall_ms"] += (time.perf_counter() - t0) * 1e3
        e1.synchronize()
        return e0.elapsed_time(e1)

    def frame_e2e(job):  # + download of the result into pinned host buffers (the Tape stays cached on the device)
        t0 = time.perf_counter()
        (job["ref"].render2D if job["dim"] == 2 else job["ref"].render3D)(job["cells"])
        job["ref"].download(job["img"], job["nrm"])
        return (time.perf_counter() - t0) * 1e3

    def step(fn):
        flush.zero_()
        torch.cuda.synchronize()
        return [fn(j) for j in jobs]

    for _ in range(args.warmup):
        step(frame)
    for j in jobs:
        j["wall_ms"] = 0.0
    clocks = ClockSampler(0)
    clocks.start()
    dev = np.array([step(frame) for _ in range(args.steps)])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, jobs, "ref")
    for _ in range(min(args.warmup, 3)):
        step(frame_e2e)
    e2e = np.array([step(frame_e2e) for _ in range(args.steps)])
    clk = clocks.stop()
    effects_ms = {}
    for j in jobs:                       # config 4: the reference's own Effects on its own frame
        if j["dim"] != 3:
            continue
        try:
            fx = oracle.RefEffects()
        except Exception:
            break
        for name, shaded in (("ssao", False), ("shaded", True)):
            fx.draw(j["ref"], shaded=shaded)
            t0 = time.perf_counter()
            for _ in range(10):
                (fx.L.ref_effects_draw_shaded if shaded else fx.L.ref_effects_draw_ssao)(fx.h, j["ref"].h)
            effects_ms[f"{j['model']}_{j['dim']}d_{j['size']}_{name}"] = (time.perf_counter() - t0) * 100.0
        fx.close()
    n_frames = len(jobs)
    h2d = sum((64 if j["dim"] == 3 else 36) for j in jobs)
    d2h = sum(j["size"] ** 2 * 4 * (2 if j["dim"] == 3 else 1) for j in jobs)
    name = lambda j: f"{j['model']}_{j['dim']}d_{j['size']}"
    line = {
        "impl": "reference", "metric": METRIC, "value": float(dev.sum(1).mean() / n_frames), "unit": "ms/frame",
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(dev.sum(1).mean()),
        "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "the reference's benchmark models as packed tapes (tests/golden/tapes)",
        "config": {"workload": "+".join(name(j) for j in jobs), "frames_per_step": n_frames,
                   "view": "2D identity, 3D T(3,2)=0.3 (reference table drivers)", "parallelism": "1 GPU",
                   "num_subtapes": SUBTAPES, "l2": "flushed between steps (256 MiB memset, untimed)",
                   "what": "unmodified reference src/context.cu + context.cpp + gpu_opcode.cu compiled for sm_100a with "
                           "-DBIG_SERVER (oracle/Makefile), driven through oracle/ref_wrap.cu",
                   "timing": "value: CUDA events on the default stream around render2D/render3D (which ends in "
                             "cudaDeviceSynchronize); wall_ms_per_frame: host clock around the same call (benchmark/stats.cpp)",
                   "wall_ms_per_frame": {name(j): j["wall_ms"] / args.steps for j in jobs},
                   "ms_per_frame": {name(j): float(dev[:, i].mean()) for i, j in enumerate(jobs)},
                   "e2e_ms_per_frame": {name(j): float(e2e[:, i].mean()) for i, j in enumerate(jobs)},
                   "e2e_protocol": "Tape resident on the device (built once), result downloaded into pinned host buffers",
                   "effects_ms": effects_ms},
        "clocks": clk,
        "e2e": {"value": float(e2e.sum(1).mean() / n_frames), "unit": "ms/frame", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h)},
    }
    if not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(workloads)
    print(json.dumps(line), flush=True)


SHARD = os.environ.get("MPRB_SHARD", "diag")      # multi-GPU split: "diag" (tile-cyclic) or "rows" (interleaved rows)


def ncu_capture(kernel: str) -> dict:
    """DRAM traffic per launch (+ what actually bounds the kernel) from the committed
    `ncu --set full` capture of this kernel, profiles/*_ncu_<kernel>*.csv (raw page export)."""
    import csv
    files = sorted((ROOT / "profiles").glob(f"*_ncu_{kernel}*.csv"))
    if not files:
        return {}
    # one "metric,unit,value" line per metric
    val, unit = {}, {}
    for row in csv.reader(files[-1].open()):
        if len(row) >= 3:
            val[row[0]], unit[row[0]] = row[2], row[1]

    def num(name, scale=None):
        try:
            v = float(val[name])
        except (KeyError, ValueError):
            return None
        if scale is not None:
            v *= {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit.get(name, "byte"), 1.0)
        return v

    rd, wr = num("dram__bytes_read.sum", 1), num("dram__bytes_write.sum", 1)
    return {"traffic": int(rd + wr) if rd is not None and wr is not None else None,
            "traffic_source": f"profiles/{files[-1].name} (one launch, bear 1024^3 frame)",
            "ncu": {"issue_active_pct": num("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                    "lsu_shared_pipe_pct": num("l1tex__data_pipe_lsu_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed"),
                    "warp_instructions": num("smsp__inst_executed.sum"),
                    "duration_ms_under_ncu": num("gpu__time_duration.sum")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="mine", choices=["mine", "reference"])
    ap.add_argument("--workload", default="prospero_2d_4096,bear_3d_1024",
                    help="comma list of <model>_<2d|3d>_<size>, or 'sweep' = the reference's table sizes "
                         "(prospero 2D 256..4096, bear 3D 256..1536)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write each workload's image (and 3D normals) of the last timed "
                         "frame as DIR/<model>_<dim>d_<size>_<image|normals>.npy, float64, < 64 MB in all")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    # NCCL takes its debug level from the environment it was loaded under: with several ranks, make sure
    # NCCL_DEBUG=INFO (communicator lines: rank / nranks) is in place before anything imports torch, by
    # replacing this process with itself once (same PID, so the launcher does not notice).
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not os.environ.get("MPRB_BENCH_REEXEC"):
        os.environ["MPRB_BENCH_REEXEC"] = "1"
        os.environ["NCCL_DEBUG"] = os.environ.get("MPRB_NCCL_DEBUG", "INFO")
        os.environ["NCCL_DEBUG_SUBSYS"] = os.environ.get("MPRB_NCCL_DEBUG_SUBSYS", "INIT")
        os.environ.pop("NCCL_DEBUG_FILE", None)
        sys.stdout.flush()
        os.execv(sys.executable, [sys.executable] + sys.argv)
    workloads = parse_workloads(args.workload)
    if args.impl == "reference":
        run_reference(args, workloads)
    else:
        run_mine(args, workloads)


if __name__ == "__main__":
    main()

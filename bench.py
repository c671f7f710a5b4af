#!/usr/bin/env python
"""bench.py -- the depth -> sort -> rasterise hot path on N B200s (BASELINE.json metric: frames/s and sorted
Msplats/s at 1920x1080; HBM GB/s against the measured roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload bonsai|garden|synth16m] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one viewer frame: full depth sort of every splat + projection + tile binning + front-to-back blend into an
RGBA8 frame (Viewer.update + Viewer.render of the reference).  Prints ONE JSON line on rank 0.

value   device-timed (CUDA events on the engine's stream), scene resident in HBM, L2 flushed between steps.
e2e     the same frames through the C ABI with HOST buffers: every frame's camera (mvp + uniforms) goes host->device and its RGBA8
        picture comes back into pinned host memory inside the timed region.  `value` is the throughput of the pipelined entry
        (gs_frame_begin / gs_frame_end, up to three frames in flight); `latency_ms` is one blocking gs_frame.
N > 1   strong scaling of ONE frame: rank r rasterises the coarse tiles with (cx + cy) % N == r; the ranks' blend kernels store
        their pixels straight into rank 0's frame over NVLink (CUDA IPC); rank 0's assembled picture is compared with a
        single-GPU render of the same frame after the timed loops (`frame_check`).
garden  the orbit of BASELINE configs[2]: step i uses frame i mod 120 of a 3-degree-per-frame orbit about cameraUp.
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

WORKLOADS = {
    # name: (splats, sh_degree, kind, seed, camera, width, height, orbit frames)   -- BASELINE.json configs[1], [2], [3]
    "bonsai": (1_200_000, 0, "bonsai", 1, "bonsai", 1920, 1080, 1),
    "garden": (5_800_000, 2, "garden", 2, "garden", 1920, 1080, 120),
    "synth16m": (16_000_000, 0, "bonsai", 3, "bonsai", 3840, 2160, 1),
    "tiny": (100_000, 0, "uniform", 0, "default", 640, 360, 1),
}
SH_BYTES = {0: 0, 1: 18, 2: 48}
ORBIT_DEGREES_PER_FRAME = 3.0
DUMP_BUDGET_BYTES = 60_000_000        # --dump-outputs: data bytes of all arrays together (under 64 MB with the .npy headers)


def workload_label(name: str) -> str:
    """One string for both arms (the driver compares the two lines' config)."""
    n, sh, kind, seed, cam, w, h, orbit = WORKLOADS[name]
    camera = f"{orbit}-frame orbit, {ORBIT_DEGREES_PER_FRAME:g} deg/frame about cameraUp" if orbit > 1 else "fixed camera"
    return f"{name}: {n} splats SH{sh} {w}x{h} {camera} (synthetic stand-in for the .ksplat, seed {seed})"


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def orbit_position(cam: dict, k: int) -> np.ndarray:
    """Camera position of orbit frame k: the demo camera rotated about cameraUp through the look-at point (SURVEY 8(d) config 3)."""
    up = np.asarray(cam["up"], np.float64)
    up /= np.linalg.norm(up)
    a = np.deg2rad(ORBIT_DEGREES_PER_FRAME * k)
    d = np.asarray(cam["position"], np.float64) - np.asarray(cam["look_at"], np.float64)
    return np.asarray(cam["look_at"], np.float64) + d * np.cos(a) + np.cross(up, d) * np.sin(a) + up * np.dot(up, d) * (1.0 - np.cos(a))


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed regions run."""

    # (no power.draw: that query is the slow one, and a sample that lands inside the ~50 ms timed window must not stall the GPU)
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu, self.first = [], None, gpu_index, 0

    def mark(self):
        """Samples from here on count (nvidia-smi is started early: on an 8-GPU box it needs seconds before its first line)."""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows[self.first:]:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def build_viewer(workload: str, rank: int, world: int, device: int, raw=None):
    from gaussiansplats3d_b200.scenes import CAMERAS, synthetic_scene
    from gaussiansplats3d_b200.viewer import Viewer
    n, sh, kind, seed, cam, w, h, _ = WORKLOADS[workload]
    if raw is None:
        raw = synthetic_scene(n, seed=seed, kind=kind, sh_degree=sh)
    c = CAMERAS[cam]
    v = Viewer(dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"], width=w, height=h,
                    sphericalHarmonicsDegree=sh, device=device, rank=rank, world_size=world))
    v.addSplatScene(raw)
    v.camera.update()
    v.updateSplatMesh()
    return v, raw


def prepared_frames(v, workload: str, frame_format: int):
    """Pre-marshalled (sort params, uniforms, render params) of every camera of the workload (1, or the 120 orbit frames)."""
    from gaussiansplats3d_b200.scenes import CAMERAS
    n, sh, kind, seed, cam, w, h, orbit = WORKLOADS[workload]
    c = CAMERAS[cam]
    out = []
    for k in range(orbit):
        if orbit > 1:
            v.camera.position = orbit_position(c, k)
            v.camera.look_at(c["look_at"])
            v.camera.update()
            v.updateSplatMesh()
        out.append(v.engine.prepare_frame(v.mvp_matrix().astype(np.float32), v.uniforms(), w, h, n, frame_format=frame_format, flip_y=True))
    return out


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: arrays = {name: (array, float dtype)} -> out_dir/<name>.npy.  The dtypes hold every value exactly (RGBA8 channels,
    u32 indexes).  When the arrays together exceed DUMP_BUDGET_BYTES, each keeps the same share of its elements, a seeded sample of
    flat positions: the same positions in every run of the same workload, so two builds' dumps compare element for element."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    total = sum(a.size * np.dtype(dt).itemsize for a, dt in arrays.values())
    keep = min(1.0, DUMP_BUDGET_BYTES / total)
    for name, (a, dt) in arrays.items():
        out = a.astype(dt)
        if keep < 1.0:
            pos = np.sort(np.random.default_rng(0).choice(a.size, int(a.size * keep), replace=False))
            out = out.reshape(-1)[pos]
        np.save(d / f"{name}.npy", out)
        print(f"[bench] {d / name}.npy: {out.size} of {a.size} elements of {name} {a.shape}, {np.dtype(dt).name}", file=sys.stderr)


# ------------------------------------------------------------------------------------------------------------------------------
def cpu_frame_seconds(workload: str, repeats: int):
    """The reference's CPU path: its own sorter (oracle/_ref, single-threaded like its one Web Worker; the C restatement when the
    compiled reference is absent) + the CPU restatement of its shaders/blend on all host cores (OpenMP; the thread count is set
    explicitly because launchers like torchrun export OMP_NUM_THREADS=1).  Orbit workloads walk the same cameras as the GPU arm."""
    import oracle
    from gaussiansplats3d_b200 import three_math as TM
    from gaussiansplats3d_b200.engine import Uniforms
    from gaussiansplats3d_b200.scenes import CAMERAS, pack_scene, synthetic_scene
    threads = oracle.set_threads(os.cpu_count() or 1)
    n, sh, kind, seed, cam, w, h, orbit = WORKLOADS[workload]
    raw = synthetic_scene(n, seed=seed, kind=kind, sh_degree=sh)
    p = pack_scene(raw)
    c = CAMERAS[cam]
    idx = np.arange(n, dtype=np.uint32)
    kind_used = "reference" if oracle.have_ref() else "port"
    sorter = oracle.ref_sort_indexes if oracle.have_ref() else oracle.port_sort_indexes
    sort_s, frame_s = [], []
    for i in range(repeats):
        camera = TM.PerspectiveCamera(50, w / h, 0.1, 1000)
        camera.position = orbit_position(c, i % orbit) if orbit > 1 else np.asarray(c["position"], np.float64)
        camera.up = np.asarray(c["up"], np.float64) / np.linalg.norm(c["up"])
        camera.look_at(c["look_at"])
        mvp = TM.multiply(camera.projectionMatrix, camera.matrixWorldInverse).astype(np.float32)
        u = Uniforms(model_view=camera.matrixWorldInverse.astype(np.float32), projection=camera.projectionMatrix.astype(np.float32),
                     camera_position=camera.position.astype(np.float32), focal=(camera.projectionMatrix[0] * 0.5 * w, camera.projectionMatrix[5] * 0.5 * h),
                     viewport=(w, h), sh_degree=p.sh_degree)
        t0 = time.perf_counter()
        order = sorter(idx, p.int_centers, None, mvp, None, None, 1 << 16, n, n, n, False, True, False)
        t1 = time.perf_counter()
        oracle.render(u, p.centers_colors, p.covariances, order, w, h, sh=p.sh, sh_degree=p.sh_degree)
        t2 = time.perf_counter()
        sort_s.append(t1 - t0)
        frame_s.append(t2 - t0)
    return dict(n=n, sort_s=sort_s, frame_s=frame_s, sort_kind=kind_used, cores=threads)


def cpu_sample_text(res: dict, steps: int) -> str:
    return (f"mean of {steps} full frames of the same workload after 1 warm-up: depth sort by the reference's own sorter_no_simd.cpp compiled natively "
            f"({res['sort_kind']}, 1 thread like its single Web Worker) + CPU restatement of its shaders/blend (port, OpenMP {res['cores']} threads); "
            f"the WASM + WebGL path itself cannot run here")


def run_reference(args):
    """--impl reference: the CPU path timed on the box's host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = WORKLOADS[args.workload][0]
    res = cpu_frame_seconds(args.workload, args.warmup + args.steps)
    fs = res["frame_s"][args.warmup:]
    ss = res["sort_s"][args.warmup:]
    total = float(np.sum(fs))
    value = len(fs) / total
    line = {
        "impl": "reference", "metric": "frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": len(fs),
        "warmup": args.warmup, "ms_per_step": 1000.0 * total / len(fs), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int32 sort keys / f32 raster", "data": "synthetic",
        "config": {"workload": workload_label(args.workload)},
        "sorted_msplats_per_sec": n / float(np.mean(ss)) / 1e6,
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": res["cores"], "kind": "port" if res["sort_kind"] == "port" else "reference",
                         "sample": cpu_sample_text(res, len(fs))},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------------------
def algorithmic_bytes(kernel: str, n: int, sh: int, w: int, h: int, instances: int, visible: int) -> float | None:
    """Compulsory HBM bytes per launch (DESIGN.md 'Kernels').  None = not an HBM-stream kernel."""
    ntd = (n + 4095) // 4096            # radix tiles of the depth sort
    chunks = (n + 2047) // 2048         # binning chunks
    table = {
        "k_depth": n * (16 + 4),                           # int32x4 centre in, distance out (identity indexes)
        "k_bucket": n * (4 + 2),                           # distance in, 16-bit key out
        "k_radix_scan[depth,0]": ntd * 256 * 8, "k_radix_scan[depth,1]": ntd * 256 * 8,
        "k_radix_hist[depth,1]": n * 2,
        "k_radix_scatter[depth,0]": n * (2 + 2 + 4),       # key in, key + index out (iota values)
        "k_radix_scatter[depth,1]": n * (2 + 4 + 4),       # key + index in, index out
        "k_project": n * (16 + 24 + SH_BYTES[sh]) + n * (48 + 8),
        "k_bin_count": n * (4 + 8 + 8) + chunks * 256 * 4,     # order + rect in, rect (by rank) out, chunk histogram out
        "k_bin_scan": chunks * 256 * 8,
        "k_bin_place": n * (4 + 8) + chunks * 256 * 4 + instances * 8,   # order + rect in, offsets in, {mask, splat} out
        "k_blend": instances * 8 + visible * 48 + w * h * 4,   # each list entry once + each visible record once + the frame
    }
    return float(table[kernel]) if kernel in table else None


def issue_with_peak(issue, clocks):
    """issue-slot roofline of the dominant kernel: peak = schedulers x SM clock (one warp instruction per scheduler per cycle)."""
    if not issue:
        return None
    try:
        mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz")
        if not mhz:
            return issue
        peak = issue["schedulers"] * mhz * 1e6 / 1e9
        return {**issue, "peak_gwarp_inst_per_s": peak, "frac": issue["achieved_gwarp_inst_per_s"] / peak, "sm_mhz": mhz}
    except Exception:
        return issue


def run_ours(args):
    import gaussiansplats3d_b200 as gs  # noqa: F401
    from gaussiansplats3d_b200 import _native as N

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    torch = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")

    K, W = args.steps, max(args.warmup, 3)
    n, sh, kind, seed, cam, width, height, orbit = WORKLOADS[args.workload]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    v, raw = build_viewer(args.workload, rank, world, local)
    e = v.engine
    frames = prepared_frames(v, args.workload, N.GS_FRAME_RGBA8)
    prep = lambda i: frames[i % len(frames)]          # noqa: E731

    gather = None
    gather_kind = None
    if world > 1:
        from gaussiansplats3d_b200.parallel import PeerGather, TileGather
        want = os.environ.get("GS_GATHER", "peer")
        if want == "peer":
            try:   # fused: ranks > 0 blend straight into rank 0's frame over NVLink (CUDA IPC); no collective on the data path
                gather = PeerGather(e, rank, world)
                gather_kind = "peer-memory stores from the blend kernel into rank 0's frame (CUDA IPC over NVLink)"
            except Exception as ex:   # e.g. IPC not permitted in this container: fall back to NCCL
                print(f"[rank {rank}] peer gather unavailable ({ex}); using NCCL all-reduce", file=sys.stderr)
                gather = None
        ok = torch.tensor([1 if gather is not None else 0], device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            if gather is not None:
                raise SystemExit("peer gather attached on some ranks only")
            gather = TileGather(e, width, height, rank, world, fmt=N.GS_FRAME_RGBA8)
            gather_kind = "NCCL all-reduce (SUM) of per-rank frames"
    peer = world > 1 and not hasattr(gather, "image")

    def step_async(i):
        e.frame_async(None, None, width, height, n, prepared=prep(i))
        if gather is not None:
            gather.all_gather()

    def barrier():
        e.synchronize()
        if dist is not None:
            torch.cuda.synchronize()
            dist.barrier()

    for i in range(W):
        step_async(i)
    barrier()
    sampler.mark()

    # ---- value: device time, scene resident, L2 flushed before every step ----------------------------------------------
    ev0 = [e.event() for _ in range(K)]
    ev1 = [e.event() for _ in range(K)]
    barrier()
    for i in range(K):
        e.flush_l2()
        ev0[i].record()
        step_async(i)
        ev1[i].record()
    barrier()
    launches = e.timings()["kernel_launches"] * K
    step_ms = np.array([ev0[i].elapsed_ms(ev1[i]) for i in range(K)])
    if args.dump_outputs and rank == 0:     # the last timed step's picture (and, on one GPU, its draw order), read back untimed
        if world > 1 and not peer:
            gather.sync_to_torch()
            picture = gather.image().cpu().numpy()
        else:
            picture = e.read_buffer(N.GS_BUF_FRAME, np.uint8, height * width * 4).reshape(height, width, 4)
        arrays = {"frame_rgba8": (picture, np.float32)}
        if world == 1:
            arrays["sorted_indexes"] = (e.read_buffer(N.GS_BUF_SORTED_INDEXES, np.uint32, n), np.float32 if n <= 1 << 24 else np.float64)
        dump_outputs(args.dump_outputs, arrays)
    total_ms = float(step_ms.sum())
    if dist is not None:
        t = torch.tensor([total_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    fps = K / (total_ms / 1000.0)

    # ---- per-kernel timeline (same frames, profiling events on, bounded to 50 steps) ------------------------------------------------
    e.set_profiling(True)
    acc: dict[str, list[float]] = {}
    for i in range(min(K, 50)):
        for _ in range(10):          # ~0.3 ms of queued GPU work: the host enqueues the whole frame (launches + event records) meanwhile,
            e.flush_l2()             # so the intervals between events are kernel time, not host launch latency; the last one flushes L2
        step_async(i)
        barrier() if dist is not None else e.synchronize()
        for name, ms in e.kernel_timings():
            acc.setdefault(name, []).append(ms)
    e.set_profiling(False)
    tm = e.timings()
    kernels = {k: float(np.mean(vv)) for k, vv in acc.items()}
    frame_kernel_ms = float(sum(kernels.values()))
    sort_ms = sum(ms for k, ms in kernels.items() if k in ("k_sort_init", "k_depth", "k_bucket") or "[depth" in k)
    dominant = max(kernels, key=kernels.get)
    peak, peak_src = peaks()
    inst, vis = int(tm["tile_instances"]), int(tm["visible_splats"])
    ab = algorithmic_bytes(dominant, n, sh, width, height, inst, vis)
    achieved = (ab / (kernels[dominant] * 1e-3) / 1e9) if ab else None
    # DRAM bytes per launch of the dominant kernel: from the committed `ncu --set full` capture of this command (profiles/); a capture of the
    # 1-GPU bonsai frame only, so it is reported for exactly that case and null otherwise
    traffic = None
    tfile = ROOT / "profiles" / "r2_kernel_traffic.json"
    if tfile.exists() and world == 1 and args.workload == "bonsai":
        tj = json.loads(tfile.read_text())
        traffic = tj.get(dominant)
    # The dominant kernel is instruction-issue bound, so the line also carries its issue-slot utilisation: warp instructions per launch
    # (same ncu capture) / measured duration / (SMs x 4 schedulers x sampled SM clock).  Same restriction as `traffic`.
    issue = None
    ifile = ROOT / "profiles" / "r2_kernel_warp_insts.json"
    try:
        if ifile.exists() and world == 1 and args.workload == "bonsai":
            wi = json.loads(ifile.read_text()).get(dominant)
            if wi:
                issue = {"warp_insts_per_launch": wi, "achieved_gwarp_inst_per_s": wi / (kernels[dominant] * 1e-3) / 1e9, "schedulers": 148 * 4}
    except Exception:      # informational only: must never cost the bench line
        issue = None
    path_bytes = n * (44 + SH_BYTES[sh]) + width * height * 4       # SURVEY 8(d): per rendered splat + framebuffer
    sort_bytes = n * 24                                             # SURVEY 8(d): 16 B centre + 4 B index in + 4 B index out

    # ---- e2e: C ABI with host buffers (pinned), copies inside the timed region -----------------------------------------------------
    # per-step host inputs = the camera (mvp + uniforms, ~3 KB).  The index list is persistent worker state exactly as in the reference's
    # default shared-memory mode (written once by gatherSceneNodesForSort, Viewer.js:2061-2074; read in place by the sorter,
    # SortWorker.js:35 `if (!useSharedMemory)`), so it is resident here too; the RGBA8 frame comes back every step.
    frames_host = [N.pinned_empty((height, width, 4), np.uint8) for _ in range(2)] if rank == 0 else [None, None]
    # (a) latency: one blocking frame per step, L2 flushed before each
    t_lat = []
    for i in range(W + min(K, 50)):
        e.flush_l2()
        barrier()
        t0 = time.perf_counter()
        if rank == 0 and (world == 1 or peer):
            e.frame_prepared(prep(i), frames_host[0])       # returns when all ranks' tiles are in and the frame is in host memory
        else:
            step_async(i)
            if world > 1 and not peer:
                gather.sync_to_torch()
                if rank == 0:
                    torch.as_tensor(frames_host[0]).copy_(gather.image(), non_blocking=True)
                torch.cuda.synchronize()
            else:
                e.synchronize()
        dt = time.perf_counter() - t0
        if dist is not None:
            tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        if i >= W:
            t_lat.append(dt)
    # (b) throughput: gs_frame_begin / gs_frame_end, frames in flight: frame i+1 is sorted and rendered while frame i's picture
    # crosses PCIe on the copy stream.  No L2 flush inside this loop (it would sit in the timed stream): the frame's working set
    # (centres, splat data, records, sort scratch, lists: > 180 MB at 1.2 M splats) exceeds the 126 MB L2 and every frame's picture leaves
    # through PCIe.  N > 1 with the NCCL fallback keeps the blocking loop.
    depth = 3      # frames in flight (N > 1 with the peer gather: rank 0's exported allocation holds two frames, the peers alternate)
    while len(frames_host) < depth:
        frames_host.append(N.pinned_empty((height, width, 4), np.uint8))

    def pipelined(count):
        for j in range(min(depth - 1, count)):
            e.frame_begin(prep(j), frames_host[j % depth])
        for i in range(count):
            if i + depth - 1 < count:
                e.frame_begin(prep(i + depth - 1), frames_host[(i + depth - 1) % depth])
            e.frame_end()

    if world == 1 or peer:       # warm-up of the pipelined entry (its second frame buffer has its own captured graph)
        if rank == 0:
            pipelined(6)
        else:
            for i in range(6):
                step_async(i)
            e.synchronize()
    barrier()
    t0 = time.perf_counter()
    if world == 1 or peer:
        if rank == 0:
            pipelined(K)
        else:
            for i in range(K):
                step_async(i)
            e.synchronize()
        e2e_mode = f"pipelined gs_frame_begin/gs_frame_end on rank 0, {depth} frames in flight over 2 device frame buffers, pinned host frames"
    else:
        for i in range(K):
            step_async(i)
            gather.sync_to_torch()
            if rank == 0:
                torch.as_tensor(frames_host[0]).copy_(gather.image(), non_blocking=True)
            torch.cuda.synchronize()
        e2e_mode = "blocking frames + NCCL all-reduce"
    t_pipe = time.perf_counter() - t0
    if dist is not None:
        tt = torch.tensor([t_pipe], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_pipe = float(tt.item())
    e2e = {"value": K / t_pipe, "unit": "frames/s", "h2d_bytes_per_step": int(64 + 3000), "d2h_bytes_per_step": int(width * height * 4),
           "ms_per_step": 1000.0 * t_pipe / K, "mode": e2e_mode, "l2": "not flushed inside the pipelined loop (working set > L2, see source)",
           "latency_ms": 1000.0 * float(np.mean(t_lat)), "latency_mode": "one blocking frame per step, L2 flushed before each"}

    # ---- N > 1: is rank 0's assembled picture THE picture?  Compared with a single-GPU render of the same frame (untimed) ---------------
    frame_check = None
    if world > 1:
        barrier()
        if rank == 0 and (peer or world == 1):
            e.frame_prepared(prep(0), frames_host[0])
        else:
            step_async(0)
            e.synchronize()
        barrier()
        if rank == 0:
            try:
                if not peer:
                    gather.sync_to_torch()
                    torch.as_tensor(frames_host[0]).copy_(gather.image())
                    torch.cuda.synchronize()
                v1, _ = build_viewer(args.workload, 0, 1, local, raw=raw)
                solo = N.pinned_empty((height, width, 4), np.uint8)
                v1.engine.frame_prepared(prepared_frames(v1, args.workload, N.GS_FRAME_RGBA8)[0], solo)
                diff = np.abs(frames_host[0].astype(np.int16) - solo.astype(np.int16))
                frame_check = {"equal_to_single_gpu_frame": bool(diff.max() == 0), "max_abs_diff_rgba8": int(diff.max()),
                               "differing_channels": int((diff != 0).sum()), "nonzero_alpha_fraction": float((solo[..., 3] > 0).mean())}
                v1.dispose()
            except Exception as ex:      # a check must never cost the bench line
                frame_check = {"error": str(ex)}
        barrier()

    # short runs end before nvidia-smi's 200 ms period has produced enough lines: keep the same frames running (untimed) until it has
    t_wait = time.perf_counter()
    extended = 0
    while True:
        need = 1 if (rank == 0 and sampler.proc is not None and len(sampler.rows) - sampler.first < 3 and time.perf_counter() - t_wait < 8.0) else 0
        if dist is not None:       # rank 0 decides for everybody (the frames below are collective)
            t = torch.tensor([need], device="cuda", dtype=torch.int32)
            dist.broadcast(t, src=0)
            need = int(t.item())
        if not need:
            break
        for i in range(50):
            step_async(i)
        barrier()
        extended += 50
    clocks = sampler.stop()

    # ---- on-chip work of the blend, the figure SURVEY 8(d) asks for beside its HBM fraction: pixels of the reference's quads
    # (+-basis1 +-basis2 parallelograms = its fragment-shader invocations, unclipped) per second of k_blend.  Untimed read-back.
    quad_pixels = None
    try:
        if world == 1:
            ps = e.read_projected(n)
            ok = ps["valid"] != 0
            quad_pixels = float(np.sum(4.0 * np.abs(ps["b1x"][ok].astype(np.float64) * ps["b2y"][ok] - ps["b1y"][ok].astype(np.float64) * ps["b2x"][ok])))
    except Exception as ex:      # a statistic must never cost the bench line
        print(f"[bench] quad-pixel statistic skipped: {ex}", file=sys.stderr)
    clocks["window"] = "timed + per-kernel + e2e regions" + (f", extended by {extended} identical untimed frames" if extended else "")

    # ---- CPU baseline beside it (rank 0, N = 1 only; bounded sample) ---------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        steps_cpu = 3
        res = cpu_frame_seconds(args.workload, 1 + steps_cpu)
        fsec, ssec = res["frame_s"][1:], res["sort_s"][1:]
        cpu = {"value": len(fsec) / float(np.sum(fsec)), "unit": "frames/s", "cores": res["cores"],
               "kind": "port" if res["sort_kind"] == "port" else "reference", "sample": cpu_sample_text(res, steps_cpu),
               "sort_msplats_per_sec": n / float(np.mean(ssec)) / 1e6}

    if rank == 0:
        if world == 1:
            par = "single GPU"
        else:
            par = (f"coarse tiles (8x4 fine tiles) interleaved diagonally over {world} GPUs; scene replicated; each rank sorts "
                   + ("only the splats that reach its tiles (subset of the depth list)" if n >= 3_000_000 else "the full depth list (replicated)")
                   + "; tile gather = " + (gather_kind or "none"))
        line = {
            "metric": "frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "ms_per_step_median": float(np.median(step_ms)), "ms_per_step_max": float(step_ms.max()),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int32 sort keys / f32 raster", "data": "synthetic",
            "config": {"workload": workload_label(args.workload), "l2": "flushed between steps (192 MiB write)", "parallelism": par,
                       "distance_map_range": 65536, "gather": gather_kind},
            "sorted_msplats_per_sec": n / (sort_ms * 1e-3) / 1e6 if sort_ms > 0 else None,
            "sort_ms": sort_ms, "kernel_ms": kernels, "tile_instances": inst, "visible_splats": vis,
            "roofline": {"kernel": dominant, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                         "traffic": traffic, "peak_source": peak_src, "launch_ms": kernels[dominant], "algorithmic_bytes": ab,
                         "issue": issue_with_peak(issue, clocks),
                         "note": "k_blend is instruction-issue bound (ncu: issue active 73 %, DRAM 1.7 %); its HBM fraction is low by construction, see `issue`"
                         if dominant == "k_blend" else None},
            "path_roofline": {"bound": "hbm", "frame_bytes": path_bytes, "frame_gbs": path_bytes / (total_ms / K * 1e-3) / 1e9,
                              "frame_frac": path_bytes / (total_ms / K * 1e-3) / 1e9 / peak, "frame_ms": total_ms / K,
                              "sort_bytes": sort_bytes, "sort_gbs": sort_bytes / (sort_ms * 1e-3) / 1e9 if sort_ms else None,
                              "sort_frac": sort_bytes / (sort_ms * 1e-3) / 1e9 / peak if sort_ms else None,
                              "note": "frame: SURVEY 8(d) bytes / device ms_per_step; sort: 24 B/splat / sum of the sort kernels' timeline"},
            "blend_work": None if not quad_pixels or "k_blend" not in kernels else
            {"quad_pixels_per_frame": quad_pixels, "gpixels_per_sec": quad_pixels / (kernels["k_blend"] * 1e-3) / 1e9,
             "note": "reference fragment invocations (unclipped quad areas of the visible splats) / k_blend time"},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "cpu_baseline": cpu, "frame_check": frame_check,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    v.dispose()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 200 for the GPU arm, 10 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="bonsai", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (RGBA8 frame; one GPU: also the sorted indexes) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    if args.impl == "reference":
        if args.steps is None:     # the CPU arm's frames take ~0.5 s each
            args.steps = 10
        run_reference(args)
    else:
        if args.steps is None:
            args.steps = 200
        run_ours(args)


if __name__ == "__main__":
    main()

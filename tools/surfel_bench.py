"""Device frame time of the TwoD (surfel) render mode beside ThreeD on bench.py's workloads.

    python tools/surfel_bench.py --workload bonsai --steps 200 [--out profiles/surfel_bench.jsonl]

Both modes render the same seeded scene and cameras (bench.py's WORKLOADS, orbit included) in one process, alternating step by
step; the L2 is flushed (gs_flush_l2) before every step and each step is timed with CUDA events on the engine's stream around one
gs_frame_async (a captured graph: sort + projection + binning + blend, RGBA8 1080p).  A second, separate pass with the per-kernel
timeline on gives the kernel split.  One JSON line per workload, with the GPU name and power limit read in the same process."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402  (workload definitions and camera orbit only)


def gpu_info() -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [c.strip() for c in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as ex:   # the line still says which GPU data are missing
        return {"gpu": None, "power_limit": None, "error": str(ex)}


def viewer(workload: str, mode: int, raw):
    from gaussiansplats3d_b200.scenes import CAMERAS
    from gaussiansplats3d_b200.viewer import Viewer
    n, sh, kind, seed, cam, w, h, _ = bench.WORKLOADS[workload]
    c = CAMERAS[cam]
    v = Viewer(dict(cameraUp=c["up"], initialCameraPosition=c["position"], initialCameraLookAt=c["look_at"], width=w, height=h,
                    sphericalHarmonicsDegree=sh, splatRenderMode=mode))
    v.addSplatScene(raw)
    v.camera.update()
    v.updateSplatMesh()
    return v


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="bonsai", choices=["bonsai", "garden", "tiny"])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None, help="append the JSON line to this file")
    a = ap.parse_args()
    if a.steps < 200 and a.workload != "tiny":
        ap.error("--steps must be >= 200 for a reportable number")
    from gaussiansplats3d_b200 import _native as N
    from gaussiansplats3d_b200.scenes import synthetic_scene
    n, sh, kind, seed, cam, w, h, orbit = bench.WORKLOADS[a.workload]
    raw = synthetic_scene(n, seed=seed, kind=kind, sh_degree=sh)
    info = gpu_info()
    modes = {"3d": viewer(a.workload, 0, raw), "2d": viewer(a.workload, 1, raw)}
    frames = {k: bench.prepared_frames(v, a.workload, N.GS_FRAME_RGBA8) for k, v in modes.items()}
    ev = {k: (v.engine.event(), v.engine.event()) for k, v in modes.items()}
    times = {k: [] for k in modes}
    for step in range(a.warmup + a.steps):
        for k, v in modes.items():
            e, prep = v.engine, frames[k][step % len(frames[k])]
            e.flush_l2()
            ev[k][0].record()
            e.frame_async(None, None, w, h, n, prepared=prep)
            ev[k][1].record()
            e.synchronize()
            if step >= a.warmup:
                times[k].append(ev[k][0].elapsed_ms(ev[k][1]))
    timeline = {}
    for k, v in modes.items():   # separate pass: the timeline records an event after every kernel (no graph replay)
        v.engine.set_profiling(True)
        acc: dict[str, list[float]] = {}
        for step in range(20):
            v.engine.flush_l2()
            v.engine.frame_async(None, None, w, h, n, prepared=frames[k][step % len(frames[k])])
            v.engine.synchronize()
            for name, ms in v.engine.kernel_timings():
                acc.setdefault(name, []).append(ms)
        v.engine.set_profiling(False)
        timeline[k] = {name: round(float(np.median(ms)) * 1000.0, 1) for name, ms in acc.items()}
        timeline[k + "_visible_splats"] = int(v.engine.timings()["visible_splats"])
    res = {"tool": "surfel_bench", "workload": a.workload, "splats": n, "sh_degree": sh, "width": w, "height": h, "cameras": orbit,
           "steps": a.steps, "l2_flushed": True, **info}
    for k, t in times.items():
        t = np.asarray(t)
        res[f"{k}_frame_ms_mean"] = round(float(t.mean()), 4)
        res[f"{k}_frame_ms_median"] = round(float(np.median(t)), 4)
    res["kernel_us_median"] = timeline
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")
    for v in modes.values():
        v.dispose()


if __name__ == "__main__":
    main()

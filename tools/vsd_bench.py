"""Time the T-LESS VSD stage on the GPU: B frames at 720x540 (T-LESS Primesense), k hypotheses, one
procedural mesh of ~30 k triangles (the T-LESS CAD models are not shipped with this repository; their
size is an assumption).  Reports, with CUDA events after warm-up, the (B*k + B) renders and the VSD-error
kernel, the same batch's template sweep (predict_pose, seeded weights) for scale, and the host path
(float64 ray caster + numpy vsd_obj arithmetic) on the same batch as the only CPU comparison available.

    python tools/vsd_bench.py [--frames 8] [--k 5] [--grid 642] [--iters 20] [--cpu-frames 1] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:       # nvidia-smi missing: keep the torch name
        q = f"{torch.cuda.get_device_name(0)}, power limit unknown ({exc})"
    return q


def time_cuda(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--grid", type=int, default=642, help="template poses swept per frame (for the sweep time)")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--cpu-frames", type=int, default=1, help="frames run through the host path (0: skip)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    assert torch.cuda.is_available(), "vsd_bench needs a CUDA device"
    from nope_b200.tless import procedural_mesh
    from nope_b200.vsd import MeshTable, render_depth, vsd_error
    from oracle.vsd_oracle import pose44, rotation, scene_depth_raw, raycast_depth, vsd_counts, error_from_counts

    H, W, B, k = 540, 720, a.frames, a.k
    K = np.array([[1075.65, 0.0, 360.0], [0.0, 1073.90, 270.0], [0.0, 0.0, 1.0]])
    verts, faces = procedural_mesh(0, n_lat=110, n_lon=140, radius=45.0)
    dev = "cuda:0"
    table = MeshTable([(verts, faces)], device=dev)
    rng = np.random.default_rng(0)
    gts, preds = [], []
    for _ in range(B):
        R = rotation(rng.normal(size=3), rng.uniform(0, 360))
        t = [rng.uniform(-60, 60), rng.uniform(-40, 40), rng.uniform(600, 900)]
        gts.append(pose44(R, t))
        preds.append([pose44(R @ rotation(rng.normal(size=3), rng.uniform(0, 40 * j)), t) for j in range(k)])
    poses = np.concatenate([np.stack([g] + p) for g, p in zip(gts, preds)])[:, :3]
    P = torch.tensor(poses, dtype=torch.float32, device=dev)
    Kt = torch.tensor(K)
    raw_np = np.stack([scene_depth_raw(verts[::1], faces, g, K, H, W, seed=i, occluder=False)
                       if i < a.cpu_frames else np.full((H, W), 7000, np.uint16) for i, g in enumerate(gts)])
    raw = torch.from_numpy(raw_np).to(dev)
    ids = [0] * len(P)
    out = {}

    def render():
        out["d"] = render_depth(table, ids, P, Kt, H, W).view(B, 1 + k, H, W)

    def error():
        d = out["d"]
        out["e"] = vsd_error(raw, torch.from_numpy(K), d[:, 0], d[:, 1:])

    render_ms = time_cuda(render, a.iters)
    error_ms = time_cuda(error, a.iters)
    both_ms = time_cuda(lambda: (render(), error()), a.iters)
    covered = int((out["d"] > 0).sum())

    from oracle import weights
    from nope_b200.model import build_model
    from nope_b200.poses import synthetic_pose_batch, relative_rotation_6d
    model = build_model(device=dev).load_state_dict(weights.make_full_state_dict(seed=0)).eval()
    _, Rg = synthetic_pose_batch(a.grid, 1)
    allR = relative_rotation_6d(Rg.numpy(), Rg.numpy()[0])[None].expand(B, -1, -1).contiguous()
    q = torch.rand(B, 3, 256, 256, generator=torch.Generator().manual_seed(0)) * 2 - 1
    qd, rd, allRd = q.to(dev), q.flip(0).to(dev), allR.to(dev)
    sweep_ms = time_cuda(lambda: model.predict_pose(qd, rd, allRd, k=k), max(3, a.iters // 4), warmup=2)

    res = {"gpu": gpu_info(), "frames": B, "k": k, "H": H, "W": W, "triangles": int(len(faces)),
           "renders": int(len(P)), "covered_pixels": covered, "render_ms": render_ms, "vsd_error_ms": error_ms,
           "render_plus_error_ms": both_ms, "renders_per_s": len(P) / (render_ms / 1e3),
           "frames_per_s": B / (both_ms / 1e3), "sweep_grid": a.grid, "sweep_ms": sweep_ms,
           "vsd_share_of_sweep": both_ms / sweep_ms}
    if a.cpu_frames > 0:
        t0 = time.perf_counter()
        errs = []
        for f in range(a.cpu_frames):
            dg, _ = raycast_depth(verts, faces, gts[f], K, H, W)
            row = []
            for p in preds[f]:
                de, _ = raycast_depth(verts, faces, p, K, H, W)
                row.append(error_from_counts(vsd_counts(raw_np[f] / 10.0, K, dg.astype(np.float32),
                                                        de.astype(np.float32))))
            errs.append(row)
        cpu_s = time.perf_counter() - t0
        res.update(cpu_frames=a.cpu_frames, cpu_seconds=cpu_s, cpu_frames_per_s=a.cpu_frames / cpu_s,
                   cpu_errors=errs, gpu_errors=out["e"][:a.cpu_frames].cpu().tolist())
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    return res


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- pose-hypotheses/s of the NOPE hot path on B200.

A "step" = one pass of the hot path for one query: the pose-conditioned UNet over the
whole pose grid + l2 scoring + top-5 (BASELINE.json configs[1]: 256x256, 642-pose
icosphere grid, batch = 1 query, fp16 UNet).  With N GPUs the grid is sharded
(weak scaling: 642 poses per GPU, global grid = 642 N) and the only collective is the
all-gather of per-shard (score, index) top-k.

  value  hypotheses/s with the encoder latents and poses already resident in HBM
  e2e    the same metric through the public API (PoseConditional.predict_pose): pinned HOST
         images + poses -> H2D -> encoder x2 -> sweep -> fused score/top-k -> D2H result
  roofline  tensor-core convolution kernel: algorithmic FLOPs / CUDA-event launch time
  cpu_baseline  the oracle (CPU port of the reference) on the host cores, bounded sample

`--impl reference` times the reference's own CPU implementation of the path (the real
reference modules when /root/reference is mounted, else the oracle port of them).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_POSES = 642
GFLOP_PER_HYP = 35.05       # SURVEY.md 8d / BASELINE.md section 3
METRIC = "pose-hypotheses/sec @256x256 (UNet sweep + l2 score + top-5)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--poses", type=int, default=N_POSES, help="poses per GPU")
    ap.add_argument("--queries", type=int, default=1, help="queries (batch) per step")
    ap.add_argument("--chunk", type=int, default=int(os.environ.get("NOPE_CHUNK", "642")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--variant", default="default", choices=["default", "ldm"],
                    help="default: template_base UNet (BASELINE configs); ldm: the LDM-variant UNetModelPose "
                         "sweep on latents (SURVEY.md 8 f2), an additional line for profiles/")
    ap.add_argument("--conv-impl", default=os.environ.get("NOPE_CONV_IMPL", "tcgen05_2cta"),
                    choices=["tcgen05", "tcgen05_2cta"])
    ap.add_argument("--precision", default=os.environ.get("NOPE_PRECISION", "fp16"),
                    choices=["fp16", "fp16_w2", "parity", "parity_fast", "bf16"],
                    help="engine precision of the headline number (config.precision); the other modes are timed "
                         "beside it under `modes` at N=1")
    ap.add_argument("--global-poses", type=int, default=0,
                    help="strong scaling (BASELINE configs[3]): a FIXED grid of this many poses sharded over the "
                         "GPUs (10248 = level-3 grid x 4 in-plane rotations); 0 = weak scaling, --poses per GPU")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra legs (other precision modes, eager-cuDNN baseline, LDM variant)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (similarity rows `sim`, "
                         "top-5 indices `topi`) as DIR/<name>.npy; the inputs are seeded, so two builds run with the "
                         "same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the B200 path; the reference arm times a sample of the grid on the host")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy, float32 kept and every other dtype as float64, at most
    DUMP_LIMIT_BYTES in all: an array that does not fit is replaced by a fixed, seeded sample of its
    flattened elements (the same sample for the same shape, so runs stay comparable).  The smallest arrays
    are written first, so only the largest ones are ever sampled."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_LIMIT_BYTES
    for name, t in sorted(arrays.items(), key=lambda kv: kv[1].numel()):
        a = t.detach().cpu().numpy()
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        room = (budget - 4096) // a.itemsize               # 4 KB: the .npy header, generously
        if a.size > room:
            keep = np.sort(np.random.default_rng(0).choice(a.size, size=max(room, 0), replace=False))
            a = a.reshape(-1)[keep]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        budget -= a.nbytes + 4096


# ---------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.idx), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except ValueError:
                continue
            for n, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm),
                "reasons": sorted(reasons)}


def ncu_traffic():
    """DRAM bytes per launch of the convolution kernel from the committed ncu capture
    (profiles/roofline_traffic.json, written by tools/summarize_ncu_raw.py), or None."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


def measured_peaks():
    """(sustained bf16 TF/s, HBM GB/s, source, burst bf16 TF/s)"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return (d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs"), "measured",
                d.get("bf16_tflops"))
    return 1400.0, 6650.0, "fallback", 1590.0     # B200_PROFILING.md fallback (sustained, burst)


# ---------------------------------------------------------------------------------------
def pick_threads(fn, candidates=(16, 32, 64)):
    """Host boxes with >100 cores run torch-CPU convs slower at full thread count than at a
    NUMA-friendly one; probe a few counts on a tiny workload and keep the fastest."""
    import torch
    n = os.cpu_count()
    cands = sorted({min(c, n) for c in candidates} | {n})
    best, best_t = n, None
    for c in cands:
        torch.set_num_threads(c)
        fn()
        t0 = time.time()
        fn()
        dt = time.time() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_baseline(seconds=12.0, chunk=16):
    """Oracle (CPU port of the reference path) on all host cores: UNet sweep in chunks of
    16 hypotheses + scoring, until ~`seconds` of work.  hyp/s."""
    import torch
    from oracle import inputs, unet_oracle as orc, weights
    sd = weights.make_unet_state_dict(seed=0)
    g = torch.Generator().manual_seed(0)
    rf = torch.randn(1, 8, 32, 32, generator=g) * 1.5
    qf = torch.randn(1, 8, 32, 32, generator=g) * 1.5
    from nope_b200.poses import synthetic_pose_batch
    poses, _ = synthetic_pose_batch(N_POSES, 1)
    done, t0 = 0, time.time()
    with torch.no_grad():
        threads = pick_threads(lambda: orc.generate_templates(sd, rf, poses[:, :4], chunk=4))
        t0 = time.time()
        while time.time() - t0 < seconds and done + chunk <= N_POSES:
            emb = orc.generate_templates(sd, rf, poses[:, done:done + chunk], chunk=chunk)
            orc.l2_similarity(qf, emb)
            done += chunk
    dt = time.time() - t0
    return {"value": done / dt, "unit": "hyp/s", "cores": threads, "kind": "port",
            "sample": f"first {done} of the {N_POSES}-pose grid, batched {chunk}/forward, "
                      f"fp32 torch-CPU oracle, {threads} of {os.cpu_count()} host threads "
                      f"(fastest of a probe), {dt:.1f} s"}


def eager_gpu_baseline(dev, chunks=(64, 128, 256, 642), reps=2):
    """SURVEY.md 8d: the reference ships no custom kernel, so the on-box GPU baseline is the same
    module in PyTorch eager (cuDNN/cuBLAS), fp16, channels_last activations AND weights.
    /root/reference does not exist on the GPU box: the oracle's torch restatement of UNet.forward runs
    on CUDA half tensors instead.  The number of hypotheses per forward is swept and the best is
    reported.  hyp/s (UNet + l2 score only, no encoder)."""
    import torch
    from oracle import unet_oracle as orc, weights
    from nope_b200.poses import synthetic_pose_batch
    sd = {}
    for k, v in weights.make_unet_state_dict(seed=0).items():
        v = v.to(dev, torch.float16)
        sd[k] = v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v
    g = torch.Generator().manual_seed(0)
    rf = (torch.randn(1, 8, 32, 32, generator=g) * 1.5).to(dev, torch.float16)
    qf = (torch.randn(1, 8, 32, 32, generator=g) * 1.5).to(dev)
    poses, _ = synthetic_pose_batch(N_POSES, 1)
    poses = poses.to(dev, torch.float16)
    prev = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    sweep = {}
    try:
        for chunk in chunks:
            x = rf.expand(chunk, -1, -1, -1).contiguous(memory_format=torch.channels_last)

            def run():
                with torch.no_grad():
                    emb = orc.unet_forward(sd, x, poses[0, :chunk])
                    orc.l2_similarity(qf, emb.float()[None])
            try:
                for _ in range(2):
                    run()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    run()
                e1.record()
                torch.cuda.synchronize()
                sweep[chunk] = chunk / (e0.elapsed_time(e1) / reps * 1e-3)
            except RuntimeError as exc:          # e.g. out of memory at the largest chunk
                sweep[chunk] = None
                torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.benchmark = prev
    ok = {c: v for c, v in sweep.items() if v}
    best = max(ok, key=ok.get)
    return {"value": ok[best], "unit": "hyp/s", "kind": "oracle port, torch-eager CUDA fp16, channels_last "
            "activations and weights, cudnn.benchmark (cuDNN/cuBLAS)", "best_chunk": best,
            "chunk_sweep_hyp_per_s": {str(c): (round(v, 1) if v else None) for c, v in sweep.items()},
            "sample": f"{reps} forwards per chunk size, UNet + l2 score"}


# what each engine precision means for parity with the fp32 reference (measured: tests/test_unet_gpu.py,
# 642-pose level-2 golden generated by the unmodified reference)
PRECISION_NOTES = {
    "fp16": "fp16 operands, fp32 accumulate/statistics; GroupNorm+SiLU fused into the conv epilogue",
    "fp16_w2": "exact weights: W = W_hi + W_lo fp16 K-segments (2x MMA work), fp16 activations",
    "parity": "split precision: exact weights + activations as fp16 (hi, lo) pairs, 3 products per tap (3x MMA work)",
    "parity_fast": "split precision on the residual stream / skips / resampled maps (fp16 (hi, lo) pairs, exact weights); "
                   "the tensor inside each ResnetBlock is a single fp16: 2 products per tap in block2, 3 elsewhere",
    "bf16": "bf16 weights and activations (BASELINE configs[2] names bf16), fp32 accumulate/statistics; embeddings "
            "1e-2 / scores 7e-3 of the fp32 reference -- outside the 1e-3 bar, as bf16 autocast is on the reference itself",
}


def workload_config(args, world):
    """The `config` both arms print: same keys and values, so the driver compares like with like."""
    strong = args.global_poses > 0
    n_global = args.global_poses if strong else args.poses * world
    per = (n_global + world - 1) // world
    if strong:
        wl = (f"configs[3]: 256x256, a FIXED {n_global}-pose grid (level-3 icosphere x 4 in-plane rotations when "
              f"10248) sharded {world}-way, batch={args.queries} query, fp16 UNet (fp32 accumulate / statistics), "
              "l2 score + top-5")
    else:
        cfg = "configs[2]" if (args.queries, args.poses) == (8, 2562) else "configs[1]"
        st = "bf16" if args.precision == "bf16" else "fp16"
        wl = (f"{cfg}: 256x256, {args.poses}-pose icosphere grid per GPU, batch={args.queries} query, "
              f"{st} UNet (fp32 accumulate / statistics), l2 score + top-5")
    return {"workload": wl, "poses_per_gpu": per, "global_poses": n_global, "queries": args.queries,
            "chunk": args.chunk, "conv_impl": args.conv_impl,
            # engine precision of the B200 arm (the reference arm always computes fp32; its `dtype` says so)
            "precision": f"{args.precision}: {PRECISION_NOTES[args.precision]}",
            "weights": "seeded random init, reference state_dict schema (305.8 M params)",
            "l2": "not flushed: each step streams 0.61 GB of fp16 weights and ~1.4 GB of "
                  "activations per chunk, >> 126 MB L2",
            "parallelism": f"pose grid sharded {world}-way, one all-gather of packed top-k records" if world > 1 else "1 GPU"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (its
    unmodified modules when /root/reference is mounted, else the oracle port of them), on the same
    workload config as our arm.  One step = the two encoder calls + the UNet sweep over a BOUNDED
    SAMPLE of the grid + scoring; the sample is sized from a probe so that the whole
    --steps/--warmup run ends within a few minutes.  `value` is the throughput of the FULL grid that
    these timings imply: N / (t_encoders + N * t_unet_per_hypothesis) -- the encoder calls are paid
    once per query, not once per sample -- and the raw sample numbers are printed beside it."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    from oracle import ref_import, unet_oracle as orc, weights
    from nope_b200.poses import synthetic_pose_batch
    cfg = workload_config(args, world)
    n_grid = cfg["poses_per_gpu"]                   # the reference has no sharding: one GPU's share of the grid
    poses, _ = synthetic_pose_batch(N_POSES, 1)
    g = torch.Generator().manual_seed(0)
    q = torch.rand(1, 3, 256, 256, generator=g) * 2 - 1
    r = torch.rand(1, 3, 256, 256, generator=g) * 2 - 1
    sd = weights.make_full_state_dict(seed=0)
    batch = 16                                      # hypotheses per UNet forward (best-effort CPU batching)
    if ref_import.reference_available():
        kind = "reference"
        model = ref_import.build_reference_model()
        model.u_net.load_state_dict(sd, strict=True)

        def encoders():
            with torch.no_grad():
                return model.u_net.encoder.encode_image(q), model.u_net.encoder.encode_image(r)

        def sweep(qf, rf, n):
            # the reference's retrieval path with the grid batched along dim 0 (its own modules)
            with torch.no_grad():
                embs = [model.u_net(rf.expand(min(batch, n - s), -1, -1, -1), poses[0, s:min(s + batch, n)])
                        for s in range(0, n, batch)]
                emb = torch.cat(embs)[None]
                d = (qf.unsqueeze(1) - emb) ** 2
                (-torch.norm(d, dim=2).sum(3).sum(2)).topk(k=min(5, n), dim=1)
    else:
        kind = "port"
        unet_sd = {k: v for k, v in sd.items() if not k.startswith("encoder.")}
        enc_sd = {k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")}

        def encoders():
            with torch.no_grad():
                return orc.encode_image(enc_sd, q), orc.encode_image(enc_sd, r)

        def sweep(qf, rf, n):
            with torch.no_grad():
                emb = orc.generate_templates(unet_sd, rf, poses[:, :n], chunk=batch)
                orc.topk_lowest_index(orc.l2_similarity(qf, emb), min(5, n))
    qf, rf = encoders()
    threads = pick_threads(lambda: sweep(qf, rf, 4))
    # probe: how many hypotheses fit in the per-step budget?
    t0 = time.time()
    sweep(qf, rf, batch)
    t_probe = (time.time() - t0) / batch
    t0 = time.time()
    encoders()
    t_enc_probe = time.time() - t0
    budget = float(os.environ.get("NOPE_REF_BUDGET_S", "150")) / max(args.steps + args.warmup, 1)
    sample = int(max(batch, min(n_grid, (budget - t_enc_probe) / max(t_probe, 1e-6))) // batch * batch)
    sample = max(batch, min(sample, n_grid))
    for _ in range(args.warmup):
        sweep(*encoders(), sample)
    t_enc = t_unet = 0.0
    for _ in range(args.steps):
        t0 = time.time()
        qf, rf = encoders()
        t1 = time.time()
        sweep(qf, rf, sample)
        t_enc += t1 - t0
        t_unet += time.time() - t1
    t_enc /= args.steps
    t_hyp = t_unet / args.steps / sample
    full_s = t_enc + n_grid * t_hyp
    v = n_grid / full_s
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "hyp/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": full_s * 1e3,
        "higher_is_better": True, "scaling": "strong" if args.global_poses else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": v, "unit": "hyp/s", "cores": threads, "kind": kind,
                         "sample": f"each step = 2 encoder calls ({t_enc * 1e3:.0f} ms) + the UNet sweep and scoring of "
                                   f"the first {sample} of the {n_grid} poses, {batch} hypotheses per forward "
                                   f"({t_hyp * 1e3:.1f} ms per hypothesis), fp32, {threads} of {os.cpu_count()} host "
                                   f"threads (fastest of a probe); value = {n_grid} / (t_enc + {n_grid} t_hyp), the "
                                   f"full-grid throughput these timings imply (sample alone: "
                                   f"{sample / (t_enc + sample * t_hyp):.1f} hyp/s)",
                         "sample_poses": sample, "t_encoders_ms": t_enc * 1e3, "t_per_hypothesis_ms": t_hyp * 1e3},
        "e2e": {"value": v, "unit": "hyp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------
def ldm_cpu_baseline(seconds=12.0, chunk=4):
    """oracle/ldm_oracle.py (CPU port of UNetModelPose.forward) + the l2 score, hyp/s."""
    import torch
    from oracle import ldm_oracle, unet_oracle as orc
    from nope_b200.synth_weights import make_ldm_state_dict
    from nope_b200.poses import synthetic_pose_batch
    sd = make_ldm_state_dict(seed=0)
    g = torch.Generator().manual_seed(0)
    rl = torch.randn(1, 4, 32, 32, generator=g)
    ql = torch.randn(1, 4, 32, 32, generator=g)
    poses, _ = synthetic_pose_batch(N_POSES, 1)
    done = 0
    with torch.no_grad():
        threads = pick_threads(lambda: ldm_oracle.ldm_sweep(sd, rl, poses[:, :2], chunk=2))
        t0 = time.time()
        while time.time() - t0 < seconds and done + chunk <= N_POSES:
            emb = ldm_oracle.ldm_sweep(sd, rl, poses[:, done:done + chunk], chunk=chunk)
            orc.l2_similarity(ql, emb)
            done += chunk
    dt = time.time() - t0
    return {"value": done / dt, "unit": "hyp/s", "cores": threads, "kind": "port",
            "sample": f"first {done} poses of the {N_POSES}-pose grid, batched {chunk}/forward, fp32 torch-CPU "
                      f"oracle of UNetModelPose, {threads} of {os.cpu_count()} host threads, {dt:.1f} s"}


def main_ldm(args):
    """LDM-variant sweep (UNetModelPose on VAE-sized latents): same metric and timing rules as main()."""
    import torch
    from nope_b200.ldm import UNetModelPose
    from nope_b200.poses import synthetic_pose_batch
    from nope_b200.synth_weights import ldm_flops_per_hyp, make_ldm_state_dict
    import torch.distributed as dist
    from nope_b200.dist import ShardedSweep
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    sharded = ShardedSweep() if world > 1 else None
    n_local = args.poses
    n = n_local * world                      # weak scaling: one grid per GPU shard
    chunk = min(args.chunk, 642)
    ldm_prec = args.precision if args.precision in ("fp16", "fp16_w2") else "fp16"
    m = UNetModelPose(device=str(dev), chunk=chunk, precision=ldm_prec)
    m.load_state_dict(make_ldm_state_dict(seed=0))
    Q = args.queries
    poses, _ = synthetic_pose_batch(n_local, Q)
    poses = poses.repeat(1, world, 1)
    g = torch.Generator().manual_seed(0)
    ref_h = torch.randn(Q, 4, 32, 32, generator=g).pin_memory()
    qry_h = torch.randn(Q, 4, 32, 32, generator=g).pin_memory()
    poses_h = poses.clone().pin_memory()
    ref_d, qry_d, poses_d = ref_h.to(dev), qry_h.to(dev), poses.to(dev)
    h2d = (ref_h.numel() + qry_h.numel() + poses_h.numel()) * 4
    d2h = Q * (5 * 8 + n * 4)

    def run(ref, pz, qry):
        if sharded is not None:
            sim, topi, _ = sharded.sweep(m, ref, pz, qry, k=5, want_emb=False)
            return {"sim": sim, "topi": topi}
        return m.sweep(ref, pz, qry, want_emb=False, k=5)

    def step_resident():
        return run(ref_d, poses_d, qry_d)

    def step_e2e():
        out = run(ref_h.to(dev, non_blocking=True), poses_h.to(dev, non_blocking=True),
                  qry_h.to(dev, non_blocking=True))
        return out["topi"].cpu(), out["sim"].cpu()

    def barrier():
        if world > 1:
            dist.barrier()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        barrier()
        t = e0.elapsed_time(e1) / steps
        if world > 1:
            tt = torch.tensor([t], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = float(tt)
        return t

    last = {}

    def step_kept():                          # the timed step, keeping its result for --dump-outputs
        last["out"] = step_resident()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(step_kept, args.steps, max(args.warmup, 3))
    launches = m.last_launch_count
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"sim": last["out"]["sim"], "topi": last["out"]["topi"]})
    ms_e2e = timed(step_e2e, args.steps, max(args.warmup, 3))
    m.profile(True)
    step_resident()
    prof = m.profile_read()
    m.profile(False)
    peak_tf, _, peak_src, _ = measured_peaks()
    gm, at = prof["gemm"], prof["attention"]
    gemm_tf = gm["flops"] / (gm["ms"] * 1e-3) / 1e12 if gm["ms"] > 0 else 0.0
    attn_tf = at["flops"] / (at["ms"] * 1e-3) / 1e12 if at["ms"] > 0 else 0.0
    fl = ldm_flops_per_hyp()
    value = Q * n / (ms * 1e-3)
    if rank != 0:
        dist.destroy_process_group()
        return
    cpu = None if (args.no_cpu_baseline or world > 1) else ldm_cpu_baseline()
    line = {
        "metric": METRIC, "value": value, "unit": "hyp/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
        "config": {
            "workload": f"LDM variant (SURVEY.md 8 f2): UNetModelPose of configs/model/vae_cin_ldm.yaml on 4x32x32 "
                        f"latents, {n_local}-pose grid per GPU, batch={Q} query, fp16 storage / fp32 accumulate, "
                        "l2 score + top-5",
            "poses_per_gpu": n_local, "global_poses": n, "queries": Q, "chunk": chunk,
            "precision": ldm_prec + (": exact weights (W_hi + W_lo K-segments, 2x the MMA work), embeddings within "
                                     "1e-3 of the fp32 reference" if ldm_prec == "fp16_w2" else
                                     ": fp16 weights and activations, fp32 accumulate (embeddings 1.08e-3)"),
            "parallelism": f"pose grid sharded {world}-way, all-gather of top-k" if world > 1 else "1 GPU",
            "weights": "seeded random init, reference state_dict schema (395.0 M params)",
            "gflop_per_hyp": fl["total"] / 1e9,
            "encoder": "none: the diffusers VAE of this variant is not in the reference tree; inputs are latents",
            "l2": "not flushed: each step streams 0.79 GB of fp16 weights and > 5 GB of activations, >> 126 MB L2",
        },
        "clocks": clocks,
        "e2e": {"value": Q * n / (ms_e2e * 1e-3), "unit": "hyp/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "UNetModelPose.sweep (pinned host latents + poses -> sweep -> top-5 -> host)"},
        "gpu_launches": int(launches * args.steps),
        "roofline": {
            "bound": "tensor", "kernel": "conv_tc2_kernel (tcgen05 implicit-GEMM conv / linear layers)",
            "achieved": gemm_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": gemm_tf / peak_tf if peak_tf else None,
            "peak_source": f"{peak_src} (sustained bf16 cuBLAS)", "traffic": None,
            "launches_per_step": gm["launches"], "gemm_ms_per_step": gm["ms"],
            "gemm_share_of_step": gm["ms"] / ms if ms else None,
            "algorithmic_tflop_per_step": gm["flops"] / 1e12,
            "attention": {"kernel": "ldm_attn_tc_kernel (tcgen05 QK^T / PV, softmax in registers)",
                          "achieved": attn_tf, "unit": "TFLOP/s", "ms_per_step": at["ms"],
                          "launches_per_step": at["launches"], "share_of_step": at["ms"] / ms if ms else None},
            "whole_step_tflops": value * fl["total"] / 1e12,
        },
        "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.variant == "ldm":
        if args.impl == "reference":
            line = {"impl": "reference", "metric": METRIC, "unit": "hyp/s", "higher_is_better": True}
            cpu = ldm_cpu_baseline(seconds=20.0)
            line.update({"value": cpu["value"], "cpu_baseline": cpu, "n_gpus": 1,
                         "config": {"workload": "LDM variant, oracle port on host cores"},
                         "e2e": {"value": cpu["value"], "unit": "hyp/s", "h2d_bytes_per_step": 0,
                                 "d2h_bytes_per_step": 0}})
            print(json.dumps(line))
            return
        main_ldm(args)
        return
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, (world, args.gpus)

    from nope_b200 import synth_weights as weights  # seeded random-init weights, reference schema
    from nope_b200.model import build_model
    from nope_b200.dist import ShardedSweep
    from nope_b200.poses import synthetic_pose_batch

    cfg = workload_config(args, world)
    strong = args.global_poses > 0
    n_global = cfg["global_poses"]
    n_local = cfg["poses_per_gpu"]
    sd = weights.make_full_state_dict(seed=0)
    model = build_model(device=str(dev), chunk=args.chunk, precision=args.precision)
    model.load_state_dict(sd).eval()
    unet = model.u_net
    unet.set_conv_impl(args.conv_impl)
    if world > 1:
        model.dist = ShardedSweep()

    # the grid: weak scaling = one icosphere grid per GPU shard (pose VALUES do not affect timing),
    # strong scaling = ONE fixed grid split contiguously over the ranks (dist.shard_range)
    Q = args.queries
    if strong:
        poses_g, _ = synthetic_pose_batch(n_global, Q)
    else:
        poses_g, _ = synthetic_pose_batch(args.poses, Q)
        poses_g = poses_g.repeat(1, world, 1)       # [Q, n_global, 6]
    g = torch.Generator().manual_seed(0)
    q_img = (torch.rand(Q, 3, 256, 256, generator=g) * 2 - 1).pin_memory()
    r_img = (torch.rand(Q, 3, 256, 256, generator=g) * 2 - 1).pin_memory()
    poses_host = poses_g.clone().pin_memory()
    h2d = q_img.numel() * 4 + r_img.numel() * 4 + poses_host.numel() * 4
    d2h = Q * (5 * 8 + n_global * 4)                # top-5 indices (int64) + similarity rows

    # ---- resident inputs for `value`
    q_feat = unet.encoder.encode_image(q_img.to(dev))
    r_feat = unet.encoder.encode_image(r_img.to(dev))
    poses_dev = poses_g.to(dev)

    def make_steps(m):
        u = m.u_net

        def step_resident():
            if world > 1:
                return m.dist.sweep(u, r_feat, poses_dev, q_feat, k=5, want_emb=False)
            out = u.sweep(r_feat, poses_dev, query_feat=q_feat, want_emb=False, k=5)
            return out["sim"], out["topi"], None

        def step_e2e():
            q = q_img.to(dev, non_blocking=True)
            r = r_img.to(dev, non_blocking=True)
            p = poses_host.to(dev, non_blocking=True)
            _, idx, sim = m.predict_pose(q, r, p, None, k=5)
            return idx.cpu(), sim.cpu()             # D2H of the step's result
        return step_resident, step_e2e

    step_resident, step_e2e = make_steps(model)
    last = {}

    def step_kept():                          # the timed step, keeping its result for --dump-outputs
        last["out"] = step_resident()

    def barrier():
        if world > 1:
            dist.barrier()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        barrier()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(step_kept, args.steps, max(args.warmup, 3))
    launches_per_step = unet.last_launch_count
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        sim, topi, _ = last["out"]
        dump_outputs(args.dump_outputs, {"sim": sim, "topi": topi})
    ms_e2e = timed(step_e2e, args.steps, max(args.warmup, 3))

    # ---- BASELINE configs[3] beside the weak-scaling headline: the FIXED 10 248-pose grid (level-3 icosphere x 4
    # in-plane rotations) split over the ranks -- the driver's `--gpus N` runs carry the strong-scaling figure too
    strong_extra = None
    if world > 1 and not strong and not args.no_extras:
        poses_s = synthetic_pose_batch(10248, Q)[0].to(dev)
        ms_s = timed(lambda: model.dist.sweep(unet, r_feat, poses_s, q_feat, k=5, want_emb=False), 3, 3)
        strong_extra = {"workload": f"configs[3]: a FIXED 10248-pose grid sharded {world}-way "
                                    f"({-(-10248 // world)} poses per GPU), batch={Q}, same timing rules, 3 steps",
                        "global_poses": 10248, "value": Q * 10248 / (ms_s * 1e-3), "unit": "hyp/s",
                        "ms_per_step": ms_s, "scaling": "strong"}
        del poses_s

    # ---- roofline of the dominant kernel (tcgen05 convolution), CUDA events per launch
    def conv_profile(u, step):
        u.profile(True)
        step()
        pr = u.profile_read()
        u.profile(False)
        return pr
    prof = conv_profile(unet, step_resident)
    peak_tf, peak_hbm, peak_src, peak_burst = measured_peaks()
    conv_s = prof["conv_ms"] * 1e-3
    conv_tf = prof["conv_alg_flops"] / conv_s / 1e12 if conv_s > 0 else 0.0      # algorithmic
    conv_exec_tf = prof["conv_flops"] / conv_s / 1e12 if conv_s > 0 else 0.0     # incl. split-precision K-segments

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    n_hyp_step = Q * n_global
    value = n_hyp_step / (ms * 1e-3)
    extras = world == 1 and not args.no_extras

    # ---- the other precision modes, same workload, resident timing (config.precision names the headline)
    modes = {args.precision: {"value": value, "ms_per_step": ms, "e2e": n_hyp_step / (ms_e2e * 1e-3),
                              "conv_algorithmic_tflops": conv_tf, "conv_executed_tflops": conv_exec_tf}}
    if extras:
        del model, unet
        torch.cuda.empty_cache()
        for mode in ("fp16", "fp16_w2", "parity", "parity_fast", "bf16"):
            if mode in modes:
                continue
            try:
                m2 = build_model(device=str(dev), chunk=args.chunk, precision=mode)
                m2.load_state_dict(sd).eval()
                sr, se = make_steps(m2)
                ms2 = timed(sr, max(3, args.steps // 2), 3)
                ms2e = timed(se, max(3, args.steps // 2), 3)
                p2 = conv_profile(m2.u_net, sr)
                modes[mode] = {"value": n_hyp_step / (ms2 * 1e-3), "ms_per_step": ms2,
                               "e2e": n_hyp_step / (ms2e * 1e-3),
                               "conv_algorithmic_tflops": p2["conv_alg_flops"] / (p2["conv_ms"] * 1e-3) / 1e12,
                               "conv_executed_tflops": p2["conv_flops"] / (p2["conv_ms"] * 1e-3) / 1e12}
                del m2
                torch.cuda.empty_cache()
            except Exception as exc:                  # informational leg only
                modes[mode] = {"unavailable": repr(exc)[:200]}
    cpu = None if (args.no_cpu_baseline or world > 1) else cpu_baseline()
    eager = None
    if not args.no_cpu_baseline and extras:
        try:
            eager = eager_gpu_baseline(dev)
        except Exception as exc:                      # informational leg only
            eager = {"unavailable": repr(exc)[:200]}
    variants = None
    if extras and not args.no_cpu_baseline:
        try:
            variants = {"ldm": ldm_summary(args, dev)}
        except Exception as exc:
            variants = {"ldm": {"unavailable": repr(exc)[:200]}}
    line = {
        "metric": METRIC, "value": value, "unit": "hyp/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "fp16", "data": "synthetic",
        "config": cfg,
        "clocks": clocks,
        "e2e": {"value": n_hyp_step / (ms_e2e * 1e-3), "unit": "hyp/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "PoseConditional.predict_pose (pinned host images -> encoder x2 -> sweep -> top-5 -> host)"},
        "gpu_launches": int(launches_per_step * args.steps),
        "roofline": {
            "bound": "tensor", "kernel": "conv_tc2_kernel (tcgen05 implicit-GEMM conv, CTA pairs; GroupNorm / SiLU / "
                                         "pose bias / residual in its epilogue)",
            "achieved": conv_tf, "peak": peak_tf, "unit": "TFLOP/s",
            "frac": conv_tf / peak_tf if peak_tf else None, "peak_source": f"{peak_src} (sustained bf16 cuBLAS)",
            "peak_burst": peak_burst, "frac_of_burst": conv_tf / peak_burst if peak_burst else None,
            "executed_tflops": conv_exec_tf,
            "traffic": ncu_traffic(), "traffic_source": "profiles/roofline_traffic.json (ncu --set full, "
            "dram__bytes_read.sum + dram__bytes_write.sum per launch, sweep convolutions)",
            "launches_per_step": prof["conv_launches"],
            "conv_ms_per_step": prof["conv_ms"], "conv_share_of_step": prof["conv_ms"] / ms if ms else None,
            "algorithmic_tflop_per_step": prof["conv_alg_flops"] / 1e12,
            "best_single_launch_tflops": prof["max_launch_tflops"],
            "whole_step_tflops": value * GFLOP_PER_HYP / 1e3,
            "whole_step_frac": value * GFLOP_PER_HYP / 1e3 / peak_tf if peak_tf else None,
            "note": "the convolution kernel also normalises / activates / adds pose bias and residual in its epilogue "
                    "(round 1 ran those as separate HBM passes and reported frac 0.87-0.90 for the bare convolution): "
                    "compare whole_step_frac, 0.71 in round 1",
        },
        "modes": modes,
        "cpu_baseline": cpu,
        "eager_gpu_baseline": eager,
        "variants": variants,
        "strong_scaling": strong_extra,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def ldm_summary(args, dev):
    """One short resident timing of the LDM variant (SURVEY.md 8 f2) for the default line's `variants`:
    the full line (e2e, clocks, cpu baseline) is `bench.py --variant ldm`."""
    import torch
    from nope_b200.ldm import UNetModelPose
    from nope_b200.poses import synthetic_pose_batch
    from nope_b200.synth_weights import ldm_flops_per_hyp, make_ldm_state_dict
    m = UNetModelPose(device=str(dev), chunk=min(args.chunk, 642))
    m.load_state_dict(make_ldm_state_dict(seed=0))
    poses, _ = synthetic_pose_batch(N_POSES, 1)
    g = torch.Generator().manual_seed(0)
    ref = torch.randn(1, 4, 32, 32, generator=g).to(dev)
    qry = torch.randn(1, 4, 32, 32, generator=g).to(dev)
    poses = poses.to(dev)
    run = lambda: m.sweep(ref, poses, qry, want_emb=False, k=5)
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    m.profile(True)
    run()
    prof = m.profile_read()
    m.profile(False)
    peak_tf, _, peak_src, peak_burst = measured_peaks()
    gm, at = prof["gemm"], prof["attention"]
    gemm_tf = gm["flops"] / (gm["ms"] * 1e-3) / 1e12 if gm["ms"] > 0 else 0.0
    fl = ldm_flops_per_hyp()
    out = {"workload": f"UNetModelPose (vae_cin_ldm.yaml) on 4x32x32 latents, {N_POSES}-pose grid, batch=1",
           "value": N_POSES / (ms * 1e-3), "unit": "hyp/s", "ms_per_step": ms, "gflop_per_hyp": fl["total"] / 1e9,
           "roofline": {"bound": "tensor", "kernel": "conv_tc2_kernel", "achieved": gemm_tf, "peak": peak_tf,
                        "unit": "TFLOP/s", "frac": gemm_tf / peak_tf if peak_tf else None,
                        "frac_of_burst": gemm_tf / peak_burst if peak_burst else None,
                        "gemm_share_of_step": gm["ms"] / ms,
                        "attention_tflops": at["flops"] / (at["ms"] * 1e-3) / 1e12 if at["ms"] > 0 else 0.0,
                        "attention_share_of_step": at["ms"] / ms},
           "full_line": "python bench.py --variant ldm"}
    del m
    torch.cuda.empty_cache()
    # exact-weights mode (the one that meets the 1e-3 embedding bar): resident timing only
    m = UNetModelPose(device=str(dev), chunk=min(args.chunk, 642), precision="fp16_w2")
    m.load_state_dict(make_ldm_state_dict(seed=0))
    run = lambda: m.sweep(ref, poses, qry, want_emb=False, k=5)
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms2 = e0.elapsed_time(e1) / 3
    out["modes"] = {"fp16": {"value": out["value"], "ms_per_step": ms},
                    "fp16_w2": {"value": N_POSES / (ms2 * 1e-3), "ms_per_step": ms2,
                                "note": "exact weights (W_hi + W_lo K-segments): embeddings 0.91e-3 vs the fp32 oracle"}}
    del m
    torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    main()

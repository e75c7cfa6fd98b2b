#!/usr/bin/env python
"""bench.py -- diffusion steps/sec of the PoseDiffusion sampling hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg3|cfg1|cfg2|cfg4|cfg5] [--dump-outputs DIR]
    (N > 1: launched by torchrun, one rank per GPU over NCCL)

A bench "step" is one full p_sample_loop of the workload: T = 100 diffusion steps of one 20-frame sequence per GPU,
the last 10 of them guided (7 000 inner Sampson/GGS iterations over 778 240 matches).  `value` counts diffusion
steps: world * sequences_per_gpu * 100 * K / (max-over-ranks device time of the K timed loops).

Output: ONE JSON line on rank 0 (see the contract in the task statement): value (inputs resident in HBM),
e2e (host buffers through the C-ABI call, H2D/D2H and match packing inside the timed region), roofline of the
dominant kernel (GGS/Sampson, HBM-bound, algorithmic 16 B per match-evaluation), cpu_baseline (the CPU oracle
port on this box's host cores, bounded sample, extrapolated), clocks, gpu_launches.
"""
from __future__ import annotations

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

import numpy as np
import torch

T_STEPS = 100
WORKLOADS = {
    # name: (frames, matches per ordered pair or 0 for GGS off, description)
    "cfg1": (5, 0, "BASELINE configs[0]: 1 sequence x 5 frames (the samples/apple demo shape), T=100, GGS off (the reference's CPU-runnable case)"),
    "cfg3": (20, 2048, "BASELINE configs[2]: 1 sequence x 20 frames per GPU, T=100, GGS on (start_step 10, 700 inner iters/step), "
                      "M=2048 uniform-random matches for each of the 380 ordered pairs (778240 matches)"),
    "cfg2": (20, 0, "BASELINE configs[1]: 1 sequence x 20 frames per GPU, T=100, GGS off (denoiser-only path)"),
    "cfg4": (20, 2048, "BASELINE configs[3]: 64 sequences x 20 frames sharded over 8 GPUs = 8 sequences per GPU (--seqs-per-gpu defaults to 8 "
                      "here), T=100, GGS on, 778240 matches per sequence; one GGS launch optimises the GPU's 8 sequences side by side"),
    "cfg5": (80, 4096, "BASELINE configs[4]: 1 sequence x 80 frames, T=100, GGS on, M=4096 x 6320 ordered pairs (25886720 matches)"),
}
FEATURES_DESC = ("widened row SURVEY 8f-2 (NOT the headline): MultiScaleImageFeatureExtractor = DINO ViT-S/16 at scales 1, 1/2, 1/3 over "
                 "20 frames of 224x224 per sequence (264 tokens per frame), the stage that produces z for the sampler")
ALGO_BYTES_PER_MATCH_EVAL = 16  # kp1.xy + kp2.xy as fp32 (SURVEY.md §8d)
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory: str, arrays: dict):
    """--dump-outputs: what the timed path returned in its last step, one float32 DIR/<name>.npy per array, so that two builds can
    be compared output for output on the same seeded inputs.  Above DUMP_LIMIT_BYTES in all, every array keeps a fixed, seeded
    sample of the rows along its first axis.  GGS-off workloads repeat to within 1e-6 of max|pose|; with GGS on, the float
    atomics of the GGS kernel's shared-memory sums change the order of additions from run to run, and the guided steps amplify
    that: two runs of one build differed by up to 2 % of max|pose| at cfg3 (1x B200, 1000 W power limit)."""
    os.makedirs(directory, exist_ok=True)
    total = sum(t.numel() * 4 for t in arrays.values())
    for name, t in arrays.items():
        a = t.detach().to(torch.float32).cpu().numpy()
        if total > DUMP_LIMIT_BYTES:
            keep = max(1, a.shape[0] * DUMP_LIMIT_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(directory, f"{name}.npy"), a)


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        load = [v for v in sm if mx and v > 0.5 * mx[0]] or sm
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# CPU arm.  The reference is Python: its unmodified `models` / `util` packages are imported from the reference checkout or
# from oracle/_ref (installed there by oracle/install_reference.py during build()) behind the pytorch3d / hydra shim of
# oracle/shims -> kind "reference".  If neither exists the oracle port (oracle/pose_oracle.py, the same operator
# sequence restated) is timed instead -> kind "port".  Bounded sample, extrapolated to the full loop.
# ----------------------------------------------------------------------------------------------------
def host_thread_candidates():
    """BASELINE.md section 3 asks for os.cpu_count() threads; PyTorch-CPU is often faster with fewer on these ~1e6-element ops,
    so the arm times a short probe with each candidate and keeps the faster (both are reported)."""
    n = os.cpu_count() or 1
    forced = os.environ.get("PDB_REF_THREADS")
    if forced:
        return [max(1, min(n, int(forced)))]
    return sorted({n, min(n, 32)}, reverse=True)


def cpu_reference_run(frames: int, per_pair: int, seed: int, budget_s: float):
    import contextlib
    import io

    from oracle import pose_oracle as po
    from oracle import ref_loader
    from posediffusion_b200 import synthetic as syn

    state = syn.random_denoiser_state(seed)
    z = syn.random_features(1, frames, seed)
    draws = syn.predraw_noise(1, frames, seed=seed)
    cfg = syn.default_ggs_cfg()
    kind = "reference" if ref_loader.reference_available() else "port"
    if kind == "reference":
        ref = ref_loader.load_reference()
        sampler = ref_loader.build_reference_sampler(ref, state)

        def denoise_loop():  # GaussianDiffusion.sample without guidance: 100 x (Denoiser.forward + DDPM update)
            with torch.no_grad():
                return sampler.sample(shape=[1, frames, 9], z=z)[0]

        def ggs_call(mean, matches, k=1):  # one geometry_guided_sampling call with iter_num = k: 2k+k+k+k+2k = 7k inner iterations
            with contextlib.redirect_stdout(io.StringIO()):  # the reference prints one line per phase
                return ref.geometry_guided_sampling(mean, 5, matches, dict(cfg, iter_num=k, min_matches=0)), 7 * k
    else:
        net = po.build_denoiser(state)
        sched = po.diffusion_schedule()

        def denoise_loop():
            return po.p_sample_loop(net, sched, z, draws, None, 0)[0]

        def ggs_call(mean, matches, k=1):
            return po.geometry_guided_sampling(mean, 5, matches, dict(cfg, iter_num=k, min_matches=0)), 7 * k

    m = syn.uniform_matches(frames, per_pair, seed=seed) if per_pair else None
    probe = {}
    for threads in host_thread_candidates():  # short probe per candidate thread count
        torch.set_num_threads(threads)
        t0 = time.perf_counter()
        if m is not None:
            ggs_call(draws[0].clone(), m)
        else:
            with torch.no_grad():
                denoise_loop()
        probe[threads] = time.perf_counter() - t0
    threads = min(probe, key=probe.get)
    torch.set_num_threads(threads)
    denoise_loop() if m is None else None  # warm-up of the path not probed above is the probe itself
    t0 = time.perf_counter()
    pose = denoise_loop()
    t_denoise = time.perf_counter() - t0
    sample = f"100 denoiser steps ({t_denoise:.2f} s)"
    t_ggs_full = 0.0
    if m is not None:
        # one guided step = one geometry_guided_sampling call = match upload / preprocessing U + 700 inner iterations.  Calls with
        # iter_num = 1 and 3 (7 and 21 inner iterations) alternate until the budget is spent; the least-squares line
        # T(call) = U + n_inner * t_iter separates the per-call cost from the per-iteration cost, and the full loop is
        # start_step x (U + 700 t_iter).
        inner_per_step = 7 * cfg["iter_num"]
        mean = pose.detach().clone()
        xs, ys = [], []
        t_start = time.perf_counter()
        while time.perf_counter() - t_start < budget_s or len(xs) < 2:
            k = 1 if len(xs) % 2 == 0 else 3
            t1 = time.perf_counter()
            mean, did = ggs_call(mean, m, k)
            ys.append(time.perf_counter() - t1)
            xs.append(did)
        t_iter, per_call = np.polyfit(np.asarray(xs, float), np.asarray(ys, float), 1)
        per_call = max(0.0, float(per_call))
        t_ggs_full = cfg["start_step"] * (per_call + inner_per_step * float(t_iter))
        sample += (f" + {int(sum(xs))} of {cfg['start_step'] * inner_per_step} inner GGS iterations in {len(xs)} calls ({sum(ys):.2f} s): "
                   f"{1e3 * t_iter:.1f} ms per inner iteration, {1e3 * per_call:.0f} ms per call (match upload), extrapolated")
    sample += "; probe s per thread count: " + ", ".join(f"{k} threads {v:.2f}" for k, v in sorted(probe.items()))
    wall = t_denoise + t_ggs_full
    return {"steps_per_s": T_STEPS / wall, "wall_s_full": wall, "sample": sample, "threads": threads, "kind": kind}


# ----------------------------------------------------------------------------------------------------
# ----------------------------------------------------------------------------------------------------
# Widened row (SURVEY 8f-2): image features.  Same contract as the headline line, metric = images/s.
# ----------------------------------------------------------------------------------------------------
VIT_GEMM_FLOPS_PER_TOKEN = 2 * (768 * 384 + 12 * (384 * 1152 + 384 * 384 + 2 * 384 * 1536))
VIT_TOKENS_PER_IMAGE = 197 + 50 + 17
VIT_SCALES = [1, 1 / 2, 1 / 3]


def cpu_features_run(n_images: int, seed: int, threads: int):
    """The oracle port of the extractor (reference wrapper arithmetic + restated hub backbone) on the host cores."""
    from oracle.dino_vit import DinoViTSmall16, multiscale_features

    torch.set_num_threads(threads)
    torch.manual_seed(seed)
    net = DinoViTSmall16().eval()
    img = torch.rand(n_images, 3, 224, 224)
    with torch.no_grad():
        multiscale_features(net, img[:1], VIT_SCALES)
        t0 = time.perf_counter()
        multiscale_features(net, img, VIT_SCALES)
        dt = time.perf_counter() - t0
    return {"images_per_s": n_images / dt, "threads": threads, "sample": f"{n_images} frames of 224x224 at 3 scales in {dt:.2f} s"}


def features_main(args):
    rank = int(os.environ.get("RANK", "0"))
    frames = 20 * args.seqs_per_gpu
    if args.impl == "reference":
        if rank != 0:
            return 0
        res = cpu_features_run(64 * max(1, args.steps), args.seed, min(os.cpu_count() or 1, int(os.environ.get("PDB_REF_THREADS", "32"))))
        print(json.dumps({"impl": "reference", "metric": "images/sec (DINO ViT-S/16 multi-scale features)", "value": res["images_per_s"],
                          "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": FEATURES_DESC},
                          "cpu_baseline": {"value": res["images_per_s"], "unit": "images/s", "cores": res["threads"], "kind": "port", "sample": res["sample"]},
                          "e2e": {"value": res["images_per_s"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return 0
    import posediffusion_b200 as pdb
    from posediffusion_b200 import _native
    from posediffusion_b200.distributed import init_from_env, sequence_seed

    rank, world, local = init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    torch.manual_seed(args.seed)
    ext = pdb.MultiScaleImageFeatureExtractor(modelname="dino_vits16", freeze=True, scale_factors=VIT_SCALES).to(dev)
    img_host = torch.rand((frames, 3, 224, 224), generator=torch.Generator().manual_seed(sequence_seed(args.seed, rank))).pin_memory()
    img_dev = img_host.to(dev)
    ctx = _native.Context.get(dev)
    ext(img_dev[:1].contiguous())  # loads the weights into the context
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(max(3, args.warmup)):
        z = ctx.extract_features(img_dev, VIT_SCALES)
    sync_all()
    ctx.profile(True)
    ctx.profile_read()
    launches0 = ctx.launch_count
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    with ClockSampler(local) as clocks:
        sync_all()
        for k in range(args.steps):
            flush.zero_()
            starts[k].record()
            z = ctx.extract_features(img_dev, VIT_SCALES)
            stops[k].record()
        sync_all()
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, stops))
    _, _, gemm_ms, gemm_n = ctx.profile_read()
    ctx.profile(False)
    launches = ctx.launch_count - launches0
    t_ms = torch.tensor([dev_ms], device=dev)
    if world > 1:
        torch.distributed.all_reduce(t_ms, op=torch.distributed.ReduceOp.MAX)
    value = frames * world * args.steps / (float(t_ms.item()) / 1000.0)
    img_np = img_host.numpy()
    ctx.extract_features_host(img_np, VIT_SCALES)
    sync_all()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        zh = ctx.extract_features_host(img_np, VIT_SCALES)
    sync_all()
    e2e_s = torch.tensor([time.perf_counter() - e0], device=dev)
    if world > 1:
        torch.distributed.all_reduce(e2e_s, op=torch.distributed.ReduceOp.MAX)
    if rank != 0:
        torch.distributed.destroy_process_group()
        return 0
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else None
    bf16 = float(peaks["bf16_tflops"]) if peaks else 2250.0
    flops_call = frames * VIT_TOKENS_PER_IMAGE * VIT_GEMM_FLOPS_PER_TOKEN
    achieved = flops_call * args.steps / (gemm_ms / 1000.0) / 1e12 if gemm_ms else None
    line = {
        "metric": "images/sec (DINO ViT-S/16 multi-scale features)", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": float(t_ms.item()) / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "tf32 tensor-core products, f32 accumulate / residual stream / softmax / LayerNorm", "data": "synthetic",
        "config": {"workload": FEATURES_DESC, "images_per_gpu": frames, "image": "224x224", "scale_factors": "1, 1/2, 1/3",
                   "l2": "flushed between timed calls (256 MiB write)", "weights": "random init (hub init law), images ~ U(0,1)"},
        "e2e": {"value": frames * world * args.steps / float(e2e_s.item()), "unit": "images/s", "h2d_bytes_per_step": int(img_host.numel() * 4),
                "d2h_bytes_per_step": int(frames * 384 * 4), "note": "C-ABI pdb_extract_features_host from pinned host memory"},
        "gpu_launches": int(launches), "clocks": clocks.summary(),
        "roofline": {"kernel": "tc_linear_kernel (tcgen05.mma kind::tf32 + TMA; all projections of the backbone)", "bound": "tensor",
                     "achieved": achieved, "peak": bf16 / 2, "unit": "TFLOP/s", "frac": achieved / (bf16 / 2) if achieved else None, "traffic": None,
                     "peak_source": ("half of the measured dense bf16 rate (MEASURED_PEAKS.json bf16_tflops): TF32 runs at half the bf16 rate"
                                     if peaks else "fallback: half of the nominal 2.25 PFLOP/s bf16 rate"),
                     "algorithmic_flops_per_call": flops_call, "gemm_launches_per_call": gemm_n // max(1, args.steps),
                     "gemm_ms_per_call": gemm_ms / max(1, args.steps),
                     "note": "fp32 operands staged by TMA (4 B/element): the 128x128 tiles are bound by operand delivery from L2, not by the tensor pipe"},
    }
    if not args.no_cpu_baseline and world == 1:
        res = cpu_features_run(96, args.seed, min(os.cpu_count() or 1, 32))
        line["cpu_baseline"] = {"value": res["images_per_s"], "unit": "images/s", "cores": res["threads"], "kind": "port", "sample": res["sample"]}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"z": z})
    print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS) + ["features"])
    ap.add_argument("--seqs-per-gpu", type=int, default=None, help="sequences per GPU (default 1; 8 for --workload cfg4)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU GGS iterations in the bounded sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ggs-layout", default="paired", choices=["plain", "paired"],
                    help="HBM layout of the packed match stream (csrc/ggs_layout.cuh); 'paired' is the library default, see DESIGN.md 4.1")
    ap.add_argument("--denoiser-engine", default="auto", choices=["auto", "fp32", "tf32"],
                    help="auto = exact-fp32 persistent kernel below 128 tokens per GPU, tcgen05/TMA tiles (TF32) at or above")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (the gathered poses; z of rank 0 for --workload "
                         "features) as DIR/<name>.npy in float32")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm times a bounded sample and computes no complete output")
    if args.seqs_per_gpu is None:
        args.seqs_per_gpu = 8 if args.workload == "cfg4" else 1
    if args.workload == "features":
        return features_main(args)
    frames, per_pair, desc = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        res = cpu_reference_run(frames, per_pair, args.seed, args.cpu_budget * max(1, args.steps))
        line = {
            "impl": "reference", "metric": "diffusion steps/sec (20-frame seq, GGS on)", "value": res["steps_per_s"],
            "unit": "diffusion steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * res["wall_s_full"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "frames": frames, "matches_per_pair": per_pair, "timesteps": T_STEPS},
            "cpu_baseline": {"value": res["steps_per_s"], "unit": "diffusion steps/s", "cores": res["threads"], "kind": res["kind"],
                             "sample": res["sample"]},
            "e2e": {"value": res["steps_per_s"], "unit": "diffusion steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------------------------
    import posediffusion_b200 as pdb
    from posediffusion_b200 import _native
    from posediffusion_b200 import synthetic as syn
    from posediffusion_b200.distributed import gather_poses, init_from_env, sequence_seed, shard_range

    rank, world, local = init_from_env("nccl")
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE {world}", file=sys.stderr)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    B = args.seqs_per_gpu
    total_seqs = B * world
    lo, hi = shard_range(total_seqs, rank, world)

    den = pdb.Denoiser(TRANSFORMER=dict(d_model=512, nhead=4, dim_feedforward=1024, num_encoder_layers=8, dropout=0.1,
                                        batch_first=True, norm_first=True))
    den.load_state_dict(syn.random_denoiser_state(args.seed), strict=True)
    den = den.to(dev)
    ctx = den.native_context()
    ctx.set_denoiser_engine(args.denoiser_engine)
    ctx.set_ggs_layout(args.ggs_layout)
    cfg = syn.default_ggs_cfg()
    cfg["verbose"] = False
    start_step = cfg["start_step"] if per_pair else 0

    # per-sequence synthetic inputs keyed by the GLOBAL sequence index (world-size invariant results)
    z_host = torch.cat([syn.random_features(1, frames, sequence_seed(args.seed, g)) for g in range(lo, hi)]).pin_memory()
    draws_host = torch.cat([syn.predraw_noise(1, frames, seed=sequence_seed(args.seed, g)) for g in range(lo, hi)], dim=1).contiguous().pin_memory()
    match_dicts = [syn.uniform_matches(frames, per_pair, seed=sequence_seed(args.seed, g)) for g in range(lo, hi)] if per_pair else None
    z_dev, draws_dev = z_host.to(dev), draws_host.to(dev)
    problems = [ctx.pack_matches(m) for m in match_dicts] if per_pair else None
    m_total = problems[0].m_total if per_pair else 0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def one_loop():
        pose, _, _ = ctx.sample_loop(z_dev, draws_dev, problems, cfg if per_pair else None, start_step, want_trail=False, want_stats=False)
        return pose

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(max(3, args.warmup)):
        pose = one_loop()
    sync_all()
    # BASELINE.md section 3: both arms must run all 7 000 inner iterations per sequence (no early exit).  Checked once, outside the
    # timed region, from the device-side statistics; recorded in the JSON line rather than asserted.
    ggs_check = None
    if per_pair:
        try:
            _, _, st = ctx.sample_loop(z_dev, draws_dev, problems, cfg, start_step, want_trail=False, want_stats=True)
            rows = _native.stats_to_numpy(st)
            ggs_check = {"inner_iterations_per_sequence": int(rows["iters"].sum()) // B, "early_exits": int(rows["dropped"].sum()),
                         "expected": start_step * 7 * cfg["iter_num"]}
        except Exception as exc:  # never let the check itself break the measurement
            ggs_check = {"error": repr(exc)[:200]}
        sync_all()

    # ---- timed region: K loops, L2 flushed between them, CUDA events on the launch stream ----
    ctx.profile(True)
    ctx.profile_read()
    launches0 = ctx.launch_count
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    wall0 = time.perf_counter()
    with ClockSampler(local) as clocks:
        sync_all()
        for k in range(args.steps):
            flush.zero_()
            starts[k].record()
            pose = one_loop()
            full = gather_poses(pose, total_seqs)  # the path's only collective (no-op at world 1)
            stops[k].record()
        sync_all()
    wall = time.perf_counter() - wall0
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, stops))
    ggs_ms, ggs_n, den_ms, den_n = ctx.profile_read()
    ctx.profile(False)
    launches = ctx.launch_count - launches0
    t_ms = torch.tensor([dev_ms], device=dev)
    if world > 1:
        torch.distributed.all_reduce(t_ms, op=torch.distributed.ReduceOp.MAX)
    dev_ms_max = float(t_ms.item())
    value = total_seqs * T_STEPS * args.steps / (dev_ms_max / 1000.0)

    # ---- end to end through the C-ABI host-buffer call: pack matches (host pass + H2D), H2D z/draws, D2H pose ----
    pose_host = torch.empty(B, frames, 9).pin_memory()
    z_np, draws_np, pose_np = z_host.numpy(), draws_host.numpy(), pose_host.numpy()

    def one_e2e():
        if per_pair:  # reference-format matches in, poses out: packing + upload overlap the unguided steps inside the call
            ctx.sample_loop_host_matches(z_np, draws_np, match_dicts, cfg, start_step, pose_np)
        else:
            ctx.sample_loop_host(z_np, draws_np, None, None, start_step, pose_np)

    one_e2e()
    sync_all()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        one_e2e()
    sync_all()
    e2e_s = torch.tensor([time.perf_counter() - e0], device=dev)
    if world > 1:
        torch.distributed.all_reduce(e2e_s, op=torch.distributed.ReduceOp.MAX)
    e2e_value = total_seqs * T_STEPS * args.steps / float(e2e_s.item())
    h2d = z_host.numel() * 4 + draws_host.numel() * 4 + (B * m_total * 16 if per_pair else 0)
    d2h = pose_host.numel() * 4

    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return 0

    peak, peak_src = read_peaks()
    line = {
        "metric": "diffusion steps/sec (20-frame seq, GGS on)" if args.workload == "cfg3" else f"diffusion steps/sec ({args.workload})",
        "value": value, "unit": "diffusion steps/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if (args.denoiser_engine == "fp32" or (args.denoiser_engine == "auto" and B * frames < 128)) else "f32 (GGS, residual stream) + tf32 tensor-core products (denoiser projections)",
        "data": "synthetic",
        "config": {"workload": desc, "frames": frames, "matches_per_pair": per_pair, "sequences_per_gpu": B, "denoiser_engine": args.denoiser_engine, "ggs_layout": args.ggs_layout, "timesteps": T_STEPS,
                   "parallelism": f"sequences sharded over {world} GPU(s), final all-gather of poses only",
                   "l2": "flushed between timed loops (256 MiB write); within a launch the match set is deliberately kept on chip when it fits",
                   "outputs": "final pose only; the optional pose_process trajectory (models/gaussian_diffuser.py:298-300, 72 KB per sequence) is not materialised in the timed loops",
                   "weights": "random init (reference init law), z ~ N(0,1), uniform-random correspondences"},
        "e2e": {"value": e2e_value, "unit": "diffusion steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "note": "C-ABI pdb_sample_loop_host_matches with pinned host buffers: reference-format float64/int64 matches are "
                        "converted on the host (48 B/match read) and uploaded as 16 B/match while the unguided steps run"},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "wall_s_timed_region": wall,
        "published_reference_note": "reference README.md:45 quotes ~60 s of sampling for a 20-frame GGS sequence on a Quadro GP100 (~1.7 steps/s, real hloc matches): other hardware, not this synthetic config, hence vs_baseline = null",
        "ggs_iteration_check": ggs_check,
        "kernel_ms_per_loop": {"ggs": ggs_ms / args.steps, "denoiser": den_ms / args.steps, "ggs_launches": ggs_n // args.steps,
                               "denoiser_launches": den_n // args.steps},
    }
    if per_pair and ggs_n:
        inner_per_launch = 7 * cfg["iter_num"]
        algo_bytes = ALGO_BYTES_PER_MATCH_EVAL * m_total * inner_per_launch * B
        achieved = algo_bytes / (ggs_ms / ggs_n / 1000.0) / 1e9
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if os.path.exists(tpath):  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
            rec = json.load(open(tpath)).get(f"ggs_entry<false>@{args.workload}")
            if rec and B == 1:
                traffic, traffic_src = rec["dram_bytes_read"] + rec["dram_bytes_write"], rec["source"]
        line["roofline"] = {
            "kernel": "ggs_entry<false> (fused Sampson error+gradient, 700 inner iterations per launch)", "bound": "hbm",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes, "avg_launch_ms": ggs_ms / ggs_n,
            "note": ("algorithmic bytes = 16 B x matches x inner iterations; at this size the CTA slices of the match set (12.45 MB total) "
                     "stay resident in shared memory for the whole launch, so DRAM traffic is ~0.2% of the algorithmic bytes by design "
                     "and the iteration is latency-chain bound (run --workload cfg5 for the HBM-streaming case: 414 MB per inner iteration)")
                    if (args.workload == "cfg3" and B == 1) else
                    "algorithmic bytes = 16 B x matches x inner iterations, streamed every inner iteration through the TMA unit's bulk-async "
                    "ring (from HBM at config 5: 414 MB per iteration; largely from L2 when the sequences' match sets fit its 126 MB)",
        }
    if not args.no_cpu_baseline and world == 1:  # reported baseline: rank 0 at N = 1 only
        res = cpu_reference_run(frames, per_pair, args.seed, args.cpu_budget)
        line["cpu_baseline"] = {"value": res["steps_per_s"], "unit": "diffusion steps/s", "cores": res["threads"], "kind": res["kind"],
                                "sample": res["sample"], "wall_s_full_extrapolated": res["wall_s_full"]}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pose": full})
    print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

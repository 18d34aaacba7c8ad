#!/usr/bin/env python
"""bench.py -- InternVLA-N1 policy-steps/sec on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Workloads (BASELINE.json `configs`, SURVEY.md §8d):
  dual_system    configs[3] (DEFAULT -- the configuration the metric is quoted on): the full dual-system step for 64
                 parallel environments on one GPU: Qwen2.5-VL-7B ViT + LLM prefill (S = 304 per env) -> 4 latent tokens ->
                 NavDP RGB-D encoder + 20-step DDPM over 32 trajectories of horizon 32 -> discrete action ids.
                 One "step" = one such call; 64 policy steps per call.
  navdp_denoise  configs[1]: NavDP diffusion denoiser only, 50 DDPM steps, 256 trajectories (8 envs x 32 samples) of
                 horizon 8, bf16.  One "step" = one full 50-step sampling call; one policy step = one environment's
                 32-trajectory sample (8 per call).
Multi-GPU: environments are independent, so every rank runs the same per-GPU workload on its own shard (weak scaling,
no data-path collective; SURVEY.md §8e).  Timing: CUDA events on the launching stream, per timed step, L2 flushed
between steps, max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "navdp_denoise": dict(kind="denoise", B=8, Ns=32, T=8, K=50,
                          desc="configs[1]: NavDP denoiser only, 50 denoise steps, 256 trajectories (8 envs x 32) of horizon 8, bf16"),
    "dual_system": dict(kind="dual", B=64, Ns=32, T=32, K=20, S=304, grid=(1, 28, 28),
                        desc="configs[3]: full dual-system step (Qwen2.5-VL-7B ViT + LLM prefill -> 4 latents -> NavDP "
                             "RGB-D encoder + 20-step DDPM, 32 samples, horizon 32 -> action ids), 64 parallel envs, bf16; "
                             "per env one 392x392 frame (784 patches -> 196 tokens) + 104 text tokens + 4 latent queries = 304"),
    "s2_prefill": dict(kind="s2", B=32, S=304, grid=(1, 28, 28),
                       desc="configs[2]: System-2 VLM forward only (Qwen2.5-VL-7B ViT + LLM prefill -> 4 latent tokens), "
                            "32 frames (392x392 -> 784 patches -> 196 tokens) x 80-token instruction + 24 template tokens + "
                            "4 latent queries = 304 tokens per env, bf16"),
    "nextdit_traj": dict(kind="nextdit", B=64, Ns=32, T=32, K=10,
                         desc="NextDiT System 1 (system1 = nextdit_async, the released DualVLN head): 64 envs x 32 trajectories "
                              "of horizon 32, condition tokens (DINOv2 ViT-S on 2 frames + MemoryEncoder + QFormer + latent "
                              "projection) + 10 flow-matching Euler steps of the 12-block trajectory DiT, guidance 1.0, bf16"),
    "ddp_train": dict(kind="train", B=32, f=6, S=304, grid=(1, 28, 28), T=32, K=20, Ns=1,
                      desc="configs[4]: InternVLA-N1 DDP training step (navdp_async branch), 32 episodes per GPU (global "
                           "batch 256 on 8 GPUs), S = 304 tokens (1 frame 392x392 + 104 text + 4 TRAJ), f = 6 selected "
                           "frames per episode (192 [goal, current] RGB-D pairs), frozen 7B System 2, trainable System 1 + "
                           "latent_queries, bucketed NCCL all-reduce of 76.8 M fp32 gradients overlapped with the System-2 "
                           "backward, fused AdamW; dropout off (see train_step.py)"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return dict(hbm=d.get("hbm_gbs", 6650.0), tf=d.get("bf16_tflops", 1590.0),
                    tf_sustained=d.get("bf16_tflops_sustained", 1400.0), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.25)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


MIN_WARMUP = int(os.environ.get("N1_BENCH_MIN_WARMUP", "3"))  # profiling runs under ncu lower this; timed runs keep >= 3


def host_threads():
    """Usable host cores: the cgroup CPU quota when there is one (a 128-core box may grant far fewer), else affinity."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            q, per = fh.read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def denoise_flops_per_sample_step(T, D=384, M=34, Ns=32, layers=16):
    # SURVEY.md §8d: decoder layer = 28 T D^2 + 4 M D^2 / Ns + 4 T^2 D + 4 T M D  (memory K/V once per env)
    return layers * (28 * T * D * D + 4 * M * D * D / Ns + 4 * T * T * D + 4 * T * M * D)


def dual_flops_per_env(wl):
    """Algorithmic FLOPs of one dual-system policy step (SURVEY.md §8d): ViT + LLM prefill + RGB-D encoder + denoiser."""
    S, n_p = wl["S"], wl["grid"][0] * wl["grid"][1] * wl["grid"][2]
    H, I, L = 3584, 18944, 28
    llm = L * (2 * S * H * (H + 2 * 512) + 2 * S * H * H + 6 * S * H * I + 4 * S * S * H / 2)
    Hv, Iv = 1280, 3420
    vit = 2 * n_p * 1176 * Hv + 32 * (2 * n_p * Hv * 3 * Hv + 2 * n_p * Hv * Hv + 6 * n_p * Hv * Iv) \
        + 2 * (n_p / 4) * 5120 * (5120 + 3584)
    D = 384
    vits = 4 * (12 * (24 * 257 * D * D + 4 * 257 * 257 * D) + 2 * 256 * 588 * D)
    den = denoise_flops_per_sample_step(wl["T"]) * wl["Ns"] * wl["K"]
    return dict(llm=llm, vit=vit, rgbd=vits, denoise=den, total=llm + vit + vits + den)


def _gemm_classes(shapes, wl, world_B):
    """Group the event-timed GEMM launches of one step by stage.  Rule: by the contraction / output widths of the model
    (decoder 3584 / 18944, vision tower 1280 / 3420 / 5120 / 1176, System 1 384-wide)."""
    def cls(sh):
        M, N, K = sh["M"], abs(sh["N"]), sh["K"]
        if N == 896 and K == 3584:
            return "s1_other"
        if K in (3584, 18944) or N in (3584, 37888, 4608) and K == 3584:
            return "llm"
        if K in (1280, 1176, 1184, 3424, 5120) or N in (1280, 3840, 6848, 5120):
            return "vit"
        if M == world_B * wl.get("Ns", 32) * wl.get("T", 32):
            return "denoiser"
        return "s1_other"
    out = {}
    for sh in shapes:
        c = out.setdefault(cls(sh), {"launches": 0, "ms": 0.0, "tflop": 0.0})
        fl = (4.0 if sh["N"] < 0 else 2.0) * sh["M"] * abs(sh["N"]) * sh["K"] * sh["count"]
        c["launches"] += sh["count"]
        c["ms"] += sh["ms"]
        c["tflop"] += fl / 1e12
    return out


def _traffic_table():
    """ncu dram__bytes_read.sum + dram__bytes_write.sum per launch of named GEMM shapes, from committed captures
    (profiles/r2_gemm_traffic.json: {"MxNxK": {"bytes": ..., "source": "profiles/..."}}); absent -> traffic null."""
    p = os.path.join(ROOT, "profiles", "r2_gemm_traffic.json")
    if os.path.exists(p):
        with open(p) as fh:
            return json.load(fh)
    return {}


def build_dual(dev, wl, rank):
    """Random-init InternVLA-N1 (Qwen2.5-VL-7B shapes + NavDP) and one step's synthetic inputs."""
    import numpy as np
    from internnav_b200.internvla_n1 import InternVLAN1ForCausalLM
    from internnav_b200.manifest import random_navdp_state_dict, random_s2_state_dict
    from internnav_b200.qwen import QWEN25VL_7B
    model = InternVLAN1ForCausalLM(QWEN25VL_7B, device=str(dev))
    model.load_parts(random_s2_state_dict(QWEN25VL_7B, seed=0, device=str(dev)), random_navdp_state_dict(seed=0))
    torch.cuda.empty_cache()
    B, S = wl["B"], wl["S"]
    t, h, w = wl["grid"]
    n_tok = t * h * w // 4
    rng = np.random.Generator(np.random.PCG64(77 + rank))
    n_text = S - 4 - n_tok - 2
    prompts = []
    for _ in range(B):
        pre = rng.integers(0, 151643, 12).tolist()
        post = rng.integers(0, 151643, n_text - 12).tolist()
        prompts.append(pre + [151652] + [151655] * n_tok + [151653] + post)
    g = torch.Generator(device="cpu").manual_seed(99 + rank)
    host = dict(
        pixels=torch.randn(B * t * h * w, 1176, generator=g).bfloat16().pin_memory(),
        rgb=torch.rand(B, 2, 224, 224, 3, generator=g).pin_memory(),
        depth=(torch.rand(B, 2, 224, 224, 1, generator=g) * 5.0).pin_memory(),
        x0=torch.randn(B * wl["Ns"], wl["T"], 3, generator=g).pin_memory(),
        nz=torch.randn(wl["K"] - 1, B * wl["Ns"], wl["T"], 3, generator=g).pin_memory())
    grids = [list(wl["grid"])] * B
    return model, prompts, grids, host


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args, wl):
    if wl["kind"] == "dual":
        return run_ours_dual(args, wl)
    if wl["kind"] == "s2":
        return run_ours_s2(args, wl)
    if wl["kind"] == "train":
        return run_ours_train(args, wl)
    if wl["kind"] == "nextdit":
        return run_ours_nextdit(args, wl)
    return run_ours_denoise(args, wl)


def _finish(args, wl, world, rank, dev, ms, ms_e2e, launches, clocks, prof, B, extra_cfg, e2e_info, algo_flops_step,
            unit="policy-steps/s", metric="InternVLA-N1 policy-steps/sec (batch RGB-D+text->action)", extra_top=None,
            shapes=None, stage_ms=None):
    import torch.distributed as dist
    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    ms_per_step = ms / args.steps
    value = world * B * args.steps / (ms / 1e3)
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    pk = peaks()
    achieved_tf = prof["gemm_flops"] / (prof["gemm_ms"] * 1e-3) / 1e12 if prof["gemm_ms"] > 0 else 0.0
    peak = pk["tf_sustained"] if ms_per_step > 50 else pk["tf"]
    cfg = {"workload": args.workload, "description": wl["desc"], "envs_per_gpu": B, "parallelism": "env-sharded x%d" % world,
           "l2": "flushed (256 MiB memset) between timed steps", "algorithmic_tflop_per_step": algo_flops_step / 1e12,
           "step_tflops_achieved": algo_flops_step / (ms_per_step * 1e-3) / 1e12}
    cfg.update(extra_cfg)
    e2e = {"value": e2e_value, "unit": unit}
    e2e.update(e2e_info)
    out = {
        "metric": metric, "value": value, "unit": unit,
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, MIN_WARMUP), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "impl": "ours", "config": cfg, "e2e": e2e, "gpu_launches": int(launches["total_launches"]), "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "n1::gemm_kernel<BN> (tcgen05, all GEMM launches of one step)",
                     "achieved": achieved_tf, "peak": peak, "unit": "TFLOP/s", "frac": achieved_tf / peak,
                     "traffic": None, "peak_source": pk["src"] + (" sustained" if ms_per_step > 50 else " burst"),
                     "gemm_launches_per_step": int(prof["gemm_launches"]), "gemm_ms_per_step": prof["gemm_ms"],
                     "gemm_share_of_step": prof["gemm_ms"] / ms_per_step},
    }
    if shapes:
        # the single dominant kernel launch shape of the step (by summed time) carries the headline roofline entry; the
        # family sum stays as `gemm_family`; `roofline_classes` gives TFLOP / ms / fraction per stage
        dom = max(shapes, key=lambda sh: sh["ms"])
        fl = (4.0 if dom["N"] < 0 else 2.0) * dom["M"] * abs(dom["N"]) * dom["K"]
        per_ms = dom["ms"] / dom["count"]
        key = "%dx%dx%d" % (dom["M"], abs(dom["N"]), dom["K"])
        tr = _traffic_table().get(key)
        fam = dict(out["roofline"])
        a_tf = fl / (per_ms * 1e-3) / 1e12
        pk1 = pk["tf"]   # a single launch is short: the burst figure is the denominator
        out["roofline"] = {"bound": "tensor", "kernel": "n1::gemm_kernel<BN,CM> (tcgen05) M x N x K = %s, %d launches per step"
                                                         % (key, dom["count"]),
                           "achieved": a_tf, "peak": pk1, "unit": "TFLOP/s", "frac": a_tf / pk1,
                           "traffic": tr["bytes"] if tr else None, "traffic_source": tr["source"] if tr else None,
                           "algorithmic_bytes": 2.0 * (dom["M"] * dom["K"] + abs(dom["N"]) * dom["K"] + dom["M"] * abs(dom["N"])
                                                       // (2 if abs(dom["N"]) == 37888 else 1)),
                           "us_per_launch": per_ms * 1e3, "ms_per_step": dom["ms"],
                           "peak_source": pk["src"] + " burst (single launch)", "gemm_family": fam}
        cl = _gemm_classes(shapes, wl, B)
        for c in cl.values():
            c["tflops"] = c["tflop"] / (c["ms"] * 1e-3) if c["ms"] > 0 else 0.0
            c["frac_of_sustained_peak"] = c["tflops"] / pk["tf_sustained"]
        out["roofline_classes"] = cl
    if stage_ms:
        out["stage_ms"] = stage_ms
    if extra_top:
        out.update(extra_top)
    if rank == 0:
        if world == 1 and not args.no_eager_baseline and wl["kind"] == "dual":
            # same-GPU, same-batch PyTorch-eager baseline (cuBLAS + SDPA), measured after our arm in this process:
            # separates "batching" from "kernels" in the speed-up (north_star's >= 10x is against eager)
            try:
                out["gpu_eager_baseline"] = eager_gpu_measure(wl, B, 2, 1, dev)
                out["gpu_eager_baseline"]["ours_over_eager"] = value / out["gpu_eager_baseline"]["value"]
            except Exception as e:  # noqa: BLE001  (the baseline leg must never cost us the bench line)
                out["gpu_eager_baseline"] = {"unavailable": repr(e)[:200]}
        if world == 1 and not args.no_cpu_baseline and wl["kind"] in ("dual", "denoise"):
            out["cpu_baseline"] = cpu_baseline(wl, budget_s=20.0)
        emit(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _timing_tools(dev, world):
    import torch.distributed as dist
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, use_events=True):
        tot = 0.0
        for _ in range(steps):
            flush.zero_()
            if use_events:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                b.synchronize()
                tot += a.elapsed_time(b)
            else:  # includes host work (D2H + numpy tail): wall clock around a synchronised region
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                tot += (time.perf_counter() - t0) * 1e3
        return tot
    return barrier, timed


def _keep_last(fn, box):
    """`fn` for a timed loop, keeping what its last call returned in box["out"] (--dump-outputs)."""
    def step():
        box["out"] = fn()
    return step


def dump_outputs(args, rank, name, out):
    """--dump-outputs DIR: the output of the last timed step as DIR/<name>.npy in float32, on rank 0.  The inputs are
    seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    if not args.dump_outputs or rank != 0:
        return
    a = out.detach().float().cpu().numpy()
    assert a.nbytes <= 64 << 20, (name, a.shape)
    os.makedirs(args.dump_outputs, exist_ok=True)
    np.save(os.path.join(args.dump_outputs, name + ".npy"), a)


def run_ours_dual(args, wl):
    import torch.distributed as dist
    from internnav_b200 import _lib
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a B200: there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model, prompts, grids, host = build_dual(dev, wl, rank)
    B = wl["B"]
    d = {k: v.to(dev) for k, v in host.items()}
    barrier, timed = _timing_tools(dev, world)
    # deployment never sees the same prompts twice: 32 rotating prompt batches (the plan cache holds 8), so every step --
    # timed or not -- builds its integer plan (mRoPE ids, splice map, cu_seqlens, RoPE table) inside the step
    sets = _prompt_sets(wl, rank, 32)
    it = [0]

    def next_prompts():
        it[0] += 1
        return sets[it[0] % len(sets)]

    def step_resident():
        lat = model.generate_latents(next_prompts(), d["pixels"], grids)
        return model.generate_traj(lat, d["rgb"], d["depth"], x_init=d["x0"], step_noise=d["nz"])

    def step_e2e():
        h2d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        return model.dual_system_step(next_prompts(), h2d["pixels"], grids, h2d["rgb"], h2d["depth"], x_init=h2d["x0"],
                                      step_noise=h2d["nz"])[1]

    for _ in range(max(args.warmup, MIN_WARMUP)):
        step_resident()
    _lib.prof_read()
    barrier()
    last = {}
    with ClockSampler(local) as clk:
        ms = timed(_keep_last(step_resident, last), args.steps)
    barrier()
    launches = _lib.prof_read()
    launches["total_launches"] //= max(args.steps, 1)
    clocks = clk.summary()
    dump_outputs(args, rank, "trajectories", last["out"])
    step_e2e()
    barrier()
    ms_e2e = timed(step_e2e, args.steps, use_events=False)
    barrier()
    _lib.prof_read()
    _lib.prof_read_shapes()
    _lib.prof_enable(True)
    step_resident()
    torch.cuda.synchronize()
    prof = _lib.prof_read()
    shapes = _lib.prof_read_shapes()
    _lib.prof_enable(False)
    # stage times of one step (CUDA events between the public calls; untimed pass)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    nav = model.model.navdp
    ev[0].record()
    feats = model._s2.visual(d["pixels"], grids)
    ev[1].record()
    lat = model._s2.prefill_latents(next_prompts(), feats, grids)
    ev[2].record()
    goal, rgbd = nav.goal_embed(lat), nav.rgbd_encoder(d["rgb"], d["depth"])
    ev[3].record()
    nav.sample(goal, rgbd, d["x0"], d["nz"])
    ev[4].record()
    torch.cuda.synchronize()
    stage_ms = {"s2_vision_tower": ev[0].elapsed_time(ev[1]), "s2_plan_and_llm_prefill": ev[1].elapsed_time(ev[2]),
                "s1_goal_and_rgbd_encoder": ev[2].elapsed_time(ev[3]), "s1_denoiser_20_steps": ev[3].elapsed_time(ev[4])}
    fl = dual_flops_per_env(wl)
    fl_stage = {"s2_vision_tower": fl["vit"] * B, "s2_plan_and_llm_prefill": fl["llm"] * B,
                "s1_goal_and_rgbd_encoder": fl["rgbd"] * B, "s1_denoiser_20_steps": fl["denoise"] * B}
    stage_ms = {k: {"ms": v, "algorithmic_tflop": fl_stage[k] / 1e12, "tflops": fl_stage[k] / (v * 1e-3) / 1e12,
                    "frac_of_sustained_peak": fl_stage[k] / (v * 1e-3) / 1e12 / peaks()["tf_sustained"]}
                for k, v in stage_ms.items()}
    _finish(args, wl, world, rank, dev, ms, ms_e2e, launches, clocks, prof, B,
            {"seq_len": wl["S"], "patches_per_env": wl["grid"][1] * wl["grid"][2], "samples_per_env": wl["Ns"],
             "horizon": wl["T"], "ddpm_steps": wl["K"], "weights": "random-init Qwen2.5-VL-7B shapes + NavDP (bf16)",
             "tflop_per_env": {k: v / 1e12 for k, v in fl.items()}, "launches_are": "per step",
             "prompts": "a different prompt batch every step (32 rotating sets, plan cache of 8): plan creation is inside "
                        "the timed region of both `value` and `e2e`"},
            {"h2d_bytes_per_step": sum(x.numel() * x.element_size() for x in host.values()),
             "d2h_bytes_per_step": B * 65 * 4,
             "api": "InternVLAN1ForCausalLM.dual_system_step (generate_latents + generate_traj + device action tail "
                    "n1_traj_to_actions; D2H = the action ids), pinned host inputs"},
            fl["total"] * B, shapes=shapes, stage_ms=stage_ms)


def _prompt_sets(wl, rank, n_sets):
    """`n_sets` different prompt batches (fresh instruction tokens): deployment never sees the same prompts twice, so the
    integer plan (mRoPE ids, splice map, cu_seqlens) is rebuilt inside every timed step."""
    import numpy as np
    B, S = wl["B"], wl["S"]
    t, h, w = wl["grid"]
    n_tok = t * h * w // 4
    n_text = S - 4 - n_tok - 2
    sets = []
    for k in range(n_sets):
        rng = np.random.Generator(np.random.PCG64([77 + rank, k]))
        prompts = []
        for _ in range(B):
            pre = rng.integers(0, 151643, 12).tolist()
            post = rng.integers(0, 151643, n_text - 12).tolist()
            prompts.append(pre + [151652] + [151655] * n_tok + [151653] + post)
        sets.append(prompts)
    return sets


def run_ours_s2(args, wl):
    """configs[2]: System-2 forward only (ViT + LLM prefill -> latents)."""
    import torch.distributed as dist
    from internnav_b200 import _lib
    from internnav_b200.manifest import random_s2_state_dict
    from internnav_b200.qwen import QWEN25VL_7B, System2
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a B200: there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    s2 = System2(QWEN25VL_7B, device=str(dev))
    s2.load_state_dict(random_s2_state_dict(QWEN25VL_7B, seed=0, device=str(dev)))
    torch.cuda.empty_cache()
    B = wl["B"]
    t, h, w = wl["grid"]
    sets = _prompt_sets(wl, rank, 8)
    grids = [list(wl["grid"])] * B
    g = torch.Generator(device="cpu").manual_seed(99 + rank)
    h_px = torch.randn(B * t * h * w, 1176, generator=g).bfloat16().pin_memory()
    d_px = h_px.to(dev)
    barrier, timed = _timing_tools(dev, world)
    it = [0]

    def step_resident():
        it[0] += 1
        return s2.generate_latents(sets[it[0] % len(sets)], d_px, grids)

    def step_e2e():
        it[0] += 1
        return s2.generate_latents(sets[it[0] % len(sets)], h_px.to(dev, non_blocking=True), grids).float().cpu()

    for _ in range(max(args.warmup, MIN_WARMUP)):
        step_resident()
    _lib.prof_read()
    barrier()
    last = {}
    with ClockSampler(local) as clk:
        ms = timed(_keep_last(step_resident, last), args.steps)
    barrier()
    launches = _lib.prof_read()
    launches["total_launches"] //= max(args.steps, 1)
    clocks = clk.summary()
    dump_outputs(args, rank, "latents", last["out"])
    step_e2e()
    barrier()
    ms_e2e = timed(step_e2e, args.steps, use_events=False)
    barrier()
    _lib.prof_read()
    _lib.prof_enable(True)
    step_resident()
    torch.cuda.synchronize()
    prof = _lib.prof_read()
    _lib.prof_enable(False)
    fl = dual_flops_per_env(dict(wl, T=32, Ns=32, K=20))
    _finish(args, wl, world, rank, dev, ms, ms_e2e, launches, clocks, prof, B,
            {"seq_len": wl["S"], "patches_per_env": h * w, "weights": "random-init Qwen2.5-VL-7B shapes (bf16)",
             "prompts": "a different prompt batch every step (8 rotating sets): plan creation is inside the timed region",
             "tflop_per_env": {"llm": fl["llm"] / 1e12, "vit": fl["vit"] / 1e12}, "launches_are": "per step"},
            {"h2d_bytes_per_step": h_px.numel() * 2, "d2h_bytes_per_step": B * 4 * 3584 * 4,
             "api": "System2.generate_latents (= InternVLAN1ForCausalLM.generate_latents), pinned host pixel_values"},
            (fl["llm"] + fl["vit"]) * B, unit="frames/s",
            metric="InternVLA-N1 System-2 forward (ViT + LLM prefill -> latents), frames/sec")


def _train_batches(wl, rank, n_sets):
    """Collated training batches (internnav_b200.training.collate_traj_batch layout) in pinned host memory."""
    B, f, T = wl["B"], wl["f"], wl["T"]
    t, h, w = wl["grid"]
    sets = _prompt_sets(wl, rank, n_sets)
    out = []
    for k, prompts in enumerate(sets):
        g = torch.Generator(device="cpu").manual_seed(1000 * rank + k)
        ids = torch.tensor([p + [151667] * 4 for p in prompts])
        batch = dict(input_ids=ids, labels=torch.full_like(ids, -100), attention_mask=torch.ones_like(ids, dtype=torch.bool),
                     t_s_pos=[len(p) for p in prompts],
                     pixel_values=torch.randn(B * t * h * w, 1176, generator=g).bfloat16().pin_memory(),
                     image_grid_thw=torch.tensor([list(wl["grid"])] * B),
                     traj_images=torch.rand(B, f, 224, 224, 3, generator=g).pin_memory(),
                     traj_depths=(torch.rand(B, f, 224, 224, generator=g) * 5.0).pin_memory(),
                     traj_poses=(torch.randn(B, f, T, 3, generator=g) * 0.5).pin_memory(),
                     video_frame_num=torch.randint(1, f + 1, (B,), generator=g))
        noise = torch.randn(B * f, T, 3, generator=g).pin_memory()
        ts = torch.randint(0, wl["K"], (B * f,), generator=g)
        out.append((batch, noise, ts))
    return out


def run_ours_train(args, wl):
    """configs[4]: one data-parallel training step per "step" (forward, backward, bucketed all-reduce, AdamW)."""
    import torch.distributed as dist
    from internnav_b200 import _lib
    from internnav_b200.internvla_n1 import InternVLAN1ForCausalLM
    from internnav_b200.manifest import random_navdp_state_dict, random_s2_state_dict
    from internnav_b200.qwen import QWEN25VL_7B
    from internnav_b200.train_step import DualSystemTrainer
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a B200: there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model = InternVLAN1ForCausalLM(QWEN25VL_7B, device=str(dev))
    s2_sd = random_s2_state_dict(QWEN25VL_7B, seed=0, device=str(dev))
    s1_sd = random_navdp_state_dict(seed=0)           # same seed on every rank: replicas start identical, as DDP requires
    model.load_parts(s2_sd, s1_sd)
    latent = s2_sd["model.latent_queries"].float()
    del s2_sd
    torch.cuda.empty_cache()
    tr = DualSystemTrainer(model, s1_sd, latent, lr=1e-4, weight_decay=0.0, max_grad_norm=1.0,
                           graph_s1=os.environ.get("N1_TRAIN_GRAPH", "1") != "0")
    B, f = wl["B"], wl["f"]
    sets = _train_batches(wl, rank, 3)
    barrier, timed = _timing_tools(dev, world)
    it = [0]
    exch = []

    def to_dev(batch):
        return {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) and k not in ("input_ids", "attention_mask", "labels",
                                                                                     "video_frame_num", "image_grid_thw") else v)
                for k, v in batch.items()}

    resident = [(to_dev(b), n.to(dev), t.to(dev)) for b, n, t in sets]

    def step_resident():
        it[0] += 1
        b, n, t = resident[it[0] % len(resident)]
        loss = tr.step(b, n, t)
        if world > 1:
            exch.append(tr.exchange_ms())
        return loss

    def step_e2e():
        it[0] += 1
        b, n, t = sets[it[0] % len(sets)]
        return float(tr.step(to_dev(b), n.to(dev, non_blocking=True), t.to(dev, non_blocking=True)))   # D2H of the loss

    for _ in range(max(args.warmup, MIN_WARMUP)):
        step_resident()
    _lib.prof_read()
    exch.clear()
    barrier()
    last = {}
    with ClockSampler(local) as clk:
        ms = timed(_keep_last(step_resident, last), args.steps)
    barrier()
    launches = _lib.prof_read()
    launches["total_launches"] //= max(args.steps, 1)
    clocks = clk.summary()
    dump_outputs(args, rank, "loss", last["out"])
    exch_t = [e for e in exch if e]
    step_e2e()
    barrier()
    ms_e2e = timed(step_e2e, args.steps, use_events=False)
    barrier()
    _lib.prof_read()
    _lib.prof_enable(True)
    step_resident()
    torch.cuda.synchronize()
    prof = _lib.prof_read()
    _lib.prof_enable(False)
    # phase breakdown of one step: device time (CUDA events) next to the host wall clock of the same step -- the System-1
    # schedule is driven from Python (one ctypes call per kernel), so a wall clock well above the device time = host-bound
    tr.profile_phases = True
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step_resident()
    t_issue = (time.perf_counter() - t0) * 1e3
    torch.cuda.synchronize()
    t_wall = (time.perf_counter() - t0) * 1e3
    phases = tr.phase_ms()
    tr.profile_phases = False
    if phases is not None:
        phases["host_issue_ms"] = t_issue
        phases["wall_ms"] = t_wall
    fl = dual_flops_per_env(dict(wl, Ns=32))
    D = 384
    vit_s = 12 * (24 * 257 * D * D + 4 * 257 * 257 * D) + 2 * 256 * 588 * D
    s1 = B * f * 2 * vit_s * (1 + 3) + 3 * B * f * denoise_flops_per_sample_step(wl["T"], Ns=1)   # RGB fwd + depth fwd/bwd; decoder fwd/bwd
    algo = (fl["llm"] + fl["vit"]) * B + s1
    n_grad = sum(g.numel() for g in tr.buckets.grads.values())
    allreduce = None
    if exch_t:
        allreduce = {"collective": "NCCL all-reduce (SUM of pre-divided fp32 buckets), torch.distributed",
                     "buckets": [int(b.numel()) * 4 for b in tr.buckets.buffers], "bytes_per_step": n_grad * 4,
                     "exposed_ms_per_step": sum(e["exposed_ms"] for e in exch_t) / len(exch_t),
                     "overlapped_launch_ms_per_step": sum(e["overlapped_launch_ms"] for e in exch_t) / len(exch_t),
                     "s2_backward_window_ms": sum(e["s2_backward_window_ms"] for e in exch_t) / len(exch_t),
                     "note": "all buckets but the one holding latent_queries are in flight during the System-2 backward; "
                             "exposed = end of that backward -> last bucket reduced (CUDA events, rank 0)"}
    host = sets[0]
    h2d = sum(v.numel() * v.element_size() for k, v in host[0].items()
              if torch.is_tensor(v) and k in ("pixel_values", "traj_images", "traj_depths", "traj_poses")) + host[1].numel() * 4
    _finish(args, wl, world, rank, dev, ms, ms_e2e, launches, clocks, prof, B,
            {"seq_len": wl["S"], "frames_per_episode": f, "global_batch": world * B, "trainable_params": n_grad,
             "optimizer": "fused AdamW (fp32 masters), max_grad_norm 1.0, dropout off", "launches_are": "per step",
             "s1_launch_mode": "CUDA graph replay" if tr.graph_s1 else "eager (one ctypes call per kernel)",
             "weights": "random-init Qwen2.5-VL-7B shapes (frozen) + NavDP (trainable)",
             "prompts": "3 rotating batches with different prompts: plan creation inside the timed region"},
            {"h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
             "api": "DualSystemTrainer.step(collated batch, noise, timesteps) -> loss; pinned host batch"},
            algo, unit="episodes/s", metric="InternVLA-N1 DDP training step, episodes/sec",
            extra_top={"allreduce": allreduce, "phase_ms": phases})


def run_ours_denoise(args, wl):
    import torch.distributed as dist
    from internnav_b200 import _lib
    from internnav_b200.manifest import random_navdp_state_dict
    from internnav_b200.navdp import NavDP_Policy_DPT_CriticSum_DAT
    from internnav_b200.postprocess import batched_traj_to_actions

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a B200: there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, Ns, T, K = wl["B"], wl["Ns"], wl["T"], wl["K"]

    model = NavDP_Policy_DPT_CriticSum_DAT(memory_size=2, predict_size=32, navdp_version=0.1, device=str(dev))
    model.load_state_dict(random_navdp_state_dict(seed=0))
    g = torch.Generator(device="cpu").manual_seed(1234 + rank)
    R = B * Ns
    # host-side (pinned) inputs of one step, as the caller of the policy holds them
    h_goal = torch.randn(B, 1, 384, generator=g).bfloat16().pin_memory()
    h_rgbd = torch.randn(B, 32, 384, generator=g).bfloat16().pin_memory()
    h_x0 = torch.randn(R, T, 3, generator=g).pin_memory()
    h_nz = torch.randn(K - 1, R, T, 3, generator=g).pin_memory()
    d_goal, d_rgbd, d_x0, d_nz = (t.to(dev) for t in (h_goal, h_rgbd, h_x0, h_nz))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_resident():
        return model.sample(d_goal, d_rgbd, d_x0, d_nz, num_steps=K)

    def step_e2e():
        goal = h_goal.to(dev, non_blocking=True)
        rgbd = h_rgbd.to(dev, non_blocking=True)
        x0 = h_x0.to(dev, non_blocking=True)
        nz = h_nz.to(dev, non_blocking=True)
        traj = model.sample(goal, rgbd, x0, nz, num_steps=K)
        return batched_traj_to_actions(traj, B)  # D2H of the trajectories + the integer tail

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, use_events=True):
        tot = 0.0
        for _ in range(steps):
            flush.zero_()
            if use_events:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                b.synchronize()
                tot += a.elapsed_time(b)
            else:  # includes host work (D2H + numpy tail): wall clock around a synchronised region
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                tot += (time.perf_counter() - t0) * 1e3
        return tot

    for _ in range(max(args.warmup, MIN_WARMUP)):
        step_resident()
    _lib.prof_read()
    barrier()
    last = {}
    with ClockSampler(local) as clk:
        ms = timed(_keep_last(step_resident, last), args.steps)
    barrier()
    launches = _lib.prof_read()
    clocks = clk.summary()
    dump_outputs(args, rank, "trajectories", last["out"])
    for _ in range(2):
        step_e2e()
    barrier()
    ms_e2e = timed(step_e2e, args.steps, use_events=False)
    barrier()

    # roofline pass for the dominant kernel (tcgen05 GEMM): per-launch CUDA events, NOT part of the timed runs above;
    # eager launches here (the timed runs replay the same launch sequence from a CUDA graph)
    _lib.prof_read()
    _lib.prof_enable(True)
    model.sample(d_goal, d_rgbd, d_x0, d_nz, num_steps=K, graph=False)
    torch.cuda.synchronize()
    prof = _lib.prof_read()
    _lib.prof_enable(False)

    launches["total_launches"] //= max(args.steps, 1)
    _finish(args, wl, world, rank, dev, ms, ms_e2e, launches, clocks, prof, B,
            {"samples_per_env": Ns, "launch_mode": "CUDA graph replay of the K-step loop (eager for the roofline pass)", "horizon": T, "ddpm_steps": K, "weights": "random-init NavDP (98.8M params)",
             "launches_are": "per step"},
            {"h2d_bytes_per_step": sum(x.numel() * x.element_size() for x in (h_goal, h_rgbd, h_x0, h_nz)),
             "d2h_bytes_per_step": B * 65 * 4,
             "api": "NavDP_Policy_DPT_CriticSum_DAT.sample + batched_traj_to_actions (device action tail), pinned host inputs"},
            denoise_flops_per_sample_step(T) * R * K)


def nextdit_flops(B, Ns, T, steps, halves=1):
    """Matrix-product + attention FLOPs of one NextDiT call: condition tokens per environment + sampler per trajectory row."""
    D, L, F = 384, 768, 1024
    vit = 2 * 257 * (12 * (4 * D * D + 8 * D * D) + 588 * D) + 12 * 4 * 257 * 257 * D
    mem = 3 * (512 * 2 * (4 * D * D + 2 * D * 2048) + 4 * 512 * 512 * D)
    qf = 3 * (32 * 2 * (4 * L * L + 2 * L * 2048 + 2 * L * L) + 512 * 2 * 2 * L * L + 4 * 32 * 32 * L + 4 * 32 * 512 * L)
    cond = 2 * vit + mem + qf + 4 * 2 * (3584 * L + L * L)
    row = 12 * 2 * (5 * D * D + 3 * D * F) + 12 * (4 * T * D + 4 * 36 * D)      # per trajectory token and evaluation
    return B * cond + halves * B * Ns * T * steps * row


def run_ours_nextdit(args, wl):
    import torch.distributed as dist
    from internnav_b200 import _lib
    from internnav_b200.manifest import random_nextdit_state_dict
    from internnav_b200.nextdit import NextDiTSystem1
    from internnav_b200.postprocess import batched_traj_to_actions

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a B200: there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, Ns, T, K = wl["B"], wl["Ns"], wl["T"], wl["K"]
    model = NextDiTSystem1(device=str(dev), num_inference_steps=K).load_state_dict(random_nextdit_state_dict(0))
    g = torch.Generator(device="cpu").manual_seed(99 + rank)
    h_lat = torch.randn(B, 4, 3584, generator=g).bfloat16().pin_memory()
    h_img = torch.rand(B, 2, 224, 224, 3, generator=g).pin_memory()
    h_x0 = torch.randn(B * Ns, T, 3, generator=g).bfloat16().pin_memory()
    d_lat, d_img, d_x0 = (t.to(dev) for t in (h_lat, h_img, h_x0))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step_resident():
        return model.generate_traj(d_lat, d_img, None, T, 1.0, K, Ns, x_init=d_x0)

    def step_e2e():
        traj = model.generate_traj(h_lat.to(dev, non_blocking=True), h_img.to(dev, non_blocking=True), None, T, 1.0, K, Ns,
                                   x_init=h_x0.to(dev, non_blocking=True))
        return batched_traj_to_actions(traj.float(), B, max_actions=4)     # device action tail, D2H = the ids

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, use_events=True):
        tot = 0.0
        for _ in range(steps):
            flush.zero_()
            if use_events:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                b.synchronize()
                tot += a.elapsed_time(b)
            else:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                tot += (time.perf_counter() - t0) * 1e3
        return tot

    for _ in range(max(args.warmup, MIN_WARMUP)):     # also captures the sampler's CUDA graph (profiler off)
        step_resident()
    _lib.prof_read()
    barrier()
    last = {}
    with ClockSampler(local) as clk:
        ms = timed(_keep_last(step_resident, last), args.steps)
    barrier()
    launches = _lib.prof_read()
    clocks = clk.summary()
    dump_outputs(args, rank, "trajectories", last["out"])
    for _ in range(2):
        step_e2e()
    barrier()
    ms_e2e = timed(step_e2e, args.steps, use_events=False)
    barrier()
    _lib.prof_read()
    _lib.prof_enable(True)                             # roofline pass: eager launches with per-GEMM events, untimed
    model.sample(model.condition_tokens(d_lat, d_img), d_x0, 1.0, K, Ns, graph=False)
    torch.cuda.synchronize()
    prof = _lib.prof_read()
    _lib.prof_enable(False)
    launches["total_launches"] //= max(args.steps, 1)
    _finish(args, wl, world, rank, dev, ms, ms_e2e, launches, clocks, prof, B,
            {"samples_per_env": Ns, "horizon": T, "euler_steps": K, "guidance_scale": 1.0,
             "launch_mode": "condition tokens eager, sampler = CUDA graph replay (eager for the roofline pass)",
             "weights": "random-init NextDiT System 1 (91.4M params)", "launches_are": "per step"},
            {"h2d_bytes_per_step": sum(x.numel() * x.element_size() for x in (h_lat, h_img, h_x0)), "d2h_bytes_per_step": B * 65 * 4,
             "api": "NextDiTSystem1.generate_traj + batched_traj_to_actions (device action tail), pinned host inputs"},
            nextdit_flops(B, Ns, T, K))


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_baseline(wl, budget_s=20.0, threads=None):
    if wl["kind"] == "dual":
        return cpu_baseline_dual(wl, budget_s, threads)
    return cpu_baseline_denoise(wl, budget_s, threads)


class DualCpuSample:
    """Reference algorithm (oracle ports, fp32 eager PyTorch) on the host cores for ONE environment of the dual-system
    step, on a bounded sample: the 7B decoder and the 32-block ViT are timed at full width for 1 and 2 layers (the
    per-layer time is the difference, scaled to 28 / 32), the RGB-D encoder runs once in full, the denoiser runs 3 of its
    K steps.  Weights are built once; measure() can be repeated.  Nothing here is part of the GPU timing."""

    def __init__(self, wl, threads=None):
        from oracle import navdp_oracle as O, qwen_oracle as Q, weights
        import numpy as np
        self.O, self.Q, self.wl = O, Q, wl
        self.threads = threads or host_threads()
        torch.set_num_threads(self.threads)
        self.grids = [list(wl["grid"])]
        self.n_p = wl["grid"][0] * wl["grid"][1] * wl["grid"][2]
        self.s2 = {}
        for depth in (1, 2):
            cfg = dict(Q.QWEN25VL_7B)
            cfg.update(v_depth=depth, fullatt=[], layers=depth)
            self.s2[depth] = (cfg, Q.make_s2_state_dict(cfg, seed=0, vocab_rows=256))
        g = torch.Generator().manual_seed(0)
        self.px = torch.randn(self.n_p, 1176, generator=g)
        self.emb = torch.randn(1, wl["S"], 3584, generator=g)
        self.pos = torch.arange(wl["S"]).view(1, 1, -1).expand(3, 1, -1)
        self.sd1 = weights.make_state_dict(0)
        self.inp = weights.make_inputs(5, B=1, T=wl["T"], Ns=wl["Ns"], K=2)

    def measure(self):
        O, Q, wl = self.O, self.Q, self.wl

        def t_of(fn, reps=1):
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            return (time.perf_counter() - t0) / reps

        with torch.no_grad():
            tv, tl = {}, {}
            for depth, (cfg, sd) in self.s2.items():
                tv[depth] = t_of(lambda: Q.vit_forward(sd, cfg, self.px, self.grids))
                tl[depth] = t_of(lambda: Q.text_forward(sd, cfg, self.emb, self.pos))
            vit_s = tv[1] + 31 * max(tv[2] - tv[1], 0.0)
            llm_s = tl[1] + 27 * max(tl[2] - tl[1], 0.0)
            rgbd_s = t_of(lambda: O.rgbd_encoder(self.sd1, self.inp["rgb"], self.inp["depth"]))
            k = torch.tensor([3])
            n_den = 3
            den_s = t_of(lambda: O.predict_noise(self.sd1, self.inp["x_init"], k, self.inp["goal"], self.inp["rgbd"]),
                         reps=n_den) * wl["K"]
        total = vit_s + llm_s + rgbd_s + den_s
        return {"value": 1.0 / total, "unit": "policy-steps/s", "cores": self.threads, "kind": "port",
                "seconds_per_env": {"vit": vit_s, "llm": llm_s, "rgbd": rgbd_s, "denoise": den_s},
                "sample": "1 env, fp32 eager oracle: ViT/LLM timed at 1 and 2 layers of 7B width (S=%d, %d patches) and "
                          "scaled to 32/28 layers; RGB-D encoder in full; %d of %d denoise steps (32 traj x T=%d) scaled"
                          % (wl["S"], self.n_p, n_den, wl["K"], wl["T"])}


def cpu_baseline_dual(wl, budget_s=20.0, threads=None):
    s = DualCpuSample(wl, threads)
    s.measure()  # warm-up (page faults, thread pool)
    return s.measure()


def cpu_baseline_denoise(wl, budget_s=20.0, threads=None):
    """The reference algorithm (oracle port, fp32 PyTorch eager) on this box's host cores, on a bounded sample of the
    same workload: 1 environment (32 trajectories) for as many denoise steps as fit the budget, scaled linearly to K."""
    from oracle import navdp_oracle as O, weights
    threads = threads or host_threads()
    torch.set_num_threads(threads)
    sd = weights.make_state_dict(0)
    T, K, Ns = wl["T"], wl["K"], wl["Ns"]
    inp = weights.make_inputs(5, B=1, T=T, Ns=Ns, K=2)
    x, goal, rgbd = inp["x_init"], inp["goal"], inp["rgbd"]
    k = torch.tensor([3])
    with torch.no_grad():
        O.predict_noise(sd, x, k, goal, rgbd)  # warm-up
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < budget_s and n < K:
            O.predict_noise(sd, x, k, goal, rgbd)
            n += 1
        dt = time.perf_counter() - t0
    per_env_call = dt / n * K
    return {"value": 1.0 / per_env_call, "unit": "policy-steps/s", "cores": threads, "kind": "port",
            "sample": "%d denoise steps of 1 env x %d trajectories x T=%d (fp32 eager oracle), scaled to %d steps" % (n, Ns, T, K)}


def run_reference(args, wl):
    """--impl reference: the reference's algorithm on the box's host cores (CPU oracle port -- the reference is Python /
    PyTorch and /root/reference cannot travel to the GPU box), same workload, metric and unit; every "step" is one
    bounded sample (see cpu_baseline); the run stops early once ~4 minutes are spent and reports the steps it did."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    if wl["kind"] not in ("dual", "denoise"):
        emit({"impl": "reference", "unavailable": "the CPU reference arm is defined for the headline workloads "
                                                  "(dual_system, navdp_denoise); %s is a secondary workload" % args.workload})
        return
    t_start = time.perf_counter()
    vals, done_w = [], 0
    if wl["kind"] == "dual":
        sample = DualCpuSample(wl)
        fn = sample.measure
    else:
        total = max(args.steps + args.warmup, 1)
        per = max(4.0, min(20.0, 120.0 / total))
        fn = lambda: cpu_baseline_denoise(wl, budget_s=per)  # noqa: E731
    for i in range(args.warmup + args.steps):
        if vals and time.perf_counter() - t_start > 240:
            break
        r = fn()
        if i >= args.warmup:
            vals.append(r)
        else:
            done_w += 1
    if not vals:
        vals.append(fn())
    v = sum(x["value"] for x in vals) / len(vals)
    cb = dict(vals[-1])
    cb["value"] = v
    out = {"metric": "InternVLA-N1 policy-steps/sec (batch RGB-D+text->action)", "value": v, "unit": "policy-steps/s",
           "impl": "reference", "n_gpus": world, "steps": len(vals), "warmup": done_w,
           "ms_per_step": 1e3 * wl["B"] / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": args.workload, "description": wl["desc"],
                      "note": "reference algorithm on host cores (CPU oracle port; /root/reference is Python and cannot travel)"},
           "cpu_baseline": cb,
           "e2e": {"value": v, "unit": "policy-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


def eager_gpu_measure(wl, batch, steps, warmup, dev=None):
    """BASELINE, not the product: the reference algorithm as batched eager PyTorch on the GPU (oracle/eager_gpu.py: bf16,
    cuBLAS Linears, SDPA attention), `batch` environments per call, device-timed like our arm.  -> dict for the JSON line."""
    import numpy as np
    from internnav_b200.manifest import random_navdp_state_dict, random_s2_state_dict
    from oracle import eager_gpu as E, navdp_oracle as O, qwen_oracle as Q
    assert wl["kind"] == "dual", "the eager-GPU baseline is defined for the dual_system workload"
    dev = dev or torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = dict(Q.QWEN25VL_7B)
    sd2 = random_s2_state_dict(cfg, seed=0, device=str(dev))
    sd1 = {k: v.to(dev, torch.bfloat16) for k, v in random_navdp_state_dict(seed=0).items()}
    t, h, w = wl["grid"]
    B = batch
    sets = _prompt_sets(dict(wl, B=B), 0, 4)
    g = torch.Generator(device="cpu").manual_seed(99)
    px = torch.randn(B * t * h * w, 1176, generator=g).bfloat16().to(dev)
    rgb = torch.rand(B, 2, 224, 224, 3, generator=g).bfloat16().to(dev)
    dep = (torch.rand(B, 2, 224, 224, 1, generator=g) * 5).bfloat16().to(dev)
    x0 = torch.randn(B * wl["Ns"], wl["T"], 3, generator=g).bfloat16().to(dev)
    nz = torch.randn(wl["K"] - 1, B * wl["Ns"], wl["T"], 3, generator=g).bfloat16().to(dev)
    it = [0]

    def step():
        it[0] += 1
        ids = torch.tensor(sets[it[0] % len(sets)])
        traj = E.dual_system_step(sd2, sd1, cfg, ids, px, wl["grid"], rgb, dep, x0, nz, K=wl["K"])
        return [O.traj_to_actions(traj[b * wl["Ns"]:(b + 1) * wl["Ns"]].clone()) for b in range(B)]

    for _ in range(max(warmup, 1)):
        step()
    torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    tot = 0.0
    for _ in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step()
        torch.cuda.synchronize()
        tot += time.perf_counter() - t0
    dt = tot / steps
    del sd2, sd1
    torch.cuda.empty_cache()
    return {"value": B / dt, "unit": "policy-steps/s", "ms_per_step": dt * 1e3, "batch": B, "steps": steps,
            "what": "reference algorithm as batched eager PyTorch on this GPU: bf16, cuBLAS (F.linear) + "
                    "F.scaled_dot_product_attention, %d envs per call, wall clock incl. the numpy action tail "
                    "(oracle/eager_gpu.py; BASELINE, none of our kernels)" % B}


def run_eager_gpu(args, wl):
    """--impl eager [--batch B]: the same-GPU PyTorch-eager baseline (default B = the workload's batch, 64)."""
    B = args.batch or wl["B"]
    r = eager_gpu_measure(wl, B, args.steps, max(args.warmup, 1))
    out = {"metric": "InternVLA-N1 policy-steps/sec (batch RGB-D+text->action)", "value": r["value"], "unit": "policy-steps/s",
           "impl": "eager_gpu", "n_gpus": 1, "steps": r["steps"], "warmup": max(args.warmup, 1), "ms_per_step": r["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": args.workload, "batch": B, "note": r["what"]}}
    emit(out)


_OUT_FD = 1


def _claim_stdout():
    """Keep stdout for the JSON line alone: library chatter written to fd 1 (e.g. NCCL's version banner) goes to stderr."""
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(out):
    """The ONE JSON line, written straight to fd 1: a rank process that leaves through NCCL/CUDA teardown without running
    Python's stdio finalisation (seen under torchrun with stdout redirected to a file) must not lose it."""
    sys.stdout.flush()
    os.write(_OUT_FD, (json.dumps(out) + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager"])
    ap.add_argument("--workload", default="dual_system", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the same-GPU PyTorch-eager baseline leg (N = 1)")
    ap.add_argument("--batch", type=int, default=0, help="--impl eager: environments per call (default: the workload's)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the output of --impl ours")
    _claim_stdout()
    wl = WORKLOADS[args.workload]
    if args.impl == "eager":
        run_eager_gpu(args, wl)
    elif args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        if not isinstance(sys.exc_info()[1], SystemExit):
            import traceback
            traceback.print_exc()
            sys.stderr.flush()
            os._exit(1)
        raise
    sys.stdout.flush()
    sys.stderr.flush()

"""Cost of train-mode dropout in the System-1 training step: the `ddp_train` per-GPU shape of bench.py (32 episodes,
f = 6 frames, frozen 7B System 2, System 1 replayed from a CUDA graph) with a p = 0 and a p = 0.1 trainer in one
process, timed in alternating windows so that both see the same clocks and neighbours.

    python scripts/bench_train_dropout.py [--steps 10] [--windows 4] [--warmup 3] [--out FILE]

Prints one JSON line: ms/step (median over windows and all window means) per trainer, the overhead of p = 0.1, a phase
breakdown (DualSystemTrainer.phase_ms) and kernel launches per step for each, and the card name and power limit read in
the same run.  bench.py keeps its `ddp_train` workload at p = 0, so its numbers stay comparable.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--windows", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--p", type=float, default=0.1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_dropout needs a B200: there is no CPU path")
    import bench
    from internnav_b200 import _lib
    from internnav_b200.internvla_n1 import InternVLAN1ForCausalLM
    from internnav_b200.manifest import random_navdp_state_dict, random_s2_state_dict
    from internnav_b200.qwen import QWEN25VL_7B
    from internnav_b200.train_step import DualSystemTrainer

    wl = bench.WORKLOADS["ddp_train"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    model = InternVLAN1ForCausalLM(QWEN25VL_7B, device=str(dev))
    s2_sd = random_s2_state_dict(QWEN25VL_7B, seed=0, device=str(dev))
    s1_sd = random_navdp_state_dict(seed=0)
    model.load_parts(s2_sd, s1_sd)
    latent = s2_sd["model.latent_queries"].float()
    del s2_sd
    torch.cuda.empty_cache()
    trainers = {p: DualSystemTrainer(model, s1_sd, latent, lr=1e-4, weight_decay=0.0, max_grad_norm=1.0, graph_s1=True,
                                     dropout=p, dropout_seed=1)
                for p in (0.0, args.p)}

    def to_dev(batch):
        return {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) and k not in ("input_ids", "attention_mask", "labels",
                                                                                     "video_frame_num", "image_grid_thw") else v)
                for k, v in batch.items()}

    resident = [(to_dev(b), n.to(dev), t.to(dev)) for b, n, t in bench._train_batches(wl, 0, 3)]
    it = [0]

    def step(tr):
        it[0] += 1
        b, n, t = resident[it[0] % len(resident)]
        model._s2.set_latent_queries(tr.latent)     # the trainers share the System-2 handle
        return tr.step(b, n, t)

    for tr in trainers.values():
        for _ in range(args.warmup):
            step(tr)
    torch.cuda.synchronize()
    times = {p: [] for p in trainers}
    launches = {p: [] for p in trainers}
    for w in range(args.windows):
        order = list(trainers) if w % 2 == 0 else list(trainers)[::-1]
        for p in order:
            tr = trainers[p]
            _lib.prof_read()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step(tr)
            e1.record()
            e1.synchronize()
            times[p].append(e0.elapsed_time(e1) / args.steps)
            launches[p].append(_lib.prof_read()["total_launches"] / args.steps)
    phases = {}
    for p, tr in trainers.items():
        tr.profile_phases = True
        step(tr)
        phases[p] = tr.phase_ms()
        tr.profile_phases = False
    med = {p: sorted(v)[len(v) // 2] for p, v in times.items()}
    base = med[0.0]
    res = {"bench": "train_dropout", "workload": "ddp_train per GPU (B=32, f=6, graph_s1)", "card": card(),
           "steps_per_window": args.steps, "windows": args.windows,
           "ms_per_step": {str(p): round(m, 3) for p, m in med.items()},
           "window_ms": {str(p): [round(x, 3) for x in v] for p, v in times.items()},
           "overhead_pct": round(100.0 * (med[args.p] - base) / base, 2),
           "launches_per_step": {str(p): sum(v) / len(v) for p, v in launches.items()},
           "phase_ms": {str(p): {k: round(x, 3) for k, x in ph.items()} for p, ph in phases.items()}}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()

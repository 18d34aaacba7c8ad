"""One optimisation step of the dual-system training (SURVEY.md §8 row a13 / config 5), navdp_async branch:

    collated batch -> System-2 TRAJ states (frozen decoder, K/V cache)        s2_train.cu
                   -> System-1 forward + backward (trainable)                train_s1.py over bwd_kernels.cu
                   -> bucketed all-reduce of the System-1 gradients          ddp.py (NCCL), in flight while ...
                   -> d loss / d TRAJ states -> d latent_queries             s2_train.cu  ... this backward runs
                   -> all-reduce of the bucket holding latent_queries, global-norm clip, fused AdamW (fp32 masters)

replacing `Trainer.training_step` -> `InternVLAN1ForCausalLM.forward(...).loss.backward()` -> DDP -> optimizer of the
reference (internnav/trainer/internvla_n1_trainer.py L206-217; scripts/train/base_train/train.py).  The trainable set is
the reference's (internvla_n1_trainer.py L118-122): every System-1 tensor except the detached RGB ViT, plus
`latent_queries`.  Gradients are accumulated directly inside the all-reduce bucket buffers (ddp.GradientBuckets).

What of HF Trainer's step is reproduced: DDP averaging, gradient accumulation (`gradient_accumulation_steps`: the
exchange happens on the last micro-batch only, like DDP's no_sync), global-norm clipping after the exchange
(`max_grad_norm=1`, train_dual_system.sh), an LR-schedule hook (`lr_schedule(step) -> lr`; `warmup_cosine` below is the
Trainer's `cosine` with `warmup_ratio`), AdamW with decoupled decay, parameters without gradient untouched.

Dropout: the reference trains in train() mode, so p = 0.1 dropout is active on the cond / action embeddings (navdp.py
L305-307), in the 16 decoder layers and in the 2 Q-former layers (attention probabilities, the three residual branches, the
FF inner activation).  `DualSystemTrainer(..., dropout=0.1)` reproduces that: every site of internnav_b200/dropout.py runs
the dropout kernels, with masks drawn from Philox4x32-10 keyed by `dropout_seed` and counted by (site, data-parallel rank,
micro-batch step) -- the contract of csrc/dropout.cuh, restated in oracle/philox.py.  The masks cannot equal torch's RNG
stream; the parity tests inject the same masks into the oracle and into the reference module
(tests/golden/s1_training_dropout_reference.npz).  `dropout=0` (the default) is the reference's step with dropout off, and
issues exactly the kernels of a trainer without dropout.  The goal compressor (dropout 0.0), both DINOv2 ViTs and the frozen
System-2 decoder have no dropout.  There is no CPU path.
"""
import math
from collections import OrderedDict

import torch

from . import _bwd, _lib
from .ddp import GradientBuckets
from .dropout import DropoutRNG
from .train_s1 import GpuOps, S1TrainStep


def warmup_cosine(base_lr, total_steps, warmup_ratio=0.03, min_ratio=0.0):
    """transformers' `cosine` schedule with linear warm-up: lr(step) for step = 0, 1, ... (step = optimizer steps done)."""
    warm = int(math.ceil(total_steps * warmup_ratio))

    def lr(step):
        if step < warm:
            return base_lr * step / max(1, warm)
        p = (step - warm) / max(1, total_steps - warm)
        return base_lr * max(min_ratio, 0.5 * (1.0 + math.cos(math.pi * min(1.0, p))))
    return lr


class DualSystemTrainer:
    def __init__(self, model, navdp_state_dict, latent_queries, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0,
                 bucket_cap_mb=100, process_group=None, max_grad_norm=None, lr_schedule=None, accumulation_steps=1,
                 graph_s1=False, dropout=0.0, dropout_seed=0):
        """model: internnav_b200.internvla_n1.InternVLAN1ForCausalLM with weights loaded (the frozen parts are used from
        it); navdp_state_dict: {reference name: tensor} for `model.navdp.*`; latent_queries [1, n_query, H].
        dropout: System 1's train-mode dropout p (0.1 reproduces the reference's training; 0 turns it off); dropout_seed:
        the key of the mask stream (each micro-batch and each data-parallel rank draws its own masks)."""
        self.model = model
        dev = model.device
        if dev.type != "cuda":
            raise RuntimeError("n1b200 has no CPU path")
        self.device = dev
        self.masters = OrderedDict()
        for k, v in navdp_state_dict.items():
            if v.is_floating_point():
                self.masters[k] = v.detach().to(dev, torch.float32).clone()
        self.latent = latent_queries.detach().to(dev, torch.float32).clone()
        dist_on = torch.distributed.is_available() and torch.distributed.is_initialized()
        rank = torch.distributed.get_rank(process_group) if dist_on else 0
        self.dropout_rng = DropoutRNG(dropout_seed, rank, dev) if dropout > 0 else None
        self._dropout_step = 0          # micro-batches run so far: the `step` word of the mask counter
        self.s1 = S1TrainStep(self.masters, GpuOps(str(dev)), dropout=dropout, rng=self.dropout_rng)
        trainable = OrderedDict((k, (tuple(v.shape), torch.float32)) for k, v in self.masters.items()
                                if not k.startswith("rgbd_encoder.rgb_model."))
        trainable["model.latent_queries"] = (tuple(self.latent.shape), torch.float32)
        self.buckets = GradientBuckets(trainable, dev, bucket_cap_mb=bucket_cap_mb, process_group=process_group)
        self.opt = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self.max_grad_norm, self.lr_schedule, self.accumulation_steps = max_grad_norm, lr_schedule, int(accumulation_steps)
        self.m = {k: torch.zeros_like(g) for k, g in self.buckets.grads.items()}
        self.v = {k: torch.zeros_like(g) for k, g in self.buckets.grads.items()}
        self.steps, self._micro, self._touched = 0, 0, set()
        self.profile_phases = False
        # graph_s1: replay the System-1 forward / backward (several thousand kernel launches driven from Python, one ctypes
        # call each: the step is host-bound without it, profiles/README.md) from a CUDA graph captured on the first step of
        # a given batch shape
        self.graph_s1, self._s1_graphs = bool(graph_s1), {}
        self._s1_views = OrderedDict((k, g) for k, g in self.buckets.grads.items() if k != "model.latent_queries")
        self.timing = {}
        import ctypes
        K = 20
        buf = (ctypes.c_float * (K * 5))()
        _lib.check(_lib.lib().n1_ddpm_tables(K, buf))
        t = torch.tensor(list(buf), dtype=torch.float32).view(K, 5)
        # column 0 = sqrt(1 - acp), so acp = 1 - col0^2   (n1_ddpm_tables layout, include/n1b200.h)
        self.alphas_cumprod = (1.0 - t[:, 0] ** 2).to(dev)

    # ------------------------------------------------------------------ pieces
    def _s2_forward(self, batch):
        m = self.model
        prompts = []
        rows = m._prompts(batch["input_ids"])
        mask = batch["attention_mask"].tolist()
        for b, row in enumerate(rows):
            t = int(batch["t_s_pos"][b])
            prompts.append([tok for i, tok in enumerate(row[:t]) if mask[b][i]])
        grid = batch["image_grid_thw"].tolist() if torch.is_tensor(batch["image_grid_thw"]) else batch["image_grid_thw"]
        return m._s2.train_forward(prompts, batch["pixel_values"], grid)

    def _s1_forward_backward(self, batch, hs, noise, timesteps, grads_into=None):
        m = self.model
        ti, td = batch["traj_images"].to(self.device), batch["traj_depths"].to(self.device)
        f = ti.shape[1]
        goal_i = ti[:, 0:1].repeat(1, f, 1, 1, 1).flatten(0, 1)
        images_dp = torch.stack([goal_i, ti.flatten(0, 1)], dim=1)
        rgb_tokens = m.model.navdp.rgb_memory_tokens(images_dp)   # frozen branch, WITHOUT former_pe (trainable: added below)
        return self.s1.forward_backward(hs, rgb_tokens, td, batch["traj_poses"], batch["video_frame_num"], noise,
                                        timesteps, self.alphas_cumprod, rgb_has_pe=False, grads_into=grads_into)

    def _s1_graphed(self, batch, hs, noise, timesteps):
        """System-1 forward / backward through a captured CUDA graph: static input buffers, gradients accumulate into the
        bucket views exactly as in the eager path.  -> (loss, set of touched names, d loss / d TRAJ states)."""
        dev = self.device
        ti, td = batch["traj_images"].to(dev), batch["traj_depths"].to(dev)
        key = (tuple(ti.shape), tuple(hs.shape), tuple(noise.shape))
        ent = self._s1_graphs.get(key)
        src = dict(ti=ti, td=td.float(), poses=batch["traj_poses"].to(dev).float(), vfn=batch["video_frame_num"].to(dev),
                   noise=noise.to(dev).float(), ts=timesteps.to(dev), hs=hs)
        if ent is None:
            st = {k: v.clone() for k, v in src.items()}

            def run():
                f = st["ti"].shape[1]
                goal_i = st["ti"][:, 0:1].repeat(1, f, 1, 1, 1).flatten(0, 1)
                images_dp = torch.stack([goal_i, st["ti"].flatten(0, 1)], dim=1)
                rgb_tokens = self.model.model.navdp.rgb_memory_tokens(images_dp)
                return self.s1.forward_backward(st["hs"], rgb_tokens, st["td"], st["poses"], st["vfn"], st["noise"], st["ts"],
                                                self.alphas_cumprod, rgb_has_pe=False, grads_into=self._s1_views)

            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                run()                         # warm-up on the capture stream: scratch buffers, cached tables
                side.synchronize()
                self.buckets.zero()           # the warm-up accumulated into the views
                before = _lib.prof_read()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
                    loss, grads, dhs = run()
                nodes = _lib.prof_read()      # kernels captured into the graph = launches of every replay
                _lib.lib().n1_prof_add(before["gemm_launches"], before["total_launches"])
            torch.cuda.current_stream(dev).wait_stream(side)
            ent = self._s1_graphs[key] = (g, st, loss, set(grads), dhs, nodes)
        g, st, loss, touched, dhs, nodes = ent
        for k, v in src.items():
            st[k].copy_(v, non_blocking=True)
        g.replay()
        _lib.lib().n1_prof_add(nodes["gemm_launches"], nodes["total_launches"])
        return loss, touched, dhs

    def _set_dropout_step(self, step):
        if self.dropout_rng is not None:
            self.dropout_rng.set_step(step)

    def loss_and_grads(self, batch, noise, timesteps, dropout_step=None):
        """Parity entry point: (loss, {name: fp32 gradient}, TRAJ states) for one batch; no exchange, no update.
        batch: the collated dict of internnav_b200.training.collate_traj_batch (tensors may live on the host).
        dropout_step: the micro-batch whose dropout masks are used (default: the next one); the counter does not advance."""
        self._set_dropout_step(self._dropout_step if dropout_step is None else dropout_step)
        hs = self._s2_forward(batch)
        loss, grads, dhs = self._s1_forward_backward(batch, hs, noise, timesteps)
        grads["model.latent_queries"] = self.model._s2.train_backward(dhs).reshape(self.latent.shape)
        return loss, grads, hs

    # ------------------------------------------------------------------ the step
    def step(self, batch, noise, timesteps):
        """One micro-batch.  On the last micro-batch of an accumulation window: exchange, clip, AdamW.  Returns the loss
        (a device scalar; no host synchronisation happens inside the step unless clipping needs the norm)."""
        dist_on = torch.distributed.is_available() and torch.distributed.is_initialized()
        if self._micro == 0:
            self.buckets.zero()
            self._touched = set()
        self._micro += 1
        last = self._micro >= self.accumulation_steps
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if dist_on else None
        pe = [torch.cuda.Event(enable_timing=True) for _ in range(5)] if self.profile_phases else None
        if pe:
            pe[0].record()
        hs = self._s2_forward(batch)
        if pe:
            pe[1].record()
        self._set_dropout_step(self._dropout_step)      # a static input of the graphed step, copied before its replay
        self._dropout_step += 1
        if self.graph_s1:
            loss, grads, dhs = self._s1_graphed(batch, hs, noise, timesteps)
        else:
            loss, grads, dhs = self._s1_forward_backward(batch, hs, noise, timesteps, grads_into=self._s1_views)
        if pe:
            pe[2].record()
        self._touched.update(grads)
        lat_view = self.buckets.grads["model.latent_queries"]
        lat_bucket = self.buckets.bucket_of("model.latent_queries")
        if last and dist_on:
            if self.accumulation_steps > 1:
                self.buckets.scale_(1.0 / self.accumulation_steps, skip=(lat_bucket,))
            # every bucket without latent_queries is complete now: exchange them while the System-2 backward runs
            ev[0].record()
            self.buckets.all_reduce(async_op=True, skip=(lat_bucket,))
            ev[1].record()
        lat_view += self.model._s2.train_backward(dhs).reshape(self.latent.shape)
        self._touched.add("model.latent_queries")
        if pe:
            pe[3].record()
        if not last:
            return loss
        if dist_on:
            if self.accumulation_steps > 1:
                self.buckets.buffers[lat_bucket].mul_(1.0 / self.accumulation_steps)
            ev[2].record()
            self.buckets.all_reduce(async_op=True, only=(lat_bucket,), append=True)
            self.buckets.wait()
            ev[3].record()
            self._events = ev
        elif self.accumulation_steps > 1:
            self.buckets.scale_(1.0 / self.accumulation_steps)
        self._micro = 0
        if self.max_grad_norm is not None:
            total = torch.sqrt(sum(b.float().pow(2).sum() for b in self.buckets.buffers))
            coef = torch.clamp(self.max_grad_norm / (total + 1e-6), max=1.0)   # torch.nn.utils.clip_grad_norm_
            for b in self.buckets.buffers:
                b.mul_(coef)
            self.last_grad_norm = total
        o = self.opt
        lr = self.lr_schedule(self.steps) if self.lr_schedule is not None else o["lr"]
        self.steps += 1
        for k, g in self.buckets.grads.items():
            if k not in self._touched:   # torch.optim skips parameters whose .grad is None (no update, no weight decay)
                continue
            master = self.latent if k == "model.latent_queries" else self.masters[k]
            _bwd.adamw(master.view(-1), None, g.view(-1), self.m[k].view(-1), self.v[k].view(-1), lr, betas=o["betas"],
                       eps=o["eps"], weight_decay=o["weight_decay"], step=self.steps)
        self.s1.refresh()
        self.model._s2.set_latent_queries(self.latent)
        if pe:
            pe[4].record()
            self._phase_events = pe
        return loss

    def phase_ms(self):
        """Device time of the phases of the last step run with `profile_phases = True` (CUDA events; synchronises)."""
        pe = getattr(self, "_phase_events", None)
        if pe is None:
            return None
        pe[4].synchronize()
        return {"s2_forward": pe[0].elapsed_time(pe[1]), "s1_forward_backward": pe[1].elapsed_time(pe[2]),
                "s2_backward": pe[2].elapsed_time(pe[3]), "exchange_clip_adamw_refresh": pe[3].elapsed_time(pe[4])}

    def exchange_ms(self):
        """CUDA-event times of the last exchanged step: (launch window of the overlapped buckets, exposed tail = from the
        end of the System-2 backward to the last bucket reduced).  Synchronises."""
        ev = getattr(self, "_events", None)
        if ev is None:
            return None
        ev[3].synchronize()
        return {"overlapped_launch_ms": ev[0].elapsed_time(ev[1]), "exposed_ms": ev[2].elapsed_time(ev[3]),
                "s2_backward_window_ms": ev[1].elapsed_time(ev[2])}

    # ------------------------------------------------------------------ dropout mask stream
    def dropout_state(self):
        """What a resumed run needs to continue the dropout mask stream (save it beside the optimizer state, as HF Trainer
        saves its RNG states): {"p", "seed", "step"}; `step` counts the micro-batches run."""
        rng = self.dropout_rng
        return {"p": self.s1.dropout, "seed": rng.seed if rng is not None else None, "step": self._dropout_step}

    def load_dropout_state(self, state):
        """Continue the mask stream of `dropout_state()` (this process keeps its own data-parallel rank)."""
        if float(state["p"]) != self.s1.dropout:
            raise ValueError("dropout p of the saved state (%r) differs from this trainer's (%r)" % (state["p"], self.s1.dropout))
        if self.dropout_rng is not None:
            self.dropout_rng.seed = int(state["seed"])
        self._dropout_step = int(state["step"])

    # ------------------------------------------------------------------ export
    def state_dict(self):
        """The trained tensors under the reference's checkpoint names (`model.navdp.*`, `model.latent_queries`)."""
        out = OrderedDict(("model.navdp." + k, v.detach().clone()) for k, v in self.masters.items())
        out["model.latent_queries"] = self.latent.detach().clone()
        return out

    def sync_model(self):
        """Push the fp32 masters into the inference handle (`model.model.navdp`), so `generate_traj` and checkpoints read
        the trained weights.  Re-packs System 1 (a few ms); call it when evaluating / saving, not every step."""
        self.model.model.navdp.load_state_dict({k: v for k, v in self.masters.items()})
        self.model._s2.set_latent_queries(self.latent)

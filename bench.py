#!/usr/bin/env python
"""bench.py -- training rays/sec of the EmerNeRF per-ray-batch hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1)
    python bench.py --impl reference ...                      (the reference's algorithm on host cores)

A *step* is one training pass of the hot path over one 8192-ray synthetic Waymo-shape pixel batch
(BASELINE.json configs[1] by default): proposal sampling -> field -> compositing -> rgb + sky losses
-> backward -> Adam on the field (and, on the steps the reference's schedule asks for it, the proposal
loss + proposal Adam).  Rays shard across ranks (weak scaling: 8192 rays per GPU); the only
collective is the gradient all-reduce.

One JSON line on stdout (rank 0): metric/value/unit/..., plus
  e2e          same metric through the public API with HOST (pinned) input batches copied H2D inside
               every step and the loss read back D2H
  roofline     the dominant kernel of the step vs the measured peak in MEASURED_PEAKS.json
  cpu_baseline the CPU oracle (restatement of the reference, oracle/) timed on this box's host cores
               on a bounded sample of the same workload
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
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "training rays/sec (8192-ray batch)"
UNIT = "rays/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=240)
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", default="static", choices=["static", "dynamic", "flow", "flow_feat"])
    ap.add_argument("--rays", type=int, default=8192, help="rays per GPU per step")
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--cpu-rays", type=int, default=256, help="rays in one CPU-baseline step (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-full-step", action="store_true", help="skip the pixel + lidar iteration timing")
    ap.add_argument("--profile-all", action="store_true", help="print the per-kernel time table of one step")
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"],
                    help="fused: emernerf_b200.optim.FusedAdam (one launch: Adam + gradient zeroing, flat buffers); "
                         "torch: torch.optim.Adam(fused=True) as builders.py builds it")
    ap.add_argument("--dp-mode", default="sharded", choices=["sharded", "allreduce"],
                    help="multi-GPU gradient exchange (emernerf_b200.distributed): reduce-scatter + sharded Adam + "
                         "all-gather, or all-reduce + replicated Adam")
    ap.add_argument("--no-defer-gather", action="store_true",
                    help="issue the field's parameter all-gather right after its Adam step instead of beside the next "
                         "step's proposal sampling")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --rays per GPU; strong: --rays in total, split over the GPUs (BASELINE configs[3,4])")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying "
                    "the captured CUDA graphs of the step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (rendered outputs, loss, "
                         "updated parameters) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the B200 arm (--impl ours)")
    return args


# ----------------------------------------------------------------------------- losses (host glue)
def pixel_losses(out, batch):
    """rgb L2 (loss/base.py:83-146, l2, coef 1) + opacity-based sky loss (loss/base.py:149-185, coef
    1e-3).  Consumers of the hot path's outputs; plain torch (SURVEY.md §8f row 2)."""
    rgb = ((out["rgb"] - batch["pixels"]) ** 2).mean()
    op = out["opacity"].squeeze(-1).clamp(1e-6, 1 - 1e-6)
    sky = torch.nn.functional.binary_cross_entropy(op, 1.0 - batch["sky_masks"]) * 1e-3
    loss = rgb + sky
    if "dino_feat" in out and "features" in batch:
        loss = loss + 0.5 * ((out["dino_feat"] - batch["features"]) ** 2).mean()
    ex = out["extras"]
    if "dynamic_density" in ex:
        loss = loss + 0.01 * ex["dynamic_density"].mean()
    if "shadow_ratio" in out:
        loss = loss + 0.01 * out["shadow_ratio"].mean()
    if "forward_pred_backward_flow" in ex:
        loss = loss + 0.01 * 0.5 * ((ex["forward_flow"].detach() + ex["forward_pred_backward_flow"]) ** 2
                                    + (ex["backward_flow"].detach() + ex["backward_pred_forward_flow"]) ** 2).mean()
    return loss


def lidar_losses(out, batch, epsilon=2.0):
    """The reference's lidar-pass losses (train_emernerf.py:772-820) as capturable tensor code: range loss
    (loss/base.py:188-269: l2 of depths normalised by 80 m over rays with 0.01 < range < 80, coef 1), line-of-sight loss
    (loss/base.py:430-464, coef 0.1, margin ``epsilon``) and the dynamic-density regulariser on lidar rays (Q13).
    (The valid-ray mask multiplies instead of indexing, so shapes are static.)"""
    gt = batch["lidar_ranges"].squeeze(-1)
    valid = ((gt > 0.01) & (gt < 80.0)).float()
    nd = lambda d: torch.clamp(d / 80.0, 0.0, 1.0)
    loss = (((nd(out["depth"].squeeze(-1)) - nd(gt)) ** 2) * valid).sum() / valid.sum().clamp_min(1.0)
    ex = out["extras"]
    w, t = ex["weights"], ex["t_vals"].detach()
    g = gt.unsqueeze(-1)
    empty = (t < g - epsilon).float()
    near = ((t > g - epsilon) & (t < g + epsilon)).float()
    sig = epsilon / 3.0
    dirac = (1.0 / (2.0 * torch.pi * sig * sig) ** 0.5) * torch.exp(-((t - g) ** 2) / (2.0 * sig * sig))
    sight = ((w.square() * empty).sum(-1, keepdim=True).mean() + ((w - dirac).square() * near).sum(-1, keepdim=True).mean())
    loss = loss + 0.1 * (sight * (gt > 0).float()).mean()
    if "dynamic_density" in ex:
        loss = loss + 0.01 * ex["dynamic_density"].mean()
    return loss


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.t_mark = index, [], None, 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.monotonic()] + [c.strip() for c in line.split(",")])

    def mark(self, wait_s: float = 10.0):
        """Called right before the timed region: nvidia-smi needs up to a few seconds for its first sample on a fresh
        box (a 0.3 s timed region used to end before it), so wait for one, then count only what comes after."""
        t_end = time.monotonic() + wait_s
        while self.proc is not None and not self.rows and time.monotonic() < t_end:
            time.sleep(0.02)
        self.t_mark = time.monotonic()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r[1:] for r in self.rows if r[0] >= self.t_mark]
        sm = sorted(int(float(r[1])) for r in rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) < 8:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- the B200 arm
class Trainer:
    def __init__(self, args, rank, world, device):
        from emernerf_b200 import configs, synthetic
        from emernerf_b200.third_party.nerfacc_prop_net import get_proposal_requires_grad_fn

        self.args, self.rank, self.world, self.device = args, rank, world, device
        self.cfg = configs.make_cfg(args.variant, num_samples=args.samples)
        self.use_graph = not args.no_graph
        self.field, self.props, self.est, self.opt = configs.build_hot_path(self.cfg, device, table_std=0.3,
                                                                            capturable=self.use_graph,
                                                                            optimizer=args.optimizer)
        self.dp = None
        if args.optimizer == "fused":
            from emernerf_b200.distributed import DataParallel

            self.dp = DataParallel([self.opt, self.est.optimizer], mode=args.dp_mode)
        self.field.train(); self.est.train()
        [p.train() for p in self.props]
        self.req_fn = get_proposal_requires_grad_fn()
        self.step_idx = 2000                     # steady state of the schedule (every ~6th call)
        feats = args.variant == "flow_feat"
        nt = self.cfg.data.num_timesteps
        # 8 distinct batches per rank, cycled (device-resident and pinned-host copies)
        self.rays = args.rays if args.scaling == "weak" else args.rays // world     # rays THIS rank renders per step
        self.host = [synthetic.pixel_batch(self.rays, nt, 3, seed=1000 * rank + i, features=feats, pin=True)
                     for i in range(8)]
        self.dev = [{k: v.to(device) for k, v in b.items()} for b in self.host]
        self.h2d_bytes = synthetic.bytes_of(self.host[0])
        # the second half of a reference training iteration: a lidar-ray pass (train_emernerf.py:748-827)
        self.lidar_dev = [{k: v.to(device) for k, v in synthetic.lidar_batch(self.rays, nt, seed=1000 * rank + i).items()}
                          for i in range(4)]
        self.params = [p for p in self.field.parameters()]
        self.prop_params = [p for m in self.props for p in m.parameters()]

    def sync_and_step(self, opt, params):
        """Average the gradients over the ranks and take the optimizer step."""
        if self.dp is not None:
            # one flat collective per group (emernerf_b200/distributed.py); the field's parameter all-gather is deferred
            # to the start of the next step, where it runs beside the proposal sampling
            self.dp.step(opt, defer_gather=(opt is self.opt and not self.args.no_defer_gather))
            return
        if self.world > 1:
            import torch.distributed as dist

            for p in params:                      # torch.optim.Adam arm: per-tensor all-reduce (round 1's recipe)
                if p.grad is not None:
                    dist.all_reduce(p.grad, op=dist.ReduceOp.AVG)
        opt.step()

    # ---- CUDA graphs: the step is ~10^2 small launches; capture it once per schedule branch
    def build_graphs(self):
        self.static = {k: torch.empty_like(v) for k, v in self.dev[0].items()}
        self.graphs, self.static_loss = {}, {}
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for prg in (False, True, False):
                self._step_body(self.static, prg)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        from emernerf_b200 import _lib

        self.graph_launches, self.static_out = {}, {}
        for prg in (False, True):
            g = torch.cuda.CUDAGraph()
            n0 = _lib.LAUNCHES
            with torch.cuda.graph(g):
                self.static_loss[prg] = self._step_body(self.static, prg)
            self.static_out[prg] = self.body_out
            self.graph_launches[prg] = _lib.LAUNCHES - n0      # library kernels inside this graph
            self.graphs[prg] = g

    def lidar_step(self, i):
        """The lidar half of a training iteration (device-resident rays): density-only render, range + line-of-sight
        losses, backward, second Adam step; the proposal schedule advances once more (Q16)."""
        prg = self.req_fn(self.step_idx)
        self.step_idx += 1
        if self.use_graph and not getattr(self, "_profiling", False):
            if not hasattr(self, "lidar_graphs"):
                self.build_lidar_graphs()
            for k, v in self.lidar_static.items():
                v.copy_(self.lidar_dev[i % 4][k], non_blocking=True)
            self.lidar_graphs[prg].replay()
            return self.lidar_loss[prg]
        return self._lidar_body(self.lidar_dev[i % 4], prg)

    def build_lidar_graphs(self):
        self.lidar_static = {k: torch.empty_like(v) for k, v in self.lidar_dev[0].items()}
        self.lidar_graphs, self.lidar_loss = {}, {}
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for prg in (False, True, False):
                self._lidar_body(self.lidar_static, prg)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for prg in (False, True):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.lidar_loss[prg] = self._lidar_body(self.lidar_static, prg)
            self.lidar_graphs[prg] = g

    def _lidar_body(self, batch, prg):
        from emernerf_b200.radiance_fields.render_utils import render_rays

        if self.dp is not None:
            self.dp.start_deferred()
        out = render_rays(self.field, self.est, self.props, batch, self.cfg, proposal_requires_grad=prg, prefix="lidar_")
        if prg:
            ploss = self.est.compute_loss(out["extras"]["trans"], 1024.0)
            self.est.optimizer.zero_grad()
            ploss.backward()
            self.sync_and_step(self.est.optimizer, self.prop_params)
        loss = lidar_losses(out, batch)
        self.opt.zero_grad()
        (loss * 1024.0).backward()
        self.sync_and_step(self.opt, self.params)
        return loss

    def step(self, i, from_host):
        prg = self.req_fn(self.step_idx)
        self.step_idx += 1
        if self.use_graph and not getattr(self, "_profiling", False):
            if not hasattr(self, "graphs"):
                self.build_graphs()
            src = self.host[i % 8] if from_host else self.dev[i % 8]
            for k, v in self.static.items():
                v.copy_(src[k], non_blocking=True)
            self.graphs[prg].replay()
            self.replayed_launches = getattr(self, "replayed_launches", 0) + self.graph_launches[prg]
            self.last_loss, self.last_out = self.static_loss[prg], self.static_out[prg]
            return self.last_loss
        if from_host:
            batch = {k: v.to(self.device, non_blocking=True) for k, v in self.host[i % 8].items()}
        else:
            batch = self.dev[i % 8]
        self.last_loss = self._step_body(batch, prg)
        self.last_out = self.body_out
        return self.last_loss

    def _step_body(self, batch, prg):
        from emernerf_b200.radiance_fields.render_utils import render_rays

        if self.dp is not None:
            self.dp.start_deferred()
        out = render_rays(self.field, self.est, self.props, batch, self.cfg, proposal_requires_grad=prg)
        if prg:
            ploss = self.est.compute_loss(out["extras"]["trans"], 1024.0)
            self.est.optimizer.zero_grad()
            ploss.backward()
            self.sync_and_step(self.est.optimizer, self.prop_params)
        loss = pixel_losses(out, batch)
        self.opt.zero_grad()
        (loss * 1024.0).backward()                # GradScaler(2**10).scale(loss), never unscaled (Q17)
        self.sync_and_step(self.opt, self.params)
        self.body_out = out                       # what render_rays returned: --dump-outputs writes it
        return loss


def timed(trainer, steps, from_host, sync):
    import torch.distributed as dist

    sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    last = None
    for i in range(steps):
        last = trainer.step(i, from_host)
        if from_host:
            last = last.item()                    # D2H read of the step's result
    ev1.record()
    sync()
    ms = ev0.elapsed_time(ev1)
    if trainer.world > 1:
        t = torch.tensor([ms], device=trainer.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return ms


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(trainer, out_dir):
    """Write what the last timed step computed as ``out_dir/<name>.npy``: every tensor ``render_rays`` returned
    (``extras.<key>`` for the per-sample extras), the loss, and every field / proposal parameter after the step's
    Adam update.  Floating arrays are written as float32 (float64 stays float64), others as float64.  Arrays larger
    than a sample size are flattened and sampled at positions drawn from a generator seeded with 0; the sample size
    starts at 2^20 elements and halves until the whole dump fits in DUMP_LIMIT_BYTES.  Both depend only on the shapes,
    so two builds run with the same arguments write the same positions.  Nothing is written unless all of it fits."""
    import numpy as np

    arrays = {"loss": trainer.last_loss}

    def add(prefix, d):
        for k, v in d.items():
            if isinstance(v, dict):
                add(f"{prefix}{k}.", v)
            elif torch.is_tensor(v):
                arrays[prefix + k] = v
            else:
                raise SystemExit(f"--dump-outputs: render output {prefix}{k} is a {type(v).__name__}, not a tensor")

    add("", trainer.last_out)
    arrays.update({f"field.{k}": v for k, v in trainer.field.named_parameters()})
    for i, p in enumerate(trainer.props):
        arrays.update({f"prop{i}.{k}": v for k, v in p.named_parameters()})

    def nbytes(t, cap):
        return min(t.numel(), cap) * (8 if t.dtype == torch.float64 or not t.is_floating_point() else 4)

    cap = 1 << 20
    while cap > 1 and sum(nbytes(t, cap) for t in arrays.values()) > DUMP_LIMIT_BYTES:
        cap //= 2
    torch.cuda.synchronize()
    out = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > cap:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        a = t.cpu().numpy()
        out[name] = a.astype(a.dtype if a.dtype == np.float64 else np.float32 if t.is_floating_point() else np.float64)
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_LIMIT_BYTES, total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return {"dir": out_dir, "arrays": len(out), "bytes": total, "sample_elements": cap}


def _safe(fn, *a):
    try:
        return fn(*a)
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"[:200]}


def time_full_step(tr, args, world, device, sync):
    """A whole reference training iteration: pixel pass + lidar pass, two (three) optimizer steps."""
    import torch.distributed as dist

    for i in range(3):
        tr.step(i, False); tr.lidar_step(i)
    sync()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    n_full = max(8, args.steps // 4)
    for i in range(n_full):
        tr.step(i, False)
        tr.lidar_step(i)
    f1.record()
    sync()
    ms_full = f0.elapsed_time(f1)
    if world > 1:
        t = torch.tensor([ms_full], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_full = t.item()
    return {"ms_per_iteration": ms_full / n_full, "iterations": n_full,
            "pixel_rays_per_s": tr.rays * world * n_full / (ms_full / 1e3),
            "rays_per_s_pixel_plus_lidar": 2 * tr.rays * world * n_full / (ms_full / 1e3),
            "what": f"one reference training iteration (train_emernerf.py:612-827): {tr.rays} pixel rays (fwd + bwd + Adam)"
                    f" + {tr.rays} lidar rays per GPU (density-only render, range + line-of-sight losses, bwd, second Adam)"}


def kernel_table(trainer, sync, steps=3):
    """Device time of every library launch (CUDA events on the launching stream, eager launches) over
    ``steps`` training steps.  Returns {(name, shape_tag): [launches, total_ms]}."""
    from emernerf_b200 import _lib

    rec = []
    trainer._profiling = True              # eager launches: events cannot be timed inside a replayed graph
    trainer.step(0, False)                 # one untimed eager step (allocator warm-up)
    sync()
    _lib.set_profile(lambda name, args: True, rec)
    for i in range(steps):
        trainer.step(i, False)
    sync()
    _lib.set_profile(None, None)
    trainer._profiling = False
    table = {}
    for name, tag, e0, e1 in rec:
        d = table.setdefault((name, tag), [0, 0.0])
        d[0] += 1
        d[1] += e0.elapsed_time(e1)
    return table


def run_ours(args):
    import torch.distributed as dist
    from emernerf_b200 import _lib

    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the B200 arm)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        if args.dump_outputs:
            # the sharded optimizer leaves each rank's copy of the parameters partly stale until the next step
            raise SystemExit("--dump-outputs needs a one-GPU run")
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    _lib.load()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()                       # before the warm-up: its first sample takes a while
    tr = Trainer(args, rank, world, device)
    for i in range(args.warmup):
        tr.step(i, False)
    if rank == 0:
        clocks.mark()
    sync()

    launches0 = _lib.LAUNCHES
    tr.replayed_launches = 0
    ms = timed(tr, args.steps, False, sync)
    launches = (_lib.LAUNCHES - launches0) + tr.replayed_launches
    dumped = dump_outputs(tr, args.dump_outputs) if args.dump_outputs else None

    e2e = None
    if not args.no_e2e:
        for i in range(2):
            tr.step(i, True)
        ms_e2e = timed(tr, args.steps, True, sync)
        e2e = {"value": tr.rays * world * args.steps / (ms_e2e / 1e3), "unit": UNIT,
               "h2d_bytes_per_step": tr.h2d_bytes, "d2h_bytes_per_step": 4,
               "ms_per_step": ms_e2e / args.steps}
    # clocks / throttle reasons sampled every 50 ms over both timed regions (device-resident and end-to-end)
    clk = clocks.stop() if rank == 0 else None

    # per-kernel device times: CUDA events around every library launch over 3 eager steps, same
    # process / inputs / clocks, right after the timed region (a replayed graph cannot be event-timed
    # per kernel).  The ncu launch list under profiles/ must agree on the kernel's SHARE.
    table = kernel_table(tr, sync, steps=3)          # every rank runs it (the steps all-reduce)

    # a whole reference training iteration: pixel pass + lidar pass, two (three) optimizer steps
    full = None
    if not args.no_full_step and world == 1:     # (one GPU only: an extra leg must not add collectives to a scaling run)
        try:
            full = time_full_step(tr, args, world, device, sync)
        except Exception as e:                       # an extra leg must never cost the headline numbers
            full = {"error": f"{type(e).__name__}: {e}"[:300]}
            torch.cuda.synchronize()


    if args.profile_all and tr.use_graph and hasattr(tr, "graphs"):
        for prg in (False, True):               # device time of each captured branch of the step
            sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                tr.graphs[prg].replay()
            e1.record()
            sync()
            if rank == 0:
                print(f"# graph replay, proposal update = {prg}: {e0.elapsed_time(e1) / 5:.3f} ms", file=sys.stderr)
    if args.profile_all and rank == 0:
        # all GPU kernels of one eager step (library + torch glue), by device time
        from torch.profiler import ProfilerActivity, profile

        tr._profiling = True
        for prg in (False, True):               # one eager step of each kind (without / with proposal update)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                tr._step_body(tr.dev[0], prg)
                torch.cuda.synchronize()
            rows = sorted(prof.key_averages(), key=lambda e: -e.device_time_total)[:40]
            tot = sum(e.device_time_total for e in prof.key_averages())
            n_launch = sum(e.count for e in prof.key_averages())
            print(f"# --- all kernels of one eager step (proposal update = {prg}): {tot / 1e3:.3f} ms device time, "
                  f"{n_launch} launches", file=sys.stderr)
            for e in rows:
                print(f"#   {e.device_time_total / 1e3:8.3f} ms n={e.count:4d}  {e.key[:110]}", file=sys.stderr)
        tr._profiling = False

    if rank != 0:
        if world > 1:                     # leave together with rank 0 (see the end of this function)
            dist.barrier()
            torch.cuda.synchronize()
            os._exit(0)
        return

    peaks = {}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"

    tot_ms = sum(v[1] for v in table.values())
    per_launch = {k: v[1] / v[0] for k, v in table.items()}
    dom = max(table, key=lambda k: table[k][1])
    grid_keys = [k for k in table if k[0] == "emer_grid_fwd"]
    grid_dom = max(grid_keys, key=lambda k: table[k][1]) if grid_keys else None
    if args.profile_all:
        for k, v in sorted(table.items(), key=lambda kv: -kv[1][1]):
            print(f"# {k[0]:26s} {k[1]:32s} n={v[0]:3d} {v[1] / 3:8.3f} ms/step {100 * v[1] / tot_ms:5.1f}%",
                  file=sys.stderr)
        print(f"# library kernels: {tot_ms / 3:.3f} ms/step of {ms / args.steps:.3f} ms/step", file=sys.stderr)

    # DRAM bytes per launch and tensor-pipe activity measured by `ncu --set full` on this build's kernels
    # (profiles/r2_dram_traffic.json, extracted from the reports summarised in profiles/r2_*_ncu_summary.md)
    try:
        NCU = json.load(open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")))
    except Exception:
        NCU = {}

    def measured(name, tag):
        e = NCU.get(f"{name}[{tag}]") or NCU.get(name) or {}
        return e.get("traffic"), e.get("tensor_pipe_active_pct")

    def layer_bytes(name, tag):
        """Algorithmic HBM bytes of one dense-layer launch: rows * (inputs + outputs) * 4."""
        import re

        m = re.match(r"k(\d+)_o(\d+)_N(\d+)", tag)
        if not m:
            return None
        k, o, n = (int(v) for v in m.groups())
        return n * (k + o) * 4

    def roofline_of(key):
        name, tag = key
        avg_ms = per_launch[key]
        traffic = measured(name, tag)[0]
        if name == "emer_grid_fwd":
            nbytes = _lib.algorithmic_bytes(tag)
        elif name == "emer_grid_bwd":
            # scatter: the corners are read-modify-written (2x the corner bytes), dy read once
            import re

            m = re.match(r"D(\d+)L(\d+)F(\d+)_N(\d+)", tag)
            d_, l_, f_, n_ = (int(v) for v in m.groups())
            nbytes = n_ * (2 * l_ * (2 ** d_) * f_ * 4 + d_ * 4 + l_ * f_ * 4)
        elif name.startswith("emer_linear"):
            nbytes = layer_bytes(name, tag)
        else:
            return None
        if not nbytes:
            return None
        ach = nbytes / (avg_ms / 1e3) / 1e9
        return {"kernel": f"{name}[{tag}]", "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach / hbm_peak, "traffic": traffic,
                # what actually crossed the DRAM pins (ncu) over the same time: the L2 serves the rest of the algorithmic bytes
                "dram_frac": (traffic / (avg_ms / 1e3) / 1e9 / hbm_peak) if traffic else None,
                "tensor_pipe_active_pct": measured(name, tag)[1], "peak_source": peak_src,
                "algorithmic_bytes_per_launch": nbytes, "avg_launch_ms": avg_ms, "launches_timed": table[key][0],
                "share_of_library_kernel_time": table[key][1] / tot_ms,
                "timing": "CUDA events around each launch, 3 eager steps after the timed region"}

    def chain_roofline(name):
        """The fused field kernels against BOTH of their bounds: tensor pipe (tf32 runs at half the measured bf16 rate;
        the 3xTF32 split executes 3 MMAs per algorithmic product) and HBM."""
        import re

        keys = [k for k in table if k[0] == name]
        if not keys:
            return None
        key = max(keys, key=lambda k: table[k][1])
        m = re.match(r"k(\d+)_f(\d+)_N(\d+)(_save)?", key[1])
        k_enc, nf, n = int(m.group(1)), int(m.group(2)), int(m.group(3))
        if name == "emer_field_fwd":
            macs = k_enc * 64 + 64 * nf + 64 * 128 + 64 * 64 + 64 * 16
            nbytes = n * 4 * (k_enc + 4 + (256 if m.group(4) else 0) + (64 if nf == 128 else 0))
        else:
            macs = 8 * 64 + 64 * 128 + 64 * 64 + nf * 64 + 64 * ((k_enc + 15) // 16 * 16)
            nbytes = n * 4 * (8 + 256 + 64 + 128 + 64 + k_enc)     # d_rgb, rgb, sigmas | saved activations | dz1, d1, dzb, d_enc
        avg_ms = per_launch[key]
        tf32_peak = float(peaks.get("bf16_tflops", 1590.0)) / 2.0
        executed = 3 * 2 * macs * n / (avg_ms / 1e3) / 1e12
        return {"kernel": f"{name}[{key[1]}]", "bound": "tensor", "achieved": executed, "peak": tf32_peak, "unit": "TFLOP/s",
                "frac": executed / tf32_peak,
                "peak_source": ("measured bf16 (MEASURED_PEAKS.json) / 2: tf32 tcgen05.mma runs at half the bf16 rate"
                                if "bf16_tflops" in peaks else "fallback 1590 / 2"),
                "algorithmic_tflops": 2 * macs * n / (avg_ms / 1e3) / 1e12,
                "executed_over_algorithmic": 3, "hbm_gbs": nbytes / (avg_ms / 1e3) / 1e9, "hbm_frac": nbytes / (avg_ms / 1e3) / 1e9 / hbm_peak,
                "algorithmic_bytes_per_launch": nbytes, "avg_launch_ms": avg_ms, "launches_timed": table[key][0],
                "share_of_library_kernel_time": table[key][1] / tot_ms, "traffic": measured(name, key[1])[0],
                "tensor_pipe_active_pct_ncu": measured(name, key[1])[1]}

    roof = roofline_of(dom)                                  # the kernel with the largest share of the step
    roof_grid = roofline_of(grid_dom) if grid_dom is not None else None   # the hash-grid gather (north star)
    dom_ms = per_launch[dom]
    by_name = {k: v[1] for k, v in table.items()}
    line = {
        "metric": METRIC, "value": tr.rays * world * args.steps / (ms / 1e3), "unit": UNIT,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic Waymo-shape rays (3 cams, 640x960, 200 timesteps), random-init MLPs, N(0,0.3) tables",
        "config": dict(workload_config(args, world),
                       l2="no explicit flush: each step streams > 1 GB of tables+activations through the 126 MB L2",
                       optimizer=args.optimizer,
                       gradient_exchange=("none (1 GPU)" if world == 1 else
                                          (f"{args.dp_mode}: one flat NCCL collective per optimizer group, "
                                           f"{tr.dp.bytes_per_step(tr.opt) / 1e6:.0f} MB sent per rank per step"
                                           if tr.dp is not None else "per-tensor all-reduce"))),
        "gpu_launches": launches,
        "dominant_kernel": {"name": f"{dom[0]}[{dom[1]}]", "share_of_library_kernel_time": by_name[dom] / tot_ms,
                            "avg_launch_ms": dom_ms},
        "cuda_graph": tr.use_graph,
        "library_kernel_ms_per_step": tot_ms / 3,
        "roofline": roof if roof is not None else (chain_roofline(dom[0]) or roof_grid), "roofline_hash_grid": roof_grid,
        "roofline_fused_chain": {"forward": _safe(chain_roofline, "emer_field_fwd"), "backward": _safe(chain_roofline, "emer_field_bwd")},
        "clocks": clk,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if dumped is not None:
        line["dumped_outputs"] = dumped
    if full is not None:
        line["full_step"] = full
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(args, steps=2, warmup=1)
        try:
            line.update(parity_vs_oracle(tr, args))     # second half of BASELINE.json's metric: PSNR vs reference
        except Exception as e:
            line["psnr_vs_reference"] = None
            line["parity_sample"] = f"failed: {type(e).__name__}: {e}"[:300]
    print(json.dumps(line))
    sys.stdout.flush()
    if world > 1:
        # captured graphs hold NCCL work: a plain destroy_process_group() was seen to hang at exit
        dist.barrier()
        torch.cuda.synchronize()
        os._exit(0)


# ----------------------------------------------------------------------------- the CPU arm
def workload_config(args, world):
    """The ``config`` both arms report: BASELINE.json's configuration the metric is quoted on."""
    per_gpu = args.rays if getattr(args, "scaling", "weak") == "weak" else args.rays // world
    return {"workload": f"BASELINE configs[{['static', 'dynamic', 'flow', 'flow_feat'].index(args.variant) + 1}]: "
                        f"default_config {args.variant} field, {per_gpu} rays x {args.samples} samples "
                        f"per GPU, proposal samples [128, 64], fwd+bwd+Adam, proposal update every ~6th step",
            "rays_per_gpu": per_gpu, "samples": args.samples, "parallelism": f"ray-sharded dp{world}"}


def cpu_baseline(args, steps, warmup):
    """The oracle (CPU restatement of the reference's Python + tcnn/nerfacc stand-ins) run as a training
    step on the host cores: same config and tables, a bounded sample of ``--cpu-rays`` rays."""
    from emernerf_b200 import configs, synthetic
    from oracle import adapters, hotpath

    # torch's intra-op pool gets SLOWER beyond ~16-32 threads on these small ops (measured: 128
    # threads -> 107 s/step vs 1.2 s/step on 8); use what helps and report the count actually used
    cores = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    cfg = configs.make_cfg(args.variant, num_samples=args.samples)
    field, props, _, _ = configs.build_hot_path(cfg, "cpu", table_std=0.3)
    fsd = adapters.cpu_state_dict(field, requires_grad=True)
    psd = [adapters.cpu_state_dict(p, requires_grad=False) for p in props]
    fspec = adapters.spec_from_module(field)
    pspec = [adapters.spec_from_module(p) for p in props]
    leaves = [v for v in fsd.values() if v.requires_grad]
    feats = args.variant == "flow_feat"

    def one(i):
        b = synthetic.pixel_batch(args.cpu_rays, cfg.data.num_timesteps, 3, seed=i, features=feats)
        out, _ = hotpath.render_rays(fsd, fspec, psd, pspec, b, num_samples=args.samples,
                                     prop_samples=cfg.nerf.propnet.num_samples_per_prop, near_plane=0.1,
                                     far_plane=1000.0, training=True)
        loss = pixel_losses(out, b)
        torch.autograd.grad(loss * 1024.0, leaves, allow_unused=True)
        return float(loss.detach())

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    for i in range(steps):
        one(i)
    dt = time.perf_counter() - t0
    return {"value": args.cpu_rays * steps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} training steps (fwd+bwd, no optimizer) of {args.cpu_rays} rays x {args.samples} "
                      f"samples, same tables/config, {dt:.1f} s", "ms_per_step": dt / steps * 1e3}


def parity_vs_oracle(tr, args, at_start=True):
    """PSNR (datasets/metrics.py:31-46: -10 log10 mse) and max relative errors of the B200 render against the CPU
    oracle -- the reference's algorithm -- on the SAME weights (the benchmark's starting state; and, for the record, the
    trainer's after the timed steps) and the same ``--cpu-rays`` Waymo-shape rays, evaluation mode (deterministic: no
    jitter, unit temporal-aggregation noise).
    Part of the cpu_baseline leg: the oracle is the checker here, never the thing measured."""
    import math

    from emernerf_b200 import synthetic
    from emernerf_b200.radiance_fields.render_utils import render_rays
    from oracle import adapters, hotpath

    from emernerf_b200 import configs

    cfg = tr.cfg
    feats = args.variant == "flow_feat"
    b = synthetic.pixel_batch(args.cpu_rays, cfg.data.num_timesteps, 3, seed=4242, features=feats)
    if at_start:
        # the benchmark's STARTING state (same seed: N(0, 0.3) tables, default-initialised MLPs), on a second model
        field, props, est, _ = configs.build_hot_path(cfg, tr.device, table_std=0.3)
    else:
        field, props, est = tr.field, tr.props, tr.est
    mods = [field, est] + list(props)
    [m.eval() for m in mods]
    with torch.no_grad():
        got = render_rays(field, est, props, {k: v.to(tr.device) for k, v in b.items()}, cfg)
    torch.cuda.synchronize()
    [m.train() for m in mods]
    fsd = adapters.cpu_state_dict(field)
    psd = [adapters.cpu_state_dict(p) for p in props]
    fspec, pspec = adapters.spec_from_module(field), [adapters.spec_from_module(p) for p in props]

    def oracle(scale=1.0):
        with torch.no_grad():
            return hotpath.render_rays(fsd, fspec, psd, pspec, b, num_samples=args.samples,
                                       prop_samples=cfg.nerf.propnet.num_samples_per_prop, near_plane=0.1,
                                       far_plane=1000.0, training=False, prop_sigma_scale=scale)[0]

    want = oracle()
    # rays whose samples do not move when the oracle's own proposal densities change in the last bits (inverse-CDF
    # resampling is ill-conditioned where a CDF is flat; tests/test_gpu_fullsize.py): depth is compared on those
    keep = hotpath.sample_stability(oracle, want["extras"]["t_vals"])

    def rel(k, sel=None):
        a, w = got[k].detach().double().cpu(), want[k].detach().double()
        if sel is not None:
            a, w = a[sel], w[sel]
        if a.numel() == 0:
            return None
        return float((a - w).abs().max() / want[k].detach().double().abs().max().clamp_min(1e-12))

    mse = float((got["rgb"].double().cpu() - want["rgb"].double()).square().mean())
    errs = {"rgb": rel("rgb"), "opacity": rel("opacity"), "depth": rel("depth", keep), "depth_all_rays": rel("depth")}
    if "dino_feat" in want:
        errs["feature"] = rel("dino_feat")
    res = {"psnr_vs_reference": (999.0 if mse == 0 else -10.0 * math.log10(mse)), "max_rel_err": errs,
           "well_conditioned_rays": f"{int(keep.sum())}/{args.cpu_rays}",
           "parity_sample": f"{args.cpu_rays} rays x {args.samples} samples, eval mode, "
                            + ("the benchmark's starting weights" if at_start else "the trainer's weights after the timed steps")
                            + "; reference = CPU oracle (the reference's Python restated, pinned by tests/golden); PSNR / rgb /"
                              " opacity over all rays, depth over the rays with well-conditioned samples"}
    if at_start:
        # for the record: the same comparison on the weights the timed steps produced.  Hundreds of lr = 0.01 Adam steps
        # towards random pixel targets leave a field whose proposal CDFs are flat almost everywhere; inverse-CDF
        # resampling is ill-conditioned there (tests/test_gpu_fullsize.py), for ANY two implementations
        try:
            after = parity_vs_oracle(tr, args, at_start=False)
            res["parity_after_training_on_random_targets"] = {k: after[k] for k in ("psnr_vs_reference", "max_rel_err",
                                                                                    "well_conditioned_rays")}
        except Exception as e:
            res["parity_after_training_on_random_targets"] = {"error": str(e)[:200]}
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    # every step is a bounded sample (--cpu-rays rays) of the workload
    steps, warmup = args.steps, max(1, min(args.warmup, 2))
    cb = cpu_baseline(args, steps=steps, warmup=warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "steps_requested": args.steps, "ms_per_step": cb["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic Waymo-shape rays (3 cams, 640x960, 200 timesteps), random-init MLPs, N(0,0.3) tables",
        "config": dict(workload_config(args, max(1, args.gpus)),
                       sample=f"CPU oracle (the reference's Python restated; tcnn / nerfacc restated) on "
                              f"{args.cpu_rays} rays x {args.samples} samples per step, fwd+bwd, no optimizer step"),
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)

#!/usr/bin/env python
"""bench.py — PFST self-training hot-path throughput on B200 (contract in the task brief).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--impl reference]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Training workloads (cfg1-cfg4 = BASELINE.json configs[0..3]; default cfg2, the config the metric is
quoted on): a "step" is one pass of the hot path (EMA teacher update, pseudo labels, ClassMix, PFGST
loss fwd+bwd, prototype accumulate / cross-rank sum / distance fwd+bwd) over one batch of synthetic
network outputs (SURVEY.md §8d), excluding the three network passes. Rank 0 prints ONE JSON line:
  value          pixels/s, whole job, inputs resident in HBM, CUDA-event timed
  plugin         the same step through the drop-in class (PFGST.forward_train) with DEVICE-resident
                 inputs — what the plugin boundary costs on top of `value`
  e2e            same metric through PFGST.forward_train with HOST (pinned) buffers:
                 H2D of every step input and D2H of the log vars inside the timed region
  roofline       dominant kernel (multi-tensor EMA, 12 B/param): bytes / CUDA-event time
                 of that launch, vs MEASURED_PEAKS.json; step_* = the whole step by SURVEY §8d bytes
  cpu_baseline   the CPU oracle (a port of the reference's path) on this box's host cores, full batch
cfg5 (configs[4]) is the mIoU evaluation sweep: 10 000 label maps sharded over the ranks, one int64
confusion-matrix all-reduce per sweep; a "step" is one sweep (strong scaling).
`--impl reference` times the CPU port alone on the full batch, same metric/config.
`--dump-outputs DIR` writes what the last timed step returned as DIR/<name>.npy (see dump_outputs), so
that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

from pfst_b200.synthetic import (EVAL_WORKLOADS, WORKLOADS, deeplab_r50_param_shapes, eval_maps,  # noqa: E402
                                 model_params, step_inputs)

METRIC = "self_training_hot_path_throughput"
EVAL_METRIC = "miou_eval_sweep_throughput"
UNIT = "pixels/s"


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def config_dict(wl) -> dict:
    """The SAME dict in both arms (the driver compares them)."""
    n_params = sum(int(np.prod(s)) for s in deeplab_r50_param_shapes(wl.C))
    return {"workload": wl.name, "batch_per_gpu": wl.B, "classes": wl.C, "image": [wl.H, wl.W],
            "feature_dim": wl.D, "params": n_params,
            "l2": "no flush: the per-step working set (parameters + maps) exceeds the 126 MB L2"}


def eval_config_dict(ew) -> dict:
    return {"workload": ew.name, "maps": ew.maps, "classes": ew.C, "image": [ew.H, ew.W],
            "l2": "no flush: the resident maps cycled per sweep exceed the 126 MB L2"}


DUMP_MAX_ELEMS = 1 << 19       # per array; 13 arrays of float64 at most stay under 64 MB
DUMP_BUDGET = 64 << 20


def dump_outputs(out_dir, arrays: dict) -> None:
    """Write each tensor as <out_dir>/<name>.npy: float64 for 64-bit and int32 sources, float32 otherwise.
    A tensor of more than DUMP_MAX_ELEMS elements is replaced by the flattened elements at DUMP_MAX_ELEMS
    sorted indices drawn from a generator seeded with 0, so every run with the same shapes samples alike."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        wide = t.dtype in (torch.float64, torch.int64, torch.int32)
        a = t.cpu().numpy().astype(np.float64 if wide else np.float32)
        total += a.nbytes
        if total > DUMP_BUDGET:
            raise RuntimeError(f"--dump-outputs: more than {DUMP_BUDGET >> 20} MB at {name}")
        np.save(d / f"{name}.npy", a)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons, sampled every 20 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, enabled: bool = True):
        self.gpu, self.rows, self.proc, self.enabled = gpu_index, [], None, enabled

    def start(self):
        if not self.enabled:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.05] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU arms
_CPU_STATE = {}


def cpu_step_time(wl, seed):
    """One oracle step on the FULL batch of the workload. Returns seconds."""
    from oracle import pfgst_loss as OL, step as ostep
    key = (wl.name, seed)
    if key not in _CPU_STATE:
        g = torch.Generator().manual_seed(seed)
        _CPU_STATE[key] = (step_inputs(wl, seed), model_params(wl.C, g), model_params(wl.C, g),
                           np.random.RandomState(seed))
    inp, student, teacher, rs = _CPU_STATE[key]
    cfg = OL.LossCfg(dilation=wl.dilation, downscale=wl.downscale if wl.downscale != 1.0 else None)
    t0 = time.perf_counter()
    ostep.hot_path_step(5000, teacher, student, inp, wl.C, loss_cfg=cfg, rng=rs)
    return time.perf_counter() - t0


def cpu_sample_text(wl):
    return (f"oracle (ATen-op-for-op port of the reference path, torch {torch.__version__} CPU): the full "
            f"{wl.B}-image batch and the full 214-tensor EMA every step, nothing extrapolated")


def run_reference(args, wl, rank):
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    for _ in range(args.warmup):
        cpu_step_time(wl, 1234)
    ts = [cpu_step_time(wl, 1234) for _ in range(args.steps)]
    t = sum(ts) / len(ts)
    value = wl.B * wl.H * wl.W / t    # one host: its cores do not multiply with the GPU count
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(wl),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": cpu_sample_text(wl)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_eval_time(ew, n_maps, seed=1234):
    """Oracle intersect_and_union (the reference's per-map histc path, metrics.py:26-86) + the
    pre-eval sum over `n_maps` maps. Returns seconds."""
    from oracle import metrics as OM
    key = ("eval", ew.name, n_maps, seed)
    if key not in _CPU_STATE:
        _CPU_STATE[key] = eval_maps(n_maps, ew.H, ew.W, ew.C, seed)
    pred, gt = _CPU_STATE[key]
    t0 = time.perf_counter()
    per_image = [OM.areas(pred[i], gt[i], ew.C, 255) for i in range(n_maps)]
    OM.metrics_from_areas(*OM.pre_eval_sum(per_image))
    return time.perf_counter() - t0


def run_eval_reference(args, ew, rank):
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    n = max(1, min(ew.maps, args.ref_eval_maps))
    for _ in range(args.warmup):
        cpu_eval_time(ew, min(n, 4))
    ts = [cpu_eval_time(ew, n) for _ in range(args.steps)]
    t = sum(ts) / len(ts)
    value = n * ew.H * ew.W / t
    line = {"impl": "reference", "metric": EVAL_METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": eval_config_dict(ew),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"oracle intersect_and_union + pre_eval sum on {n} of the {ew.maps} maps per step "
                                       "(throughput is per map, the sweep is a loop over maps)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- GPU arm
class HostFeed:
    """The e2e leg's inputs live in pinned HOST memory. Every step's tensors (the data batch and
    the network outputs the replay segmentor 'produces') cross PCIe inside the timed region; the
    copies of step k+1 run on a copy stream while step k computes (two device slots)."""

    def __init__(self, pinned: dict, device):
        self.pinned = pinned
        self.slots = [{k: torch.empty_like(v, device=device) for k, v in pinned.items()} for _ in range(2)]
        self.stream = torch.cuda.Stream(device=device)
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.free = [torch.cuda.Event() for _ in range(2)]
        self.used = [False, False]
        self.cur = 0
        self.bytes_per_step = sum(v.numel() * v.element_size() for v in pinned.values())
        self.bytes_copied = 0

    def issue(self, slot: int) -> None:
        if self.used[slot]:
            self.stream.wait_event(self.free[slot])        # the step that read this slot has finished
        with torch.cuda.stream(self.stream):
            for k, v in self.pinned.items():
                self.slots[slot][k].copy_(v, non_blocking=True)
                self.bytes_copied += v.numel() * v.element_size()
        self.ready[slot].record(self.stream)

    def acquire(self, slot: int) -> dict:
        torch.cuda.current_stream().wait_event(self.ready[slot])
        self.cur = slot
        return self.slots[slot]

    def release(self, slot: int) -> None:
        self.free[slot].record(torch.cuda.current_stream())
        self.used[slot] = True


class ReplaySegmentor(torch.nn.Module):
    """Stands in for the DeepLabV3+ R50-D8 segmentor in the plugin / e2e legs: it owns a parameter
    list of the real shapes (so the EMA runs over the true 214 tensors) and 'produces' the network
    outputs from the current feed slot. Its decode loss is a 0-dim tensor of the feed (no kernel
    of its own: the three cuDNN passes are not part of the measured path)."""
    FEED = None      # class attribute: shared by the student and its deep-copied teacher

    def __init__(self, wl, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.params = torch.nn.ParameterList([torch.nn.Parameter(p) for p in model_params(wl.C, g)])
        self.calls = 0
        self.num_classes = wl.C
        self.train_cfg, self.test_cfg = {}, {}

    def _fetch(self, key):
        feed = ReplaySegmentor.FEED
        return feed.slots[feed.cur][key]

    def encode_decode(self, img, img_metas):
        logits = self._fetch("ema_logits")
        feats = self._fetch("x_ema")
        return logits, {"feats": feats, "decoded_features": feats, "seg_logits": logits}

    def forward_train(self, img, img_metas, gt, seg_weight=None, return_feats=False, return_decoded_feats=False,
                      return_logits=False, return_states=False):
        first = self.calls % 2 == 0
        self.calls += 1
        out = {"decode.loss_ce": self._fetch("loss_ce").detach().requires_grad_(True)}
        if first:     # source pass: decoded features + logits of the source image
            x = self._fetch("x_src").detach().requires_grad_(True)
            out.update(features=x, decoded_features=x, logits=self._fetch("logits_src"))
        else:         # mixed pass: logits of the mixed image (gradient target of the sim losses)
            out.update(features=None, logits=self._fetch("logits_trg").detach().requires_grad_(True))
        return out


def build_plugin(wl, seed, dev):
    from pfst_b200.uda import PFGST
    factory = lambda: ReplaySegmentor(wl, seed)  # noqa: E731
    return PFGST(model=factory, max_iters=40000, alpha=0.999, pseudo_threshold=0.98, pseudo_weight_ignore_top=0,
                 pseudo_weight_ignore_bottom=0, imnet_feature_dist_lambda=0, imnet_feature_dist_classes=None,
                 imnet_feature_dist_scale_min_ratio=None, mix='class', blur=False, color_jitter_strength=0.2,
                 color_jitter_probability=1.0, print_grad_magnitude=False, trg_loss_weight=1.,
                 use_decoded_feats=True, thre_type='all', compute_vis=False,
                 prototypes=dict(weight=0.1),
                 aux_losses=[dict(type='PFGSTLoss', kernel_size=3, dilation=wl.dilation, top_k=3,
                                  weights={'src_pos': 0.1, 'src_neg': 0.1, 'sim_pos': 0.1, 'sim_neg': 0.1,
                                           'src_pos_std': 0.1, 'src_neg_std': 0.1},
                                  sim_type='cosine', feat_level=None, detach_unfold=True,
                                  downscale=wl.downscale if wl.downscale != 1.0 else None)]).to(dev)


def run_ours(args, wl, rank, world, local_rank):
    import torch.distributed as dist
    from pfst_b200 import ops
    from pfst_b200.step import SelfTrainingStep, algorithmic_bytes

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    ops.device_check()
    seed = 1234 + rank
    g = torch.Generator().manual_seed(seed)
    np.random.seed(seed)
    host = step_inputs(wl, seed)
    inp = {k: v.to(dev) for k, v in host.items()}
    student = [p.to(dev) for p in model_params(wl.C, g)]
    teacher = [p.to(dev) for p in model_params(wl.C, g)]
    n_params = sum(p.numel() for p in student)
    step = SelfTrainingStep(teacher, student, wl.C, wl.D, dev, dilation=wl.dilation,
                            downscale=wl.downscale if wl.downscale != 1.0 else None, max_batch=max(wl.B, 64),
                            graphs=not args.no_graphs)

    def one(it):
        out = step.run(it, inp["img"], inp["target_img_strong_aug"], inp["gt"], inp["ema_logits"],
                       inp["logits_trg"], inp["x_src"], inp["x_ema"])
        # the next batch's labels are known before its network passes: their class-presence bits
        # (M1 part 1, one kernel + a 36-byte D2H) are prefetched so the host never waits for them
        step.prefetch(inp["gt"])
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warmup = max(args.warmup, 3)
    for i in range(warmup):
        one(i)
    sampler = ClockSampler(local_rank, enabled=rank == 0)   # one nvidia-smi poller per job
    ema_pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                 for _ in range(args.steps)]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    t_wall0 = time.time()
    ev0.record()
    for k in range(args.steps):
        step.ema_events = ema_pairs[k]
        out = one(warmup + k + 1)
    ev1.record()
    barrier()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1)
    step.ema_events = None
    if args.dump_outputs and rank == 0:
        # before the EMA launches below move the teacher on: it is the step's in-place output
        out = {k: v for k, v in out.items() if v is not None}
        out["teacher"] = torch.cat([p.reshape(-1) for p in teacher])
        dump_outputs(args.dump_outputs, out)
        del out
    ms = ev0.elapsed_time(ev1)
    try:
        ema_overlapped_ms = statistics.mean(a.elapsed_time(b) for a, b in ema_pairs)
    except (ValueError, RuntimeError):
        ema_overlapped_ms = None
    # The dominant kernel (multi-tensor EMA) runs on its own stream inside the step and shares
    # HBM with the other kernels there, so its roofline point is taken from launches of the
    # SAME kernel/grid timed alone, on the launching stream (523 MB per launch: nothing fits in L2).
    coeffs = ops.ema_coeffs(5000, 0.999)
    alone = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
    for _ in range(3):
        step.table.update(*coeffs, blocks_per_sm=step.ema_blocks_per_sm)
    torch.cuda.synchronize()
    for a, b in alone:
        a.record()
        step.table.update(*coeffs, blocks_per_sm=step.ema_blocks_per_sm)
        b.record()
    torch.cuda.synchronize()
    ema_ms = statistics.mean(a.elapsed_time(b) for a, b in alone)
    reduce_mode = "peer board: one-shot NVLink all-reduce inside proto_finalize" if step.bank.peer is not None else \
        ("ncclAllReduce" if world > 1 else "none (single rank)")
    if step.bank.peer is not None:
        step.bank.peer.check()

    # ---- plugin + e2e legs: the PFGST drop-in class -----------------------------------------
    pinned = {k: v.pin_memory() for k, v in host.items()}
    pinned["logits_src"] = (2.0 * torch.randn(host["logits_trg"].shape, generator=g)).pin_memory()
    pinned["target_img"] = torch.randn(host["img"].shape, generator=g).pin_memory()
    pinned["loss_ce"] = torch.rand((), generator=g).pin_memory()
    net_keys = ("ema_logits", "x_ema", "x_src", "logits_src", "logits_trg", "loss_ce")
    batch_keys = ("img", "gt", "target_img", "target_img_strong_aug")
    feed = HostFeed({k: pinned[k] for k in net_keys + batch_keys}, dev)
    ReplaySegmentor.FEED = feed
    model = build_plugin(wl, seed, dev)
    metas = [{'img_norm_cfg': {'mean': [0., 0., 0.], 'std': [1., 1., 1.]}}] * wl.B

    # (1) device-resident inputs: slot 0 is filled once, outside the timed region
    feed.issue(0)
    d = feed.acquire(0)
    torch.cuda.synchronize()

    def plugin_step():
        return model.forward_train(d["img"], metas, d["gt"], d["target_img"], metas, d["target_img_strong_aug"])[0]

    plugin_steps = max(3, args.steps)
    for _ in range(warmup):
        plugin_step()
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(plugin_steps):
        lv = plugin_step()
    float(lv["loss"])                 # the log variables are read back once at the end (one D2H for the interval)
    p1.record()
    barrier()
    plugin_ms = p0.elapsed_time(p1)

    # (2) e2e: host (pinned) buffers in, log vars out
    step_no = [0]

    def e2e_step():
        slot = step_no[0] % 2
        step_no[0] += 1
        dd = feed.acquire(slot)                   # this step's inputs have crossed PCIe
        feed.issue(slot ^ 1)                      # the next step's copies overlap this step's compute
        log_vars, _ = model.forward_train(dd["img"], metas, dd["gt"], dd["target_img"], metas,
                                          dd["target_img_strong_aug"])
        feed.release(slot)
        return log_vars

    e2e_steps = max(3, min(args.steps, 20))
    feed.used = [False, False]
    feed.issue(0)
    for _ in range(8):                            # both feed slots: two eager passes + graph capture each
        float(e2e_step()["loss"])
    barrier()
    feed.bytes_copied = 0
    d2h_before = model.d2h_bytes()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        lv = e2e_step()
        float(lv["loss"])                         # the step's result is read on the host every step
    torch.cuda.current_stream().wait_stream(feed.stream)   # the look-ahead copy belongs to the timed region too
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    h2d = feed.bytes_copied / e2e_steps           # counted from the tensors copied in the timed region
    d2h = (model.d2h_bytes() - d2h_before) / e2e_steps

    times = torch.tensor([ms, e2e_ms, plugin_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms, plugin_ms = times.tolist()
    model.close()
    step.close()                   # collective: graphs and peer boards go before the process group
    if rank != 0:
        return
    px = wl.B * wl.H * wl.W
    value = px * world * args.steps / (ms * 1e-3)
    e2e_value = px * world * e2e_steps / (e2e_ms * 1e-3)
    peak, peak_src = measured_peak()
    ab = algorithmic_bytes(wl.B, wl.C, wl.H, wl.W, wl.D, inp["x_src"].shape[2], inp["x_src"].shape[3], n_params)
    step_bytes = sum(ab.values())
    achieved = ab["ema"] / (ema_ms * 1e-3) / 1e9
    traffic = None
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists():
        traffic = json.loads(tp.read_text()).get("ema_multi_kernel")
    us_step = ms / args.steps * 1e3
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(wl),
            "notes": {"step": "EMA + pseudo-label + ClassMix + PFGST loss fwd/bwd + prototypes fwd/bwd (+ cross-rank sum)",
                      "cuda_graphs": not args.no_graphs, "proto_reduce": reduce_mode},
            "iters_per_s": args.steps / (ms * 1e-3),
            "step_bytes": step_bytes, "step_gbs_per_gpu": step_bytes / (us_step * 1e-6) / 1e9,
            "step_frac_of_peak": step_bytes / (us_step * 1e-6) / 1e9 / peak,
            "step_frac_of_nominal_8tbs": step_bytes / (us_step * 1e-6) / 1e9 / 8000.0,
            "clocks": clocks,
            "plugin": {"value": px * world * plugin_steps / (plugin_ms * 1e-3), "unit": UNIT,
                       "ms_per_step": plugin_ms / plugin_steps, "steps": plugin_steps,
                       "vs_step": (plugin_ms / plugin_steps) / (ms / args.steps),
                       "api": "pfst_b200.uda.PFGST.forward_train, inputs resident in HBM, log vars read once at the end"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps,
                    "h2d_gbs_per_rank": h2d / (e2e_ms / e2e_steps * 1e-3) / 1e9,
                    "api": "pfst_b200.uda.PFGST.forward_train (plugin class) with pinned host buffers; copies of step "
                           "k+1 overlap step k (copy stream, two device slots); log vars read on the host every step"},
            "gpu_launches": SelfTrainingStep.KERNEL_LAUNCHES * args.steps,
            "roofline": {"bound": "hbm", "kernel": "ema_multi_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "bytes_per_launch": ab["ema"], "us_per_launch": ema_ms * 1e3,
                         "timed": "20 launches alone after the timed steps (same grid as in the step: %s)" % (
                             "%d blocks/SM" % step.ema_blocks_per_sm if step.ema_blocks_per_sm else "one block per 4096-float chunk"),
                         "us_per_launch_overlapped_in_step": None if ema_overlapped_ms is None else ema_overlapped_ms * 1e3}}
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        cpu_step_time(wl, 1234)                                 # warm-up (allocator, thread pools)
        ts = [cpu_step_time(wl, 1234) for _ in range(2)]
        t_full = sum(ts) / len(ts)
        line["cpu_baseline"] = {"value": px / t_full, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                "sample": cpu_sample_text(wl) + f" (2 steps after 1 warm-up, {t_full:.2f} s each)"}
    print(json.dumps(line), flush=True)


def run_eval_ours(args, ew, rank, world, local_rank):
    """cfg5: the rank's contiguous shard of the sweep (evaluation.shard_range), `resident` distinct
    maps kept in HBM and cycled, the (C+1)^2 int64 matrix all-reduced once per sweep."""
    import torch.distributed as dist
    from pfst_b200 import ops
    from pfst_b200.evaluation import metrics as M

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    ops.device_check()
    lo, hi = M.shard_range(ew.maps, rank, world)
    n_local = hi - lo
    batch = args.eval_batch
    res = max(batch, min(args.eval_resident, n_local) // batch * batch)
    pred, gt = eval_maps(res, ew.H, ew.W, ew.C, seed=1234 + rank)
    d_pred, d_gt = torch.from_numpy(pred).to(dev), torch.from_numpy(gt).to(dev)
    meter = M.ConfusionMeter(ew.C, device=dev)
    launches = [0]

    def sweep():
        meter.conf.zero_()
        done = 0
        while done < n_local:
            i = done % res
            n = min(batch, n_local - done, res - i)
            meter.update(d_pred[i:i + n], d_gt[i:i + n])
            launches[0] += 1
            done += n
        meter.all_reduce()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        sweep()
    sampler = ClockSampler(local_rank, enabled=rank == 0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    t0 = time.time()
    launches[0] = 0
    ev0.record()
    for _ in range(args.steps):
        sweep()
    ev1.record()
    barrier()
    clocks = sampler.stop(t0, time.time())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"confusion": meter.conf})
    ms = ev0.elapsed_time(ev1)
    n_launch = launches[0]
    total = int(meter.conf.sum())
    miou = float(np.nanmean(meter.metrics()["IoU"]))
    # dominant (only) kernel: one launch over `batch` maps, timed alone
    pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
    for k, (a, b) in enumerate(pairs):
        i = (k * batch) % res
        a.record(); meter.update(d_pred[i:i + batch], d_gt[i:i + batch]); b.record()
    torch.cuda.synchronize()
    k_ms = statistics.mean(a.elapsed_time(b) for a, b in pairs)

    # e2e: evaluation.intersect_and_union_batch on HOST arrays (pinned), result read on the host
    e2e_maps = min(n_local, args.eval_e2e_maps, res)
    h_pred, h_gt = torch.from_numpy(pred[:e2e_maps]).pin_memory(), torch.from_numpy(gt[:e2e_maps]).pin_memory()

    def e2e_sweep():
        tot = None
        for i in range(0, e2e_maps, batch):
            a = M.intersect_and_union_batch(h_pred[i:i + batch], h_gt[i:i + batch], ew.C, 255).sum(0)
            tot = a if tot is None else tot + a
        return tot.cpu()

    e2e_sweep()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_steps = max(1, min(args.steps, 5))
    e0.record()
    for _ in range(e2e_steps):
        areas = e2e_sweep()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    times = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms = times.tolist()
    if rank != 0:
        return
    px = ew.H * ew.W
    peak, peak_src = measured_peak()
    bytes_per_launch = 9 * px * batch
    achieved = bytes_per_launch / (k_ms * 1e-3) / 1e9
    line = {"metric": EVAL_METRIC, "value": ew.maps * px * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": eval_config_dict(ew),
            "notes": {"step": f"one sweep: {ew.maps} maps sharded over {world} rank(s) ({n_local} on rank 0), "
                              f"{batch} maps per launch, {res} distinct maps resident per GPU and cycled, then ONE int64 "
                              f"(C+1)^2 all-reduce", "counted_pixels_last_sweep": total, "mIoU": miou,
                      "maps_per_s": ew.maps * args.steps / (ms * 1e-3)},
            "clocks": clocks,
            "e2e": {"value": e2e_maps * world * px * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": int(9 * px * e2e_maps), "d2h_bytes_per_step": int(areas.numel() * 8),
                    "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps,
                    "api": f"pfst_b200.evaluation.intersect_and_union_batch on pinned host arrays (int64 pred + uint8 gt), "
                           f"{e2e_maps} maps per rank per step (bounded sample of the shard), areas read on the host"},
            "gpu_launches": n_launch,
            "roofline": {"bound": "hbm", "kernel": "confusion_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                         "bytes_per_launch": bytes_per_launch, "us_per_launch": k_ms * 1e3,
                         "timed": f"20 launches alone ({batch} maps each: 9 B/px = int64 pred + uint8 gt)"},
            "sweep_gbs_per_gpu": n_local * 9 * px * args.steps / (ms * 1e-3) / 1e9}
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        n = max(1, min(ew.maps, args.ref_eval_maps))
        cpu_eval_time(ew, min(n, 4))
        t = cpu_eval_time(ew, n)
        line["cpu_baseline"] = {"value": n * px / t, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"oracle intersect_and_union + pre_eval sum on {n} of the {ew.maps} maps ({t:.2f} s)"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS) + sorted(EVAL_WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel eagerly (no CUDA-graph segments)")
    ap.add_argument("--eval-batch", type=int, default=16, help="cfg5: maps per launch")
    ap.add_argument("--eval-resident", type=int, default=64, help="cfg5: distinct maps kept in HBM per GPU")
    ap.add_argument("--eval-e2e-maps", type=int, default=64, help="cfg5: maps per rank per e2e step")
    ap.add_argument("--ref-eval-maps", type=int, default=64, help="cfg5: maps per step of the CPU arms")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0; GPU arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    is_eval = args.workload in EVAL_WORKLOADS
    wl = EVAL_WORKLOADS[args.workload] if is_eval else WORKLOADS[args.workload]
    if args.impl == "reference":
        (run_eval_reference if is_eval else run_reference)(args, wl, rank)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        (run_eval_ours if is_eval else run_ours)(args, wl, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()

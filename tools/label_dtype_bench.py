"""int64 vs uint8 label maps through SelfTrainingStep(graphs=True), cfg1-cfg4 at full size.

For every config: the uint8 step is first checked against the int64 step on the same seeded inputs
(labels, masks, mixed image and weight bit-identical; mu and the proto loss within 1e-5; whenever both
runs' dot maps equal the dots kernel launched alone, DESIGN.md 3.2, also the losses and the logits gradient
bit-identical and grad_x_src within 1e-5), then both are timed with CUDA events, alternating int64 and uint8 legs (warm-up + --steps
each, --rounds alternations). One JSON line per config: us/step per dtype (median and spread of the
legs), algorithmic bytes per dtype (step.algorithmic_bytes), the achieved GB/s, the host-to-device
bytes of gt per step, and the card name and power limit read in the same run.

    python tools/label_dtype_bench.py [--configs cfg1,cfg2,cfg3,cfg4] [--steps 200] [--warmup 20] [--rounds 3]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from pfst_b200 import ops                                               # noqa: E402
from pfst_b200.step import SelfTrainingStep, algorithmic_bytes          # noqa: E402
from pfst_b200.synthetic import WORKLOADS, model_params, step_inputs    # noqa: E402


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (x.strip() for x in out.split(","))
        return {"gpu": name, "power_limit": power}
    except Exception as exc:                     # the numbers are still printed, without the card
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unavailable ({exc})"}


def make_step(wl, dev, graphs=True):
    g = torch.Generator().manual_seed(1234)
    student = [p.to(dev) for p in model_params(wl.C, g)]
    teacher = [p.to(dev) for p in model_params(wl.C, g)]
    down = wl.downscale if wl.downscale != 1.0 else None
    step = SelfTrainingStep(teacher, student, wl.C, wl.D, dev, dilation=wl.dilation, downscale=down,
                            max_batch=max(wl.B, 64), graphs=graphs)
    return step, sum(p.numel() for p in student)


def run(step, it, inp, gt):
    return step.run(it, inp["img"], inp["target_img_strong_aug"], gt, inp["ema_logits"], inp["logits_trg"],
                    inp["x_src"], inp["x_ema"])


def check(wl, inp, dev) -> dict:
    outs = {}
    for dt in (torch.int64, torch.uint8):
        step, _ = make_step(wl, dev)
        np.random.seed(5)
        o = run(step, 0, inp, inp["gt"].to(dt))
        np.random.seed(6)
        o = run(step, 1, inp, inp["gt"].to(dt))
        torch.cuda.synchronize()
        outs[dt] = {k: v.clone() for k, v in o.items()}
        b, geo = next(iter(step._bufs.values()))
        ref = torch.empty_like(b.dots)
        ops.neigh_dots_slot(inp["x_ema"], geo.dilation // geo.up, 0, ref)
        ops.neigh_dots_slot(inp["x_src"], geo.dilation // geo.up, 1, ref)
        torch.cuda.synchronize()
        outs[dt]["dots_exact"] = torch.equal(b.dots, ref)
        step.release_graphs()
    a, b = outs[torch.int64], outs[torch.uint8]
    for k in ("pseudo_label", "mixed_lbl", "mix_masks"):
        assert torch.equal(b[k], a[k].to(torch.uint8)), k
    for k in ("mixed_img", "pseudo_weight", "pseudo_conf"):
        assert torch.equal(a[k], b[k]), k
    rel = lambda k: float((a[k] - b[k]).abs().max() / a[k].abs().max().clamp_min(1e-30))   # noqa: E731
    for k in ("mu", "proto_loss"):
        assert rel(k) <= 1e-5, k
    dots_exact = a["dots_exact"] and b["dots_exact"]
    if dots_exact:
        for k in ("losses", "grad_logits_trg"):
            assert torch.equal(a[k], b[k]), k
        assert rel("grad_x_src") <= 1e-5, "grad_x_src"
    # with inexact dot maps (DESIGN.md 3.2) what depends on them differs whatever the label dtype: recorded
    return {"dots_exact": {"int64": a["dots_exact"], "uint8": b["dots_exact"]},
            "losses_bit_identical": torch.equal(a["losses"], b["losses"]),
            "grad_logits_bit_identical": torch.equal(a["grad_logits_trg"], b["grad_logits_trg"]),
            "grad_x_src_max_rel_diff": rel("grad_x_src"), "mu_max_rel_diff": rel("mu")}


def time_leg(step, inp, gt, it0, warmup, steps) -> float:
    for i in range(warmup):
        run(step, it0 + i, inp, gt)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for i in range(steps):
        run(step, it0 + warmup + i, inp, gt)
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) * 1e3 / steps


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg1,cfg2,cfg3,cfg4")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("label_dtype_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    ops.device_check()
    hw = card()
    for name in args.configs.split(","):
        wl = WORKLOADS[name]
        inp = {k: v.to(dev) for k, v in step_inputs(wl, 1234).items()}
        parity = check(wl, inp, dev)
        steps, n_params = {}, None
        gts = {torch.int64: inp["gt"], torch.uint8: inp["gt"].to(torch.uint8)}
        for dt in gts:
            steps[dt], n_params = make_step(wl, dev)
        legs = {torch.int64: [], torch.uint8: []}
        it = {torch.int64: 0, torch.uint8: 0}
        np.random.seed(7)
        for _ in range(args.rounds):
            for dt in (torch.int64, torch.uint8):
                legs[dt].append(time_leg(steps[dt], inp, gts[dt], it[dt], args.warmup, args.steps))
                it[dt] += args.warmup + args.steps
        h, w = inp["x_src"].shape[2:]
        line = {"config": name, "workload": wl.name, "steps_per_leg": args.steps, "warmup_per_leg": args.warmup,
                "rounds": args.rounds, **hw, "parity": parity}
        for dt, tag in ((torch.int64, "int64"), (torch.uint8, "uint8")):
            us = sorted(legs[dt])
            ab = sum(algorithmic_bytes(wl.B, wl.C, wl.H, wl.W, wl.D, h, w, n_params,
                                       label_bytes=gts[dt].element_size()).values())
            med = us[len(us) // 2]
            line[tag] = {"us_per_step_median": round(med, 2), "us_per_step_legs": [round(u, 2) for u in legs[dt]],
                         "spread_us": round(us[-1] - us[0], 2), "algorithmic_bytes": ab,
                         "GB_per_s": round(ab / (med * 1e-6) / 1e9, 1),
                         "gt_h2d_bytes_per_step": gts[dt].numel() * gts[dt].element_size()}
        line["uint8_speedup"] = round(line["int64"]["us_per_step_median"] / line["uint8"]["us_per_step_median"], 4)
        print(json.dumps(line), flush=True)
        for s in steps.values():
            s.release_graphs()
        del steps, inp
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

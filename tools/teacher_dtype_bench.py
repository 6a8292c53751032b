"""fp32 vs bf16 teacher outputs (ema_logits, x_ema) through SelfTrainingStep(graphs=True), cfg1-cfg4 at full size.

For every config: the bf16 step is first checked against the fp32 step on the upcast tensors (pseudo labels, conf,
mixed image, weights and masks bit-identical; mu and the proto loss within 1e-5; whenever both runs' dot maps equal the
dots kernel launched alone, DESIGN.md 3.2, also the dot maps bit-identical and the losses and both student gradients
within 1e-5),
then three legs are timed with CUDA events, alternated (warm-up + --steps each, --rounds alternations):
  fp32     teacher outputs in fp32;
  bf16     teacher outputs in bf16, handed over as they are;
  upcast   teacher outputs in bf16, upcast with .float() inside the timed region (the workaround without this path).
One JSON line per config: us/step per leg (median and spread), algorithmic bytes (step.algorithmic_bytes with
teacher_bytes 4 / 2), and the card name, power limit and clocks read in the same run.

    python tools/teacher_dtype_bench.py [--configs cfg1,cfg2,cfg3,cfg4] [--steps 200] [--warmup 20] [--rounds 3]
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
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(("gpu", "power_limit", "sm_clock", "sm_clock_max"), (x.strip() for x in out.split(","))))
    except Exception as exc:                     # the numbers are still printed, without the card
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unavailable ({exc})"}


def make_step(wl, dev):
    g = torch.Generator().manual_seed(1234)
    student = [p.to(dev) for p in model_params(wl.C, g)]
    teacher = [p.to(dev) for p in model_params(wl.C, g)]
    down = wl.downscale if wl.downscale != 1.0 else None
    step = SelfTrainingStep(teacher, student, wl.C, wl.D, dev, dilation=wl.dilation, downscale=down,
                            max_batch=max(wl.B, 64), graphs=True)
    return step, sum(p.numel() for p in student)


def run(step, it, inp, el, xe, upcast=False):
    if upcast:
        el, xe = el.float(), xe.float()
    return step.run(it, inp["img"], inp["target_img_strong_aug"], inp["gt"], el, inp["logits_trg"], inp["x_src"], xe)


def check(wl, inp, el16, xe16, dev) -> dict:
    outs = []
    for el, xe in ((el16.float(), xe16.float()), (el16, xe16)):
        step, _ = make_step(wl, dev)
        for it in (0, 1):
            np.random.seed(5 + it)
            o = run(step, it, inp, el, xe)
        torch.cuda.synchronize()
        outs.append({k: v.clone() for k, v in o.items()})
        b, geo = next(iter(step._bufs.values()))
        ref = torch.empty_like(b.dots)
        ops.neigh_dots_slot(xe, geo.dilation // geo.up, 0, ref)
        ops.neigh_dots_slot(inp["x_src"], geo.dilation // geo.up, 1, ref)
        torch.cuda.synchronize()
        outs[-1]["dots"] = b.dots.clone()
        outs[-1]["dots_exact"] = torch.equal(b.dots, ref)
        step.release_graphs()
    a, b = outs
    for k in ("pseudo_label", "pseudo_conf", "count", "mixed_lbl", "mixed_img", "pseudo_weight", "mix_masks"):
        assert torch.equal(a[k], b[k]), k
    rel = lambda k: float((a[k] - b[k]).abs().max() / a[k].abs().max().clamp_min(1e-30))   # noqa: E731
    diffs = {k: rel(k) for k in ("mu", "proto_loss", "losses", "grad_logits_trg", "grad_x_src")}
    assert diffs["mu"] <= 1e-5 and diffs["proto_loss"] <= 1e-5, diffs
    dots_exact = a["dots_exact"] and b["dots_exact"]
    if dots_exact:
        assert torch.equal(a["dots"], b["dots"])
        for k in ("losses", "grad_logits_trg", "grad_x_src"):
            assert diffs[k] <= 1e-5, (k, diffs[k])
    # with inexact dot maps (DESIGN.md 3.2) what depends on them differs whatever the teacher dtype: recorded
    return {"dots_exact": {"fp32": a["dots_exact"], "bf16": b["dots_exact"]}, "max_rel_diff": diffs}


def time_leg(step, inp, el, xe, upcast, it0, warmup, steps) -> float:
    for i in range(warmup):
        run(step, it0 + i, inp, el, xe, upcast)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for i in range(steps):
        run(step, it0 + warmup + i, inp, el, xe, upcast)
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
        sys.exit("teacher_dtype_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    ops.device_check()
    for name in args.configs.split(","):
        wl = WORKLOADS[name]
        inp = {k: v.to(dev) for k, v in step_inputs(wl, 1234).items()}
        el16, xe16 = inp["ema_logits"].bfloat16(), inp["x_ema"].bfloat16()
        el32, xe32 = el16.float(), xe16.float()
        parity = check(wl, inp, el16, xe16, dev)
        legs_in = {"fp32": (el32, xe32, False), "bf16": (el16, xe16, False), "upcast": (el16, xe16, True)}
        steps, n_params = {}, None
        for leg in legs_in:
            steps[leg], n_params = make_step(wl, dev)
        legs = {leg: [] for leg in legs_in}
        it = {leg: 0 for leg in legs_in}
        np.random.seed(7)
        for _ in range(args.rounds):
            for leg, (el, xe, up) in legs_in.items():
                legs[leg].append(time_leg(steps[leg], inp, el, xe, up, it[leg], args.warmup, args.steps))
                it[leg] += args.warmup + args.steps
        h, w = inp["x_src"].shape[2:]
        line = {"config": name, "workload": wl.name, "steps_per_leg": args.steps, "warmup_per_leg": args.warmup,
                "rounds": args.rounds, **card(), "parity": parity}
        for leg in legs_in:
            us = sorted(legs[leg])
            tb = 2 if leg == "bf16" else 4
            ab = sum(algorithmic_bytes(wl.B, wl.C, wl.H, wl.W, wl.D, h, w, n_params, teacher_bytes=tb).values())
            line[leg] = {"us_per_step_median": round(us[len(us) // 2], 2),
                         "us_per_step_legs": [round(u, 2) for u in legs[leg]],
                         "spread_us": round(us[-1] - us[0], 2), "algorithmic_bytes": ab}
        print(json.dumps(line), flush=True)
        for s in steps.values():
            s.release_graphs()
        del steps, inp
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

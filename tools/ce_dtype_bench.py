"""Decode-head loss (upsample_cross_entropy) on fp32 vs 16-bit student logits, forward + backward through autograd.

For every geometry the 16-bit call is first checked against the `.float()` path on the same logits (accuracy
bit-identical, loss within 1e-7 relative, logits gradient bit-identical on all but 1e-3 of the elements and
within one 16-bit ulp except where the contributions nearly cancel, there within 2^-20 of its largest
magnitude: the fp32 atomics' order), then three legs are timed with CUDA events, alternated (--warmup + --iters calls each,
--rounds alternations):
  fp32     fp32 logits;
  direct   16-bit logits handed over as they are;
  upcast   16-bit logits through `.float()` inside the timed region (the workaround without the 16-bit path:
           a cast kernel in the forward; the multiply and the cast's backward in the backward).
Geometries: the decode head of cfg1-cfg4 (H/4 logits, the factor-4 kernel) and an auxiliary FCN head on the
same batches (H/8 logits, the general kernel). Labels are int64 with ignored bands, pixel weights are fp32, and
every call reads its own replica of the inputs, so that one round's working set exceeds the 126 MB L2.
One JSON line per geometry: us per call for each leg (median and spread over the rounds), bytes per call
computed from the shapes, and the card's name and power limit read in the same run.

    python tools/ce_dtype_bench.py [--dtype bf16|fp16] [--iters 200] [--warmup 20] [--rounds 5]
"""
from __future__ import annotations

import argparse
import json
import math
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from pfst_b200 import ops                                       # noqa: E402
from pfst_b200.losses import upsample_cross_entropy             # noqa: E402
from pfst_b200.synthetic import WORKLOADS                       # noqa: E402

L2_BYTES = 126 << 20


def card() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(("gpu", "power_limit", "sm_clock", "sm_clock_max"), (x.strip() for x in out.split(","))))
    except Exception as exc:                     # the numbers are still printed, without the card
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unavailable ({exc})"}


def make_inputs(B, C, H, W, factor, dtype, dev, seed=1234):
    """-> replicas [(z32, z16, label, weight)], one per call of a round."""
    g = torch.Generator().manual_seed(seed)
    lh, lw = H // factor, W // factor
    per = B * C * lh * lw * (4 + 2) + B * H * W * (8 + 4)
    reps = max(2, math.ceil(2 * L2_BYTES / per))
    out = []
    for _ in range(reps):
        z16 = (2.0 * torch.randn((B, C, lh, lw), generator=g)).to(dtype)
        label = torch.randint(0, C, (B, 1, H, W), generator=g)
        label[:, :, 3::17] = 255
        weight = torch.rand((B, H, W), generator=g)
        out.append(tuple(t.to(dev) for t in (z16.float(), z16, label, weight)))
    return out


def call(z, label, weight, upcast):
    x = z.detach().requires_grad_(True)
    loss, acc = upsample_cross_entropy(x.float() if upcast else x, label, weight)
    loss.backward()
    return loss, acc, x.grad


def ordered16(t):
    i = t.contiguous().view(torch.int16).to(torch.int32)
    return torch.where(i < 0, -(i & 0x7fff), i)


def parity(reps) -> dict:
    z32, z16, label, weight = reps[0]
    l_d, a_d, g_d = call(z16, label, weight, False)
    l_u, a_u, g_u = call(z16, label, weight, True)
    assert torch.equal(a_d, a_u), (float(a_d), float(a_u))
    rel = abs(float(l_d) - float(l_u)) / abs(float(l_u))
    assert rel <= 1e-7, rel
    assert g_d.dtype == g_u.dtype == z16.dtype
    d = (ordered16(g_d) - ordered16(g_u)).abs()
    n_off = int((d != 0).sum())
    assert n_off <= max(4, d.numel() // 1000), n_off
    # more than one ulp only where the contributions nearly cancel (fp32 atomics-order noise of the fp32 path)
    far = d > 1
    err = float((g_d.float() - g_u.float())[far].abs().max()) if far.any() else 0.0
    scale = float(g_u.float().abs().max())
    assert err <= 2.0 ** -20 * scale, (int(d.max()), err, scale)
    return {"acc_identical": True, "loss_rel_diff": rel, "grad_max_ulp": int(d.max()), "grad_elems_off": n_off,
            "grad_elems_over_1ulp": int(far.sum()), "grad_over_1ulp_max_abs_err_rel_to_max": err / scale,
            "grad_elems": d.numel()}


def time_leg(reps, leg, warmup, iters) -> float:
    upcast = leg == "upcast"
    idx = 0 if leg == "fp32" else 1
    for i in range(warmup):
        r = reps[i % len(reps)]
        call(r[idx], r[2], r[3], upcast)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for i in range(iters):
        r = reps[i % len(reps)]
        call(r[idx], r[2], r[3], upcast)
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) * 1e3 / iters


def bytes_per_call(B, C, H, W, factor, leg, es) -> int:
    """Algorithmic bytes: the kernel reads the logits, labels and weights once and writes the fp32 gradient
    (zeroed first); the backward reads it and writes the logits' gradient. `upcast` adds the forward cast
    (16-bit read, fp32 write) and its backward (fp32 read, 16-bit write)."""
    n = B * C * (H // factor) * (W // factor)
    core = B * H * W * (8 + 4) + 2 * 4 * n + 4 * n     # labels, weights; fp32 gradient zeroed, written, read
    if leg == "direct":
        return core + es * n + es * n
    out = core + 4 * n + 4 * n                           # fp32 logits read, fp32 gradient written
    return out if leg == "fp32" else out + (es + 4) * n + (4 + es) * n


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg1,cfg2,cfg3,cfg4")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ce_dtype_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    ops.device_check()
    dtype = {"bf16": torch.bfloat16, "fp16": torch.float16}[args.dtype]
    es = 2
    info = card()
    for name in args.configs.split(","):
        wl = WORKLOADS[name]
        for head, factor in (("decode", 4), ("aux_fcn", 8)):
            reps = make_inputs(wl.B, wl.C, wl.H, wl.W, factor, dtype, dev)
            par = parity(reps)
            legs = {leg: [] for leg in ("fp32", "direct", "upcast")}
            for _ in range(args.rounds):
                for leg in legs:
                    legs[leg].append(time_leg(reps, leg, args.warmup, args.iters))
            line = {"config": name, "head": head, "factor": factor, "shape": [wl.B, wl.C, wl.H, wl.W],
                    "dtype": args.dtype, "replicas": len(reps), "iters_per_leg": args.iters,
                    "warmup_per_leg": args.warmup, "rounds": args.rounds, **info, "parity": par}
            for leg, us in legs.items():
                s = sorted(us)
                line[leg] = {"us_per_call_median": round(s[len(s) // 2], 2), "us_per_call_rounds": [round(u, 2) for u in us],
                             "spread_us": round(s[-1] - s[0], 2),
                             "bytes_per_call": bytes_per_call(wl.B, wl.C, wl.H, wl.W, factor, leg, es)}
            print(json.dumps(line), flush=True)
            del reps
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

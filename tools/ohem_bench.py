"""Decode-head loss with an OHEM pixel sampler: the fused path against the reference's op sequence on the GPU.

For every geometry and sampler mode (thresh=0.7, or thresh=None; min_kept=100000 as in mmseg's configs) the
legs are first checked against each other, then timed with CUDA events, alternated (--warmup + --iters calls
each, --rounds alternations), forward + backward through autograd:
  fused      decode_head_losses(seg_logit, seg_label, sampler=OHEMPixelSampler(...)): the map on the device
             (pfst_ohem_weight) from the low-resolution logits, then the fused loss fed that map;
  reference  F.interpolate -> oracle OHEMPixelSampler.sample (soft-max or per-pixel loss, sort, the host
             synchronisation of max(min_threshold, thresh)) -> F.cross_entropy * map -> mean, and accuracy;
  ce         the fused loss without a sampler (for scale);
  sampler    ops.ohem_weight alone (forward only): its algorithmic bytes over its time give its share of the
             HBM peak (7.7 TB/s, the B200 data sheet).
Parity: the fused map may differ from the reference's only at pixels whose float64 key lies within 1e-6
relative of the float64 threshold; the loss is compared with the reference's on the same map.
Geometries: the decode heads of cfg2, cfg3 and cfg4 (H/4 logits) and the factor-8 auxiliary head of cfg2.
Labels are int64 with ignored bands; every call reads its own replica of the inputs, so one round's working set
exceeds the 126 MB L2. One JSON line per geometry and mode, with the card's name and power limit read in the
same run.

    python tools/ohem_bench.py [--iters 100] [--warmup 10] [--rounds 5]
"""
from __future__ import annotations

import argparse
import json
import math
import subprocess
import sys
from pathlib import Path
from types import SimpleNamespace

import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from oracle import ohem as OO, weighted_ce as OC                # noqa: E402
from pfst_b200 import ops                                       # noqa: E402
from pfst_b200.losses import OHEMPixelSampler, decode_head_losses   # noqa: E402
from pfst_b200.synthetic import WORKLOADS                       # noqa: E402

L2_BYTES = 126 << 20
HBM_PEAK = 7.7e12
MIN_KEPT, THRESH = 100000, 0.7
GEOMETRIES = (("cfg2", "decode", 4), ("cfg3", "decode", 4), ("cfg4", "decode", 4), ("cfg2", "aux_fcn", 8))


def card() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(("gpu", "power_limit", "sm_clock", "sm_clock_max"), (x.strip() for x in out.split(","))))
    except Exception as exc:                     # the numbers are still printed, without the card
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unavailable ({exc})"}


def make_inputs(B, C, H, W, factor, dev, seed=1234):
    g = torch.Generator().manual_seed(seed)
    lh, lw = H // factor, W // factor
    per = B * C * lh * lw * 4 + B * H * W * 8
    reps = max(2, math.ceil(2 * L2_BYTES / per))
    out = []
    for _ in range(reps):
        z = 2.0 * torch.randn((B, C, lh, lw), generator=g)
        label = torch.randint(0, C, (B, 1, H, W), generator=g)
        label[:, :, 3::17] = 255
        out.append((z.to(dev), label.to(dev)))
    return out


def call(leg, z, label, sampler, ref_sampler):
    x = z.detach().requires_grad_(True)
    if leg == "fused":
        out = decode_head_losses(x, label, sampler=sampler)
        loss, acc = out["loss_ce"], out["acc_seg"]
    elif leg == "ce":
        out = decode_head_losses(x, label)
        loss, acc = out["loss_ce"], out["acc_seg"]
    else:
        loss, acc, _ = OO.decode_head_losses(x, label, ref_sampler)
    loss.backward()
    return loss, acc


def parity(reps, sampler, ref_sampler) -> dict:
    z, label = reps[0]
    w, _, _ = ops.ohem_weight(z, label, thresh=sampler.thresh, min_kept=sampler.min_kept)
    up64 = F.interpolate(z.double(), label.shape[2:], None, "bilinear", False)
    want = ref_sampler.sample(up64, label)
    lab = label[:, 0]
    valid = lab != 255
    if sampler.thresh is not None:
        key = torch.softmax(up64, 1).gather(1, torch.where(valid, lab, 0)[:, None])[:, 0]
    else:
        key = F.cross_entropy(up64, lab, reduction="none", ignore_index=255)
    srt = key[valid].sort()[0]
    n, kept = srt.numel(), sampler.min_kept * z.shape[0]
    if sampler.thresh is not None:
        kth = float(srt[min(kept, n - 1)])
        thr = sampler.thresh if sampler.thresh > kth else kth
    else:
        thr = float(srt[n - kept]) if kept < n else None
    diff = w.double() != want
    near = (key - thr).abs() <= 1e-6 * abs(thr) if thr is not None else torch.zeros_like(diff)
    assert not bool((diff & ~near).any()), (int(diff.sum()), int((diff & ~near).sum()))
    l_f, a_f = call("fused", z, label, sampler, ref_sampler)
    l_r, a_r, _ = OC.decode_head_losses(z.double(), label, w.double())     # float64, the fused path's map
    rel = abs(float(l_f) - float(l_r)) / abs(float(l_r))
    assert rel <= 1e-5, rel
    return {"pixels": diff.numel(), "map_pixels_differing": int(diff.sum()), "pixels_near_threshold": int(near.sum()),
            "kept": int(w.sum()), "valid": n, "loss_rel_diff_vs_float64": rel}


def time_leg(reps, leg, sampler, ref_sampler, warmup, iters) -> float:
    def one(i):
        z, label = reps[i % len(reps)]
        if leg == "sampler":
            ops.ohem_weight(z, label, thresh=sampler.thresh, min_kept=sampler.min_kept)
        else:
            call(leg, z, label, sampler, ref_sampler)
    for i in range(warmup):
        one(i)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for i in range(iters):
        one(i)
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) * 1e3 / iters


def sampler_bytes(B, C, H, W, factor, topk) -> int:
    """Algorithmic bytes of pfst_ohem_weight: the key pass reads the low-res logits and the int64 labels and
    writes a 4-byte key per pixel; three radix passes read the keys; top-k reads them once more for the tie
    count; the weight pass reads them and writes the fp32 map."""
    N = B * H * W
    return B * C * (H // factor) * (W // factor) * 4 + N * (8 + 4) + 3 * 4 * N + (4 * N if topk else 0) + 8 * N


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ohem_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    ops.device_check()
    info = card()
    head = SimpleNamespace(ignore_index=255, loss_decode=OO.CrossEntropyLoss())
    for name, hname, factor in GEOMETRIES:
        wl = WORKLOADS[name]
        reps = make_inputs(wl.B, wl.C, wl.H, wl.W, factor, dev)
        for mode, thresh in (("thresh", THRESH), ("topk", None)):
            sampler = OHEMPixelSampler(head, thresh=thresh, min_kept=MIN_KEPT)
            ref_sampler = OO.OHEMPixelSampler(head, thresh=thresh, min_kept=MIN_KEPT)
            par = parity(reps, sampler, ref_sampler)
            legs = {leg: [] for leg in ("fused", "reference", "ce", "sampler")}
            for _ in range(args.rounds):
                for leg in legs:
                    legs[leg].append(time_leg(reps, leg, sampler, ref_sampler, args.warmup, args.iters))
            line = {"config": name, "head": hname, "factor": factor, "shape": [wl.B, wl.C, wl.H, wl.W], "mode": mode,
                    "thresh": thresh, "min_kept": MIN_KEPT, "replicas": len(reps), "iters_per_leg": args.iters,
                    "warmup_per_leg": args.warmup, "rounds": args.rounds, **info, "parity": par}
            for leg, us in legs.items():
                s = sorted(us)
                line[leg] = {"us_per_call_median": round(s[len(s) // 2], 2),
                             "us_per_call_rounds": [round(u, 2) for u in us], "spread_us": round(s[-1] - s[0], 2)}
            nbytes = sampler_bytes(wl.B, wl.C, wl.H, wl.W, factor, mode == "topk")
            t = line["sampler"]["us_per_call_median"] * 1e-6
            line["sampler"].update({"bytes_per_call": nbytes, "hbm_share_of_peak": round(nbytes / t / HBM_PEAK, 3)})
            print(json.dumps(line), flush=True)
        del reps
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

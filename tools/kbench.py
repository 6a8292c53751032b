"""Per-kernel micro-benchmark: achieved HBM GB/s of every kernel on its BASELINE shape.

Development tool (bench.py is the contract benchmark). Each kernel is timed with
CUDA events on the launching stream, L2 flushed (256 MB memset) before every
timed launch, median of `--iters` launches after warm-up.

    python tools/kbench.py [--workload cfg2] [--iters 20] [--only ema,pl,...]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from pfst_b200 import ops  # noqa: E402
from pfst_b200.synthetic import WORKLOADS, model_params, step_inputs, eval_maps  # noqa: E402


def peak_gbs() -> float:
    p = Path(__file__).resolve().parent.parent / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"])
    return 6650.0


class Timer:
    """Times `fn(i)` (i = rotating buffer-set index) as a CUDA graph of `reps` launches so
    that host launch overhead does not pollute kernels that run for a few microseconds.
    The rotating sets are sized by the caller to exceed L2 in total; in addition L2 is
    flushed (256 MB memset) before every timed graph replay."""

    def __init__(self, dev, use_graph=True):
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.use_graph = use_graph

    def time(self, fn, sets=1, iters=20, warmup=3, reps=8):
        for i in range(warmup):
            fn(i % sets)
        torch.cuda.synchronize()
        if not self.use_graph:
            reps = 1
            run = lambda: fn(0)
        else:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(sets):
                    fn(i)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for i in range(reps):
                    fn(i % sets)
            run = graph.replay
        ts = []
        for _ in range(iters):
            self.flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            run()
            e.record()
            e.synchronize()
            ts.append(s.elapsed_time(e) * 1e-3 / reps)
        return statistics.median(ts), min(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--only", default="")
    ap.add_argument("--no-graph", action="store_true", help="plain launches (use under ncu)")
    ap.add_argument("--reps", type=int, default=8)
    args = ap.parse_args()
    only = set(filter(None, args.only.split(",")))
    dev = torch.device("cuda:0")
    ops.device_check()
    wl = WORKLOADS[args.workload]
    T = Timer(dev, use_graph=not args.no_graph)
    peak = peak_gbs()
    R = args.reps          # rotating buffer sets == launches per graph: nothing is re-read from L2
    keep = []              # keeps every output of a captured launch alive (distinct addresses)

    def report(name, nbytes, fn):
        keep.clear()
        med, best = T.time(fn, sets=R, iters=args.iters, reps=R)
        row = dict(kernel=name, bytes=nbytes, us_median=round(med * 1e6, 2), us_best=round(best * 1e6, 2),
                   gbs=round(nbytes / med / 1e9, 1), frac_of_measured_peak=round(nbytes / med / 1e9 / peak, 4))
        print(json.dumps(row), flush=True)

    want = lambda n: (not only) or (n in only)
    g = torch.Generator().manual_seed(1234)
    B, C, H, W = wl.B, wl.C, wl.H, wl.W
    P = B * H * W

    if want("ema"):
        student = [p.to(dev) for p in model_params(C, g)]
        teacher = [p.to(dev) for p in model_params(C, g)]
        table = ops.EmaTable(teacher, student)
        a, b = ops.ema_coeffs(5000, 0.999)
        report("ema", 12 * table.total, lambda i: table.update(a, b))
        del student, teacher, table

    inp = step_inputs(wl)
    if want("pl") or want("mix"):
        logits = [inp["ema_logits"].to(dev) + 0.0 for _ in range(R)]
        report("pl", (4 * C + 12) * P, lambda i: keep.append(ops.pseudo_label(logits[i], 0.98)))
        lab, conf, count, _ = ops.pseudo_label(logits[0], 0.98)
    if want("presence") or want("mix"):
        gts = [inp["gt"].to(dev) + 0 for _ in range(R)]
        pres = torch.empty(9, dtype=torch.int32, device=dev)
        report("presence", 8 * P, lambda i: ops.class_presence(gts[i], out=pres))
    if want("mix"):
        del logits
        imgs = [inp["img"].to(dev) + 0.0 for _ in range(R)]
        trgs = [inp["target_img_strong_aug"].to(dev) + 0.0 for _ in range(R)]
        labs = [lab + 0 for _ in range(R)]
        chosen = torch.zeros((B, 8), dtype=torch.int32, device=dev)
        chosen[:, 0] = 0b010101
        # gt 8 + img 12 + trg 12 + pl 8 read; img 12 + lbl 8 + w 4 + mask 8 written  (thre_type='all')
        report("mix", 80 * P, lambda i: keep.append(ops.class_mix(gts[i], chosen, imgs[i], trgs[i], labs[i],
                                                                  count=count, ps_size=P)))
        del imgs, trgs, labs
    keep.clear()

    if want("feat"):
        # the feature-tensor passes (cold: R rotating copies of each 67 MB tensor)
        from pfst_b200 import _lib
        from pfst_b200.prototypes import PrototypeBank
        D, h, w = wl.D, inp["x_src"].shape[2], inp["x_src"].shape[3]
        p = B * h * w
        dil = wl.dilation
        xs = [inp["x_src"].to(dev) + 0.0 for _ in range(R)]
        gt = inp["gt"].to(dev)
        lab3 = gt[:, 0].contiguous()
        bank = PrototypeBank(C, D, dev)
        report("proto_accum(order+stream)", 4 * D * p, lambda i: bank.accumulate(xs[i], lab3))
        report("proto_order", 8 * p, lambda i: bank.order(lab3, B, h, w))
        report("proto_accum_ordered", 4 * D * p, lambda i: bank.accumulate_ordered(xs[i]))
        report("proto_accum_single_launch", 4 * D * p, lambda i: bank.accumulate_single_launch(xs[i], lab3))
        mu = bank.finalize()
        geo = ops.LossGeometry(inp["logits_trg"].shape, inp["x_src"].shape, gt.shape,
                               wl.downscale if wl.downscale != 1.0 else None, dil)
        fd = geo.dilation // geo.up
        dots, ks = ops.neigh_dots_slot(xs[0], fd, 0)
        report("neigh_dots_slot", 4 * D * p, lambda i: ops.neigh_dots_slot(xs[i], fd, 1, dots))
        ops.neigh_dots_slot(xs[1 % R], fd, 1, dots)
        dist = torch.empty((B, h, w), dtype=torch.float32, device=dev)
        acc = torch.empty(4, dtype=torch.float64, device=dev)
        ploss = torch.empty(1, dtype=torch.float32, device=dev)

        def dist_fwd(i):
            _lib.call("pfst_proto_dist_fwd", xs[i].data_ptr(), B, D, h, w, lab3.data_ptr(), _lib.DT_I64, H, W,
                      mu.data_ptr(), bank.seen.data_ptr(), C, dist.data_ptr(), acc.data_ptr(), ploss.data_ptr(),
                      ops._stream())
        report("proto_dist_fwd", 4 * D * p, dist_fwd)
        logits = inp["logits_trg"].to(dev)
        mix = (torch.rand((B, 1, H, W), generator=g) < 0.5).long().to(dev)
        w6 = (0.1,) * 6
        st = {}

        def loss_fwd(i):
            st["v"] = ops.pfgst_loss_fwd(dots, ks, geo, logits, gt, mix, 3, w6, want_vis=False)
        report("pfgst_loss_fwd(prep+stats)", (2 * 5 * 4 * ks + 9 * 4 * 2) * p, loss_fwd)
        gout = torch.ones(6, dtype=torch.float32, device=dev)
        report("pfgst_loss_bwd", (2 * 5 * 4 + 9 * 4) * p,
               lambda i: keep.append(ops.pfgst_loss_bwd(dots, ks, geo, logits, gt, mix, 3, w6, st["v"][1], gout)))
        coef, _ = ops.pfgst_loss_bwd(dots, ks, geo, logits, gt, mix, 3, w6, st["v"][1], gout)
        keep.clear()
        grads = [torch.empty_like(xs[0]) for _ in range(R)]
        report("neigh_grad", 8 * D * p, lambda i: ops.neigh_grad(xs[i], coef, fd, out=grads[i]))
        dist_fwd(0)
        gl = torch.full((1,), 0.1, dtype=torch.float32, device=dev)
        pr = dict(labels=lab3, mu=mu, seen=bank.seen, dist=dist, acc=acc, grad_loss=gl)
        report("neigh_grad_proto", 8 * D * p, lambda i: ops.neigh_grad(xs[i], coef, fd, out=grads[i], proto=pr))

        def dist_bwd(i):
            _lib.call("pfst_proto_dist_bwd", xs[i].data_ptr(), B, D, h, w, lab3.data_ptr(), _lib.DT_I64, H, W,
                      mu.data_ptr(), bank.seen.data_ptr(), C, dist.data_ptr(), acc.data_ptr(), gl.data_ptr(),
                      grads[i].data_ptr(), 0, ops._stream())
        report("proto_dist_bwd", 8 * D * p, dist_bwd)
        del xs, grads
    keep.clear()

    if want("thr"):
        # offline class-wise thresholds: GPU radix select (incl. host permutation + H2D of the index)
        import time
        import numpy as np
        from pfst_b200.pseudo_labeling import cal_threshold
        lg = inp["ema_logits"].to(dev)
        ratios = [0.2, 0.5, 0.8]
        cal_threshold(lg, 0.5, ratios, np.random.RandomState(0))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            cal_threshold(lg, 0.5, ratios, np.random.RandomState(0))
        torch.cuda.synchronize()
        t_gpu = (time.perf_counter() - t0) / 5
        print(json.dumps({"kernel": "class thresholds (sample 0.5 of %d px, incl. host permutation + H2D of the index)" % P,
                          "ms_gpu_path": round(t_gpu * 1e3, 2)}), flush=True)

    if want("ce"):
        # decode-head loss: fused kernel vs the PyTorch op sequence of the reference (both on this GPU)
        import torch.nn.functional as F
        from pfst_b200.losses import upsample_cross_entropy
        lh, lw = H // 4, W // 4
        zs = [(2.0 * torch.randn((B, C, lh, lw), generator=g)).to(dev).requires_grad_(True) for _ in range(R)]
        lab = inp["gt"].to(dev)
        wgt = torch.rand((B, H, W), generator=g).to(dev)
        nbytes = 2 * 4 * C * B * lh * lw + (8 + 4) * P

        def fused(i):
            loss, acc = upsample_cross_entropy(zs[i], lab, wgt)
            loss.backward()
            zs[i].grad = None
        report("weighted_ce fused fwd+bwd", nbytes, fused)

        def torch_ref(i):
            up = F.interpolate(zs[i], (H, W), mode="bilinear", align_corners=False)
            loss = (F.cross_entropy(up, lab[:, 0], reduction="none", ignore_index=255) * wgt).mean()
            (up.argmax(1) == lab[:, 0]).float().sum()
            loss.backward()
            zs[i].grad = None
        report("weighted_ce torch ops fwd+bwd (reference sequence, same GPU)", nbytes, torch_ref)
        del zs
    keep.clear()

    if want("conf"):
        n = 16
        pred, gt = eval_maps(n, 1024, 1024, 6, seed=1)
        dps = [torch.from_numpy(pred).to(dev) + 0 for _ in range(R)]
        dgs = [torch.from_numpy(gt).to(dev) + 0 for _ in range(R)]
        out = torch.zeros((1, 7, 7), dtype=torch.int64, device=dev)
        report("conf_i64_u8", 9 * n * 1024 * 1024, lambda i: ops.confusion_accum(dps[i], dgs[i], 6, out=out))
        outp = torch.zeros((n, 7, 7), dtype=torch.int64, device=dev)
        report("conf_per_image", 9 * n * 1024 * 1024,
               lambda i: ops.confusion_accum(dps[i], dgs[i], 6, per_image=True, out=outp))
        dp8 = [d.to(torch.uint8) for d in dps]
        report("conf_u8_u8", 2 * n * 1024 * 1024, lambda i: ops.confusion_accum(dp8[i], dgs[i], 6, out=out))
        # blocky (realistic) maps and a many-class case
        from pfst_b200.synthetic import blocky_labels
        bl = [blocky_labels(n, 1024, 1024, 6, g)[:, 0].to(dev) for _ in range(2)]
        report("conf_blocky", 16 * n * 1024 * 1024, lambda i: ops.confusion_accum(bl[0], bl[1], 6, out=out))
        p33, g33 = eval_maps(n, 1024, 1024, 33, seed=2)
        d33, l33 = torch.from_numpy(p33).to(dev), torch.from_numpy(g33).to(dev)
        out33 = torch.zeros((1, 34, 34), dtype=torch.int64, device=dev)
        report("conf_c33_random", 9 * n * 1024 * 1024, lambda i: ops.confusion_accum(d33, l33, 33, out=out33))
    keep.clear()

    if want("evallogits"):
        # on-device evaluation input path: fused arg-max + confusion vs arg-max kernel -> confusion kernel
        from pfst_b200.synthetic import blocky_labels, teacher_logits
        n = 8
        lgs = [teacher_logits(n, 6, 1024, 1024, g).to(dev) for _ in range(min(R, 4))]
        gts8 = [blocky_labels(n, 1024, 1024, 6, g)[:, 0].to(torch.uint8).to(dev) for _ in range(min(R, 4))]
        outp = torch.zeros((n, 7, 7), dtype=torch.int64, device=dev)
        px = n * 1024 * 1024
        report("argmax_confusion fused (blocky gt)", (4 * 6 + 1) * px,
               lambda i: ops.argmax_confusion(lgs[i % len(lgs)], gts8[i % len(lgs)], 6, per_image=True, out=outp))

        def two_kernels(i):
            lab = ops.pseudo_label(lgs[i % len(lgs)], 0.0)[0]
            ops.confusion_accum(lab, gts8[i % len(lgs)], 6, per_image=True, out=outp)
        report("argmax kernel -> confusion kernel (same bytes counted)", (4 * 6 + 1) * px, two_kernels)
        rnd = [torch.randn((n, 6, 1024, 1024), generator=g).to(dev) for _ in range(2)]
        rgt = torch.randint(0, 6, (n, 1024, 1024), generator=g).to(torch.uint8).to(dev)
        report("argmax_confusion fused (noise logits, random gt)", (4 * 6 + 1) * px,
               lambda i: ops.argmax_confusion(rnd[i % 2], rgt, 6, per_image=True, out=outp))
        report("argmax only (u8 map out)", (4 * 6 + 1) * px,
               lambda i: keep.append(ops.argmax_confusion(rnd[i % 2], None, return_pred=torch.uint8)))
        del lgs, gts8, rnd
    keep.clear()

    if want("blur"):
        # strong_transform's Gaussian blur of the mixed image (kornia GaussianBlur2d, 51x51 at 512^2)
        imgs = [inp["img"].to(dev) + 0.0 for _ in range(R)]
        outs = [torch.empty_like(imgs[0]) for _ in range(R)]
        for name, sig in (("sigma 1.15 (15 taps)", [1.15] * B), ("sigma 0.65 (9 taps)", [0.65] * B),
                          ("sigma 0.15 (1 tap)", [0.15] * B)):
            report("gaussian_blur " + name, 8 * 3 * P, lambda i: ops.gaussian_blur(imgs[i], sig, out=outs[i]))
        del imgs, outs
    keep.clear()

    if want("sa"):
        # StrongAugmentation on uint8 HWC images: 3 B read + 3 B written per pixel
        from pfst_b200.pipelines import StrongAugmentation
        from pfst_b200 import ops as _ops
        u8 = [torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8).to(dev) for _ in range(R)]
        o8 = [torch.empty_like(u8[0]) for _ in range(R)]
        full = [[(_ops.SA_CONVERT, 1, 12.5), (_ops.SA_SATURATION, 1.3, 0), (_ops.SA_HUE, 9, 0),
                 (_ops.SA_CONVERT, 1.2, 0)]] * B
        light = [[(_ops.SA_CONVERT, 1, 12.5)]] * B
        aug = StrongAugmentation()
        report("photometric_u8 (all four distortions)", 6 * P, lambda i: aug.apply_batch(u8[i], full, out=o8[i]))
        report("photometric_u8 (brightness only)", 6 * P, lambda i: aug.apply_batch(u8[i], light, out=o8[i]))
        del u8, o8
        # colour jitter of the mixed image (kornia ColorJitter restated): 12 B read + 12 B written per pixel
        fimg = [inp["img"].to(dev) + 0.0 for _ in range(R)]
        fout = [torch.empty_like(fimg[0]) for _ in range(R)]
        fac, order = [(0.9, 1.1, 1.15, 0.1)] * B, [[2, 0, 3, 1]] * B
        mean, std = [123.675, 116.28, 103.53], [58.395, 57.12, 57.375]
        report("color_jitter (four transforms, denorm/renorm)", 24 * P,
               lambda i: _ops.color_jitter(fimg[i], fac, order, mean, std, out=fout[i]))
        report("color_jitter (brightness + contrast only)", 24 * P,
               lambda i: _ops.color_jitter(fimg[i], fac, [[0, 1]] * B, mean, std, out=fout[i]))
        del fimg, fout
    print(json.dumps({"peak_gbs": peak, "workload": wl.name, "graph": not args.no_graph}))


if __name__ == "__main__":
    main()

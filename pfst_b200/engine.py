"""PluginEngine — the launch groups of the hot path as the PFGST drop-in issues them.

`PFGST.forward_train` (rsiseg/models/uda/pfgst.py:179-356) has three network passes in its
middle, so the kernels of this package fall into three groups, each entered once per
iteration with the tensors the surrounding passes have just produced:

  teacher_outputs   after the teacher pass ④ : pseudo_label(ema_logits) ║ neigh_dots(x_ema)
                    -> label sort -> proto_accum(x_ema) -> proto_finalize (with the cross-rank
                    peer exchange when distributed)                       S1/S2, L2, P1, P2
  (ClassMix M1/M2 is one eager launch in forward_train: its outputs feed the mixed pass ⑧)
  aux_forward       after the mixed pass ⑧   : neigh_dots(x_src) -> proto_dist_fwd ║ loss
                    statistics (prep + fwd)                               L1-L6, P3 forward
  aux_backward      inside total_loss.backward(): upstream gradients packed into one vector,
                    loss backward, neigh_grad + proto_dist_bwd in one pass  backward of ⑨

The first two groups have fixed input/output addresses per (shape, input pointer) key and are
replayed as CUDA graphs after two eager passes; a trainer whose allocator keeps moving the
network outputs simply stays on the eager launches. The backward group writes into fresh
tensors (autograd may keep or steal them), so it stays eager: three launches.

The EMA update (E2) runs on its own stream from the start of the iteration and is joined
right before the teacher pass — the reference's order (pfgst.py:203-208 before :255).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import _lib, ops
from ._lib import PfstError
from .prototypes import PrototypeBank

LOSS_KEYS = ("loss_src_pos_mean", "loss_src_neg_mean", "loss_src_pos_std", "loss_src_neg_std",
             "loss_sim_pos", "loss_sim_neg")


class _GraphCache:
    """CUDA graphs keyed by (shapes, input addresses): two eager passes, then capture (two
    executable instances used alternately). Gives up (eager for good) when the keys keep changing."""
    MAX_SETS, MAX_MISSES, INSTANCES = 8, 24, 2

    def __init__(self, enabled: bool):
        self.enabled = enabled
        self.seen: dict = {}
        self.graphs: dict = {}
        self.misses = 0
        self.turn = 0

    def run(self, key, fn) -> None:
        if not self.enabled:
            fn()
            return
        g = self.graphs.get(key)
        if g is None:
            n = self.seen.get(key, 0)
            if n < 2 or self.misses >= self.MAX_MISSES:
                if n == 0:
                    self.misses += 1
                    if len(self.seen) > 4 * self.MAX_SETS:
                        self.seen.clear()
                self.seen[key] = n + 1
                fn()
                return
            while len(self.graphs) >= self.MAX_SETS:
                self.graphs.pop(next(iter(self.graphs)))
            g = []
            for _ in range(self.INSTANCES):
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr, capture_error_mode="thread_local"):
                    fn()
                g.append(gr)
            self.graphs[key] = g
        self.turn += 1
        g[self.turn % len(g)].replay()

    def clear(self) -> None:
        self.graphs.clear()
        self.seen.clear()


class PluginEngine:
    def __init__(self, device, num_classes: int, loss_cfg: Optional[dict], proto_cfg: Optional[dict],
                 alpha: float = 0.999, group=None, graphs: Optional[bool] = None):
        self.device = torch.device(device)
        self.C = int(num_classes)
        self.loss_cfg = loss_cfg          # dict(top_k, dilation, downscale, w6)
        self.proto_cfg = proto_cfg        # dict(weight, alpha, conf_threshold) or None
        self.alpha = float(alpha)
        self.group = group
        if graphs is None:
            graphs = os.environ.get("PFST_PLUGIN_GRAPHS", "1") != "0"
        self._ga, self._gb = _GraphCache(graphs), _GraphCache(graphs)
        self.bank: Optional[PrototypeBank] = None
        self._side = torch.cuda.Stream(device=self.device)
        self._ema_stream = torch.cuda.Stream(device=self.device)
        self._ev = [torch.cuda.Event() for _ in range(8)]
        self._bufs: dict = {}
        self._gout = torch.zeros(8, dtype=torch.float32, device=self.device)
        self._token = 0
        self._fwd = None                  # state of the last aux_forward, consumed by aux_backward
        self.ema_blocks_per_sm = int(os.environ.get("PFST_PLUGIN_EMA_BLOCKS_PER_SM", "0"))
        self._ema_pending = False

    # ------------------------------------------------------------------------------- E1/E2
    def launch_ema(self, table: ops.EmaTable, it: int) -> None:
        """E1 (it == 0: teacher <- student) / E2 on the EMA stream, forked from the current one."""
        main = torch.cuda.current_stream()
        self._ev[0].record(main)
        es = self._ema_stream
        es.wait_event(self._ev[0])
        if it == 0:
            table.update(0.0, 1.0, mode=1, blocks_per_sm=self.ema_blocks_per_sm, stream=es.cuda_stream)
        else:
            table.update(*ops.ema_coeffs(it, self.alpha), blocks_per_sm=self.ema_blocks_per_sm, stream=es.cuda_stream)
        self._ev[1].record(es)
        self._ema_pending = True

    def wait_ema(self) -> None:
        """The teacher pass (and anything else that reads the teacher's weights) comes after this."""
        if self._ema_pending:
            torch.cuda.current_stream().wait_event(self._ev[1])
            self._ema_pending = False

    # ------------------------------------------------------------------------- group 1 (S,P)
    def _bank(self, D: int) -> PrototypeBank:
        if self.bank is None:
            import torch.distributed as dist
            self.bank = PrototypeBank(self.C, D, self.device, alpha=self.proto_cfg.get('alpha', self.alpha),
                                      group=self.group)
            if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1 \
                    and os.environ.get("PFST_PEER_REDUCE", "1") != "0":
                self.bank.attach_peer_board()
        return self.bank

    def teacher_outputs(self, ema_logits: torch.Tensor, x_ema: Optional[torch.Tensor], thr: float,
                        thr_vec: Optional[torch.Tensor], want_part: bool, geo: Optional[ops.LossGeometry],
                        label_dtype: torch.dtype = torch.int64):
        """-> (pseudo_label (B,H,W) of label_dtype (int64 or uint8, the dtype of the batch's gt), pseudo_prob
        fp32, count int64[1], part-weight|None). x_ema: the (B,D,h,w) teacher features (None: no loss /
        prototypes on features)."""
        if label_dtype not in ops.LABEL_DTYPES:
            raise TypeError(f"label maps must be torch.int64 or torch.uint8, got {label_dtype}")
        B, Cc, H, W = ema_logits.shape
        ops._dev(ema_logits, "ema_logits", torch.float32)
        use_x = x_ema is not None and (self.loss_cfg is not None or self.proto_cfg is not None)
        if use_x:
            ops._dev(x_ema, "x_ema", torch.float32)
        skey = ("a", tuple(ema_logits.shape), None if not use_x else tuple(x_ema.shape), want_part, label_dtype)
        b = self._bufs.get(skey)
        if b is None:
            e = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.device)  # noqa: E731
            b = dict(label=e((B, H, W), label_dtype), conf=e((B, H, W), torch.float32), count=e((1,), torch.int64),
                     wpart=e((B, H, W), torch.float32) if want_part else None, dots=None, ks=0)
            if use_x and self.loss_cfg is not None:
                Bf, D, h, w = x_ema.shape
                b["ks"] = ops.neigh_dots_splits(Bf, D, h, w)
                b["dots"] = e((b["ks"], 2, Bf, 5, h, w), torch.float32)
            self._bufs[skey] = b
        bank = self._bank(x_ema.shape[1]) if (use_x and self.proto_cfg is not None) else None
        conf_thr = None if self.proto_cfg is None else self.proto_cfg.get('conf_threshold', None)

        def launch():
            main = torch.cuda.current_stream()
            dots_here = b["dots"] is not None
            if dots_here:
                self._ev[2].record(main)
                self._side.wait_event(self._ev[2])
                with torch.cuda.stream(self._side):
                    ops.neigh_dots_slot(x_ema, geo.dilation // geo.up, 0, b["dots"])
                    self._ev[3].record(self._side)
            _lib.call("pfst_pseudo_label_lbl", ema_logits.data_ptr(), B, Cc, H * W, float(thr),
                      None if thr_vec is None else thr_vec.data_ptr(), 0, -1, b["label"].data_ptr(),
                      ops._TORCH2DT[label_dtype], b["conf"].data_ptr(), None if b["wpart"] is None else b["wpart"].data_ptr(),
                      b["count"].data_ptr(), main.cuda_stream)
            masked = bank is not None and bank.masked(x_ema.shape[2], x_ema.shape[3], x_ema)
            if dots_here and not masked:
                main.wait_event(self._ev[3])             # the label sort never runs next to a TMA dots kernel (step.py)
            if bank is not None:
                Bf, D, h, w = x_ema.shape
                cf = b["conf"] if conf_thr is not None else None
                ct = conf_thr if conf_thr is not None else 0.0
                if masked:                               # few classes: one masked launch, runs next to dots(x_ema)
                    bank.accumulate(x_ema, b["label"], cf, ct)
                else:
                    bank.order(b["label"], Bf, h, w, cf, ct)
                    bank.accumulate_ordered(x_ema)       # x_ema again: L2 hits
                bank.finalize_captured(main.cuda_stream)
            if dots_here and masked:
                main.wait_event(self._ev[3])             # join the dots branch

        key = skey + (ema_logits.data_ptr(), None if not use_x else x_ema.data_ptr(), float(thr),
                      None if thr_vec is None else thr_vec.data_ptr())
        self._ga.run(key, launch)
        if bank is not None:
            bank.iter += 1
        self._a = b
        return b["label"], b["conf"], b["count"], b["wpart"]

    # ------------------------------------------------------------------------- group 3 (L,P3)
    def aux_forward(self, logits_trg, x_src, gt, mix_masks, geo: ops.LossGeometry, want_vis: bool):
        """Loss statistics (+ prototype distance) of this iteration. -> (losses fp32[6] buffer,
        weighted prototype loss fp32[1] buffer | None, density | None, eroded | None)."""
        plan = self.aux_plan(logits_trg, x_src, gt, mix_masks, geo, want_vis)
        self.aux_run(plan)
        b = plan["b"]
        return b["losses"], (b["ploss_w"] if plan["bank"] is not None else None), b["density"], b["eroded"]

    def aux_plan(self, logits_trg, x_src, gt, mix_masks, geo: ops.LossGeometry, want_vis: bool) -> dict:
        """Validates the inputs and binds the launch group to its (persistent) output buffers without
        launching anything: plan['b']['losses'] (fp32[6]) and plan['b']['ploss_w'] (fp32[1]) are where
        `aux_run(plan)` will leave the six losses and the weighted prototype distance."""
        cfg = self.loss_cfg
        a = self._a
        if a is None or a["dots"] is None:
            raise PfstError("aux_forward without teacher_outputs(x_ema) in this iteration")
        for name, t, dt in (("logits_trg", logits_trg, torch.float32), ("x_src", x_src, torch.float32)):
            ops._dev(t, name, dt)
        ldt = ops._labels(gt, "gt")                  # int64 or uint8; mix_masks shares gt's dtype
        ops._labels(mix_masks, "mix_masks", like=gt)
        Bf, D, h, w = x_src.shape
        if a["dots"].shape[2:] != (Bf, 5, h, w):
            raise PfstError("PFGSTLoss: x_ema / x_src shape mismatch")
        bank = self.bank if self.proto_cfg is not None else None
        skey = ("b", tuple(logits_trg.shape), tuple(x_src.shape), tuple(gt.shape), want_vis, gt.dtype)
        b = self._bufs.get(skey)
        if b is None:
            e = lambda shape, dt: torch.empty(shape, dtype=dt, device=self.device)  # noqa: E731
            ws_bytes = int(_lib.load().pfst_pfgst_loss_ws_bytes(geo.B, geo.C, geo.fh, geo.fw, geo.up))
            b = dict(ws=e((ws_bytes,), torch.uint8), stats=e((16,), torch.float64), losses=e((6,), torch.float32),
                     dist=e((Bf, h, w), torch.float32), acc=e((4,), torch.float64), ploss=e((1,), torch.float32),
                     ploss_w=e((1,), torch.float32),
                     density=e((geo.B, 1, geo.gh, geo.gw), torch.float32) if want_vis else None,
                     eroded=e((geo.B, 1, geo.gh, geo.gw), torch.uint8) if want_vis else None)
            b["loss_views"] = [b["losses"][i] for i in range(6)]      # 0-dim views handed to the log ledger
            b["ploss_view"] = b["ploss_w"][0]
            self._bufs[skey] = b
        H, W = gt.shape[-2], gt.shape[-1]
        dots, ks = a["dots"], a["ks"]
        w6 = ops._w6(cfg["w6"])
        common = (dots.data_ptr(), ks, geo.B, geo.fh, geo.fw, geo.up, logits_trg.data_ptr(), geo.C, geo.lh, geo.lw,
                  geo.lscale, geo.lscale, gt.data_ptr(), mix_masks.data_ptr(), geo.gt_h, geo.gt_w, geo.dilation,
                  int(cfg["top_k"]), w6, b["ws"].data_ptr(), b["stats"].data_ptr())
        pw = (C.c_float * 1)(float(self.proto_cfg.get('weight', 0.1))) if bank is not None else None
        pp = (C.c_void_p * 1)(b["ploss"].data_ptr())

        def launch():
            main = torch.cuda.current_stream()
            self._ev[4].record(main)
            self._side.wait_event(self._ev[4])
            with torch.cuda.stream(self._side):
                ops.neigh_dots_slot(x_src, geo.dilation // geo.up, 1, dots)
                self._ev[5].record(self._side)
                if bank is not None:
                    _lib.call("pfst_proto_dist_fwd_lbl", x_src.data_ptr(), Bf, D, h, w, gt.data_ptr(), ldt, H, W,
                              bank.mu.data_ptr(), bank.seen.data_ptr(), self.C, b["dist"].data_ptr(),
                              b["acc"].data_ptr(), b["ploss"].data_ptr(), self._side.cuda_stream)
                    _lib.call("pfst_pack_scalars", pp, pw, 1, b["ploss_w"].data_ptr(), self._side.cuda_stream)
                    self._ev[6].record(self._side)
            main.wait_event(self._ev[5])
            _lib.call("pfst_pfgst_loss_fwd_lbl", *common, b["losses"].data_ptr(),
                      None if b["density"] is None else b["density"].data_ptr(),
                      None if b["eroded"] is None else b["eroded"].data_ptr(), *ops.SHIPPED_LOSS_ARGS, ldt, main.cuda_stream)
            if bank is not None:
                main.wait_event(self._ev[6])

        key = skey + (logits_trg.data_ptr(), x_src.data_ptr(), gt.data_ptr(), mix_masks.data_ptr(), dots.data_ptr(),
                      bank is not None)
        return dict(key=key, launch=launch, common=common, w6=w6, b=b, geo=geo, bank=bank, keep=(pw, pp),
                    shapes=(Bf, D, h, w, H, W), ldt=ldt)

    def aux_run(self, plan: dict) -> None:
        self._gb.run(plan["key"], plan["launch"])
        self._token += 1
        plan["token"] = self._token
        self._fwd = plan

    def aux_backward(self, token: int, grads, logits_trg, x_src, gt, need_logits: bool, need_x: bool,
                     scale=(1.0, 1.0)):
        """grads: 7 upstream gradients (0-dim CUDA fp32 tensors or None) of the six losses and of
        the weighted prototype loss. -> (grad_logits | None, grad_x | None), fresh tensors."""
        f = self._fwd
        if f is None or f["token"] != token:
            raise PfstError("backward of an auxiliary-loss tail whose buffers a later forward_train has reused "
                            "(call backward once, in the iteration that produced the loss)")
        s = torch.cuda.current_stream().cuda_stream
        ptrs = (C.c_void_p * 7)()
        keep = []
        for i, g in enumerate(grads):
            if g is None:
                continue
            if not g.is_cuda or g.dtype != torch.float32 or g.numel() != 1:
                g = g.to(device=self.device, dtype=torch.float32).reshape(())
            keep.append(g)
            ptrs[i] = g.data_ptr()
        bank, b, geo = f["bank"], f["b"], f["geo"]
        wa, wp = float(scale[0]), float(scale[1])
        wts = (C.c_float * 7)(wa, wa, wa, wa, wa, wa,
                              wp * float(self.proto_cfg.get('weight', 0.1)) if bank is not None else 0.0)
        _lib.call("pfst_pack_scalars", ptrs, wts, 7, self._gout.data_ptr(), s)
        Bf, D, h, w, H, W = f["shapes"]
        coef = torch.empty((Bf, 9, h, w), dtype=torch.float32, device=self.device)
        glog = torch.empty_like(logits_trg) if need_logits else None
        _lib.call("pfst_pfgst_loss_bwd_lbl", *f["common"], self._gout.data_ptr(), coef.data_ptr(),
                  None if glog is None else glog.data_ptr(), *ops.SHIPPED_LOSS_ARGS, f["ldt"], s)
        gx = None
        if need_x:
            gx = torch.empty_like(x_src)
            d = geo.dilation // geo.up
            if bank is not None:
                _lib.call("pfst_neigh_grad_proto_lbl", x_src.data_ptr(), coef.data_ptr(), Bf, D, h, w, d,
                          gt.data_ptr(), f["ldt"], H, W, bank.mu.data_ptr(), bank.seen.data_ptr(), self.C, b["dist"].data_ptr(),
                          b["acc"].data_ptr(), self._gout.data_ptr() + 24, gx.data_ptr(), s)
            else:
                _lib.call("pfst_neigh_grad", x_src.data_ptr(), coef.data_ptr(), Bf, D, h, w, d, gx.data_ptr(), s)
        return glog, gx

    def close(self) -> None:
        """Collective on multi-rank runs (before destroy_process_group)."""
        torch.cuda.synchronize(self.device)
        self._ga.clear()
        self._gb.clear()
        if self.bank is not None and self.bank.peer is not None:
            self.bank.peer.close()
            self.bank.peer = None


class StepTotalFn(torch.autograd.Function):
    """total_loss of one PFGST.forward_train iteration (pfgst.py:237,310,342,344) as ONE autograd
    node: forward = the auxiliary launch group (loss statistics + prototype distance) followed by
    ONE gather launch that writes every log variable of the iteration into the ledger row and
    forms total = 0 + clean + mix * trg_loss_weight + aux (+ proto); backward hands the upstream
    gradient to the loss scalars of the segmentor and runs the auxiliary backward kernels for
    logits_trg / x_src."""

    @staticmethod
    def forward(ctx, eng, rec, plan, gt, idx, logits_trg, x_src, *vals):
        if plan is not None:
            eng.aux_run(plan)
        total = torch.empty((), dtype=torch.float32, device=eng.device)
        rec.launch(total)
        ctx.eng, ctx.rec, ctx.idx = eng, rec, idx
        ctx.token = plan["token"] if plan is not None else None
        ctx.gt = gt
        if plan is not None:
            ctx.save_for_backward(logits_trg, x_src)
        return total

    @staticmethod
    def backward(ctx, g):
        rec = ctx.rec
        out = []
        for j, i in enumerate(ctx.idx):
            if not ctx.needs_input_grad[7 + j]:
                out.append(None)
                continue
            w = rec.segment_weight(i)
            out.append(g if w == 1.0 else g * w)
        glog = gx = None
        if ctx.token is not None:
            logits_trg, x_src = ctx.saved_tensors
            w_aux, w_proto = rec.aux_weights
            glog, gx = ctx.eng.aux_backward(ctx.token, [g] * 7, logits_trg, x_src, ctx.gt, ctx.needs_input_grad[5],
                                            ctx.needs_input_grad[6], scale=(w_aux, w_proto))
        return (None, None, None, None, None, glog, gx, *out)

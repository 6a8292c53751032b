"""SelfTrainingStep — the whole per-iteration hot path as one sync-light launch
sequence (SURVEY.md §3.2 steps ①②⑤⑥⑦⑨⑩ + north_star P1-P3), given the outputs of the
three network passes. It issues the same kernels as the PFGST drop-in
(pfst_b200/uda/pfgst.py) but calls the forward/backward kernels directly instead of
through autograd, into buffers allocated once, so that no PyTorch kernel and no allocator
call sits between them:

  aux       presence(gt) -> D2H 36 B -> [event]   (own stream)         M1 part 1
  segment A pseudo_label(ema_logits)                                   S1/S2
            neigh_dots(x_ema)            -> dots slot 0                L2
            proto_accum(x_ema, label)    (x_ema re-read from L2)       P1
  eager     EMA update (1 launch, all tensors) on its own stream       E2
            proto_finalize (in place, re-zeroes packed)                P2   (single rank)
            [host: wait event, np.random.choice per image, H2D 256 B]  M1 part 2
  segment B class_mix                                                  M2
            neigh_dots(x_src)            -> dots slot 1                L2
            proto_dist_fwd(x_src, gt)    (x_src re-read from L2)       P3
            pfgst_loss_fwd (prep + statistics)                         L1,L3-L6
            pfgst_loss_bwd                                             backward
            neigh_grad + proto_dist_bwd  (one pass: read x_src, write grad_x)

With more than one rank the NCCL all-reduce of the packed [sums|counts] buffer is issued
(async) right after segment A and segment B is split around it: B1 = everything that does not
need the prototypes (ClassMix, neigh_dots(x_src), the loss statistics and their backward
maps), then proto_finalize — the only place that waits for the all-reduce — then B2 =
prototype distance + the fused backward pass. The collective's latency is hidden behind B1.

Independent kernels run on forked streams so that the latency-bound ones (label sort,
loss statistics, tiny maps) overlap the bandwidth-bound ones: the EMA update (independent
of everything else in the step) runs on its own stream across the whole step, the
pseudo-label kernel next to neigh_dots(x_ema), ClassMix next to neigh_dots(x_src), and the
prototype distance next to the loss statistics; everything is joined before run() returns.
The only host round trip is the 36-byte class-presence read, hidden behind segment A.
With ``graphs=True`` segments A and B are captured once per set of input addresses into CUDA graphs and replayed (the launch-bound part of the step: 10 kernels and
3 memsets become two graph launches). Used by bench.py and __graft_entry__.smoke(); a
trainer that owns its autograd graph can call it in place of the aux-loss section of
forward_train.
"""
from __future__ import annotations

import os
from typing import Optional

import numpy as np
import torch

from . import ops
from .prototypes import PrototypeBank
from .utils.dacs_transforms import ClassMixPlan

W6_DEFAULT = (0.1, 0.1, 0.1, 0.1, 0.1, 0.1)   # src_pos, src_neg, src_pos_std, src_neg_std, sim_pos, sim_neg


class _Buffers:
    """Every output / workspace of one step for a fixed set of input shapes."""

    def __init__(self, dev, B, C, H, W, img_shape, logits_shape, feat_shape, geo: ops.LossGeometry,
                 label_dtype=torch.int64):
        f32, i64 = torch.float32, torch.int64
        e = lambda shape, dt: torch.empty(shape, dtype=dt, device=dev)  # noqa: E731
        # the label maps follow gt's dtype (int64 or uint8)
        self.label, self.conf, self.count = e((B, H, W), label_dtype), e((B, H, W), f32), e((1,), i64)
        self.mixed_img, self.mixed_lbl = e(img_shape, f32), e((B, 1, H, W), label_dtype)
        self.weight, self.mix_mask = e((B, H, W), f32), e((B, 1, H, W), label_dtype)
        Bf, D, h, w = feat_shape
        self.ks = ops.neigh_dots_splits(Bf, D, h, w)
        self.dots = e((self.ks, 2, Bf, 5, h, w), f32)
        self.ws = e((ops.pfgst_loss_ws_bytes(geo),), torch.uint8)
        self.stats, self.losses = e((16,), torch.float64), e((6,), f32)
        self.dist, self.acc, self.ploss = e((Bf, h, w), f32), e((4,), torch.float64), e((1,), f32)
        self.coef, self.grad_logits, self.grad_x = e((Bf, 9, h, w), f32), e(logits_shape, f32), e(feat_shape, f32)


class SelfTrainingStep:
    # launches of THIS library's kernels per run(): presence, pseudo-label, dots(x_ema), proto
    # order + accum, EMA, finalize, mix, dots(x_src), dist fwd, loss prep, loss fwd, loss bwd,
    # grad+dist bwd; memsets, copies and NCCL are not counted
    KERNEL_LAUNCHES = 14
    # executable-graph instances used alternately: launching an instance that is still running makes
    # the host wait for it, so with one instance the host could never run ahead of the device
    GRAPH_INSTANCES = int(os.environ.get("PFST_GRAPH_INSTANCES", "2"))
    # graphs are keyed by the input addresses (a trainer whose allocator hands the network outputs
    # back at the same addresses replays; new addresses trigger a new capture): bounded cache
    MAX_GRAPH_SETS = 8

    def __init__(self, teacher_params, student_params, num_classes: int, feat_dim: int, device,
                 alpha: float = 0.999, pseudo_threshold: float = 0.98, dilation: int = 2, top_k: int = 3,
                 downscale: Optional[float] = 0.5, weights6=W6_DEFAULT, proto_weight: float = 0.1,
                 max_batch: int = 64, group=None, graphs: bool = False,
                 split_for_allreduce: Optional[bool] = None):
        self.device = torch.device(device)
        self.alpha, self.thr = alpha, pseudo_threshold
        self.dilation, self.top_k, self.downscale = dilation, top_k, downscale
        self.w6 = tuple(float(v) for v in weights6)
        self.proto_weight = float(proto_weight)
        self.C, self.D = num_classes, feat_dim
        self.table = ops.EmaTable(teacher_params, student_params)
        self.plan = ClassMixPlan(self.device, max_batch=max_batch)
        self.bank = PrototypeBank(num_classes, feat_dim, self.device, alpha=alpha, group=group)
        self.gout = torch.ones(6, dtype=torch.float32, device=self.device)
        self.gproto = torch.full((1,), self.proto_weight, dtype=torch.float32, device=self.device)
        self.ema_events = None    # optional (start, end) CUDA events around the EMA launch
        self.graphs = bool(graphs)
        self.split_for_allreduce = split_for_allreduce   # None: split segment B only when world_size > 1
        self.ema_blocks_per_sm = int(os.environ.get("PFST_EMA_BLOCKS_PER_SM", "2"))
        self.nccl_in_graph = os.environ.get("PFST_NCCL_IN_GRAPH", "1") != "0"
        # multi-rank P2: one-shot all-reduce over NVLink peer memory inside the finalise kernel
        # (csrc/peer.cu); PFST_PEER_REDUCE=0 falls back to ncclAllReduce between two kernels
        self.peer_reduce = os.environ.get("PFST_PEER_REDUCE", "1") != "0"
        self.split_bwd = os.environ.get("PFST_SPLIT_BWD", "0") == "1"    # loss backward as two launches (coef | grad_logits)
        self._bufs = {}           # shape key -> _Buffers
        self._graphs = {}         # pointer key -> (graph A, graph B)
        # fork/join plumbing: one side stream for the second branch of a segment, one for the EMA
        # The EMA is a full-grid kernel on a lowest-priority stream and every branch of the step DAG is captured on
        # high-priority streams: the EMA's short blocks (4096 floats each) soak up whatever SM slots and HBM
        # bandwidth the DAG leaves free, and a DAG kernel that becomes ready gets the next slots that retire.
        # Measured against the bounded persistent grid (2 blocks/SM, PFST_EMA_BACKGROUND=0): cfg1 135.8 -> 131.6,
        # cfg2 244.3 -> 239.4, cfg3 357.7 -> 348.7 us per step.
        self.ema_background = os.environ.get("PFST_EMA_BACKGROUND", "1") == "1"
        hp = dict(priority=-1) if self.ema_background else {}
        if self.ema_background:
            self.ema_blocks_per_sm = int(os.environ.get("PFST_EMA_BG_BLOCKS", "0"))
        self._side = torch.cuda.Stream(device=self.device, **hp)
        self._hi = torch.cuda.Stream(device=self.device, **hp)
        self._ema_stream = torch.cuda.Stream(device=self.device)
        self._aux = torch.cuda.Stream(device=self.device, priority=-1)   # tiny, latency-critical for the host
        self._comm = torch.cuda.Stream(device=self.device, **hp)
        self._ev = [torch.cuda.Event() for _ in range(10)]
        self._world = None        # world size, resolved on first use
        self._prefetched = None   # data_ptr of the gt whose presence bits are in flight
        self._step_count = 0
        self._ema_it = None       # iteration whose EMA update_teacher() has already launched

    # ------------------------------------------------------------------ segments
    def _segment_a(self, b: _Buffers, ema_logits, x_ema, geo):
        main = torch.cuda.current_stream()
        fork, join = self._ev[0], self._ev[1]
        fork.record(main)
        self._side.wait_event(fork)
        with torch.cuda.stream(self._side):                       # branch 2: L2 on x_ema
            ops.neigh_dots_slot(x_ema, geo.dilation // geo.up, 0, b.dots)
            join.record(self._side)
        ops.launch_pseudo_label(ema_logits, self.thr, None, 0, -1, b.label, b.conf, None, b.count, ops._stream())
        if self.bank.masked(x_ema.shape[2], x_ema.shape[3], x_ema):
            self.bank.accumulate(x_ema, b.label)                  # one masked launch next to dots(x_ema)
            main.wait_event(join)
            return
        main.wait_event(join)                                     # the sort never runs next to a TMA dots kernel
        self.bank.order(b.label, x_ema.shape[0], x_ema.shape[2], x_ema.shape[3])   # label sort: 1 block / tile
        self.bank.accumulate_ordered(x_ema)                       # x_ema again: L2 hits

    def _segment_b(self, b: _Buffers, img, trg_img, gt, chosen, logits_trg, x_src, geo, part="all", mu_ready=None):
        """part 'all': the whole segment (single rank: the prototypes are final before it starts).
        Multi-rank: 'b1' = everything that does not need the prototypes (runs while the NCCL
        all-reduce is in flight), then proto_finalize, then 'b2' = distance forward + fused backward."""
        main = torch.cuda.current_stream()
        s = main.cuda_stream
        bank = self.bank
        fork, dots_done, join = self._ev[2], self._ev[3], self._ev[4]

        def dist_fwd():
            ops.launch_proto_dist_fwd(x_src, gt, bank.mu, bank.seen, b.dist, b.acc, b.ploss, ops._stream())

        if part in ("all", "b1"):
            fork.record(main)
            self._side.wait_event(fork)
            with torch.cuda.stream(self._side):                   # branch 2: the x_src passes
                ops.neigh_dots_slot(x_src, geo.dilation // geo.up, 1, b.dots)
                dots_done.record(self._side)
                if part == "all":
                    if mu_ready is not None:                      # prototypes come from another branch
                        self._side.wait_event(mu_ready)
                    dist_fwd()
                    join.record(self._side)
            ops.launch_class_mix(gt, chosen, img, trg_img, b.label, None, b.count, b.label.numel(), 0, 0,
                                 b.mixed_img, b.mixed_lbl, b.weight, b.mix_mask, s)
            main.wait_event(dots_done)
            loss = self._loss_args(b, gt, logits_trg, geo)
            ops.launch_pfgst_loss_fwd(loss, b.losses, None, None, s)
            # backward of (sum of the six losses + proto_weight * proto loss)
            ops.launch_pfgst_loss_bwd(loss, self.gout, b.coef, b.grad_logits, s)
            if part == "all":
                main.wait_event(join)
        if part == "b2":
            dist_fwd()
        if part in ("all", "b2"):
            ops.launch_neigh_grad_proto(x_src, b.coef, geo.dilation // geo.up, gt, bank.mu, bank.seen, b.dist, b.acc,
                                        self.gproto, b.grad_x, s)

    def _loss_args(self, b: _Buffers, gt, logits_trg, geo):
        return ops.pfgst_loss_args(b.dots, b.ks, geo, logits_trg, gt, b.mix_mask, self.top_k, self.w6, b.ws, b.stats)

    def _multi_rank(self) -> bool:
        if self._world is None:
            import torch.distributed as dist
            self._world = dist.get_world_size(self.bank.group) if dist.is_available() and dist.is_initialized() else 1
            if self._world > 1:
                # first use on every rank (they construct and step symmetrically): one eager collective
                # so that NCCL's lazy communicator set-up never happens inside a graph capture
                dist.all_reduce(torch.zeros(1, device=self.device), group=self.bank.group)
                if self.peer_reduce:
                    self.bank.attach_peer_board()          # collective: IPC handles exchanged once
        return self._world > 1

    def _whole_step(self, b, args_a, args_b, reduce: bool = False):
        """The whole step as ONE stream-ordered DAG (one CUDA graph per step) with its true data
        dependencies — three branches forked from the current stream:

          side    neigh_dots(x_ema) -> [label sort done] -> neigh_dots(x_src)      (inputs only)
          proto   [pseudo_label, dots(x_ema)] -> label sort -> proto_accum(x_ema) -> (cross-rank sum)
                  -> proto_finalize -> [dots(x_src)] -> proto_dist_fwd(x_src)      P1, P2, P3 forward
          main    pseudo_label -> class_mix -> [dots(x_src)] -> loss prep/fwd -> loss bwd ->
                  [proto] -> neigh_grad + proto_dist_bwd                          S, M2, L, backward

        ClassMix and the loss statistics never wait for the prototypes; only the fused backward pass
        does. reduce=True (multi-rank): the cross-rank sum is the peer-board exchange inside the
        finalise kernel (csrc/peer.cu) or, without a board, an ncclAllReduce in front of it.

        Ordering rule found the hard way (DESIGN.md §3.2): the label-sort kernel (`proto_accum_kernel<1>`)
        must never be resident next to a TMA neighbourhood kernel — launched at the same instant inside a
        graph, the dots kernel then returns sums with a few channel boxes wrong (reproducible at 1024^2,
        cause not established). The sort therefore sits BETWEEN the two dots kernels: it waits for
        dots(x_ema) and dots(x_src) waits for it; tests/test_gpu_step_fused.py checks every replay."""
        ema_logits, x_ema, geo = args_a
        img, trg_img, gt, chosen, logits_trg, x_src, _ = args_b
        Bf, _, h, w = x_src.shape
        bank = self.bank
        cur = torch.cuda.current_stream()
        main = cur
        fork, dots_ema, dots_src, pl_done, proto_done, sort_done = (self._ev[i] for i in (0, 1, 2, 3, 4, 8))
        fork.record(cur)
        if self.ema_background:
            main = self._hi
            main.wait_event(fork)
        s = main.cuda_stream
        self._side.wait_event(fork)
        with torch.cuda.stream(self._side):
            ops.neigh_dots_slot(x_ema, geo.dilation // geo.up, 0, b.dots)
            dots_ema.record(self._side)
        ops.launch_pseudo_label(ema_logits, self.thr, None, 0, -1, b.label, b.conf, None, b.count, s)
        pl_done.record(main)
        unsafe = os.environ.get("PFST_DAG_UNSAFE") == "1"           # reproduces DESIGN.md 3.2 (tools/dots_replay_check.py)
        masked = bank.masked(h, w, x_ema)      # few classes: no sort kernel -> nothing to keep away from the TMA kernels
        self._comm.wait_event(pl_done)
        if not masked:
            if not unsafe:
                self._comm.wait_event(dots_ema)
            with torch.cuda.stream(self._comm):
                bank.order(b.label, Bf, h, w)                         # label sort: 1 block / tile
                sort_done.record(self._comm)
            if not unsafe:
                self._side.wait_event(sort_done)
        with torch.cuda.stream(self._side):
            ops.neigh_dots_slot(x_src, geo.dilation // geo.up, 1, b.dots)
            dots_src.record(self._side)
        with torch.cuda.stream(self._comm):
            if masked:
                bank.accumulate(x_ema, b.label)                       # one masked launch (x_ema: L2 hits after dots)
            else:
                bank.accumulate_ordered(x_ema)                        # x_ema again: L2 hits
            if reduce and bank.peer is None:
                import torch.distributed as dist
                dist.all_reduce(bank.packed, op=dist.ReduceOp.SUM, group=bank.group)
            bank.finalize_captured(self._comm.cuda_stream, local_only=not reduce)
            self._comm.wait_event(dots_src)
            ops.launch_proto_dist_fwd(x_src, gt, bank.mu, bank.seen, b.dist, b.acc, b.ploss, self._comm.cuda_stream)
            proto_done.record(self._comm)
        ops.launch_class_mix(gt, chosen, img, trg_img, b.label, None, b.count, b.label.numel(), 0, 0, b.mixed_img,
                             b.mixed_lbl, b.weight, b.mix_mask, s)
        main.wait_event(dots_src)
        loss = self._loss_args(b, gt, logits_trg, geo)
        ops.launch_pfgst_loss_fwd(loss, b.losses, None, None, s)
        if self.split_bwd:
            # the x_src gradient pass only needs the coefficient maps: grad_logits on the idle side stream
            stats_done, logits_done = self._ev[9], self._ev[0]
            stats_done.record(main)
            self._side.wait_event(stats_done)
            ops.launch_pfgst_loss_bwd(loss, self.gout, None, b.grad_logits, self._side.cuda_stream)
            logits_done.record(self._side)
            ops.launch_pfgst_loss_bwd(loss, self.gout, b.coef, None, s)
        else:
            ops.launch_pfgst_loss_bwd(loss, self.gout, b.coef, b.grad_logits, s)
        main.wait_event(proto_done)
        ops.launch_neigh_grad_proto(x_src, b.coef, geo.dilation // geo.up, gt, bank.mu, bank.seen, b.dist, b.acc,
                                    self.gproto, b.grad_x, s)
        if self.split_bwd:
            main.wait_event(logits_done)
        if main is not cur:
            self._ev[9].record(main)
            cur.wait_event(self._ev[9])

    def _captured(self, key, b, args_a, args_b, parts):
        """CUDA graphs for one set of input addresses, captured after a warm-up pass on a side
        stream (CUDA needs first-use initialisation outside a capture). Single rank: [whole step];
        multi-rank: [A, B1, B2] with the all-reduce and proto_finalize between them."""
        if key in self._graphs:
            return self._graphs[key]
        while len(self._graphs) >= self.MAX_GRAPH_SETS:        # inputs keep moving: forget the oldest capture
            self._graphs.pop(next(iter(self._graphs)))
        bank = self.bank
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        snap = [t.clone() for t in (bank.packed, bank.mu, bank.seen, bank.counts, bank.iter_state)]
        with torch.cuda.stream(side):              # warm-up: module load, cudaFuncSetAttribute
            # (no collective in the warm-up: a rank that re-captures alone must not issue an
            # all-reduce its peers do not match; the communicator is initialised in _multi_rank())
            if parts == ("all",) or parts == ("reduce",):
                self._whole_step(b, args_a, args_b, reduce=False)
            else:
                self._segment_a(b, *args_a)
                for part in parts:
                    self._segment_b(b, *args_b, part=part)
        torch.cuda.current_stream().wait_stream(side)
        for t, c in zip((bank.packed, bank.mu, bank.seen, bank.counts, bank.iter_state), snap):
            t.copy_(c)                             # the warm-up touched the prototype bank
        sets = []
        for _ in range(self.GRAPH_INSTANCES):      # ping-pong instances: an executable graph cannot overlap itself
            if parts == ("all",) or parts == ("reduce",):
                graphs = [torch.cuda.CUDAGraph()]
                with torch.cuda.graph(graphs[0]):
                    self._whole_step(b, args_a, args_b, reduce=parts == ("reduce",))
            else:
                graphs = [torch.cuda.CUDAGraph() for _ in range(1 + len(parts))]
                with torch.cuda.graph(graphs[0]):
                    self._segment_a(b, *args_a)
                for g, part in zip(graphs[1:], parts):
                    with torch.cuda.graph(g):
                        self._segment_b(b, *args_b, part=part)
            sets.append(graphs)
        graphs = sets
        self._graphs[key] = graphs
        return graphs

    def close(self) -> None:
        """Collective teardown on multi-rank runs (every rank calls it, before
        destroy_process_group): drops the graphs, then unmaps / frees the peer boards."""
        self.release_graphs()
        if self.bank.peer is not None:
            self.bank.peer.close()
            self.bank.peer = None

    def release_graphs(self) -> None:
        """Drop the captured CUDA graphs. On multi-rank runs they contain NCCL work: release them
        (or the whole object) BEFORE destroying the process group, or the communicator teardown
        can wait forever for resources the graphs still hold."""
        torch.cuda.synchronize(self.device)
        self._graphs.clear()

    def prefetch(self, gt, wait_stream: Optional[torch.cuda.Stream] = None) -> None:
        """M1 part 1 for the NEXT run(): class-presence kernel + its 36-byte D2H on the auxiliary
        stream. `gt` is known as soon as the batch is loaded (long before the network passes that
        precede the hot path), so a trainer calls this early — e.g. right after enqueueing the
        previous step — and run() then never blocks the host: it only finds the bits already there.
        `gt` must already be materialised on the device, or `wait_stream` must be the stream that
        produces it (the auxiliary stream then waits for the work enqueued there so far)."""
        if wait_stream is not None:
            self._ev[7].record(wait_stream)
            self._aux.wait_event(self._ev[7])
        self.plan.start(gt, self._aux)
        self._prefetched = (gt.data_ptr(), tuple(gt.shape))

    def update_teacher(self, it: int) -> None:
        """E1/E2 of iteration `it` — call it BEFORE the teacher forward of that iteration, as the
        reference does (pfgst.py:203-208 precede the teacher pass :255); `teacher_ready()` then makes
        the current stream wait for it. run(it, ...) joins the same launch instead of issuing its
        own. Without this call run() launches the update itself, which is only correct when the
        teacher outputs passed to run() did not come from a forward of this iteration's teacher
        (synthetic network outputs, as in bench.py)."""
        self._launch_ema(it, torch.cuda.current_stream())
        self._ema_it = it

    def teacher_ready(self) -> None:
        torch.cuda.current_stream().wait_event(self._ev[6])

    def _launch_ema(self, it: int, main) -> None:
        """E2 on its own stream (bounded persistent grid): independent of everything else in the
        step, forked from `main` here and joined at the end of run()."""
        ema_fork, ema_done = self._ev[5], self._ev[6]
        ema_fork.record(main)
        es = self._ema_stream
        es.wait_event(ema_fork)
        if self.ema_events is not None:
            self.ema_events[0].record(es)
        if it == 0:
            self.table.update(0.0, 1.0, mode=1, blocks_per_sm=self.ema_blocks_per_sm, stream=es.cuda_stream)
        else:
            self.table.update(*ops.ema_coeffs(it, self.alpha), blocks_per_sm=self.ema_blocks_per_sm,
                              stream=es.cuda_stream)
        if self.ema_events is not None:
            self.ema_events[1].record(es)
        ema_done.record(es)

    # ----------------------------------------------------------------------- run
    def run(self, it: int, img, trg_img, gt, ema_logits, logits_trg, x_src, x_ema, rng=np.random):
        """gt: int64 or uint8; the pseudo labels, ClassMix labels and masks returned have its dtype.
        ema_logits / x_ema: the teacher's outputs in fp32, fp16 or bf16, each in the dtype the teacher pass
        produced (a pass under torch.autocast); every other tensor is fp32."""
        B, H, W = gt.shape[0], gt.shape[-2], gt.shape[-1]
        ops._labels(gt, "gt")
        for name, t, dt in (("img", img, torch.float32), ("target_img", trg_img, torch.float32),
                            ("logits_trg", logits_trg, torch.float32), ("x_src", x_src, torch.float32)):
            ops._dev(t, name, dt)
        ops._teacher(ema_logits, "ema_logits")
        ops._teacher(x_ema, "x_ema")
        skey = (tuple(img.shape), tuple(ema_logits.shape), tuple(logits_trg.shape), tuple(x_src.shape), gt.dtype,
                ema_logits.dtype, x_ema.dtype)
        ent = self._bufs.get(skey)
        if ent is None:
            geo = ops.LossGeometry(logits_trg.shape, x_src.shape, gt.shape, self.downscale, self.dilation)
            ent = (_Buffers(self.device, B, self.C, H, W, img.shape, logits_trg.shape, x_src.shape, geo, gt.dtype),
                   geo)
            self._bufs[skey] = ent
        b, geo = ent
        main = torch.cuda.current_stream()
        # M1: presence bits (prefetched, or computed now on the auxiliary stream), host draw, H2D
        if self._prefetched != (gt.data_ptr(), tuple(gt.shape)):
            self.plan.drop_pending()                   # a prefetch for another batch must not shift the FIFO
            self.prefetch(gt, wait_stream=main)
        self._prefetched = None
        args_a = (ema_logits, x_ema, geo)
        chosen_buf = self.plan._chosen[:B]
        args_b = (img, trg_img, gt, chosen_buf, logits_trg, x_src, geo)
        split = self._multi_rank() if self.split_for_allreduce is None else bool(self.split_for_allreduce)
        # multi-rank: one graph with the collective inside ("reduce"), or three graphs around an
        # eagerly issued all-reduce ("b1","b2") when NCCL graph capture is switched off
        in_one = self._multi_rank() and (self.bank.peer is not None or (self.graphs and self.nccl_in_graph))
        parts = (("reduce",) if in_one else ("b1", "b2")) if split else ("all",)
        graphs = None
        if self.graphs:
            pkey = skey + parts + tuple(t.data_ptr() for t in (img, trg_img, gt, ema_logits, logits_trg, x_src, x_ema))
            sets = self._captured(pkey, b, args_a, args_b, parts)
            graphs = sets[self._step_count % len(sets)]
        self._step_count += 1
        self.plan.choose(rng)                          # waits for the 36-byte copy only
        if self._ema_it != it:                         # not already issued by update_teacher(it)
            self._launch_ema(it, main)                 # E2 on its own stream, joined below
        self._ema_it = None
        if len(parts) == 1:
            # S1/S2, L2(x_ema), P1 -> (all-reduce) P2 -> M2, L2(x_src), P3, L1/L3-L6, backward
            if graphs:
                graphs[0].replay()
            else:
                self._whole_step(b, args_a, args_b, reduce=parts == ("reduce",))
            self.bank.iter += 1
        else:
            if graphs:
                graphs[0].replay()
            else:
                self._segment_a(b, *args_a)
            work = self.bank.all_reduce()             # async NCCL all-reduce of [sums|counts]
            for i, part in enumerate(parts):
                if part == "b2":
                    self.bank.finalize(work, main.cuda_stream)   # P2: the only wait for the all-reduce
                if graphs:
                    graphs[1 + i].replay()
                else:
                    self._segment_b(b, *args_b, part=part)
        mu = self.bank.mu
        main.wait_event(self._ev[6])
        return dict(losses=b.losses, proto_loss=b.ploss, pseudo_label=b.label, pseudo_conf=b.conf, count=b.count,
                    mixed_img=b.mixed_img, mixed_lbl=b.mixed_lbl, pseudo_weight=b.weight, mix_masks=b.mix_mask,
                    grad_x_src=b.grad_x, grad_logits_trg=b.grad_logits, mu=mu)


def algorithmic_bytes(B: int, C: int, H: int, W: int, D: int, h: int, w: int, n_params: int,
                      label_bytes: int = 8, teacher_bytes: int = 4) -> dict:
    """Algorithmic HBM bytes per step and per kernel family — exactly SURVEY.md §8(d)'s figures
    (cfg2: 1.3115 GB): K_ema 12 B/param; K_pl (4C+12) B/px; K_mask+K_mix 84 B/px (presence read 8
    + mix reads 44 + writes 32); K_sim fwd two feature tensors; K_loss bwd read x_src + write grad;
    K_proto one feature read + the labels; K_dist fwd+bwd 3 feature-sized passes. The small loss
    maps (dots, coefficient maps, ~3.7 MB at cfg2) are not counted. label_bytes = bytes of one
    label-map element (8: int64, 1: uint8): the pseudo-label write, the presence read of gt, the two
    label reads and the two label-map writes of the mix, and the label gather of K_proto. teacher_bytes =
    bytes of one element of the teacher's outputs (4: fp32, 2: fp16 / bf16): the ema_logits read of K_pl,
    the x_ema half of K_sim fwd and the feature read of K_proto."""
    P, p, lb, tb = B * H * W, B * h * w, int(label_bytes), int(teacher_bytes)
    return {
        "ema": 12 * n_params,
        "pseudo_label": (tb * C + 4 + lb) * P,
        "class_presence_and_mix": (44 + 5 * lb) * P,
        "neigh_dots": (tb + 4) * D * p,
        "proto_accum": tb * D * p + lb * p,
        "neigh_grad": 2 * 4 * D * p,
        "proto_dist_fwd_bwd": 3 * 4 * D * p,
    }

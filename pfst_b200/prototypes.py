"""Class prototypes (P1-P3): pseudo-feature accumulation, prototype bank and the
feature-to-prototype distance loss. north_star extension — the reference has no
prototype code; the loss is PFGST.masked_feat_dist (rsiseg/models/uda/pfgst.py:168-177)
with f2 = mu[label]. Kernels: csrc/proto.cu.

Multi-GPU: `PrototypeBank.update` accumulates sums (C,D) and counts (C) into ONE
packed fp32 buffer which is exactly the NCCL all-reduce payload (the accumulation
kernel's atomics write straight into it — no pack/copy step).
"""
from __future__ import annotations

import os

from typing import Optional

import torch

from . import _lib, ops
from ._lib import PfstError


def _lab3(labels: torch.Tensor) -> torch.Tensor:
    """(B,1,H,W) or (B,H,W) label map, int64 or uint8 -> contiguous (B,H,W) of the same dtype."""
    if labels.dim() == 4:
        labels = labels[:, 0]
    return labels.contiguous()


class PeerBoard:
    """The multi-rank side of P2: every rank's prototype "board" (inbox + flags) in NVLink peer
    memory, mapped into this process through CUDA IPC handles exchanged over the process group
    (plumbing only: one all_gather_object at construction). `PrototypeBank.finalize_captured`
    then runs pfst_proto_finalize_peer — push, token wait, rank-ordered sum and finalise in ONE
    kernel (csrc/peer.cu) — so no collective call sits on the step's critical path."""

    def __init__(self, num_classes: int, dim: int, device, group=None, timeout_s: float = 10.0):
        import ctypes as C
        import torch.distributed as dist
        self.device = torch.device(device)
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.timeout_ns = int(timeout_s * 1e9)
        lib = _lib.load()
        nbytes = int(lib.pfst_peer_board_bytes(num_classes, dim, self.world, None, None))
        if nbytes <= 0:
            raise PfstError(f"peer board: unsupported C={num_classes}, D={dim}, ranks={self.world}")
        with torch.cuda.device(self.device):
            ptr, handle = C.c_void_p(), C.create_string_buffer(64)
            _lib.call("pfst_peer_alloc", nbytes, C.byref(ptr), handle)
            self._own = ptr.value
            handles = [None] * self.world
            dist.all_gather_object(handles, (self.rank, bytes(handle.raw)), group=group)
            self._opened, bases = [], []
            for r, h in sorted(handles):
                if r == self.rank:
                    bases.append(self._own)
                    continue
                q = C.c_void_p()
                _lib.call("pfst_peer_open", C.create_string_buffer(h, 64), C.byref(q))
                self._opened.append(q.value)
                bases.append(q.value)
        self.boards = torch.tensor(bases, dtype=torch.int64, device=self.device)
        self.status = torch.zeros(2, dtype=torch.int64, device=self.device)
        dist.barrier(group=group)          # every board is mapped everywhere before the first push

    def check(self) -> None:
        """Synchronises; raises if a peer's token did not arrive in time during any step so far."""
        if int(self.status[0].item()) != 0:
            raise PfstError("peer all-reduce: a rank did not publish its prototype chunk within the timeout; "
                            "the prototypes of that step are invalid")

    def close(self) -> None:
        """Collective teardown: nobody unmaps or frees a board a peer may still push into."""
        import torch.distributed as dist
        if self._own is None:
            return
        torch.cuda.synchronize(self.device)
        if dist.is_initialized():
            dist.barrier(group=self.group)
        with torch.cuda.device(self.device):
            for q in self._opened:
                _lib.call("pfst_peer_close", q)
            _lib.call("pfst_peer_free", self._own)
        self._opened, self._own = [], None


class PrototypeBank:
    def __init__(self, num_classes: int, dim: int, device, alpha: float = 0.999, group=None,
                 comm_stream: Optional[torch.cuda.Stream] = None):
        self.peer = None             # PeerBoard: finalize_captured then includes the cross-rank sum
        self.C, self.D = int(num_classes), int(dim)
        self.device = torch.device(device)
        self.alpha = float(alpha)
        self.group = group
        self.iter = 0
        self.packed = torch.zeros(self.C * self.D + self.C, dtype=torch.float32, device=self.device)
        self.mu = torch.zeros((self.C, self.D), dtype=torch.float32, device=self.device)
        self.seen = torch.zeros(self.C, dtype=torch.uint8, device=self.device)
        self.counts = torch.zeros(self.C, dtype=torch.int64, device=self.device)
        self.comm_stream = comm_stream
        self._order_key, self._order_ws = None, None
        self.iter_state = torch.zeros(2, dtype=torch.int64, device=self.device)   # device copy of `iter` (+ counter)

    # P1
    def accumulate(self, feats: torch.Tensor, labels: torch.Tensor, conf: Optional[torch.Tensor] = None,
                   conf_thr: float = 0.0) -> None:
        """packed += [class sums | class counts] of `feats` (fp32, fp16 or bf16) over `labels`. Few classes (`masked`): one
        launch. Otherwise two: the label sort (once per image tile) and the streaming segment-reduce
        (`order` / `accumulate_ordered` can also be issued separately)."""
        ops._teacher(feats, "feats")        # before the label sort is launched
        B, D, h, w = feats.shape
        if self.masked(h, w, feats):        # few classes: one masked-accumulation launch, no sort
            self.accumulate_single_launch(feats, labels, conf, conf_thr)
            return
        self.order(labels, B, h, w, conf, conf_thr)
        self.accumulate_ordered(feats)

    MASKED_MAX_PIXELS = int(os.environ.get("PFST_MASKED_MAX_PIXELS", "16384"))

    def masked(self, h: int, w: int, feats: Optional[torch.Tensor] = None) -> bool:
        """True when `accumulate` for (h, w) feature maps is the single masked-accumulation launch
        (C <= 8, h*w % 4 == 0, not a small plane): no label-sort kernel exists then, so a scheduler has
        nothing to keep away from the TMA neighbourhood kernels (DESIGN.md 3.2)."""
        if feats is not None:
            if feats.data_ptr() % 16:
                return False      # the library then takes the self-contained sort + stream kernel
            # Measured inside the step (background EMA, DESIGN.md 4): the masked launch wins while the batch is
            # too small to fill the GPU with streaming blocks (cfg1, 2 x 4096 px: 131 vs 137 us per step, the
            # sort runs on two blocks); from 32 k feature pixels on the sort + bulk-copy stream kernel
            # interferes less with the kernels next to it (cfg2 228 vs 240 us, cfg3 343 vs 349 us)
            if feats.shape[0] * int(h) * int(w) > self.MASKED_MAX_PIXELS:
                return False
        return bool(_lib.load().pfst_proto_accum_is_masked(self.C, int(h), int(w)))

    def order(self, labels: torch.Tensor, B: int, h: int, w: int, conf: Optional[torch.Tensor] = None,
              conf_thr: float = 0.0) -> None:
        """Class-sorted pixel lists of every (image, tile) into the cached workspace; adds the pixel
        counts to `packed`."""
        labels = _lab3(labels)
        key = (B, h, w)
        if self._order_key != key:
            nbytes = int(_lib.load().pfst_proto_order_ws_bytes(B, h, w, self.C))
            if nbytes <= 0:
                raise PfstError(f"prototype accumulation does not support B={B}, h={h}, w={w}, C={self.C}")
            self._order_ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self._order_key = key
        _lib.call("pfst_proto_order", labels.data_ptr(), ops._labels(labels, "labels"), B, h, w, labels.shape[-2],
                  labels.shape[-1], ops._opt(conf, "conf", torch.float32), float(conf_thr), self.C,
                  self.packed.data_ptr() + 4 * self.C * self.D, self._order_ws.data_ptr(), ops._stream())

    def accumulate_ordered(self, feats: torch.Tensor) -> None:
        B, D, h, w = feats.shape
        if D != self.D:
            raise ValueError("feature dim mismatch")
        if self._order_key != (B, h, w):
            raise PfstError("accumulate_ordered: call order() for this batch geometry first")
        _lib.call("pfst_proto_accum_ordered", feats.data_ptr(), ops._teacher(feats, "feats"), B, D, h, w, self.C,
                  self._order_ws.data_ptr(), self.packed.data_ptr(), ops._stream())

    def accumulate_single_launch(self, feats: torch.Tensor, labels: torch.Tensor,
                                 conf: Optional[torch.Tensor] = None, conf_thr: float = 0.0) -> None:
        """The self-contained kernel (every streaming block sorts its own tile): no workspace."""
        labels = _lab3(labels)
        B, D, h, w = feats.shape
        if D != self.D:
            raise ValueError("feature dim mismatch")
        _lib.call("pfst_proto_accum", feats.data_ptr(), ops._teacher(feats, "feats"), B, D, h, w,
                  labels.data_ptr(), ops._labels(labels, "labels"), labels.shape[-2], labels.shape[-1],
                  ops._opt(conf, "conf", torch.float32), float(conf_thr), self.C, self.packed.data_ptr(),
                  ops._stream())

    def all_reduce(self):
        """Sum the packed [sums | counts] buffer over ranks (NCCL). Returns the async work
        handle (or None); `finalize` waits on it."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self.group) == 1:
            return None
        if self.peer is not None:          # the finalise kernel itself sums over the ranks
            return None
        return dist.all_reduce(self.packed, op=dist.ReduceOp.SUM, group=self.group, async_op=True)

    # P2
    def finalize(self, work=None, stream: Optional[int] = None) -> torch.Tensor:
        """In place (mu / seen keep their addresses); the kernel also zeroes `packed` for the next
        step's accumulation and advances the device-resident iteration, from which it derives the
        prototype-EMA coefficients — no per-step host argument, so the launch is graph-capturable
        (`finalize_captured` below is the same call without the host bookkeeping)."""
        if work is not None:
            work.wait()
        self.finalize_captured(ops._stream() if stream is None else stream)
        self.iter += 1
        return self.mu

    def attach_peer_board(self, timeout_s: float = 10.0) -> "PeerBoard":
        """Collective (every rank of `group` calls it): from now on `finalize_captured` sums the
        packed buffers of all ranks over NVLink peer memory inside the finalise kernel."""
        if self.peer is None:
            self.peer = PeerBoard(self.C, self.D, self.device, self.group, timeout_s)
        return self.peer

    def finalize_captured(self, stream: int, local_only: bool = False) -> None:
        if self.peer is not None and not local_only:
            pb = self.peer
            _lib.call("pfst_proto_finalize_peer", self.packed.data_ptr(), self.C, self.D, self.mu.data_ptr(),
                      self.seen.data_ptr(), float(self.alpha), self.iter_state.data_ptr(), self.mu.data_ptr(),
                      self.counts.data_ptr(), self.seen.data_ptr(), pb.boards.data_ptr(), pb.rank, pb.world,
                      pb.status.data_ptr(), pb.timeout_ns, stream)
            return
        _lib.call("pfst_proto_finalize", self.packed.data_ptr(), self.C, self.D, self.mu.data_ptr(),
                  self.seen.data_ptr(), float(self.alpha), self.iter_state.data_ptr(), self.mu.data_ptr(),
                  self.counts.data_ptr(), self.seen.data_ptr(), 1, stream)

    def update(self, feats, labels, conf=None, conf_thr: float = 0.0) -> torch.Tensor:
        self.accumulate(feats, labels, conf, conf_thr)
        return self.finalize(self.all_reduce())


class _ProtoDistFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, labels, mu, seen):
        feats = feats.contiguous()
        B, _, h, w = feats.shape
        dev = feats.device
        dist = torch.empty((B, h, w), dtype=torch.float32, device=dev)
        acc = torch.empty(4, dtype=torch.float64, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        ops._dev(feats, "feats", torch.float32)
        ops._labels(labels, "labels")
        ops._dev(mu, "mu", torch.float32)
        ops._opt(seen, "seen", torch.uint8)
        ops.launch_proto_dist_fwd(feats, labels, mu, seen, dist, acc, loss, ops._stream())
        ctx.save_for_backward(feats, labels, mu, seen, dist, acc)
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        feats, labels, mu, seen, dist, acc = ctx.saved_tensors
        B, D, h, w = feats.shape
        grad = torch.empty_like(feats)
        g = grad_out.reshape(1).contiguous().float()
        _lib.call("pfst_proto_dist_bwd", feats.data_ptr(), B, D, h, w, labels.data_ptr(),
                  ops._labels(labels, "labels"), labels.shape[-2],
                  labels.shape[-1], mu.data_ptr(), None if seen is None else seen.data_ptr(), mu.shape[0],
                  dist.data_ptr(), acc.data_ptr(), g.data_ptr(), grad.data_ptr(), 0, ops._stream())
        return grad, None, None, None


def proto_dist_loss(feats: torch.Tensor, labels: torch.Tensor, mu: torch.Tensor,
                    seen: Optional[torch.Tensor] = None) -> torch.Tensor:
    """mean_valid ||f_n - mu[y_n]||_2 (mu is treated as a constant, like the detached
    ImageNet features of masked_feat_dist's original use)."""
    return _ProtoDistFn.apply(feats, _lab3(labels), mu.detach().contiguous(), seen)


def proto_dist_all(feats: torch.Tensor, mu: torch.Tensor) -> torch.Tensor:
    B, D, h, w = feats.shape
    C = mu.shape[0]
    out = torch.empty((B, C, h, w), dtype=torch.float32, device=feats.device)
    _lib.call("pfst_proto_dist_all", ops._dev(feats, "feats", torch.float32), B, D, h, w,
              ops._dev(mu, "mu", torch.float32), C, out.data_ptr(), ops._stream())
    return out


class _FeatDistFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, f1, f2, mask):
        f1, f2 = f1.contiguous(), f2.contiguous()
        B, D, h, w = f1.shape
        dev = f1.device
        dist = torch.empty((B, h, w), dtype=torch.float32, device=dev)
        acc = torch.empty(4, dtype=torch.float64, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        _lib.call("pfst_feat_dist_fwd", ops._dev(f1, "f1", torch.float32), ops._dev(f2, "f2", torch.float32),
                  None if mask is None else mask.data_ptr(), B, D, h, w, dist.data_ptr(), acc.data_ptr(),
                  loss.data_ptr(), ops._stream())
        ctx.save_for_backward(f1, f2, dist, acc)
        ctx.mask = mask
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        f1, f2, dist, acc = ctx.saved_tensors
        B, D, h, w = f1.shape
        g1 = torch.empty_like(f1) if ctx.needs_input_grad[0] else None
        g2 = torch.empty_like(f2) if ctx.needs_input_grad[1] else None
        g = grad_out.reshape(1).contiguous().float()
        if g1 is not None or g2 is not None:
            _lib.call("pfst_feat_dist_bwd", f1.data_ptr(), f2.data_ptr(),
                      None if ctx.mask is None else ctx.mask.data_ptr(), B, D, h, w, dist.data_ptr(), acc.data_ptr(),
                      g.data_ptr(), None if g1 is None else g1.data_ptr(), None if g2 is None else g2.data_ptr(),
                      ops._stream())
        return g1, g2, None


def masked_feat_dist(f1: torch.Tensor, f2: torch.Tensor, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """PFGST.masked_feat_dist (rsiseg/models/uda/pfgst.py:168-177): mean over the masked pixels of
    ||f1 - f2||_2 along the channel dim; one forward and one backward launch (csrc/feat_dist.cu)."""
    if f1.shape != f2.shape or f1.dim() != 4:
        raise ValueError("masked_feat_dist: f1 / f2 must be (B,D,h,w) tensors of the same shape")
    m = None
    if mask is not None:
        B, _, h, w = f1.shape
        if mask.numel() != B * h * w:
            raise ValueError("masked_feat_dist: mask must be (B,1,h,w)")
        m = (mask if mask.dtype in (torch.bool, torch.uint8) else mask != 0).contiguous().view(torch.uint8)
        ops._dev(m, "mask", torch.uint8)
    return _FeatDistFn.apply(f1, f2, m)

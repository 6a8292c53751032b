"""SelfTrainingStep (fused launch sequence, eager and CUDA-graph replay) against the CPU
oracle step, and the fused/split kernels it relies on against their unfused forms:
pfst_neigh_dots_slot vs pfst_neigh_dots, pfst_neigh_grad_proto vs pfst_neigh_grad +
pfst_proto_dist_bwd (bit-exact), in-place prototype finalize."""
import numpy as np
import pytest
import torch

from oracle import step as ostep
from pfst_b200 import _lib, ops, prototypes as P
from pfst_b200.step import SelfTrainingStep
from pfst_b200.synthetic import WORKLOADS, blocky_labels, step_inputs

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("B,D,h,w,dil", [(2, 64, 64, 64, 2), (3, 24, 32, 48, 1), (2, 16, 15, 15, 2), (1, 40, 16, 20, 4)])
def test_dots_slot_matches_pair_launch(cuda, B, D, h, w, dil):
    g = torch.Generator().manual_seed(1)
    xa = torch.relu(torch.randn((B, D, h, w), generator=g)).to(cuda)
    xb = torch.relu(torch.randn((B, D, h, w), generator=g)).to(cuda)
    pair, ks2 = ops.neigh_dots(xa, xb, dil)
    slots, ks1 = ops.neigh_dots_slot(xa, dil, 0)
    ops.neigh_dots_slot(xb, dil, 1, slots)
    a, b = pair.double().sum(0), slots.double().sum(0)          # merge the channel splits
    assert a.shape == b.shape == (2, B, 5, h, w)
    assert (a - b).abs().max() <= 1e-5 * a.abs().max()


@pytest.mark.parametrize("B,D,h,w,dil,C,H,W", [(2, 64, 64, 64, 2, 6, 512, 512), (2, 48, 32, 32, 1, 33, 64, 64),
                                                (3, 16, 15, 15, 2, 33, 120, 120), (1, 520, 16, 32, 2, 4, 64, 128)])
def test_fused_grad_proto_is_bit_identical_to_two_tagged_passes(cuda, B, D, h, w, dil, C, H, W):
    g = torch.Generator().manual_seed(2)
    x = torch.relu(torch.randn((B, D, h, w), generator=g)).to(cuda)
    coef = torch.randn((B, 9, h, w), generator=g).to(cuda)
    labels = blocky_labels(B, H, W, C, g, min_rect=2, max_rect=max(4, H // 2))[:, 0].contiguous().to(cuda)
    mu = torch.randn((C, D), generator=g).to(cuda)
    seen = torch.ones(C, dtype=torch.uint8)
    seen[C - 1] = 0
    seen = seen.to(cuda)
    dist = torch.empty((B, h, w), dtype=torch.float32, device=cuda)
    acc = torch.empty(4, dtype=torch.float64, device=cuda)
    loss = torch.empty(1, dtype=torch.float32, device=cuda)
    _lib.call("pfst_proto_dist_fwd", x.data_ptr(), B, D, h, w, labels.data_ptr(), _lib.DT_I64, H, W, mu.data_ptr(),
              seen.data_ptr(), C, dist.data_ptr(), acc.data_ptr(), loss.data_ptr(), ops._stream())
    gl = torch.full((1,), 0.37, dtype=torch.float32, device=cuda)
    two = ops.neigh_grad(x, coef, dil)
    _lib.call("pfst_proto_dist_bwd", x.data_ptr(), B, D, h, w, labels.data_ptr(), _lib.DT_I64, H, W, mu.data_ptr(),
              seen.data_ptr(), C, dist.data_ptr(), acc.data_ptr(), gl.data_ptr(), two.data_ptr(), 1, ops._stream())
    one = ops.neigh_grad(x, coef, dil, proto=dict(labels=labels, mu=mu, seen=seen, dist=dist, acc=acc, grad_loss=gl))
    assert torch.equal(one, two)
    assert float(one.abs().sum()) > 0


def test_finalize_in_place_resets_packed(cuda):
    C, D = 5, 48
    g = torch.Generator().manual_seed(3)
    bank = P.PrototypeBank(C, D, cuda)
    for it in range(3):
        feats = torch.relu(torch.randn((2, D, 8, 8), generator=g)).to(cuda)
        labels = blocky_labels(2, 64, 64, C, g, min_rect=2, max_rect=32).to(cuda)
        mu_ptr = bank.mu.data_ptr()
        bank.update(feats, labels)
        assert bank.mu.data_ptr() == mu_ptr                    # graph-friendly: address is stable
        assert float(bank.packed.abs().sum()) == 0.0           # re-zeroed by the finalize kernel


def _check_step(cuda, wl_name, graphs, iters=(0, 1, 2), split=None):
    wl = WORKLOADS[wl_name]
    host = step_inputs(wl, 1234)
    g = torch.Generator().manual_seed(7)
    shapes = [(), (5,), (4097,), (16, 3, 3, 3), (513,)]
    student = [0.02 * torch.randn(s, generator=g) for s in shapes]
    teacher = [0.02 * torch.randn(s, generator=g) for s in shapes]
    d_student, d_teacher = [p.to(cuda) for p in student], [p.to(cuda) for p in teacher]
    inp = {k: v.to(cuda) for k, v in host.items()}
    step = SelfTrainingStep(d_teacher, d_student, wl.C, wl.D, cuda, dilation=wl.dilation,
                            downscale=wl.downscale if wl.downscale != 1.0 else None, graphs=graphs,
                            split_for_allreduce=split)
    from oracle import pfgst_loss as OL
    cfg = OL.LossCfg(dilation=wl.dilation, downscale=wl.downscale if wl.downscale != 1.0 else None)
    proto_state = None
    for it in iters:
        np.random.seed(100 + it)
        out = step.run(it, inp["img"], inp["target_img_strong_aug"], inp["gt"], inp["ema_logits"],
                       inp["logits_trg"], inp["x_src"], inp["x_ema"])
        rs = np.random.RandomState(100 + it)
        ref = ostep.hot_path_step(it, teacher, student, host, wl.C, loss_cfg=cfg, proto_state=proto_state, rng=rs)
        proto_state = ref["proto_state"]
        torch.cuda.synchronize()
        for a, b in zip(d_teacher, teacher):
            assert torch.equal(a.cpu(), b), "EMA mismatch"
        assert torch.equal(out["mix_masks"].cpu(), ref["mix_masks"])
        assert torch.equal(out["pseudo_label"].cpu(), ref["pseudo_label"])
        safe = (ref["pseudo_conf"] - np.float32(0.98)).abs() > 1e-6
        assert torch.equal(out["pseudo_conf"].cpu().ge(0.98)[safe], ref["large"][safe])
        assert torch.equal(out["mixed_lbl"].cpu(), ref["mixed_lbl"])
        assert torch.equal(out["mixed_img"].cpu(), ref["mixed_img"])
        wo, wr = out["pseudo_weight"].cpu(), ref["pseudo_weight"].reshape(out["pseudo_weight"].shape)
        assert (wo - wr).abs().max() <= 1e-6
        lo, lr = out["losses"].cpu(), ref["losses"]
        assert torch.all((lo - lr).abs() <= 1e-5 * lr.abs() + 1e-9), (it, lo, lr)
        po, pr = float(out["proto_loss"].cpu()), float(ref["proto_loss"])
        assert abs(po - pr) <= 1e-5 * abs(pr), (po, pr)
        mo, mr = out["mu"].cpu(), ref["mu"]
        assert (mo - mr).abs().max() <= 1e-5 * mr.abs().max()
        for key in ("grad_x_src", "grad_logits_trg"):
            go, gr = out[key].cpu(), ref[key]
            if gr is None:
                gr = torch.zeros_like(go)
            assert (go - gr).abs().max() <= 1e-5 * gr.abs().max() + 1e-12, (it, key)


@pytest.mark.parametrize("graphs", [False, True])
@pytest.mark.parametrize("wl_name", ["tiny", "tiny33"])
def test_selftraining_step_matches_oracle(cuda, wl_name, graphs):
    _check_step(cuda, wl_name, graphs)


@pytest.mark.parametrize("graphs", [False, True])
def test_step_split_around_the_allreduce_matches_oracle(cuda, graphs):
    """The multi-rank schedule (segment B split around proto_finalize) on one rank."""
    _check_step(cuda, "tiny", graphs, split=True)


def test_graph_replay_is_bit_identical_to_eager(cuda):
    wl = WORKLOADS["tiny"]
    inp = {k: v.to(cuda) for k, v in step_inputs(wl, 99).items()}
    outs = []
    for graphs in (False, True):
        g = torch.Generator().manual_seed(5)
        stu = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in [(300,), (7, 5)]]
        tea = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in [(300,), (7, 5)]]
        step = SelfTrainingStep(tea, stu, wl.C, wl.D, cuda, graphs=graphs)
        res = []
        for it in range(4):
            np.random.seed(it)
            o = step.run(it, inp["img"], inp["target_img_strong_aug"], inp["gt"], inp["ema_logits"],
                         inp["logits_trg"], inp["x_src"], inp["x_ema"])
            res.append({k: v.clone() for k, v in o.items() if k in
                        ("losses", "pseudo_label", "mixed_img", "mix_masks", "grad_logits_trg", "pseudo_weight")})
        outs.append(res)
    for a, b in zip(*outs):
        for k in a:
            assert torch.equal(a[k], b[k]), k


def test_update_teacher_precedes_the_teacher_forward(cuda):
    """pfgst.py:203-208 update the EMA teacher BEFORE the teacher pass of the same iteration
    (:255). With `update_teacher(it)` + `teacher_ready()` in front of a teacher forward that
    really reads the teacher's weights, two iterations equal the oracle loop in that order."""
    from oracle import ema as oema
    wl = WORKLOADS["tiny"]
    host = step_inputs(wl, 77)
    g = torch.Generator().manual_seed(8)
    shapes = [(wl.C,), (33,)]
    student = [torch.randn(s, generator=g) for s in shapes]
    teacher = [torch.randn(s, generator=g) for s in shapes]
    d_student, d_teacher = [p.to(cuda) for p in student], [p.to(cuda) for p in teacher]
    inp = {k: v.to(cuda) for k, v in host.items()}
    step = SelfTrainingStep(d_teacher, d_student, wl.C, wl.D, cuda, dilation=wl.dilation, downscale=wl.downscale)

    def teacher_forward(params, base):          # a 'network' whose output depends on the teacher's weights
        return (base + 3.0 * params[0].view(1, -1, 1, 1)).contiguous()

    state = None
    for it in range(3):
        with torch.no_grad():                                     # the optimizer moved the student
            for p, q in zip(student, d_student):
                p.add_(0.1 * (it + 1))
                q.add_(0.1 * (it + 1))
        step.update_teacher(it)
        step.teacher_ready()
        ema_logits = teacher_forward(d_teacher, inp["ema_logits"])
        np.random.seed(300 + it)
        out = step.run(it, inp["img"], inp["target_img_strong_aug"], inp["gt"], ema_logits, inp["logits_trg"],
                       inp["x_src"], inp["x_ema"])
        # oracle, reference order: EMA first, then the teacher pass, then the rest of the step
        if it == 0:
            oema.ema_init(teacher, student)
        else:
            oema.ema_update(teacher, student, it, 0.999)
        h = dict(host)
        h["ema_logits"] = teacher_forward(teacher, host["ema_logits"])
        frozen = [t.clone() for t in teacher]
        ref = ostep.hot_path_step(it, frozen, [t.clone() for t in frozen], h, wl.C, proto_state=state,
                                  rng=np.random.RandomState(300 + it))    # (its own EMA of identical tensors is a no-op)
        state = ref["proto_state"]
        torch.cuda.synchronize()
        for a, b in zip(d_teacher, teacher):
            assert torch.equal(a.cpu(), b)
        assert torch.equal(out["pseudo_label"].cpu(), ref["pseudo_label"]), it
        assert torch.equal(out["mixed_lbl"].cpu(), ref["mixed_lbl"])


@pytest.mark.parametrize("name", ["cfg2", "cfg3", "cfg4"])
def test_graph_replays_keep_the_dot_maps_exact(cuda, name):
    """Regression (DESIGN.md §3.2): inside the one-graph DAG every kernel starts the instant its
    dependencies allow. With the label sort resident next to a TMA dots kernel the dots came back
    with a few channel boxes wrong at 1024^2 (cfg3) — on random replays, within tolerance of
    nothing. The schedule now keeps the two apart; here every replay's dot maps must be
    bit-identical to the same kernel launched alone, and the gradient equal to the eager launch
    sequence."""
    wl = WORKLOADS[name]
    inp = {k: v.to(cuda) for k, v in step_inputs(wl, 1234).items()}
    down = wl.downscale if wl.downscale != 1.0 else None
    outs = {}
    for graphs in (False, True):
        g = torch.Generator().manual_seed(3)
        shapes = [(64, 3, 3, 3), (wl.C,), (100003,)]
        student = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in shapes]
        teacher = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in shapes]
        step = SelfTrainingStep(teacher, student, wl.C, wl.D, cuda, dilation=wl.dilation, downscale=down,
                                max_batch=max(wl.B, 64), graphs=graphs)
        for it in range(8 if graphs else 2):
            np.random.seed(5)
            out = step.run(it, inp["img"], inp["target_img_strong_aug"], inp["gt"], inp["ema_logits"],
                           inp["logits_trg"], inp["x_src"], inp["x_ema"])
            torch.cuda.synchronize()
            b, geo = next(iter(step._bufs.values()))
            d = geo.dilation // geo.up
            ref = torch.empty_like(b.dots)
            ops.neigh_dots_slot(inp["x_ema"], d, 0, ref)
            ops.neigh_dots_slot(inp["x_src"], d, 1, ref)
            torch.cuda.synchronize()
            assert torch.equal(b.dots, ref), (name, graphs, it)
            if it == 1:
                outs[graphs] = {k: out[k].clone() for k in ("losses", "grad_x_src", "grad_logits_trg", "mixed_lbl")}
    a, b_ = outs[False], outs[True]
    assert torch.equal(a["mixed_lbl"], b_["mixed_lbl"]) and torch.equal(a["losses"], b_["losses"])
    assert torch.equal(a["grad_logits_trg"], b_["grad_logits_trg"])
    assert (a["grad_x_src"] - b_["grad_x_src"]).abs().max() <= 1e-6 * a["grad_x_src"].abs().max()

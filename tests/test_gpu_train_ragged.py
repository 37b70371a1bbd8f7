"""GPU tests of training on padded batches with per-pair keypoint counts (num_keypoints0/1): the ragged loss-side
kernels against torch / float64 autograd, and whole training steps in both train_precisions against the same pairs run
one at a time, un-padded, through the CPU oracle.  A padded batch with counts must train exactly like its pairs
(DESIGN.md 3.9): the padding's values and the ground truth outside each pair's valid block do not matter."""
import math

import pytest
import torch
import torch.nn.functional as F

from glue_factory_colon_b200 import LightGlue, _abi
from glue_factory_colon_b200._abi import ptr
from glue_factory_colon_b200.padding import pad_and_stack, pad_to_length
from glue_factory_colon_b200.synthetic import make_pairs, to_device
from oracle import loss_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CONF = {"n_layers": 3, "filter_threshold": 0.0, "loss": {"gamma": 1.0, "fn": "nll", "nll_balancing": 0.5}}
N0S, N1S = [300, 129, 1], [260, 260, 77]  # 129 and 260 cross a 128-row tile boundary
LEN0, LEN1 = 320, 280                     # every pair is padded
LOSS_KEYS = ("total", "last", "assignment_nll", "nll_pos", "nll_neg", "num_matchable", "num_unmatchable", "row_norm",
             "confidence")


def _st():
    return torch.cuda.current_stream(DEV).cuda_stream


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _pairs(n0s, n1s, seed=7):
    return [make_pairs(B=1, n0=a, n1=b, seed=seed + i, with_gt=True) for i, (a, b) in enumerate(zip(n0s, n1s))]


def _padded(pairs, len0, len1, fill="random", adversarial=True, seed=123):
    """The pairs padded with padding.pad_and_stack plus the counts.  fill: "random" (the reference's padding modes) or
    "zeros".  adversarial: the padded ground truth points at real keypoints (gt_matches = 0) and gt_assignment is True
    on padded rows and columns; otherwise it is -1 / False."""
    torch.manual_seed(seed)
    kp = dict(mode="random_c", bounds=(0.0, 480.0)) if fill == "random" else dict(mode="zeros")
    ds = dict(mode="random", bounds=(-0.2, 0.2)) if fill == "random" else dict(mode="zeros")
    data = {}
    for i, L in ((0, len0), (1, len1)):
        data[f"keypoints{i}"] = pad_and_stack([p[f"keypoints{i}"][0] for p in pairs], L, -2, **kp)
        data[f"descriptors{i}"] = pad_and_stack([p[f"descriptors{i}"][0] for p in pairs], L, -2, **ds)
        data[f"view{i}"] = {"image_size": torch.cat([p[f"view{i}"]["image_size"] for p in pairs])}
        data[f"num_keypoints{i}"] = torch.tensor([p[f"keypoints{i}"].shape[1] for p in pairs], dtype=torch.int32)
        data[f"gt_matches{i}"] = pad_and_stack([p[f"gt_matches{i}"][0] for p in pairs], L, -1,
                                               mode="zeros" if adversarial else "minus_one")
    ga_mode = "ones" if adversarial else "zeros"
    data["gt_assignment"] = torch.stack([pad_to_length(pad_to_length(p["gt_assignment"][0], len1, -1, mode=ga_mode),
                                                       len0, -2, mode=ga_mode) for p in pairs])
    return data


def _model(train_precision, checkpointed=False, seed=5, train=True, precision="fp32"):
    torch.manual_seed(seed)
    model = LightGlue({**CONF, "checkpointed": checkpointed, "train_precision": train_precision,
                       "precision": precision}).to(DEV)
    return model.train(train)


def _step(data_c, train_precision, checkpointed=False):
    model = _model(train_precision, checkpointed)
    data = to_device(data_c, DEV)
    data["descriptors0"].requires_grad_(True)
    data["descriptors1"].requires_grad_(True)
    model.zero_grad(set_to_none=True)
    pred = model(data)
    losses, _ = model.loss(pred, data)
    losses["total"].mean().backward()
    grads = {k: p.grad for k, p in model.named_parameters()}
    return pred, {k: v.detach() for k, v in losses.items()}, grads, (data["descriptors0"].grad, data["descriptors1"].grad)


def _oracle_pairs(pairs, dtype):
    """Per pair, un-padded: a training step through the CPU oracle with autograd -> (losses per pair [B] each,
    mean over pairs of the parameter gradients, [d descriptors0 / B per pair], [d descriptors1 / B per pair])."""
    sd = {k: v.clone() for k, v in _model("fp32").state_dict().items()}
    B = len(pairs)
    losses, grads, gd0, gd1 = {}, {}, [], []
    for pair in pairs:
        leaves = {k: v.detach().cpu().to(dtype).clone().requires_grad_(True) for k, v in sd.items()
                  if v.is_floating_point() and k != "confidence_thresholds"}
        d = dict(pair)
        d["descriptors0"] = pair["descriptors0"].to(dtype).clone().requires_grad_(True)
        d["descriptors1"] = pair["descriptors1"].to(dtype).clone().requires_grad_(True)
        pred = loss_oracle.forward_collect(leaves, CONF, d, keep_graph=True, dtype=dtype)
        ls, _ = loss_oracle.loss(leaves, CONF, pred, d, True, keep_graph=True)
        ls["total"].mean().backward()
        for k, v in ls.items():
            losses.setdefault(k, []).append(v.detach().double().reshape(-1))
        for k, v in leaves.items():
            grads[k] = grads.get(k, 0.0) + v.grad.double() / B
        gd0.append(d["descriptors0"].grad[0].double() / B)
        gd1.append(d["descriptors1"].grad[0].double() / B)
    return {k: torch.cat(v) for k, v in losses.items()}, grads, gd0, gd1


def _valid_rows(gd, counts):
    return torch.cat([gd[b, : int(c)] for b, c in enumerate(counts)])


def _padded_rows_are_zero(gd, counts):
    return all(float(gd[b, int(c):].abs().max()) == 0.0 for b, c in enumerate(counts) if int(c) < gd.shape[1])


# ---- kernels --------------------------------------------------------------------------------------------------


def test_loss_reduce_ragged_against_torch():
    lib = _abi.load()
    g = torch.Generator().manual_seed(3)
    B, R, C = 4, 201, 150
    counts = [(200, 149), (77, 130), (0, 5), (129, 0)]
    la = ((torch.randn(B, R, C, generator=g) * 3).round() / 2 - 4.0)  # quantised: plenty of exact ties
    la[1, 7, 5] = float("nan")
    la[0, :, 11] = -float("inf")
    gt = torch.rand(B, R - 1, C - 1, generator=g) < 0.02  # True outside the valid blocks too: must be ignored
    lens = torch.tensor(counts, dtype=torch.int32).reshape(-1).to(DEV)
    rows = torch.full((3, B, R - 1), 7.0, device=DEV)
    ra = torch.full((B, R - 1), 7, device=DEV, dtype=torch.int32)
    ca = torch.full((B, C - 1), 7, device=DEV, dtype=torch.int32)
    la_d, gt_d = la.to(DEV), gt.to(DEV)
    rc = lib.lgb200_loss_reduce_ragged(ptr(la_d), B, R, C, ptr(lens), ptr(gt_d), ptr(rows[0]), ptr(rows[1]), ptr(rows[2]),
                                       ptr(ra), ptr(ca), _st())
    assert rc == 0, lib.lgb200_error_string(rc)
    rows, ra, ca = rows.cpu(), ra.cpu(), ca.cpu()
    for b, (n0, n1) in enumerate(counts):
        ri, ci = list(range(n0)) + [R - 1], list(range(n1)) + [C - 1]
        lb = la[b][ri][:, ci]  # the pair un-padded, dustbins last
        inner, gb = lb[:-1, :-1], gt[b, :n0, :n1]
        ok = ~torch.isnan(inner).any(-1)
        torch.testing.assert_close(rows[0, b, :n0][ok], torch.where(gb, inner, torch.zeros_like(inner)).sum(-1)[ok],
                                   atol=1e-4, rtol=1e-5)
        assert torch.equal(rows[1, b, :n0], gb.float().sum(-1))
        torch.testing.assert_close(rows[2, b, :n0][ok], lb[:-1].exp().sum(-1)[ok], atol=1e-5, rtol=1e-5)
        ref_ra = lb[:-1].max(-1).indices
        ref_ca = lb[:, :-1].max(-2).indices
        assert torch.equal(ra[b, :n0].long(), torch.where(ref_ra == n1, C - 1, ref_ra)), b
        assert torch.equal(ca[b, :n1].long(), torch.where(ref_ca == n0, R - 1, ref_ca)), b
        # past the counts: zero sums, arg-maximum -1
        assert float(rows[:, b, n0:].abs().max() if n0 < R - 1 else 0.0) == 0.0
        assert bool((ra[b, n0:] == -1).all()) and bool((ca[b, n1:] == -1).all())


def test_assign_dsim_ragged_against_autograd():
    lib = _abi.load()
    B, m, n, Lp = 3, 150, 131, 256
    counts = [(150, 131), (77, 40), (0, 12)]
    g = torch.Generator().manual_seed(3)
    sim_full = torch.randn(B, m, n, generator=g) * 2
    gt = torch.rand(B, m, n, generator=g) < 0.02  # True outside the valid blocks: never read
    gpos = torch.randn(B, generator=g).double()
    ref = torch.zeros(B, m, n, dtype=torch.float64)
    lse = torch.zeros(2 * B, Lp, dtype=torch.float64)
    gm = torch.zeros(B, m, n, dtype=torch.bool)
    for b, (n0, n1) in enumerate(counts):
        if n0 == 0 or n1 == 0:
            continue
        s = sim_full[b, :n0, :n1].double().requires_grad_(True)
        la = F.log_softmax(s, 1) + F.log_softmax(s, 0)
        ((la * gt[b, :n0, :n1]).sum() * gpos[b]).backward()
        ref[b, :n0, :n1] = s.grad
        lse[2 * b, :n0] = torch.logsumexp(s.detach(), 1)
        lse[2 * b + 1, :n1] = torch.logsumexp(s.detach(), 0)
        gm[b, :n0, :n1] = gt[b, :n0, :n1]
    sim = sim_full.clone()
    for b, (n0, n1) in enumerate(counts):  # outside the valid blocks: NaN, must not be read
        sim[b, n0:] = float("nan")
        sim[b, :, n1:] = float("nan")
    sim_d = sim.to(DEV).contiguous()
    r = (gpos[:, None] * gm.sum(2)).float().to(DEV).contiguous()
    c = (gpos[:, None] * gm.sum(1)).float().to(DEV).contiguous()
    lens = torch.tensor(counts, dtype=torch.int32).reshape(-1).to(DEV)
    lse_d, gt_d, gpos_d = lse.float().to(DEV), gt.to(DEV), gpos.float().to(DEV)  # (kept alive across the launch)
    rc = lib.lgb200_assign_dsim_ragged(ptr(sim_d), B, m, n, ptr(lse_d), Lp, ptr(lens), ptr(gt_d), ptr(gpos_d), ptr(r),
                                       ptr(c), _st())
    assert rc == 0, lib.lgb200_error_string(rc)
    out = sim_d.cpu()
    assert _rel(out, ref) < 1e-5
    for b, (n0, n1) in enumerate(counts):
        assert float(out[b, n0:].abs().max() if n0 < m else 0.0) == 0.0
        assert float(out[b, :, n1:].abs().max() if n1 < n else 0.0) == 0.0


@pytest.mark.parametrize("m,n", [(200, 179), (384, 130)], ids=["ragged", "wide"])
def test_ragged_assign_loss_equals_scores_plus_reduce_ragged(m, n):
    """lgb200_assign_loss with per-pair counts against lgb200_assign_scores + lgb200_loss_reduce_ragged on the same
    operands: arg-maxima identical (-1 past the counts), sums to fp32 rounding (the bounds of
    test_fused_assign_loss_equals_scores_plus_reduce)."""
    lib = _abi.load()
    g = torch.Generator().manual_seed(m + n)
    counts = [(m, n), (m - 71, 129), (0, 33), (5, 0), (130, n - 1)]
    B = len(counts)
    Lp = ((max(m, n) + 127) // 128) * 128
    S = 2 * B
    md = (torch.randn(S, Lp, 256, generator=g) * 0.35).to(DEV).to(torch.bfloat16)  # finite values past the counts
    z = (torch.randn(S, Lp, generator=g) * 2).to(DEV)
    z[0, 3] = 30.0
    z[1, 5] = -30.0
    lens = torch.tensor(counts, dtype=torch.int32).reshape(-1).to(DEV)
    lse = torch.zeros(S, Lp, device=DEV)
    assert lib.lgb200_assign_lse(_abi.BF16, ptr(md), S, Lp, ptr(lens), ptr(lse), _st()) == 0
    R, C = m + 1, n + 1
    gt = (torch.rand(B, m, n, generator=g) < 0.01).to(DEV)  # True outside the valid blocks as well
    sc = torch.empty(B, R, C, device=DEV)
    assert lib.lgb200_assign_scores(_abi.BF16, ptr(md), ptr(z), ptr(lse), B, Lp, ptr(lens), R, C, ptr(sc), None, _st()) == 0
    ref_rows = torch.zeros(3, B, m, device=DEV)
    ref_ra = torch.zeros(B, m, device=DEV, dtype=torch.int32)
    ref_ca = torch.zeros(B, n, device=DEV, dtype=torch.int32)
    assert lib.lgb200_loss_reduce_ragged(ptr(sc), B, R, C, ptr(lens), ptr(gt), ptr(ref_rows[0]), ptr(ref_rows[1]),
                                         ptr(ref_rows[2]), ptr(ref_ra), ptr(ref_ca), _st()) == 0
    rows = torch.full((3, B, m), 7.0, device=DEV)
    ra = torch.zeros(B, m, device=DEV, dtype=torch.int32)
    ca = torch.zeros(B, n, device=DEV, dtype=torch.int32)
    ws = torch.empty(B * (R + C), device=DEV, dtype=torch.int64)
    rc = lib.lgb200_assign_loss(_abi.BF16, ptr(md), ptr(z), ptr(lse), B, Lp, ptr(lens), R, C, ptr(gt), ptr(rows[0]),
                                ptr(rows[1]), ptr(rows[2]), ptr(ra), ptr(ca), ptr(ws), _st())
    assert rc == 0, lib.lgb200_error_string(rc)
    assert torch.equal(rows[1], ref_rows[1])
    torch.testing.assert_close(rows[0], ref_rows[0], atol=1e-4, rtol=1e-5)
    torch.testing.assert_close(rows[2], ref_rows[2], atol=1e-5, rtol=1e-4)
    assert torch.equal(ra, ref_ra) and torch.equal(ca, ref_ca)
    # an empty side: rows past the count -1, the rows of a pair without columns take the dustbin
    assert bool((ra[2] == -1).all()) and bool((ca[3] == -1).all())
    assert bool((ra[3, :5] == n).all()) and bool((ra[3, 5:] == -1).all())


# ---- whole training steps -----------------------------------------------------------------------------------------


@pytest.mark.parametrize("train_precision", ["fp32", "bf16"])
def test_ragged_training_step_against_the_oracle_per_pair(train_precision):
    """fp32: every parameter gradient and both descriptor gradients within 2e-3 (norm-wise) of the mean over pairs of
    the float64 oracle's per-pair gradients, losses within the tolerances of test_gpu_loss.py.  bf16: within 2x of the
    oracle's own bf16 deviation (median tensor, all parameters, descriptors), worst tensor below 0.25, and the forward
    bit-equal to the no-grad bf16 forward with the same counts.  Descriptor gradients are exactly 0 on padded rows;
    kept and checkpointed steps are bit-equal."""
    pairs = _pairs(N0S, N1S)
    data_c = _padded(pairs, LEN0, LEN1)
    pred, losses, grads, gd = _step(data_c, train_precision)
    assert set(losses) == set(LOSS_KEYS)
    l_o, grads_o, gd0_o, gd1_o = _oracle_pairs(pairs, torch.float64)
    for k, p in grads.items():
        assert p is not None and torch.isfinite(p).all(), k
    assert _padded_rows_are_zero(gd[0], N0S) and _padded_rows_are_zero(gd[1], N1S)
    gv0, gv1 = _valid_rows(gd[0], N0S), _valid_rows(gd[1], N1S)
    if train_precision == "fp32":
        for k in LOSS_KEYS:
            torch.testing.assert_close(losses[k].reshape(-1).cpu().double(), l_o[k], atol=5e-4, rtol=1e-4,
                                       msg=lambda msg: f"{k}: {msg}")
        worst = max((_rel(grads[k], grads_o[k]), k) for k in grads_o)
        print(f"ragged fp32 step: worst parameter {worst}, d0 {_rel(gv0, torch.cat(gd0_o)):.2e}, "
              f"d1 {_rel(gv1, torch.cat(gd1_o)):.2e}")
        assert worst[0] < 2e-3, worst
        assert _rel(gv0, torch.cat(gd0_o)) < 2e-3 and _rel(gv1, torch.cat(gd1_o)) < 2e-3
    else:
        _, grads_b, gd0_b, gd1_b = _oracle_pairs(pairs, torch.bfloat16)

        def figures(gp, g0, g1):
            errs = sorted(_rel(gp[k], grads_o[k]) for k in grads_o)
            num = sum(float((gp[k].detach().double().cpu() - grads_o[k]).norm() ** 2) for k in grads_o)
            den = sum(float(grads_o[k].norm() ** 2) for k in grads_o)
            return errs[-1], errs[len(errs) // 2], math.sqrt(num / den), _rel(g0, torch.cat(gd0_o)), _rel(g1, torch.cat(gd1_o))

        env = figures(grads_b, torch.cat(gd0_b), torch.cat(gd1_b))
        got = figures(grads, gv0, gv1)
        print(f"ragged bf16 step: oracle bf16 {tuple(f'{x:.3g}' for x in env)}, ours {tuple(f'{x:.3g}' for x in got)}")
        assert got[0] < 0.25, got
        for i in range(1, 5):
            assert got[i] <= 2.0 * env[i], (i, got, env)
        for k in ("total", "nll_pos", "nll_neg", "confidence", "row_norm"):
            torch.testing.assert_close(losses[k].reshape(-1).cpu().double(), l_o[k], atol=0.05, rtol=0.02,
                                       msg=lambda msg: f"{k}: {msg}")
        # forward: bit-equal to the no-grad bf16 forward with the same counts
        model = _model("bf16", precision="bf16")
        with torch.no_grad():
            ref = model(to_device(data_c, DEV))
        for key in ("log_assignment", "matches0", "matches1", "matching_scores0", "matching_scores1"):
            assert torch.equal(pred[key].detach(), ref[key]), key
        for i, cnts in ((0, N0S), (1, N1S)):
            for b, cnt in enumerate(cnts):
                assert torch.equal(pred[f"ref_descriptors{i}"][b, :, :cnt].detach(), ref[f"ref_descriptors{i}"][b, :, :cnt])
    # the inference layout of a padded batch: dustbins at R-1 / C-1, padded entries 0, matches -1, scores 0
    la = pred["log_assignment"].detach()
    for b, (n0, n1) in enumerate(zip(N0S, N1S)):
        assert float(la[b, n0:-1].abs().max()) == 0.0 and float(la[b, :, n1:-1].abs().max()) == 0.0
        assert bool((pred["matches0"][b, n0:] == -1).all()) and bool((pred["matches1"][b, n1:] == -1).all())
        assert float(pred["matching_scores0"][b, n0:].abs().max()) == 0.0
    # kept and checkpointed: bit-equal
    _, losses_c, grads_c, gd_c = _step(data_c, train_precision, checkpointed=True)
    for k in LOSS_KEYS:
        assert torch.equal(losses_c[k], losses[k]), k
    for k in grads:
        assert torch.equal(grads_c[k], grads[k]), k
    assert torch.equal(gd_c[0], gd[0]) and torch.equal(gd_c[1], gd[1])


@pytest.mark.parametrize("train_precision", ["fp32", "bf16"])
def test_padding_values_and_padded_ground_truth_do_not_matter(train_precision):
    pairs = _pairs(N0S, N1S)
    runs = [_step(_padded(pairs, LEN0, LEN1, fill, adv), train_precision)
            for fill, adv in (("random", True), ("zeros", False), ("random", False))]
    pred0, losses0, grads0, gd0 = runs[0]
    for pred, losses, grads, gd in runs[1:]:
        for k in LOSS_KEYS:
            assert torch.equal(losses[k], losses0[k]), k
        for k in grads0:
            assert torch.equal(grads[k], grads0[k]), k
        assert torch.equal(gd[0], gd0[0]) and torch.equal(gd[1], gd0[1])
        for key in ("log_assignment", "matches0", "matches1", "matching_scores0", "matching_scores1"):
            assert torch.equal(pred[key], pred0[key]), key
        for i, cnts in ((0, N0S), (1, N1S)):
            for b, cnt in enumerate(cnts):
                assert torch.equal(pred[f"ref_descriptors{i}"][b, :, :cnt], pred0[f"ref_descriptors{i}"][b, :, :cnt])


@pytest.mark.parametrize("train_precision", ["fp32", "bf16"])
def test_full_counts_change_nothing(train_precision):
    data_c = make_pairs(B=2, n0=200, n1=170, seed=4, with_gt=True)
    pred_a, losses_a, grads_a, gd_a = _step(data_c, train_precision)
    full = dict(data_c, num_keypoints0=torch.tensor([200, 200]), num_keypoints1=torch.tensor([170, 170]))
    pred_b, losses_b, grads_b, gd_b = _step(full, train_precision)
    for k in LOSS_KEYS:
        assert torch.equal(losses_a[k], losses_b[k]), k
    for k in grads_a:
        assert torch.equal(grads_a[k], grads_b[k]), k
    assert torch.equal(gd_a[0], gd_b[0]) and torch.equal(gd_a[1], gd_b[1])
    for key in ("log_assignment", "matches0", "matches1", "ref_descriptors0", "ref_descriptors1"):
        assert torch.equal(pred_a[key], pred_b[key]), key


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_loss_and_metrics_with_counts_are_per_pair(precision):
    """no_grad validation of a padded batch with counts: losses and metrics against oracle/loss_oracle.loss on each
    pair un-padded (the same prediction cut to the pair, dustbins moved to its last row / column)."""
    pairs = _pairs(N0S, N1S, seed=21)
    data_c = _padded(pairs, LEN0, LEN1)
    model = _model("fp32", train=False, precision=precision)
    sd = model.state_dict()
    with torch.no_grad():
        pred = model(to_device(data_c, DEV))
        losses, metrics = model.loss(pred, to_device(data_c, DEV))
    assert set(losses) == set(LOSS_KEYS) - {"confidence"}
    for b, (n0, n1) in enumerate(zip(N0S, N1S)):
        ri, ci = list(range(n0)) + [LEN0], list(range(n1)) + [LEN1]
        pred_b = {
            "ref_descriptors0": pred["ref_descriptors0"][b:b + 1, :, :n0].cpu(),
            "ref_descriptors1": pred["ref_descriptors1"][b:b + 1, :, :n1].cpu(),
            "log_assignment": pred["log_assignment"][b].cpu()[ri][:, ci][None],
            "matches0": pred["matches0"][b:b + 1, :n0].cpu(),
            "matching_scores0": pred["matching_scores0"][b:b + 1, :n0].cpu(),
        }
        ref_l, ref_m = loss_oracle.loss(sd, CONF, pred_b, pairs[b], False)
        for k, v in ref_l.items():
            got = losses[k][b].cpu().float()
            if precision == "fp32":
                torch.testing.assert_close(got, v.reshape(()).float(), atol=5e-4, rtol=1e-4, msg=lambda m: f"{b} {k}: {m}")
            else:
                torch.testing.assert_close(got, v.reshape(()).float(), atol=0.05, rtol=0.02, msg=lambda m: f"{b} {k}: {m}")
        assert set(ref_m) == set(metrics)
        for k, v in ref_m.items():
            torch.testing.assert_close(metrics[k][b].cpu(), v.reshape(()), atol=1e-5, rtol=1e-5, msg=lambda m: f"{b} {k}: {m}")


@pytest.mark.parametrize("train_precision", ["fp32", "bf16"])
def test_empty_sides_train_and_leave_the_other_pairs_alone(train_precision):
    n0s, n1s = [200, 0, 57, 0], [140, 140, 0, 0]
    pairs = _pairs(n0s, n1s, seed=31)
    _, losses, grads, gd = _step(_padded(pairs, 208, 144), train_precision)
    for k in LOSS_KEYS:
        assert torch.isfinite(losses[k]).all(), k
    for k, g in grads.items():
        assert torch.isfinite(g).all(), k
    assert torch.isfinite(gd[0]).all() and torch.isfinite(gd[1]).all()
    assert _padded_rows_are_zero(gd[0], n0s) and _padded_rows_are_zero(gd[1], n1s)
    full = _pairs([200] * 4, [140] * 4, seed=31)  # pair 0 identical, pairs 1-3 at full counts
    _, losses_f, _, _ = _step(_padded(full, 208, 144), train_precision)
    for k in LOSS_KEYS:
        assert torch.equal(losses[k][0], losses_f[k][0]), k


@pytest.mark.parametrize("train_precision", ["fp32", "bf16"])
def test_ragged_training_reduces_the_loss(train_precision):
    model = _model(train_precision, seed=0)
    data = to_device(_padded(_pairs([128, 90], [100, 128], seed=4), 144, 136), DEV)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    hist = []
    for _ in range(6):
        opt.zero_grad(set_to_none=True)
        losses, _ = model.loss(model(data), data)
        loss = losses["total"].mean()
        loss.backward()
        opt.step()
        hist.append(float(loss.detach()))
    assert all(math.isfinite(x) for x in hist) and hist[-1] < hist[0] - 0.05, hist

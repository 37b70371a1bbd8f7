"""GPU tests of training through `log_assignment`, `matching_scores0/1` and the keypoints: lgb200_assign_bwd against
float64 autograd of the double softmax with dustbins, and whole training steps whose loss reads those outputs and whose
keypoints (scales, orientations) require grad, against autograd through the float64 CPU oracle -- its filter_matches
included -- in both train_precisions, on full and on padded batches."""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

from glue_factory_colon_b200 import LightGlue, _abi
from glue_factory_colon_b200._abi import ptr
from glue_factory_colon_b200.padding import pad_and_stack, pad_to_length
from glue_factory_colon_b200.synthetic import make_pairs, to_device
from oracle import lightglue_oracle, loss_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CONF = {"n_layers": 3, "filter_threshold": 0.1, "loss": {"gamma": 1.0, "fn": "nll", "nll_balancing": 0.5}}
KPT_KEYS = ("keypoints0", "keypoints1", "scales0", "scales1", "oris0", "oris1")


def _st():
    return torch.cuda.current_stream(DEV).cuda_stream


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


# ---- the kernel -------------------------------------------------------------------------------------------------


def _assign_bwd(G, sim, lse, Lp, lens, z):
    """lgb200_assign_bwd on device copies -> (d sim, dz0, dz1) on the CPU."""
    lib = _abi.load()
    B, m, n = sim.shape
    G_d, sim_d, lse_d, z_d = G.to(DEV), sim.to(DEV).contiguous(), lse.to(DEV), z.to(DEV)
    lens_d = None if lens is None else torch.tensor(lens, dtype=torch.int32).reshape(-1).to(DEV)
    dz0, dz1 = torch.full((B, m), 7.0, device=DEV), torch.full((B, n), 7.0, device=DEV)
    n_ws = ctypes.c_longlong(0)
    assert lib.lgb200_assign_bwd_workspace(B, m, n, ctypes.byref(n_ws)) == 0
    ws = torch.full((n_ws.value,), float("nan"), device=DEV)
    rc = lib.lgb200_assign_bwd(ptr(G_d), ptr(sim_d), B, m, n, ptr(lse_d), Lp, ptr(lens_d), ptr(z_d), ptr(dz0), ptr(dz1),
                               ptr(ws), _st())
    assert rc == 0, lib.lgb200_error_string(rc)
    torch.cuda.synchronize()
    return sim_d.cpu(), dz0.cpu(), dz1.cpu()


@pytest.mark.parametrize("B,m,n,Lp,counts", [
    (2, 150, 131, 256, None),
    (2, 2048, 2048, 2048, None),
    (3, 320, 280, 384, [(300, 260), (129, 260), (0, 77)]),
], ids=["small", "2048", "ragged"])
def test_assign_bwd_against_autograd(B, m, n, Lp, counts):
    """d sim within the 1e-5 relative bound of test_assign_dsim_against_autograd, dz within 1e-5, exact zeros outside
    the valid blocks (where every input holds NaN: nothing there may be read), and two runs bit-equal."""
    g = torch.Generator().manual_seed(m + n)
    sim_full = torch.randn(B, m, n, generator=g) * 2
    z = torch.randn(2 * B, Lp, generator=g) * 2
    G_full = torch.randn(B, m + 1, n + 1, generator=g)  # dense, dustbin row / column included
    cnt = counts or [(m, n)] * B
    ref_ds = torch.zeros(B, m, n, dtype=torch.float64)
    ref_dz0, ref_dz1 = torch.zeros(B, m, dtype=torch.float64), torch.zeros(B, n, dtype=torch.float64)
    lse = torch.full((2 * B, Lp), float("nan"))
    sim, G = sim_full.clone(), G_full.clone()
    for b, (n0, n1) in enumerate(cnt):
        s = sim_full[b, :n0, :n1].double().requires_grad_(True)
        z0 = z[2 * b, :n0].double().requires_grad_(True)
        z1 = z[2 * b + 1, :n1].double().requires_grad_(True)
        ri, ci = list(range(n0)) + [m], list(range(n1)) + [n]
        Gb = G_full[b][ri][:, ci].double()
        la = torch.zeros(n0 + 1, n1 + 1, dtype=torch.float64)
        if n0 > 0 and n1 > 0:
            la[:n0, :n1] = F.log_softmax(s, 1) + F.log_softmax(s, 0) + F.logsigmoid(z0)[:, None] + F.logsigmoid(z1)[None]
            lse[2 * b, :n0] = torch.logsumexp(s.detach(), 1).float()
            lse[2 * b + 1, :n1] = torch.logsumexp(s.detach(), 0).float()
        la[:n0, n1] = F.logsigmoid(-z0)
        la[n0, :n1] = F.logsigmoid(-z1)
        (la * Gb).sum().backward()
        if s.grad is not None:
            ref_ds[b, :n0, :n1] = s.grad
        ref_dz0[b, :n0] = z0.grad if z0.grad is not None else 0.0
        ref_dz1[b, :n1] = z1.grad if z1.grad is not None else 0.0
        # outside the valid block (and its dustbin entries): NaN, must not be read
        sim[b, n0:], sim[b, :, n1:] = float("nan"), float("nan")
        G[b, n0:m], G[b, :, n1:n] = float("nan"), float("nan")
        G[b, m, n] = float("nan")
        z[2 * b, n0:], z[2 * b + 1, n1:] = float("nan"), float("nan")
    out = _assign_bwd(G, sim, lse, Lp, counts, z)
    ds, dz0, dz1 = out
    e = (_rel(ds, ref_ds), _rel(dz0, ref_dz0), _rel(dz1, ref_dz1))
    print(f"assign_bwd {B}x{m}x{n}: d sim {e[0]:.2e}, dz0 {e[1]:.2e}, dz1 {e[2]:.2e}")
    assert e[0] < 1e-5 and e[1] < 1e-5 and e[2] < 1e-5, e
    for b, (n0, n1) in enumerate(cnt):
        assert float(ds[b, n0:].abs().max() if n0 < m else 0.0) == 0.0
        assert float(ds[b, :, n1:].abs().max() if n1 < n else 0.0) == 0.0
        assert float(dz0[b, n0:].abs().max() if n0 < m else 0.0) == 0.0
        assert float(dz1[b, n1:].abs().max() if n1 < n else 0.0) == 0.0
    again = _assign_bwd(G, sim, lse, Lp, counts, z)
    for x, y in zip(out, again):
        assert torch.equal(x, y)


# ---- whole training steps ---------------------------------------------------------------------------------------

# name -> (make_pairs arguments, conf, checkpointed, integer keypoints with ties and a square extent, image_size).
# The seeds are chosen so that every row and column arg-maximum of the float64 log_assignment leads the runner-up by
# more than 1.5e-3: the kernels' fp32 mutual pairs are then the oracle's.
CASES = {
    "size_kept": (dict(n0=170, n1=150, seed=27), {}, False, False, True),
    "nosize_ties_checkpointed": (dict(n0=170, n1=150, seed=27), {}, True, True, False),
    "scale_ori_dim128": (dict(n0=160, n1=140, scale_ori=True, dim=128, seed=41),
                         {"input_dim": 128, "add_scale_ori": True}, False, False, True),
}


def _case_data(name, seed=None):
    kw, _, _, ties, with_size = CASES[name]
    kw = dict(kw) if seed is None else dict(kw, seed=seed)
    data = make_pairs(B=2, with_gt=True, **kw)
    if ties:  # integer pixel coordinates in [0, 63]: ties at the maxima / minima, extent 64 x 64 (W = H)
        for i in (0, 1):
            k = (data[f"keypoints{i}"] / 10.0).floor().clamp(0, 63)
            k[:, 0], k[:, 1] = 0.0, 63.0
            k[:, 2, 0], k[:, 3, 1] = 63.0, 0.0
            data[f"keypoints{i}"] = k
    if not with_size:
        data["view0"], data["view1"] = {}, {}
    return data


def _extra_weights(B, m, n, seed=3):
    """Seeded W [B,m+1,n+1], v [B,m], u [B,n] of the extra loss terms sum W.la + sum v.ms0 + sum u.ms1."""
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, m + 1, n + 1, generator=g) * 1e-3, torch.randn(B, m, generator=g) * 0.1,
            torch.randn(B, n, generator=g) * 0.1)


def _conf(name, **over):
    return {**CONF, **CASES[name][1], "checkpointed": CASES[name][2], **over}


def _model(conf, seed=5):
    torch.manual_seed(seed)
    return LightGlue(conf).to(DEV).train()


def _leaves(data):
    return [k for k in KPT_KEYS + ("descriptors0", "descriptors1") if k in data]


def _step(conf, data_c, extra=True, kpt_grad=True, seed=5):
    """One training step: LightGlue.loss's total (mean over pairs) plus, with `extra`, sum W.la + sum v.ms0 +
    sum u.ms1 -> (pred, parameter gradients, input gradients)."""
    model = _model(conf, seed)
    data = to_device(data_c, DEV)
    for k in _leaves(data):
        if kpt_grad or k.startswith("desc"):
            data[k].requires_grad_(True)
    model.zero_grad(set_to_none=True)
    pred = model(data)
    losses, _ = model.loss(pred, data)
    loss = losses["total"].mean()
    if extra:
        B, m, n = pred["log_assignment"].shape[0], pred["matches0"].shape[1], pred["matches1"].shape[1]
        W, v, u = (t.to(DEV) for t in _extra_weights(B, m, n))
        loss = loss + (W * pred["log_assignment"]).sum() + (v * pred["matching_scores0"]).sum() + \
            (u * pred["matching_scores1"]).sum()
    loss.backward()
    grads = {k: p.grad for k, p in model.named_parameters()}
    return pred, grads, {k: data[k].grad for k in _leaves(data) if data[k].grad is not None}


def _oracle_step(conf, data_c, dtype, seed=5):
    """The same step through the CPU oracle with torch autograd -> (pred, parameter gradients, input gradients)."""
    sd = _model(conf, seed).state_dict()
    leaves = {k: v.detach().cpu().to(dtype).clone().requires_grad_(True) for k, v in sd.items()
              if v.is_floating_point() and k != "confidence_thresholds"}
    d = dict(data_c)
    for k in _leaves(d):
        d[k] = data_c[k].to(dtype).clone().requires_grad_(True)
    pred = loss_oracle.forward_collect(leaves, conf, d, keep_graph=True, dtype=dtype)
    ls, _ = loss_oracle.loss(leaves, conf, pred, d, True, keep_graph=True)
    B, m, n = pred["log_assignment"].shape[0], pred["matches0"].shape[1], pred["matches1"].shape[1]
    W, v, u = (t.to(dtype) for t in _extra_weights(B, m, n))
    loss = ls["total"].mean() + (W * pred["log_assignment"]).sum() + (v * pred["matching_scores0"]).sum() + \
        (u * pred["matching_scores1"]).sum()
    loss.backward()
    return pred, {k: v.grad.double() for k, v in leaves.items()}, {k: d[k].grad.double() for k in _leaves(d)}


def _mutual(la):
    """The raw mutual pairs (every mutual pair, whatever its score) of each pair's log_assignment [B,m+1,n+1]."""
    out = [lightglue_oracle.filter_matches(la[b].detach().double().cpu(), -1.0) for b in range(la.shape[0])]
    return torch.stack([o[0] for o in out]), torch.stack([o[1] for o in out])


@pytest.mark.parametrize("name", sorted(CASES))
def test_fp32_step_against_the_oracle(name):
    """Every parameter gradient and every input gradient (descriptors, keypoints, scales, orientations) within 2e-3
    (norm-wise) of float64 autograd through the oracle, whose mutual pairs are the kernels' exactly."""
    data_c = _case_data(name)
    conf = _conf(name)
    pred, grads, gin = _step(conf, data_c)
    pred_o, grads_o, gin_o = _oracle_step(conf, data_c, torch.float64)
    for a, b in zip(_mutual(pred["log_assignment"]), _mutual(pred_o["log_assignment"])):
        assert torch.equal(a, b), "the fixture must give the oracle's mutual pairs"
    assert _rel(pred["log_assignment"], pred_o["log_assignment"]) < 1e-4
    assert _rel(pred["matching_scores0"], pred_o["matching_scores0"]) < 1e-4
    worst = max((_rel(grads[k], grads_o[k]), k) for k in grads_o)
    ins = {k: _rel(gin[k], gin_o[k]) for k in gin_o}
    print(f"{name}: worst parameter {worst}, inputs " + ", ".join(f"{k} {e:.2e}" for k, e in ins.items()))
    assert worst[0] < 2e-3, worst
    assert set(gin) == set(gin_o) and max(ins.values()) < 2e-3, ins


def _figures(grads, gin, grads_o, gin_o):
    """(worst parameter, median parameter, all parameters together, worst input) relative errors."""
    errs = sorted(_rel(grads[k], grads_o[k]) for k in grads_o)
    num = sum(float((grads[k].detach().double().cpu() - grads_o[k]).norm() ** 2) for k in grads_o)
    den = sum(float(grads_o[k].norm() ** 2) for k in grads_o)
    return errs[-1], errs[len(errs) // 2], math.sqrt(num / den), max(_rel(gin[k], gin_o[k]) for k in gin_o)


@pytest.mark.parametrize("name", sorted(CASES))
def test_bf16_step_within_the_oracles_own_bf16_envelope(name):
    """train_precision="bf16": median, all-parameter and input figures within 2x of the oracle's own deviation when it
    runs the step in torch.bfloat16; the worst parameter below 0.25 or 2x the oracle's worst (test_gpu_train_bf16.py's
    bounds)."""
    data_c = _case_data(name)
    conf = _conf(name)
    _, grads_o, gin_o = _oracle_step(conf, data_c, torch.float64)
    _, grads_b, gin_b = _oracle_step(conf, data_c, torch.bfloat16)
    pred, grads, gin = _step(_conf(name, train_precision="bf16"), data_c)
    env, got = _figures(grads_b, gin_b, grads_o, gin_o), _figures(grads, gin, grads_o, gin_o)
    print(f"{name} bf16: oracle bf16 {tuple(f'{x:.3g}' for x in env)}, ours {tuple(f'{x:.3g}' for x in got)}")
    assert got[0] < max(0.25, 2.0 * env[0]), (got, env)
    for i in range(1, 4):
        assert got[i] <= 2.0 * env[i], (i, got, env)


# padded batches with counts: N0S x N1S padded to LEN0 x LEN1, no image_size (the extent of the valid points)
N0S, N1S = [170, 129, 1], [150, 150, 77]
LEN0, LEN1 = 192, 176


def _pairs():
    return [_case_data("nosize_ties_checkpointed", seed=40 + i) for i in range(3)]


def _per_pair(data):
    """Each pair of a padded batch cut to its counts (the un-padded pair)."""
    out = []
    for b, (n0, n1) in enumerate(zip(N0S, N1S)):
        d = {k: data[k][b:b + 1, :(n0 if k.endswith("0") else n1)]
             for k in ("keypoints0", "keypoints1", "descriptors0", "descriptors1", "gt_matches0", "gt_matches1")}
        d["gt_assignment"] = data["gt_assignment"][b:b + 1, :n0, :n1]
        d["view0"], d["view1"] = {}, {}
        out.append(d)
    return out


def _padded(pairs, fill, seed=123):
    torch.manual_seed(seed)
    kp = dict(mode="random_c", bounds=(0.0, 480.0)) if fill == "random" else dict(mode="zeros")
    ds = dict(mode="random", bounds=(-0.2, 0.2)) if fill == "random" else dict(mode="zeros")
    data = {"view0": {}, "view1": {}}
    for i, (L, ns) in enumerate(((LEN0, N0S), (LEN1, N1S))):
        data[f"keypoints{i}"] = pad_and_stack([p[f"keypoints{i}"][0, :c] for p, c in zip(pairs, ns)], L, -2, **kp)
        data[f"descriptors{i}"] = pad_and_stack([p[f"descriptors{i}"][0, :c] for p, c in zip(pairs, ns)], L, -2, **ds)
        data[f"num_keypoints{i}"] = torch.tensor(ns, dtype=torch.int32)
        gms = []
        for p, c, co in zip(pairs, ns, N1S if i == 0 else N0S):
            gm = p[f"gt_matches{i}"][0, :c].clone()
            gms.append(torch.where(gm >= co, -1, gm))  # partners cut off by the other side's count: unmatchable
        data[f"gt_matches{i}"] = pad_and_stack(gms, L, -1, mode="zeros")
    data["gt_assignment"] = torch.stack([pad_to_length(pad_to_length(p["gt_assignment"][0, :a, :b], LEN1, -1,
                                                                     mode="ones"), LEN0, -2, mode="ones")
                                         for p, a, b in zip(pairs, N0S, N1S)])
    return data


@pytest.mark.parametrize("train_precision", ["fp32", "bf16"])
def test_padded_batch_with_counts(train_precision):
    """fp32: parameter and input gradients of the padded step equal the per-pair oracle steps (un-padded, each with
    the pair's cut of W, v, u; parameter gradients summed over pairs) within 2e-3.  Both precisions: input gradients
    exactly 0 on padded rows, everything bit-equal whatever the padding holds."""
    conf = _conf("nosize_ties_checkpointed", train_precision=train_precision)
    pairs = _pairs()
    runs = [_step(conf, _padded(pairs, fill)) for fill in ("random", "zeros")]
    pred, grads, gin = runs[0]
    for k in _leaves(gin):
        cnts = N0S if k.endswith("0") else N1S
        assert all(float(gin[k][b, c:].abs().max()) == 0.0 for b, c in enumerate(cnts) if c < gin[k].shape[1]), k
    pred_z, grads_z, gin_z = runs[1]
    for k in grads:
        assert torch.equal(grads[k], grads_z[k]), k
    for k in gin:
        assert torch.equal(gin[k], gin_z[k]), k
    for k in ("log_assignment", "matches0", "matches1", "matching_scores0", "matching_scores1"):
        assert torch.equal(pred[k], pred_z[k]), k
    if train_precision == "bf16":
        return
    padded = _padded(pairs, "random")
    W, v, u = _extra_weights(len(N0S), LEN0, LEN1)
    grads_o, gin_o = {}, {k: [] for k in gin}
    B = len(N0S)
    for b, d in enumerate(_per_pair(padded)):
        n0, n1 = N0S[b], N1S[b]
        sd = _model(conf).state_dict()
        leaves = {k: t.detach().cpu().double().clone().requires_grad_(True) for k, t in sd.items()
                  if t.is_floating_point() and k != "confidence_thresholds"}
        for k in _leaves(d):
            d[k] = d[k].double().clone().requires_grad_(True)
        pr = loss_oracle.forward_collect(leaves, conf, d, keep_graph=True, dtype=torch.float64)
        ls, _ = loss_oracle.loss(leaves, conf, pr, d, True, keep_graph=True)
        ri, ci = list(range(n0)) + [LEN0], list(range(n1)) + [LEN1]
        loss = ls["total"].mean() / B + (W[b][ri][:, ci].double() * pr["log_assignment"][0]).sum() + \
            (v[b, :n0].double() * pr["matching_scores0"][0]).sum() + (u[b, :n1].double() * pr["matching_scores1"][0]).sum()
        loss.backward()
        for k, t in leaves.items():
            grads_o[k] = grads_o.get(k, 0.0) + t.grad
        for k in gin:
            gin_o[k].append(d[k].grad[0])
    worst = max((_rel(grads[k], grads_o[k]), k) for k in grads_o)
    ins = {k: _rel(torch.cat([gin[k][b, :c] for b, c in enumerate(N0S if k.endswith("0") else N1S)]),
                   torch.cat(gin_o[k])) for k in gin}
    print(f"padded fp32: worst parameter {worst}, inputs " + ", ".join(f"{k} {e:.2e}" for k, e in ins.items()))
    assert worst[0] < 2e-3, worst
    assert max(ins.values()) < 2e-3, ins


def test_outputs_and_todays_loss_do_not_change():
    """The forward outputs are bit-equal whether or not the loss reads them, and a step with today's loss launches
    exactly the two keypoint-gradient kernels more when the keypoints require grad, nothing else."""
    lib = _abi.load()
    data_c = _case_data("size_kept")
    conf = _conf("size_kept")
    pred_a, _, _ = _step(conf, data_c, extra=True)
    pred_b, _, _ = _step(conf, data_c, extra=False)
    for k in ("log_assignment", "matches0", "matches1", "matching_scores0", "matching_scores1", "ref_descriptors0"):
        assert torch.equal(pred_a[k].detach(), pred_b[k].detach()), k
    counts = []
    for kpt_grad in (False, True, False):
        torch.cuda.synchronize()
        c0 = lib.lgb200_launch_count()
        _step(conf, data_c, extra=False, kpt_grad=kpt_grad)
        torch.cuda.synchronize()
        counts.append(lib.lgb200_launch_count() - c0)
    assert counts[0] == counts[2] and counts[1] == counts[0] + 2, counts


@pytest.mark.parametrize("train_precision", ["fp32", "bf16"])
def test_training_on_log_assignment_alone_reduces_it(train_precision):
    """Six Adam steps on an NLL read from pred["log_assignment"] only (not LightGlue.loss)."""
    data = to_device(_case_data("size_kept", seed=4), DEV)
    model = _model(_conf("size_kept", train_precision=train_precision), seed=0)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    gt = data["gt_assignment"]
    hist = []
    for _ in range(6):
        opt.zero_grad(set_to_none=True)
        la = model(data)["log_assignment"]
        loss = -(la[:, :-1, :-1] * gt).sum() / gt.sum()
        loss.backward()
        opt.step()
        hist.append(float(loss.detach()))
    assert all(math.isfinite(x) for x in hist) and hist[-1] < hist[0] - 0.05, hist

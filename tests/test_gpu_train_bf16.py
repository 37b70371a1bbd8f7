"""GPU tests of bf16 mixed-precision training (conf.train_precision = "bf16"): the bf16 attention backward
(lgb200_attention_bwd_bf16) against float64 autograd on the same bf16-rounded inputs, the training forward against the
no-grad bf16 forward, and a whole training step against autograd through the CPU oracle, with the oracle's own bf16
deviation as the bound."""
import ctypes
import math

import pytest
import torch

from glue_factory_colon_b200 import LightGlue, _abi
from glue_factory_colon_b200._abi import ptr
from glue_factory_colon_b200.synthetic import make_pairs, to_device
from helpers import oracle_training_step

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _st():
    return torch.cuda.current_stream(DEV).cuda_stream


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _bwd16(q, k, v, dctx, lens_d, kv_xor):
    """bf16 forward (lgb200_attention) + lgb200_attention_bwd_bf16 -> dq, dk, dv (fp32 [S,4,Lp,64])."""
    lib = _abi.load()
    S, _, Lp, _ = q.shape
    ctx = torch.zeros(S, Lp, 256, device=DEV, dtype=torch.bfloat16)
    assert lib.lgb200_attention(_abi.BF16, ptr(q), ptr(k), ptr(v), S, Lp, ptr(lens_d), kv_xor, ptr(ctx), _st()) == 0
    dq, dk, dv = (torch.full((S, 4, Lp, 64), 7.0, device=DEV) for _ in range(3))
    n_ws = ctypes.c_longlong(0)
    assert lib.lgb200_attention_bwd_bf16_workspace(S, Lp, ctypes.byref(n_ws)) == 0
    ws = torch.full((n_ws.value,), float("nan"), device=DEV)
    rc = lib.lgb200_attention_bwd_bf16(ptr(q), ptr(k), ptr(v), ptr(ctx), ptr(dctx), S, Lp, ptr(lens_d), kv_xor, ptr(dq),
                                       ptr(dk), ptr(dv), ptr(ws), _st())
    assert rc == 0, lib.lgb200_error_string(rc)
    return dq, dk, dv


def _ref_grads(q, k, v, dctx, ln, kv_xor):
    """float64 autograd of the attention (q in the log2 domain) on the given (bf16-rounded) inputs."""
    S, _, Lp, _ = q.shape
    qd, kd, vd = (t.double().cpu().requires_grad_(True) for t in (q, k, v))
    ctx_ref = torch.zeros(S, Lp, 256, dtype=torch.float64)
    for s in range(S):
        so = s ^ kv_xor
        nq, nk = int(ln[s]), int(ln[so])
        if nq == 0 or nk == 0:
            continue
        a = torch.softmax(qd[s, :, :nq] @ kd[so, :, :nk].transpose(-1, -2) * math.log(2.0), -1)
        ctx_ref[s, :nq] = (a @ vd[so, :, :nk]).permute(1, 0, 2).reshape(nq, 256)
    (ctx_ref * dctx.double().cpu()).sum().backward()
    return qd.grad, kd.grad, vd.grad


@pytest.mark.parametrize("kv_xor", [0, 1], ids=["self", "cross"])
@pytest.mark.parametrize("lens,gscale", [(None, 1.0), ([200, 131, 64, 256], 1.0), ([70, 0, 129, 5], 1.0),
                                         ([200, 131, 64, 256], 3e-9), (None, 7e3)],
                         ids=["full", "ragged", "empty_side", "ragged_tiny_gradient", "full_large_gradient"])
def test_attention_bwd_bf16_against_autograd(kv_xor, lens, gscale):
    """Norm-wise errors against float64 on the same bf16 inputs: P and D are rounded to bf16 once per element before
    their products (8 mantissa bits), so the expected order is 1e-2.  Measured on a B200 (self-attention cases): dq
    3.0e-3 - 3.2e-3, dk 2.8e-3 - 3.0e-3, dv 2.3e-3 - 2.4e-3; the bound 2e-2 leaves room for other seeds."""
    S, Lp = 4, 256
    g = torch.Generator().manual_seed(11 + kv_xor)
    q = (torch.randn(S, 4, Lp, 64, generator=g) * 0.6).to(DEV, torch.bfloat16)
    k = (torch.randn(S, 4, Lp, 64, generator=g) * 0.6).to(DEV, torch.bfloat16)
    v = torch.randn(S, 4, Lp, 64, generator=g).to(DEV, torch.bfloat16)
    if kv_xor:
        k = q  # cross block: to_qk feeds both sides, one tensor
    dctx = (torch.randn(S, Lp, 256, generator=g) * torch.rand(S, Lp, 1, generator=g) ** 4 * gscale).to(DEV)
    ln = torch.tensor(lens if lens is not None else [Lp] * S)
    lens_d = None if lens is None else ln.to(DEV, torch.int32)
    rq, rk, rv = _ref_grads(q, k, v, dctx, ln, kv_xor)
    dq, dk, dv = _bwd16(q, k, v, dctx, lens_d, kv_xor)
    if kv_xor:  # one tensor on both sides: its gradient is dq + dk
        checks = (("dq+dk", dq + dk, rq + rk), ("dv", dv, rv))
    else:
        checks = (("dq", dq, rq), ("dk", dk, rk), ("dv", dv, rv))
    for name, got, ref in checks:
        assert torch.isfinite(got).all(), name
        e = _rel(got, ref)
        print(f"bf16 attention bwd {name}: {e:.2e}")
        assert e < 2e-2, f"{name}: {e}"
    for got in (dq, dk, dv):
        for s in range(S):  # rows past the valid count carry no gradient
            assert float(got[s, :, int(ln[s]):].abs().max() if int(ln[s]) < Lp else 0.0) == 0.0


def test_attention_bwd_bf16_error_does_not_grow_with_length():
    """2 x 2048 keys with same-sign sums (non-zero means), against 2 x 256 keys of the same distributions: the tensor
    core rounds its fp32 accumulator toward zero after every MMA; the kernel folds its TMEM accumulators into
    round-to-nearest running sums every 4 tiles, so neither the norm-wise nor the one-sided (mean) error grows with the
    number of keys."""
    res = {}
    for Lp in (256, 2048):
        S = 2
        g = torch.Generator().manual_seed(1)
        q = (torch.randn(S, 4, Lp, 64, generator=g) * 0.6).to(DEV, torch.bfloat16)
        k = (torch.randn(S, 4, Lp, 64, generator=g) * 0.6).to(DEV, torch.bfloat16)
        v = (torch.randn(S, 4, Lp, 64, generator=g) + 0.5).to(DEV, torch.bfloat16)
        dctx = (torch.randn(S, Lp, 256, generator=g) * 1e-3 + 5e-4).to(DEV)
        qd, kd, vd = (t.double().requires_grad_(True) for t in (q, k, v))
        a = torch.softmax(qd @ kd.transpose(-1, -2) * math.log(2.0), -1)
        ((a @ vd).permute(0, 2, 1, 3).reshape(S, Lp, 256) * dctx.double()).sum().backward()
        got = _bwd16(q, k, v, dctx, None, 0)
        for name, gg, ref in zip(("dq", "dk", "dv"), got, (qd.grad, kd.grad, vd.grad)):
            d = gg.double() - ref
            res[(Lp, name)] = (float(d.norm() / ref.norm()), abs(float(d.mean() / ref.abs().mean())))
    print({k: tuple(f"{x:.2e}" for x in v) for k, v in res.items()})
    for name in ("dq", "dk", "dv"):
        (n256, b256), (n2048, b2048) = res[(256, name)], res[(2048, name)]
        assert n2048 < 1.5 * n256 + 1e-3, f"{name}: norm-wise {n256:.2e} at 256 keys, {n2048:.2e} at 2048"
        assert b2048 < 2.0 * b256 + 1e-3, f"{name}: one-sided {b256:.2e} at 256 keys, {b2048:.2e} at 2048"


def _data(B=2, n0=200, n1=170, seed=4):
    data = to_device(make_pairs(B=B, n0=n0, n1=n1, seed=seed, with_gt=True), DEV)
    data["descriptors0"].requires_grad_(True)
    data["descriptors1"].requires_grad_(True)
    return data


def test_bf16_training_forward_equals_the_no_grad_bf16_forward():
    torch.manual_seed(3)
    model = LightGlue({"n_layers": 3, "precision": "bf16", "train_precision": "bf16", "filter_threshold": 0.0})
    model = model.to(DEV).train()
    data = _data()
    pred = model(data)
    assert pred["ref_descriptors0"].requires_grad
    losses, _ = model.loss(pred, data)
    with torch.no_grad():
        ref = model(data)
        ref_losses, _ = model.loss(ref, data)
    for key in ("ref_descriptors0", "ref_descriptors1", "log_assignment", "matches0", "matches1"):
        assert pred[key].dtype == ref[key].dtype and torch.equal(pred[key].detach(), ref[key]), key
    torch.testing.assert_close(losses["total"].detach(), ref_losses["total"], rtol=1e-5, atol=0.0)


def _oracle_figures(gp, gd, grads_o, gd_o):
    """Norm-wise relative errors of a step's gradients (gp: {name: gradient}, gd: (d desc0, d desc1)) against float64:
    (worst tensor, median tensor, all parameters together, d descriptors0, d descriptors1)."""
    errs = sorted(_rel(gp[k], grads_o[k]) for k in grads_o)
    num = sum(float((gp[k].detach().double().cpu() - grads_o[k].double()).norm() ** 2) for k in grads_o)
    den = sum(float(grads_o[k].double().norm() ** 2) for k in grads_o)
    return errs[-1], errs[len(errs) // 2], math.sqrt(num / den), _rel(gd[0], gd_o[0]), _rel(gd[1], gd_o[1])


def _bf16_step(fx, checkpointed, data_c):
    torch.manual_seed(fx["seed"])
    model = LightGlue({**fx["conf"], "checkpointed": checkpointed, "train_precision": "bf16"}).to(DEV).train()
    data = to_device(data_c, DEV)
    data["descriptors0"].requires_grad_(True)
    data["descriptors1"].requires_grad_(True)
    model.zero_grad(set_to_none=True)
    losses, _ = model.loss(model(data), data)
    losses["total"].mean().backward()
    return model, losses, data


@pytest.mark.parametrize("name", ["grad_train", "grad_train_sift"])
def test_bf16_training_step_within_the_oracles_own_bf16_envelope(name, golden_dir):
    """Every parameter gradient and both descriptor gradients against autograd through the float64 CPU oracle.  The
    bound is the oracle's own deviation when it runs the same step in torch.bfloat16: within 2x of it for the median
    tensor, all parameters together and the descriptors; the worst tensor below 0.25.  Kept and checkpointed steps give
    bit-equal gradients (the same deterministic kernels and cuBLAS calls on the same inputs)."""
    fx = torch.load(golden_dir / f"{name}.pt", weights_only=False)
    torch.manual_seed(fx["seed"])
    sd = {k: v.clone() for k, v in LightGlue(fx["conf"]).state_dict().items()}
    data_c = make_pairs(with_gt=True, **fx["data_kwargs"])
    total_o, grads_o, gd0_o, gd1_o = oracle_training_step(sd, fx["conf"], data_c, dtype=torch.float64)
    total_b, grads_b, gd0_b, gd1_b = oracle_training_step(sd, fx["conf"], data_c, dtype=torch.bfloat16)
    env = _oracle_figures(grads_b, (gd0_b, gd1_b), grads_o, (gd0_o, gd1_o))

    model, losses, data = _bf16_step(fx, False, data_c)
    named = dict(model.named_parameters())
    assert set(named) == set(grads_o)
    for k, p in named.items():
        assert p.grad is not None, f"{k} received no gradient"
        assert torch.isfinite(p.grad).all(), k
    assert torch.isfinite(data["descriptors0"].grad).all() and torch.isfinite(data["descriptors1"].grad).all()
    got = _oracle_figures({k: p.grad for k, p in named.items()}, (data["descriptors0"].grad, data["descriptors1"].grad),
                          grads_o, (gd0_o, gd1_o))
    print(f"{name}: bf16 oracle (worst, median, all, d0, d1) = {tuple(f'{x:.3g}' for x in env)}, loss "
          f"{_rel(total_b, total_o):.2e}; train_precision=bf16 = {tuple(f'{x:.3g}' for x in got)}, loss "
          f"{_rel(losses['total'].detach(), total_o):.2e}")
    assert got[0] < 0.25, f"worst tensor {got[0]:.3g}"
    for i, what in ((1, "median tensor"), (2, "all parameters"), (3, "d descriptors0"), (4, "d descriptors1")):
        assert got[i] <= 2.0 * env[i], f"{what}: {got[i]:.3g} vs the oracle's bf16 {env[i]:.3g}"

    model_c, losses_c, data_cp = _bf16_step(fx, True, data_c)
    assert torch.equal(losses_c["total"], losses["total"])
    for k, p in model_c.named_parameters():
        assert torch.equal(p.grad, named[k].grad), f"{k}: kept and checkpointed gradients differ"
    assert torch.equal(data_cp["descriptors0"].grad, data["descriptors0"].grad)
    assert torch.equal(data_cp["descriptors1"].grad, data["descriptors1"].grad)


def test_bf16_training_reduces_the_loss():
    torch.manual_seed(0)
    model = LightGlue({"n_layers": 3, "filter_threshold": 0.0, "train_precision": "bf16"}).to(DEV).train()
    data = to_device(make_pairs(B=2, n0=128, n1=100, seed=4, with_gt=True), DEV)
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

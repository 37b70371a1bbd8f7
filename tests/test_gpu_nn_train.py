"""Training through the nearest-neighbour matcher (`loss: "N_pair"`): lgb200_npair_loss_bwd against float64 autograd of
the reference loss, whole steps against float64 autograd of the reference forward and loss, values unchanged by the
graph, padded batches with counts, the temperature alone, determinism, and a short training run."""
import pytest
import torch
import torch.nn.functional as F

from helpers import ROOT  # noqa: F401  (puts the repository on sys.path)
from oracle import nn_oracle

from glue_factory_colon_b200.synthetic import make_pairs, to_device

pytestmark = pytest.mark.gpu
TOL = 1e-4  # max |got - float64| <= TOL * max |float64 gradient|


def _matcher(T=1.0):
    from glue_factory_colon_b200.nearest_neighbor_matcher import NearestNeighborMatcher

    m = NearestNeighborMatcher({"loss": "N_pair"}).cuda().train()
    with torch.no_grad():
        m.temperature.fill_(T)
    return m


def _rel(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return (got - ref).abs().max().item() / ref.abs().max().item()


def _check(got, ref, what):
    assert got.shape == ref.shape, what
    err = _rel(got, ref)
    assert err <= TOL, f"{what}: max |d| = {err:.3g} x max |g64|"
    return err


def _step(model, data):
    losses, _ = model.loss(model(data), data)
    losses["total"].mean().backward()
    return losses


def _float64_step(data, T, descriptors_grad=True, valid=None):
    """float64 autograd of the reference forward (its einsum) and N_pair loss, `total.mean().backward()`.  valid
    [B, N, M] (optional): the similarity is 0 outside it, as the matcher writes it for a padded batch with counts."""
    x0 = data["descriptors0"].detach().cpu().double().requires_grad_(descriptors_grad)
    x1 = data["descriptors1"].detach().cpu().double().requires_grad_(descriptors_grad)
    t = torch.tensor(T, dtype=torch.float64, requires_grad=True)
    sim = torch.einsum("bnd,bmd->bnm", x0, x1)
    if valid is not None:
        sim = torch.where(valid, sim, 0.0)
    pred = nn_oracle.forward({}, {}, sim=sim)
    nn_oracle.npair_loss(pred["similarity"], data["gt_assignment"].cpu(), t)["total"].mean().backward()
    return x0.grad, x1.grad, t.grad


def _sim_case(B, N, M):
    """Similarity of unit descriptors and ground truth.  Pair 0: three exact duplicate descriptors (entries +-1/16, so
    that the similarity is exactly 1 and the clamp holds) that are ground-truth matches, a row and a column with several
    ground-truth entries.  Pair 1: no ground truth at all."""
    data = make_pairs(B, N, M, seed=N + M, with_gt=True)
    d0, d1, gt = data["descriptors0"], data["descriptors1"], data["gt_assignment"].clone()
    d0[0, :3] = torch.randint(0, 2, (3, 256), generator=torch.Generator().manual_seed(N)) / 8.0 - 1 / 16
    d1[0, :3] = d0[0, :3]
    gt[0, :3] = False
    gt[0, :, :3] = False
    gt[0, 0, 0] = gt[0, 1, 1] = gt[0, 2, 2] = True
    gt[0, 5, 3:7] = True
    gt[0, 8:12, 9] = True
    if B > 1:
        gt[1] = False
    return torch.einsum("bnd,bmd->bnm", d0.cuda(), d1.cuda()), gt


@pytest.mark.parametrize("shape", [(1, 37, 53), (3, 300, 260), (2, 2048, 2048)])
@pytest.mark.parametrize("T", [0.3, 1.0, 5.0])
def test_npair_bwd_kernel_against_float64_autograd(shape, T):
    B, N, M = shape
    sim, gt = _sim_case(B, N, M)
    assert ((2 * (1 - sim[0, [0, 1, 2], [0, 1, 2]])) < 1e-6).all()  # the duplicates are clamped entries
    g = torch.randn(B, generator=torch.Generator().manual_seed(1)) + 2.0
    model = _matcher(T)
    s = sim.clone().requires_grad_()
    losses, _ = model.loss({"similarity": s}, {"gt_assignment": gt})
    (losses["total"] * g.cuda()).sum().backward()
    # float64 autograd of the reference loss on the same (upcast) similarity
    s64 = sim.cpu().double().requires_grad_()
    t64 = torch.tensor(T, dtype=torch.float64, requires_grad=True)
    (nn_oracle.npair_loss(s64, gt, t64)["total"] * g.double()).sum().backward()
    # the same in fp32 torch autograd on the GPU, for scale
    s32 = sim.clone().requires_grad_()
    t32 = torch.tensor(T, device="cuda", requires_grad=True)
    (nn_oracle.npair_loss(s32, gt.cuda(), t32)["total"] * g.cuda()).sum().backward()
    e_sim, e_t = _check(s.grad, s64.grad, "d sim"), _check(model.temperature.grad, t64.grad, "d T")
    print(f"\n{shape} T={T}: kernel d sim {e_sim:.2e}, d T {e_t:.2e}; fp32 torch autograd d sim "
          f"{_rel(s32.grad, s64.grad):.2e}, d T {_rel(t32.grad, t64.grad):.2e} (x max |g64|)")
    assert (s.grad[0, [0, 1, 2], [0, 1, 2]] == 0).all()  # clamped: no gradient through the similarity
    if B > 1:
        assert (s.grad[1] == 0).all()  # no ground truth: nll = 0 whatever the similarity


@pytest.mark.parametrize("dim", [256, 128])
def test_training_step_against_float64_autograd(dim):
    data = make_pairs(2, 300, 260, dim=dim, seed=7, with_gt=True)
    dd = to_device(data, "cuda")
    d0, d1 = dd["descriptors0"].requires_grad_(), dd["descriptors1"].requires_grad_()
    model = _matcher(1.3)
    _step(model, dd)
    assert d0.grad.dtype == torch.float32 and d1.grad.shape == (2, 260, dim)
    r0, r1, rt = _float64_step(data, 1.3)
    _check(d0.grad, r0, "d descriptors0")
    _check(d1.grad, r1, "d descriptors1")
    _check(model.temperature.grad, rt, "d temperature")


def test_values_are_unchanged_by_the_graph():
    data = to_device(make_pairs(2, 300, 260, seed=9, with_gt=True), "cuda")
    model = _matcher(0.7)
    for mode in ("train", "eval"):
        model.train(mode == "train")
        with torch.no_grad():
            ref = model(data)
            ref_l, ref_m = model.loss(ref, data)
        plain = model(data)  # grad enabled, descriptors without requires_grad
        plain_l, plain_m = model.loss(plain, data)
        assert all(v.grad_fn is None and not v.requires_grad for v in plain.values())
        assert plain_l["total"].grad_fn is not None  # the temperature requires grad
        leaf = dict(data, descriptors0=data["descriptors0"].clone().requires_grad_(),
                    descriptors1=data["descriptors1"].clone().requires_grad_())
        out = model(leaf)
        out_l, out_m = model.loss(out, leaf)
        assert out["similarity"].grad_fn is not None and out_l["total"].grad_fn is not None
        assert out["log_assignment"].grad_fn is None and not out["log_assignment"].requires_grad
        assert out_l["n_pair_temperature"].requires_grad and not ref_l["n_pair_temperature"].requires_grad
        for got in (plain, out):
            assert got.keys() == ref.keys() and all(torch.equal(got[k].detach(), ref[k]) for k in ref)
        for got_l, got_m in ((plain_l, plain_m), (out_l, out_m)):
            assert got_l.keys() == ref_l.keys() and all(torch.equal(got_l[k].detach(), ref_l[k]) for k in ref_l)
            assert got_m.keys() == ref_m.keys() and all(torch.equal(got_m[k], ref_m[k]) for k in ref_m)
        with torch.no_grad():  # descriptors that require grad under no_grad: no graph anywhere
            ng = model(leaf)
            ng_l, _ = model.loss(ng, leaf)
        assert all(not v.requires_grad for v in [*ng.values(), *ng_l.values()])


def test_padded_batch_with_counts():
    data = make_pairs(2, 300, 260, seed=11, with_gt=True)
    n0, n1 = torch.tensor([300, 171]), torch.tensor([260, 143])
    valid = (torch.arange(300)[None, :, None] < n0[:, None, None]) & (torch.arange(260)[None, None] < n1[:, None, None])
    data["gt_assignment"] &= valid

    def run(padding):
        dd = to_device(data, "cuda")
        d0, d1 = dd["descriptors0"].clone(), dd["descriptors1"].clone()
        d0[1, 171:], d1[1, 143:] = padding(d0[1, 171:]), padding(d1[1, 143:])
        dd.update(descriptors0=d0.requires_grad_(), descriptors1=d1.requires_grad_(), num_keypoints0=n0,
                  num_keypoints1=n1)
        model = _matcher(1.1)
        losses = _step(model, dd)
        return d0.grad, d1.grad, model.temperature.grad, losses

    rnd = run(lambda x: 3 * torch.randn_like(x))
    zero = run(torch.zeros_like)
    assert (rnd[0][1, 171:] == 0).all() and (rnd[1][1, 143:] == 0).all()
    for a, b in zip(rnd[:3], zero[:3]):
        assert torch.equal(a, b)
    assert all(torch.equal(rnd[3][k], zero[3][k]) for k in rnd[3])
    # what `loss` differentiates: the similarity with zeros outside each pair's valid block
    r0, r1, rt = _float64_step(data, 1.1, valid=valid)
    _check(rnd[0], r0, "d descriptors0")
    _check(rnd[1], r1, "d descriptors1")
    _check(rnd[2], rt, "d temperature")


def test_temperature_only():
    data = make_pairs(2, 300, 260, seed=13, with_gt=True)
    dd = to_device(data, "cuda")
    model = _matcher(2.0)
    pred = model(dd)
    assert pred["similarity"].grad_fn is None and not pred["similarity"].requires_grad
    losses, _ = model.loss(pred, dd)
    losses["total"].mean().backward()
    _, _, rt = _float64_step(data, 2.0, descriptors_grad=False)
    _check(model.temperature.grad, rt, "d temperature")


def test_backward_is_deterministic():
    dd = to_device(make_pairs(2, 1024, 1100, seed=15, with_gt=True), "cuda")
    grads = []
    for _ in range(2):
        d0, d1 = dd["descriptors0"].clone().requires_grad_(), dd["descriptors1"].clone().requires_grad_()
        model = _matcher(1.7)
        _step(model, dict(dd, descriptors0=d0, descriptors1=d1))
        grads.append((d0.grad, d1.grad, model.temperature.grad))
    assert all(torch.equal(a, b) for a, b in zip(*grads))


def test_six_adam_steps_lower_the_loss():
    data = to_device(make_pairs(4, 256, 240, dim=64, seed=17, with_gt=True), "cuda")
    torch.manual_seed(0)
    extractor = torch.nn.Linear(64, 128).cuda()
    model = _matcher(1.0)
    opt = torch.optim.Adam([*extractor.parameters(), *model.parameters()], lr=1e-2)
    hist = []
    for _ in range(6):
        opt.zero_grad()
        f0 = F.normalize(extractor(data["descriptors0"]), dim=-1)
        f1 = F.normalize(extractor(data["descriptors1"]), dim=-1)
        losses = _step(model, dict(data, descriptors0=f0, descriptors1=f1))
        assert extractor.weight.grad.abs().sum() > 0 and model.temperature.grad != 0
        opt.step()
        hist.append(float(losses["total"].mean().detach()))
    assert hist[-1] < hist[0], hist

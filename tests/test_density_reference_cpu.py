"""The float64 proposal-density reference (``density_reference.py``) against the oracle's ``HashMLPDensityField`` and against finite
differences, and the proposal field's construction-time refusals.  No GPU needed."""
import pytest
import torch

import density_reference as dref

from cropnerf_b200.density_fields import HashMLPDensityField
from cropnerf_b200.field_components import SceneContraction, hash_scalings
from oracle import nerfstudio_torch as ns


def _oracle_field(case):
    H = case.W1.shape[0]
    f = ns.HashMLPDensityField(case.aabb, hidden_dim=H, num_levels=case.num_levels, max_res=int(case.scalings[-1]) + 1,
                               log2_hashmap_size=case.log2_hashmap_size, spatial_distortion=ns.SceneContraction() if case.contraction else None,
                               average_init_density=case.avg)
    f.encoding.scalings.copy_(torch.tensor(case.scalings))
    net = f.mlp_base[1]
    with torch.no_grad():
        f.encoding.hash_table.copy_(case.table)
        net.layers[0].weight.copy_(case.W1)
        net.layers[0].bias.copy_(case.b1)
        net.layers[1].weight.copy_(case.W2)
        net.layers[1].bias.copy_(case.b2)
    return f


def _oracle_samples(case):
    R, S = case.R, case.S
    fr = ns.Frustums(case.origins[:, None, :].expand(R, S, 3), case.directions[:, None, :].expand(R, S, 3), case.starts[..., None],
                     case.ends[..., None], torch.ones(R, S, 1))
    return ns.RaySamples(fr)


@pytest.mark.parametrize("contraction", [True, False])
@pytest.mark.parametrize("L,H", [(5, 16), (8, 64)])
def test_reference_in_float32_is_the_oracle(L, H, contraction):
    case = dref.make_case(29, 37, L, H, contraction, seed=L + H)
    assert case.scalings == hash_scalings(L, 16, 2048).tolist()
    dd = torch.randn(case.R * case.S, generator=torch.Generator().manual_seed(1))
    ref = dref.evaluate(case, dd, dtype=torch.float32)
    oracle = _oracle_field(case)
    d, _ = oracle.get_density(_oracle_samples(case))
    (d.reshape(-1) * dd).sum().backward()
    assert (ref["density"] != 0).all() if contraction else (ref["density"] == 0).any()  # without contraction, rays leave the box
    err = ((ref["density"] - d.detach().reshape(-1)).abs() / (d.detach().reshape(-1).abs() + 1e-30)).max().item()
    assert err <= 1e-6, f"density: {err:.3e}"
    net = oracle.mlp_base[1]
    grads = {"table": oracle.encoding.hash_table.grad, "W1": net.layers[0].weight.grad, "b1": net.layers[0].bias.grad,
             "W2": net.layers[1].weight.grad, "b2": net.layers[1].bias.grad}
    for k, g in grads.items():
        err = (ref[k] - g).abs().max().item() / g.abs().max().item()
        assert err <= 1e-6, f"{k}: {err:.3e}"


@pytest.mark.parametrize("contraction", [True, False])
def test_reference_ray_gradients_match_finite_differences(contraction):
    """The reference's d origins / d directions are autograd through the float64 warp with the float32 cells held fixed; gradcheck
    differentiates the same function numerically.  Rays 1 and 2 are the far ray and the zero-length frustums."""
    case = dref.make_case(5, 8, 5, 16, contraction, seed=3)
    idx = dref.corners(case)
    off = idx["offsets"][idx["selector"]]
    assert idx["selector"].sum() >= 10 and ((off > 0.01) & (off < 0.99)).float().mean() > 0.9  # mostly away from cell faces
    params = [getattr(case, k).double() for k in ("table", "W1", "b1", "W2", "b2")]
    dd = torch.randn(case.R * case.S, generator=torch.Generator().manual_seed(2), dtype=torch.float64)

    def f(o, d):
        return (dref.forward(case, idx, *params, origins=o, directions=d)[0] * dd).sum()

    o = case.origins.double().requires_grad_(True)
    d = case.directions.double().requires_grad_(True)
    assert torch.autograd.gradcheck(f, (o, d), eps=1e-7, atol=1e-6, rtol=1e-5)
    ref = dref.evaluate(case, dd, ray_grads=True)
    go, gd = torch.autograd.grad(f(o, d), (o, d))
    assert torch.equal(ref["origins"], go) and torch.equal(ref["directions"], gd)
    assert go.abs().max() > 0 and gd.abs().max() > 0
    # with the rays given, the value is the float32 cell's: the same densities as without ray gradients
    assert torch.equal(ref["density"], dref.evaluate(case)["density"])


@pytest.mark.parametrize("kw", [dict(num_layers=3), dict(features_per_level=4), dict(num_levels=17), dict(hidden_dim=8), dict(hidden_dim=48),
                                dict(hidden_dim=128)], ids=lambda kw: "-".join(f"{k}={v}" for k, v in kw.items()))
def test_proposal_field_refuses_uncompiled_architectures_at_construction(kw):
    with pytest.raises(ValueError):
        HashMLPDensityField(torch.tensor([[-1.0] * 3, [1.0] * 3]), spatial_distortion=SceneContraction(), **kw)


@pytest.mark.parametrize("H", [16, 32, 64])
def test_proposal_field_accepts_compiled_widths(H):
    f = HashMLPDensityField(torch.tensor([[-1.0] * 3, [1.0] * 3]), hidden_dim=H, num_levels=12)
    assert f.mlp_base[1].layers[0].weight.shape == (H, 24)

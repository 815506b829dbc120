"""The proposal-network density operator (``csrc/density_field.cu``) at every compiled (levels, hidden width) specialisation against the
float64 reference of ``density_reference.py``: forward densities, the table / MLP parameter gradients, the gradient reaching the encoded
features and the rays, the kept-feature forward / backward pair, the fused training step at a non-default proposal shape, and the
configurations the operator refuses.

Which kernel runs (``DISPATCH`` / ``launch_bwd``): the forward is ``k_density_fwd<8|16, H>``; the backward is the tensor-core kernel
``k_density_bwd_tc`` for hidden 16 with <= 7 levels (mixed precision: bf16 operands in its MLP parameter-gradient contraction) and the
SIMT kernel ``k_density_bwd<8|16, H>`` otherwise, in either precision.  4096 x 256 samples are more than the forward's (16 CTAs / SM)
and the SIMT backward's (8 CTAs / SM) grid caps, so the grid-stride loops run several rounds.

Bounds: every test records its largest errors as test properties (``pytest --junitxml``).  Each bound below is at most 10x the largest
error observed over the cases it covers, measured on one NVIDIA B200 (1000 W power limit); the observation is noted beside it."""
import ctypes as C
import dataclasses

import pytest
import torch

import density_reference as dref
from helpers import product_bundle, product_model

from cropnerf_b200 import _lib as L
from cropnerf_b200 import engine, ops, synthetic
from cropnerf_b200.density_fields import HashMLPDensityField
from cropnerf_b200.field_components import SceneContraction
from oracle import cases

pytestmark = pytest.mark.gpu

TOL_FWD = 1e-5    # |d - d_ref| <= TOL_FWD * (|d_ref| + FLOOR); observed 6.1e-6 (MLP output ~ -15: expf of an fp32 sum of that size), else 3.1e-7
FLOOR = 1e-12
TOL_BWD = 5e-5    # max |g - g_ref| <= TOL_BWD * max |g_ref| per parameter tensor (exact mode, and mixed on the SIMT kernels); observed 5.1e-6
TOL_FEAT = 1e-6   # kept encoded features, same form as TOL_BWD (a blend can cancel to ~0); observed 1.4e-7
TOL_RAYS = 3e-6   # d origins / d directions, same form as TOL_BWD; observed 3.4e-7
MIXED_L2 = 2e-2   # mixed tensor-core backward: relative L2 of the MLP parameter gradients, the suite's bound; observed 8.8e-4
CNB_ERR_ARG, CNB_ERR_UNSUPPORTED = -1, -3  # include/cropnerf_b200.h
PARAMS = ("table", "W1", "b1", "W2", "b2")

# (levels, hidden): every DISPATCH entry, with both sides of the tensor-core / SIMT boundary (L = 7 / 8 at hidden 16)
MATRIX = [(1, 16), (5, 16), (7, 16), (8, 16), (3, 32), (8, 32), (8, 64), (9, 16), (16, 16), (12, 32), (12, 64), (16, 64)]


def _tensor_core(nl, H):
    return H == 16 and nl <= 7


def _d_density(n, seed):
    """Upstream gradient of both signs, mostly positive (as the interlevel loss gives), with exact zeros the kernels skip."""
    g = torch.Generator().manual_seed(seed)
    dd = torch.rand(n, generator=g) * 2.0 - 0.5
    dd[torch.rand(n, generator=g) < 0.1] = 0.0
    return dd


def _module(case, dev, precision="fp32"):
    nl, H = case.num_levels, case.W1.shape[0]
    net = HashMLPDensityField(case.aabb.to(dev), hidden_dim=H, num_levels=nl, max_res=2048, log2_hashmap_size=case.log2_hashmap_size,
                              spatial_distortion=SceneContraction() if case.contraction else None, average_init_density=case.avg,
                              precision=precision).to(dev)
    assert net.encoding._scalings_host == case.scalings
    lin = net.mlp_base[1].layers
    params = {"table": net.encoding.hash_table, "W1": lin[0].weight, "b1": lin[0].bias, "W2": lin[1].weight, "b2": lin[1].bias}
    with torch.no_grad():
        for k, p in params.items():
            p.copy_(getattr(case, k))
    return net, params


def _run(case, dev, dd, precision="fp32", ray_grads=False):
    """density_from_layout -> backward of sum(density * dd): the public operator path (cnb_density_field_fwd / _bwd / _bwd_rays)."""
    net, params = _module(case, dev, precision)
    o = case.origins.to(dev).requires_grad_(ray_grads)
    d = case.directions.to(dev).requires_grad_(ray_grads)
    density = net.density_from_layout((o, d, case.starts.to(dev), case.ends.to(dev), None, case.R, case.S, case.S))
    (density * dd.to(dev)).sum().backward()
    res = {"density": density.detach(), **{k: p.grad for k, p in params.items()}}
    if ray_grads:
        res["origins"], res["directions"] = o.grad, d.grad
    return res


def _reference(case, dd, dev, ray_grads=False):
    # the float64 half runs on the GPU: the benchmark-sized cases gather 10^8 corner values
    return dref.evaluate(case, dd, ray_grads=ray_grads, device=dev)


def _rel_fwd(a, ref):
    return ((a.double() - ref).abs() / (ref.abs() + FLOOR)).max().item()


def _rel_max(a, ref):
    return (a.double() - ref).abs().max().item() / ref.abs().max().item()


def _rel_l2(a, ref):
    return (a.double() - ref).norm().item() / ref.norm().item()


def _check(res, ref, record, precision="fp32", tensor_core=True):
    err = _rel_fwd(res["density"], ref["density"])
    record("err_density", err)
    assert err <= TOL_FWD, f"density: {err:.3e}"
    assert torch.equal(res["density"] == 0, ref["density"] == 0), "samples outside the box: exactly zero density"
    for k in PARAMS:
        g, gr = res[k], ref[k]
        assert gr.abs().max() > 0, k
        if precision == "mixed" and tensor_core and k != "table":
            err = _rel_l2(g, gr)
            record(f"l2_{k}", err)
            assert err <= MIXED_L2, f"mixed {k}: relative L2 {err:.3e}"
        else:
            err = _rel_max(g, gr)
            record(f"err_{k}", err)
            assert err <= TOL_BWD, f"{precision} {k}: {err:.3e}"


@pytest.mark.parametrize("precision", ["fp32", "mixed"])
@pytest.mark.parametrize("contraction", [True, False], ids=["contract", "aabb"])
@pytest.mark.parametrize("nl,H", MATRIX)
def test_matrix(dev, record_property, nl, H, contraction, precision):
    """37 rays x 53 samples (1961: not a multiple of the 128-sample tile), with a far ray and a ray of zero-length frustums."""
    case = dref.make_case(37, 53, nl, H, contraction, seed=100 * nl + H)
    dd = _d_density(case.R * case.S, seed=nl + H)
    _check(_run(case, dev, dd, precision), _reference(case, dd, dev), record_property, precision, _tensor_core(nl, H))


@pytest.mark.parametrize("R,S", [(1, 1), (129, 1), (2, 200)])
@pytest.mark.parametrize("nl,H", [(5, 16), (8, 16), (8, 64), (12, 32), (16, 64)])
def test_ragged_tiles(dev, record_property, nl, H, R, S):
    """One sample, and 129 samples whose last tile holds one."""
    case = dref.make_case(R, S, nl, H, True, seed=R + S)
    dd = torch.linspace(0.5, 1.5, R * S)  # no zero: the lone sample must take part
    _check(_run(case, dev, dd), _reference(case, dd, dev), record_property)


@pytest.mark.parametrize("nl,H,precision", [(5, 16, "fp32"), (5, 16, "mixed"), (8, 64, "fp32"), (16, 64, "fp32")])
def test_benchmark_size(dev, record_property, nl, H, precision):
    """4096 rays x 256 samples (a benchmark step's first proposal level): several rounds of every grid-stride loop."""
    case = dref.make_case(4096, 256, nl, H, True, seed=7 + nl)
    dd = _d_density(case.R * case.S, seed=8)
    _check(_run(case, dev, dd, precision), _reference(case, dd, dev), record_property, precision, _tensor_core(nl, H))


@pytest.mark.parametrize("shift", [15.0, -15.0])
@pytest.mark.parametrize("nl,H", [(5, 16), (8, 64)])
def test_trunc_exp_clamp(dev, record_property, nl, H, shift):
    """MLP outputs around +-15: about half the samples take trunc_exp's clamped gradient exp(+-15).  avg = 0.5."""
    case = dref.make_case(37, 53, nl, H, True, seed=5, avg=0.5, out_shift=shift)
    dd = _d_density(case.R * case.S, seed=6)
    ref = _reference(case, dd, dev)
    clamped = (ref["out"].abs() > 15).float().mean().item()
    assert 0.2 < clamped < 0.8, clamped
    _check(_run(case, dev, dd), ref, record_property)


@pytest.mark.parametrize("nl,H", [(5, 16), (8, 64)])
def test_density_fn_zero_length_frustums(dev, record_property, nl, H):
    """Field.density_fn(positions): one zero-length frustum per point (R = N rays of one sample), inside and outside the box."""
    case = dref.make_case(1, 1, nl, H, False, seed=9)
    g = torch.Generator().manual_seed(10)
    pos = (torch.rand((3001, 3), generator=g) * 2 - 1) * 1.2
    case = dataclasses.replace(case, origins=pos, directions=torch.ones_like(pos), starts=torch.zeros(3001, 1), ends=torch.zeros(3001, 1))
    dd = _d_density(3001, seed=11)
    net, params = _module(case, dev)
    density = net.density_fn(pos.to(dev))
    assert density.shape == (3001, 1)
    (density[:, 0] * dd.to(dev)).sum().backward()
    res = {"density": density.detach()[:, 0], **{k: p.grad for k, p in params.items()}}
    ref = _reference(case, dd, dev)
    assert (ref["density"] == 0).any() and (ref["density"] != 0).any()
    _check(res, ref, record_property)


def test_empty_batch(dev):
    case = dref.make_case(0, 16, 5, 16, True)
    res = _run(case, dev, torch.zeros(0))
    assert res["density"].shape == (0,)
    assert all(float(res[k].abs().max()) == 0.0 for k in PARAMS)


# ---------------------------------------------------------------------------------------------------------------------------------------
# C ABI entries without a Python path of their own


def _abi(case, dev, precision=L.PREC_FP32, grads=True):
    """cnb_density_field + cnb_samples of a case; the tensors they point to stay alive in the returned dict."""
    t = {k: getattr(case, k).to(dev).contiguous() for k in PARAMS + ("origins", "directions", "starts", "ends")}
    g = {k: torch.zeros_like(t[k]) for k in PARAMS} if grads else {k: None for k in PARAMS}
    f = L.DensityField()
    f.grid = L.make_grid(t["table"], g["table"], case.num_levels, case.log2_hashmap_size, case.scalings)
    f.mlp = L.make_mlp([t["W1"], t["W2"]], [t["b1"], t["b2"]], L.ACT_NONE, [g["W1"], g["W2"]], [g["b1"], g["b2"]])
    f.warp = L.make_warp(case.contraction, case.aabb.tolist())
    f.average_init_density = case.avg
    f.precision = precision
    sm = ops.make_samples(t["origins"], t["directions"], t["starts"], t["ends"], None, case.R, case.S, case.S)
    return {"f": f, "sm": sm, "t": t, "g": g}


@pytest.mark.parametrize("precision", ["fp32", "mixed"])
@pytest.mark.parametrize("nl", [1, 5, 7])
def test_kept_features(dev, record_property, nl, precision):
    """cnb_density_field_fwd_keep writes the encoded features level-major [L][N] float2; cnb_density_field_bwd_kept consumes them."""
    case = dref.make_case(37, 53, nl, 16, True, seed=20 + nl)
    N = case.R * case.S
    dd = _d_density(N, seed=21)
    ref = _reference(case, dd, dev)
    a = _abi(case, dev, L.PREC_MIXED if precision == "mixed" else L.PREC_FP32)
    density = torch.empty(N, device=dev)
    feat = torch.empty((nl, N, 2), device=dev)
    st = L.stream_ptr(dev)
    assert L.lib().cnb_density_field_kept_supported(C.byref(a["f"])) == 1
    L.check(L.lib().cnb_density_field_fwd_keep(C.byref(a["f"]), C.byref(a["sm"]), density.data_ptr(), feat.data_ptr(), st), "fwd_keep")
    err = _rel_max(feat.permute(1, 0, 2).reshape(N, 2 * nl), ref["feat"])
    record_property("err_feat", err)
    assert err <= TOL_FEAT, f"kept features: {err:.3e}"
    ddv = dd.to(dev)
    L.check(L.lib().cnb_density_field_bwd_kept(C.byref(a["f"]), C.byref(a["sm"]), ddv.data_ptr(), feat.data_ptr(), st), "bwd_kept")
    _check({"density": density, **a["g"]}, ref, record_property, precision, True)


@pytest.mark.parametrize("nl,H", [(1, 16), (7, 16), (8, 16), (9, 16), (5, 32), (7, 64), (16, 64)])
def test_kept_supported_exactly_for_the_tensor_core_backward(dev, nl, H):
    case = dref.make_case(5, 7, nl, H, True)
    a = _abi(case, dev)
    supported = L.lib().cnb_density_field_kept_supported(C.byref(a["f"]))
    assert supported == int(_tensor_core(nl, H))
    if supported:
        return
    N = case.R * case.S
    dd = torch.ones(N, device=dev)
    feat = torch.zeros((nl, N, 2), device=dev)
    rc = L.lib().cnb_density_field_bwd_kept(C.byref(a["f"]), C.byref(a["sm"]), dd.data_ptr(), feat.data_ptr(), L.stream_ptr(dev))
    assert rc == CNB_ERR_ARG and "kept-feature" in L.last_error()
    torch.cuda.synchronize()
    assert all(float(g.abs().max()) == 0.0 for g in a["g"].values()), "a refused call writes nothing"


@pytest.mark.parametrize("contraction", [True, False], ids=["contract", "aabb"])
@pytest.mark.parametrize("nl,H", [(5, 16), (8, 64)])
def test_ray_gradients(dev, record_property, nl, H, contraction):
    """cnb_density_field_bwd_rays: the feature gradient it leaves in its scratch ([N, 2L]), then d origins / d directions."""
    case = dref.make_case(37, 53, nl, H, contraction, seed=30 + nl)
    N = case.R * case.S
    dd = _d_density(N, seed=31)
    ref = _reference(case, dd, dev, ray_grads=True)
    res = _run(case, dev, dd, ray_grads=True)
    _check(res, ref, record_property)
    for k in ("origins", "directions"):
        err = _rel_max(res[k], ref[k])
        record_property(f"err_{k}", err)
        assert err <= TOL_RAYS, f"d {k}: {err:.3e}"
    a = _abi(case, dev)
    scratch = torch.empty((N, 2 * nl), device=dev)
    d_o, d_d = torch.zeros((case.R, 3), device=dev), torch.zeros((case.R, 3), device=dev)
    ddv = dd.to(dev)
    L.check(L.lib().cnb_density_field_bwd_rays(C.byref(a["f"]), C.byref(a["sm"]), ddv.data_ptr(), scratch.data_ptr(), d_o.data_ptr(),
                                               d_d.data_ptr(), L.stream_ptr(dev)), "bwd_rays")
    err = _rel_max(scratch, ref["d_feat"])
    record_property("err_d_feat", err)
    assert err <= TOL_BWD, f"d features: {err:.3e}"


def test_refusals(dev):
    """Configurations outside the compiled kernels return a named error and write nothing."""
    case = dref.make_case(5, 7, 5, 16, True)
    N = case.R * case.S
    st = L.stream_ptr(dev)

    def fwd(a):
        out = torch.full((N,), -7.0, device=dev)
        rc = L.lib().cnb_density_field_fwd(C.byref(a["f"]), C.byref(a["sm"]), out.data_ptr(), None, st)
        torch.cuda.synchronize()
        assert bool((out == -7.0).all()), "a refused call writes nothing"
        return rc, L.last_error()

    for H in (8, 48, 128):  # hidden widths without a kernel, past the Python constructor's check
        rc, msg = fwd(_abi(dataclasses.replace(case, W1=torch.zeros(H, 10), b1=torch.zeros(H), W2=torch.zeros(1, H)), dev, grads=False))
        assert rc == CNB_ERR_UNSUPPORTED and f"hidden width {H} not compiled" in msg, (rc, msg)
    a = _abi(case, dev, grads=False)
    a["f"].mlp.num_layers = 3
    rc, msg = fwd(a)
    assert rc == CNB_ERR_UNSUPPORTED and "2L->H->1" in msg, (rc, msg)
    a = _abi(case, dev, grads=False)
    a["f"].grid.num_levels = 17
    rc, msg = fwd(a)
    assert rc == CNB_ERR_ARG and "num_levels 17" in msg, (rc, msg)
    # level resolution >= 65535: the forward runs, the backward's aggregated scatter refuses
    net = HashMLPDensityField(torch.tensor([[-1.0] * 3, [1.0] * 3], device=dev), hidden_dim=16, num_levels=2, max_res=70000,
                              log2_hashmap_size=14, spatial_distortion=SceneContraction()).to(dev)
    assert net.encoding._scalings_host[-1] >= 65535
    rays = dref.make_case(5, 7, 2, 16, True)
    density = net.density_from_layout((rays.origins.to(dev), rays.directions.to(dev), rays.starts.to(dev), rays.ends.to(dev), None, 5, 7, 7))
    assert bool(torch.isfinite(density).all())
    with pytest.raises(RuntimeError, match="too large for the aggregated scatter"):
        density.sum().backward()
    assert net.encoding.hash_table.grad is None or float(net.encoding.hash_table.grad.abs().max()) == 0.0


def test_fused_train_step_at_the_nerfstudio_default_proposal_shape(dev):
    """Both proposal networks at nerfstudio's HashMLPDensityField default (8 levels, hidden 64): the training step's proposal backward is
    cnb_density_field_bwd (no kept features, SIMT kernel) inside cnb_train_step, against the per-module autograd operators."""
    prop = {"hidden_dim": 64, "log2_hashmap_size": 14, "num_levels": 8, "max_res": 512, "use_linear": False}
    cfg = cases.make_config(dict(proposal_net_args_list=[prop, dict(prop, max_res=1024)]))
    oracle, state = cases.build_oracle(cfg, 20, 0, 0.5)
    R = 256
    rays = synthetic.make_rays(R, seed=6, num_cameras=20)
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    jit = synthetic.make_jitter(R, 3, seed=2)
    results = []
    for use_fused in (True, False):
        model = product_model(cfg, state, 20, dev, True)
        assert all(n.mlp_base[1].layers[0].weight.shape == (64, 16) for n in model.proposal_networks)
        feed = synthetic.JitterFeed(jit)
        model.proposal_sampler.initial_sampler.rand_fn = feed
        model.proposal_sampler.pdf_sampler.rand_fn = feed
        tr = engine.Trainer(model, fused=use_fused)
        assert tr._use_fused() == use_fused
        grads = {}
        orig = tr.optimizer_step

        def spy(step, tr=tr, grads=grads, orig=orig, **kw):
            for name, g in tr.groups.items():
                grads[name] = g.grad.clone()
            orig(step, **kw)

        tr.optimizer_step = spy
        stats = tr.train_iteration(500, product_bundle(rays, dev), targets)
        results.append((stats, grads))
    (sa, ga), (sb, gb) = results
    for k in ("rgb_loss", "semantics_loss", "interlevel_loss", "distortion"):
        a, b = float(sa[k]), float(sb[k])
        assert abs(a - b) <= 1e-5 * abs(b) + 1e-7, f"{k}: fused {a} vs modular {b}"
    assert gb["proposal_networks"].abs().max().item() > 0
    for name in ga:
        err = (ga[name] - gb[name]).abs().max().item() / (gb[name].abs().max().item() + 1e-20)
        assert err < 1e-4, f"grad group {name}: {err:.3e}"

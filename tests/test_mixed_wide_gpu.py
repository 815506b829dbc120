"""Mixed precision for the FruitField of the reference's `fruit_nerf_big` / `fruit_nerf_huge` presets (geo_feat_dim 30, a three-layer 128-wide
semantic MLP): the tcgen05 MLP operator (csrc/mlp_mixed.cu) against torch fp32 autograd, and the field / models built on it against the fp32
oracle, with the tolerances the base mixed mode is held to (DESIGN section 2)."""
import ctypes as C

import pytest
import torch

from helpers import assert_close, product_bundle, product_model

from cropnerf_b200 import _lib as L
from cropnerf_b200 import engine, synthetic
from cropnerf_b200.field_components import FieldHeadNames
from oracle import cases

pytestmark = pytest.mark.gpu

RTOL_MIXED = 2e-3
CNB_ERR_UNSUPPORTED = -3   # include/cropnerf_b200.h
BIG_PRESET = dict(geo_feat_dim=30, hidden_dim_semantics=128, num_layers_semantic=3, max_res=4096)

# (dims, out_activation): the base, semantic and RGB MLPs of the big / huge presets
SHAPES = [((32, 64, 31), L.ACT_NONE), ((30, 128, 128, 64), L.ACT_NONE), ((78, 64, 64, 3), L.ACT_SIGMOID)]


def _mlp_params(dims, dev, seed):
    g = torch.Generator().manual_seed(seed)
    Ws, bs = [], []
    for i in range(len(dims) - 1):
        lin = torch.nn.Linear(dims[i], dims[i + 1])
        with torch.no_grad():
            lin.weight.copy_(torch.empty_like(lin.weight).uniform_(-1, 1, generator=g) * (6.0 / dims[i]) ** 0.5 * 0.5)
            lin.bias.copy_(torch.empty_like(lin.bias).uniform_(-0.2, 0.2, generator=g))
        Ws.append(lin.weight.detach().to(dev).contiguous())
        bs.append(lin.bias.detach().to(dev).contiguous())
    return Ws, bs


def _torch_mlp(x, Ws, bs, act, fp16_operands=False):
    """fp16_operands: the function the operator evaluates -- inputs, weights and kept hidden activations rounded to fp16, the rest in float64 --
    so that its ReLU masks are the operator's (cast gradients pass through unchanged)."""
    r = (lambda t: t.half().double()) if fp16_operands else (lambda t: t)  # noqa: E731
    h = r(x)
    for i, (W, b) in enumerate(zip(Ws, bs)):
        h = h @ r(W).t() + (b.double() if fp16_operands else b)
        if i < len(Ws) - 1:
            h = r(torch.relu(h))
    return torch.sigmoid(h) if act == L.ACT_SIGMOID else h


def _rel_l2(a, b):
    return (a.double() - b.double()).norm().item() / (b.double().norm().item() + 1e-30)


@pytest.mark.parametrize("n", [1, 127, 129, 4099, 196608])
@pytest.mark.parametrize("shape", SHAPES, ids=["base", "semantic", "rgb"])
def test_operator_matches_torch_fp32(dev, shape, n):
    dims, act = shape
    Ws, bs = _mlp_params(dims, dev, seed=len(dims) * 7 + dims[0])
    g = torch.Generator().manual_seed(n)
    # x with a row stride wider than its width (the field hands over column slices of wider rows)
    stride = dims[0] + 3
    xs = (torch.rand((n, stride), generator=g) * 2 - 1).to(dev)
    x = xs[:, : dims[0]]
    dy = torch.randn((n, dims[-1]), generator=g).to(dev)
    dWs = [torch.zeros_like(W) for W in Ws]
    dbs = [torch.zeros_like(b) for b in bs]
    m = L.make_mlp(Ws, bs, act, dWs, dbs)
    lib = L.lib()
    floats = lib.cnb_mlp_mixed_scratch_floats(C.byref(m), n, 1)
    assert floats > 0 and floats >= lib.cnb_mlp_mixed_scratch_floats(C.byref(m), n, 0)
    scratch = torch.empty((floats,), device=dev, dtype=torch.float32)
    y = torch.empty((n, dims[-1]), device=dev, dtype=torch.float32)
    dx = torch.empty((n, dims[0] + 1), device=dev, dtype=torch.float32)
    st = L.stream_ptr(dev)
    L.check(lib.cnb_mlp_mixed_fwd(C.byref(m), xs.data_ptr(), stride, n, y.data_ptr(), scratch.data_ptr(), 1, st), "mlp_mixed_fwd")
    L.check(lib.cnb_mlp_mixed_bwd(C.byref(m), xs.data_ptr(), stride, y.data_ptr(), dy.data_ptr(), n, dx.data_ptr(), dims[0] + 1, scratch.data_ptr(), st),
            "mlp_mixed_bwd")
    # inference forward: its own (smaller) scratch, same numbers
    y_inf = torch.empty_like(y)
    s_inf = torch.empty((max(1, lib.cnb_mlp_mixed_scratch_floats(C.byref(m), n, 0)),), device=dev, dtype=torch.float32)
    L.check(lib.cnb_mlp_mixed_fwd(C.byref(m), xs.data_ptr(), stride, n, y_inf.data_ptr(), s_inf.data_ptr(), 0, st), "mlp_mixed_fwd inference")
    torch.cuda.synchronize()
    assert torch.equal(y, y_inf)

    xr = x.detach().clone().requires_grad_(True)
    Wr = [W.clone().requires_grad_(True) for W in Ws]
    br = [b.clone().requires_grad_(True) for b in bs]
    yr = _torch_mlp(xr, Wr, br, act)
    (yr * dy).sum().backward()
    scale = yr.detach().abs().max().item()
    err = (y - yr.detach()).abs().max().item()
    assert err <= 2e-3 * scale, f"forward max error {err:.3e} vs output scale {scale:.3e}"
    # The gradients are those of the function the operator evaluated: its ReLU masks come from its stored fp16 activations.  Where the fp16
    # forward and the fp32 one disagree on the sign of a hidden unit near zero, the masks differ and that row's contribution is off by its
    # full size (relative L2 ~ sqrt(flipped fraction); measured up to 4 % for dX, which is per row, and 2 % for dW at 127 rows).  So every
    # gradient is held to the bf16 bound against the autograd of THAT function (fp16-rounded operands and kept activations, float64
    # arithmetic), and to 5e-2 against fp32.
    xh = x.detach().clone().requires_grad_(True)
    Wh = [W.clone().requires_grad_(True) for W in Ws]
    bh = [b.clone().requires_grad_(True) for b in bs]
    (_torch_mlp(xh, Wh, bh, act, fp16_operands=True) * dy.double()).sum().backward()
    grads = [("dX", dx[:, : dims[0]], xh.grad, xr.grad)]
    for i in range(len(Ws)):
        grads += [(f"dW{i}", dWs[i], Wh[i].grad, Wr[i].grad), (f"db{i}", dbs[i], bh[i].grad, br[i].grad)]
    for name, got, ref16, ref32 in grads:
        assert _rel_l2(got, ref16) <= 2e-2, f"{name} relative L2 vs the fp16-operand function {_rel_l2(got, ref16):.3e}"
        assert _rel_l2(got, ref32) <= 5e-2, f"{name} relative L2 vs fp32 {_rel_l2(got, ref32):.3e}"


def test_operator_refuses_shapes_outside_support(dev):
    """Layers wider than 128 are refused with the shape in the message, never computed wrongly."""
    lib = L.lib()
    for dims in ((30, 256, 64), (256, 64, 3), (64, 129)):
        Ws, bs = _mlp_params(dims, dev, seed=1)
        m = L.make_mlp(Ws, bs, L.ACT_NONE)
        n = 256
        x = torch.randn((n, dims[0]), device=dev)
        y = torch.full((n, dims[-1]), 7.0, device=dev)
        scratch = torch.empty((1 << 20,), device=dev)
        assert lib.cnb_mlp_mixed_scratch_floats(C.byref(m), n, 1) == 0
        rc = lib.cnb_mlp_mixed_fwd(C.byref(m), x.data_ptr(), dims[0], n, y.data_ptr(), scratch.data_ptr(), 1, L.stream_ptr(dev))
        assert rc == CNB_ERR_UNSUPPORTED
        assert "->".join(str(d) for d in dims) in L.last_error()
        assert bool((y == 7.0).all())


def _field_samples(R, S, seed):
    rays = synthetic.make_rays(R, seed=seed, num_cameras=20)
    g = torch.Generator().manual_seed(seed)
    edges = torch.sort(torch.rand((R, S + 1), generator=g) * 3.0, dim=-1).values
    edges[0] = torch.linspace(0, 2000.0, S + 1)  # far samples: contraction branch
    return rays, edges


def _field_pair(dev, training, contraction=True):
    cfg = cases.make_config(dict(log2_hashmap_size=14, disable_scene_contraction=not contraction, **BIG_PRESET))
    oracle, state = cases.build_oracle(cfg, 20, seed=0, table_scale=0.5)
    oracle.train(training)
    model = product_model(cfg, state, 20, dev, training, precision="mixed")
    return oracle, model


@pytest.mark.parametrize("contraction", [True, False])
@pytest.mark.parametrize("training", [False, True])
def test_field_forward_mixed_big(dev, training, contraction):
    R, S = 200, 48
    oracle, model = _field_pair(dev, training, contraction)
    rays, edges = _field_samples(R, S, 3)
    rs = cases.oracle_bundle(rays).get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    with torch.set_grad_enabled(training):
        out_ref = oracle.field(rs)
        e = edges.to(dev)
        out = model.field(product_bundle(rays, dev).get_ray_samples(e[:, :-1, None], e[:, 1:, None]))
    assert_close(out[FieldHeadNames.RGB], out_ref["rgb"].detach(), RTOL_MIXED, "mixed rgb", floor=1e-1)
    assert_close(out[FieldHeadNames.DENSITY], out_ref["density"].detach(), 1e-2, "mixed density", floor=1e-2, frac=0.999)
    assert_close(out[FieldHeadNames.SEMANTICS], out_ref["semantics"].detach(), 1e-2, "mixed semantics", floor=1e-1)
    assert torch.equal(model.field._sample_locations.cpu(), oracle.field._sample_locations.detach())


@pytest.mark.parametrize("R,S", [(160, 48), (37, 21), (9, 5)])
def test_field_backward_mixed_big(dev, R, S):
    oracle, model = _field_pair(dev, True)
    rays, edges = _field_samples(R, S, 3)
    rs = cases.oracle_bundle(rays).get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    out_ref = oracle.field(rs)
    e = edges.to(dev)
    out = model.field(product_bundle(rays, dev).get_ray_samples(e[:, :-1, None], e[:, 1:, None]))
    g = torch.Generator().manual_seed(11)
    gd, gr, gs = torch.randn((R, S, 1), generator=g) * 0.01, torch.randn((R, S, 3), generator=g), torch.randn((R, S, 1), generator=g)
    (out_ref["density"] * gd).sum().add((out_ref["rgb"] * gr).sum()).add((out_ref["semantics"] * gs).sum()).backward()
    (out[FieldHeadNames.DENSITY] * gd.to(dev)).sum().add((out[FieldHeadNames.RGB] * gr.to(dev)).sum()).add(
        (out[FieldHeadNames.SEMANTICS] * gs.to(dev)).sum()).backward()
    ref_params = dict(oracle.field.named_parameters())
    worst = {}
    for name, p in model.field.named_parameters():
        gr_ = ref_params[name].grad
        assert gr_ is not None and p.grad is not None, name
        worst[name] = _rel_l2(p.grad.cpu(), gr_)
    tol = 4e-2 if R * S >= 500 else 6e-2
    bad = {k: v for k, v in worst.items() if not v < tol}
    assert not bad, f"mixed backward relative L2 errors: {bad} (all: {worst})"


@pytest.mark.parametrize("training", [False, True])
def test_get_density_get_outputs_split_mixed_big(dev, training):
    R, S = 96, 48
    oracle, model = _field_pair(dev, training)
    rays, edges = _field_samples(R, S, 5)
    e = edges.to(dev)
    rs = product_bundle(rays, dev).get_ray_samples(e[:, :-1, None], e[:, 1:, None])
    with torch.set_grad_enabled(training):
        density, emb = model.field.get_density(rs)
        heads = model.field.get_outputs(rs, density_embedding=emb)
        full = model.field(rs)
    assert emb.shape == (R, S, 30) and density.shape == (R, S, 1)
    assert torch.equal(density, full[FieldHeadNames.DENSITY]) and torch.equal(heads[FieldHeadNames.RGB], full[FieldHeadNames.RGB])
    assert torch.equal(heads[FieldHeadNames.SEMANTICS], full[FieldHeadNames.SEMANTICS])
    rs_o = cases.oracle_bundle(rays).get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    with torch.no_grad():
        _, emb_ref = oracle.field.get_density(rs_o)
    assert (emb.detach().cpu() - emb_ref).abs().max().item() <= 2e-2 * max(1.0, emb_ref.abs().max().item())


def _preset_cfg(preset, log2_hashmap_size=15):
    big = dict(BIG_PRESET, num_nerf_samples_per_ray=128, num_proposal_samples_per_ray=(512, 256), proposal_weights_anneal_max_num_iters=5000,
               log2_hashmap_size=log2_hashmap_size)
    if preset == "huge":   # fruit_nerf_config.py:141-150: 7-level second proposal grid, (512, 512) + 64 samples, max_res 8192
        big.update(num_nerf_samples_per_ray=64, num_proposal_samples_per_ray=(512, 512), max_res=8192, proposal_net_args_list=[
            {"hidden_dim": 16, "log2_hashmap_size": 13, "num_levels": 5, "max_res": 512, "use_linear": False},
            {"hidden_dim": 16, "log2_hashmap_size": 13, "num_levels": 7, "max_res": 2048, "use_linear": False}])
    return cases.make_config(big)


@pytest.mark.parametrize("preset", ["big", "huge"])
@pytest.mark.parametrize("training", [False, True])
def test_preset_model_mixed_vs_oracle(dev, training, preset):
    cfg = _preset_cfg(preset)
    num_images, R = 20, 96
    oracle, state = cases.build_oracle(cfg, num_images, 0, 0.5)
    oracle.train(training)
    rays = synthetic.make_rays(R, seed=4, num_cameras=num_images)
    model = product_model(cfg, state, num_images, dev, training, precision="mixed")
    if not training:
        with torch.no_grad():
            ref = oracle(cases.oracle_bundle(rays))
            out = model(product_bundle(rays, dev))
        assert_close(out["rgb"], ref["rgb"], RTOL_MIXED, "mixed rgb", floor=1e-1)
        assert_close(out["accumulation"], ref["accumulation"], RTOL_MIXED, "mixed accumulation", floor=1e-1)
        agree = (out["semantics_colormap"].cpu() == ref["semantics_colormap"]).float().mean().item()
        assert agree >= 0.999, agree
        d_rel = ((out["depth"].cpu() - ref["depth"]).abs() / (ref["depth"].abs() + 1e-3)).flatten()
        print(f"{preset} mixed depth: {float((d_rel <= RTOL_MIXED).float().mean()):.4f} of rays within {RTOL_MIXED} relative")
        return
    jit = synthetic.make_jitter(R, 3, seed=2)
    for mdl in (oracle, model):
        feed = synthetic.JitterFeed(jit)
        mdl.proposal_sampler.initial_sampler.rand_fn = feed
        mdl.proposal_sampler.pdf_sampler.rand_fn = feed
    oracle.set_anneal(2500)
    for cb in model.get_training_callbacks():
        if "BEFORE_TRAIN_ITERATION" in cb.where_to_run:
            cb.func(2500)
    targets = synthetic.make_targets(R, seed=3)
    ref = oracle(cases.oracle_bundle(rays))
    loss_ref = oracle.get_loss_dict(ref, targets)
    sum(loss_ref.values()).backward()
    out = model(product_bundle(rays, dev))
    loss = model.get_loss_dict(out, {k: v.to(dev) for k, v in targets.items()})
    for k, v in loss.items():
        r = float(loss_ref[k])
        assert abs(float(v) - r) <= 1e-3 * abs(r) + 1e-8, f"{k}: {float(v)} vs {r}"
    sum(loss.values()).backward()
    ref_params = dict(oracle.named_parameters())
    checked = 0
    for name, p in model.named_parameters():
        gr = ref_params[name].grad if name in ref_params else None
        if gr is None or p.grad is None:
            continue
        gn, rn = p.grad.double().norm().item(), gr.double().norm().item()
        assert abs(gn - rn) <= 4e-2 * rn + 1e-12, f"grad norm {name}: {gn} vs {rn}"
        checked += 1
    assert checked >= 20


def _big_models(dev, n=2, num_images=20):
    cfg = _preset_cfg("big")
    _, state = cases.build_oracle(cfg, num_images, 0, 0.5)
    return [product_model(cfg, state, num_images, dev, True, precision="mixed") for _ in range(n)]


def test_fused_train_step_equals_modular_mixed_big(dev):
    """cnb_train_step and the per-module autograd operators run the same kernels: identical losses, gradients to fp32 atomic noise."""
    R = 256
    fused, modular = _big_models(dev)
    rays = synthetic.make_rays(R, seed=6, num_cameras=20)
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    jit = synthetic.make_jitter(R, 3, seed=2)
    results = []
    for model, use_fused in ((fused, True), (modular, False)):
        feed = synthetic.JitterFeed(jit)
        model.proposal_sampler.initial_sampler.rand_fn = feed
        model.proposal_sampler.pdf_sampler.rand_fn = feed
        tr = engine.Trainer(model, fused=use_fused)
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
    for k in ("rgb_loss", "semantics_loss", "interlevel_loss", "distortion", "psnr"):
        a, b = float(sa[k]), float(sb[k])
        assert abs(a - b) <= 1e-5 * abs(b) + 1e-7, f"{k}: fused {a} vs modular {b}"
    for name in ga:
        scale = gb[name].abs().max().item() + 1e-20
        err = (ga[name] - gb[name]).abs().max().item() / scale
        assert err < 2e-3, f"grad group {name}: {err:.3e}"
        assert gb[name].abs().max().item() > 0


def test_fused_render_equals_modular_mixed_big(dev):
    fused, modular = _big_models(dev)
    for m in (fused, modular):
        m.eval()
    modular.fused_render = False
    rays = synthetic.make_rays(777, seed=4, num_cameras=20)
    with torch.no_grad():
        a = fused(product_bundle(rays, dev))
        b = modular(product_bundle(rays, dev))
    for k in ("rgb", "accumulation", "depth", "semantics", "semantics_colormap"):
        assert torch.equal(a[k], b[k]), f"{k}: max diff {(a[k].float() - b[k].float()).abs().max().item()}"


def test_cuda_graph_radam_step_equals_eager_mixed_big(dev):
    R = 256
    a, b = _big_models(dev)
    rays = synthetic.make_rays(R, seed=6, num_cameras=20)
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    jit = synthetic.make_jitter(R, 3, seed=2)
    stats, params = [], []
    for model, graph in ((a, True), (b, False)):
        feed = synthetic.JitterFeed(jit)
        model.proposal_sampler.initial_sampler.rand_fn = feed
        model.proposal_sampler.pdf_sampler.rand_fn = feed
        tr = engine.Trainer(model, optimizers=engine.BIG_PRESET_OPTIMIZERS, cuda_graph=graph, force_proposal_update=True)
        for step in (6000, 6001, 6002):   # past the preset's 5000 anneal iterations, which run eagerly
            feed.reset()
            st = tr.train_iteration(step, product_bundle(rays, dev), targets)
        stats.append({k: float(v) for k, v in st.items()})
        params.append({n: g.flat.clone() for n, g in tr.groups.items()})
        if graph:
            assert len(tr._graphs) == 1
    for k in ("rgb_loss", "semantics_loss", "interlevel_loss", "distortion"):
        assert abs(stats[0][k] - stats[1][k]) <= 2e-4 * abs(stats[1][k]) + 1e-7, (k, stats[0][k], stats[1][k])
    for n in params[0]:
        assert (params[0][n] - params[1][n]).abs().max().item() < 5e-2, n


def test_in_step_camera_optimizer_mixed_big(dev):
    """SO3xR3 inside cnb_train_step (ray gradients through the row-major d(features) of this path) against the autograd route."""
    from cropnerf_b200.fruit_nerf import CameraOptimizer

    R, num_images = 256, 12
    cfg = _preset_cfg("big")
    _, state = cases.build_oracle(cfg, num_images, 0, 0.5)
    rays = synthetic.make_rays(R, seed=6, num_cameras=num_images)
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    jit = synthetic.make_jitter(R, 3, seed=2)
    g = torch.Generator().manual_seed(5)
    pose0 = torch.randn((num_images, 6), generator=g) * 0.02
    got = []
    for eager in (True, False):
        model = product_model(cfg, state, num_images, dev, True, precision="mixed")
        model.camera_optimizer = CameraOptimizer(num_images, "SO3xR3").to(dev)
        with torch.no_grad():
            model.camera_optimizer.pose_adjustment.copy_(pose0.to(dev))
        feed = synthetic.JitterFeed(jit)
        model.proposal_sampler.initial_sampler.rand_fn = feed
        model.proposal_sampler.pdf_sampler.rand_fn = feed
        tr = engine.Trainer(model, force_proposal_update=True)
        tr._camopt_eager = eager
        grads = {}
        orig = tr.optimizer_step

        def spy(step, tr=tr, grads=grads, orig=orig, **kw):
            for name, grp in tr.groups.items():
                grads[name] = grp.grad.clone()
            orig(step, **kw)

        tr.optimizer_step = spy
        stats = tr.train_iteration(2000, product_bundle(rays, dev), targets)
        got.append(({k: float(v) for k, v in stats.items()}, grads))
    (sa, ga), (sb, gb) = got
    for k in ("rgb_loss", "semantics_loss", "interlevel_loss"):
        assert abs(sa[k] - sb[k]) <= 1e-5 * abs(sa[k]) + 1e-8, (k, sa[k], sb[k])
    for name in ("camera_opt", "fields", "proposal_networks"):
        a, b = ga[name].double(), gb[name].double()
        err = (a - b).norm().item() / (a.norm().item() + 1e-30)
        assert err <= 5e-3, (name, err)
        assert a.abs().max().item() > 0

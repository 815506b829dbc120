"""fp16 field tables (FruitField table_precision="fp16") at the fruit_nerf_big / _huge shapes.

Key invariant: a field with fp16 tables computes exactly what the fp32-table path computes on a table holding hash_table.half().float().  The
kernels are compared with that rounded table bit for bit; whole models are compared with a model whose fp32 table is already fp16-representable,
where only the order of the red.global table-gradient scatter may differ."""
import ctypes as C

import pytest
import torch

from helpers import assert_close, product_bundle, product_model

from cropnerf_b200 import _lib as L
from cropnerf_b200 import engine, export, ops, synthetic
from cropnerf_b200.checkpoint import load_nerfstudio_checkpoint
from cropnerf_b200.field_components import hash_scalings
from oracle import cases

pytestmark = pytest.mark.gpu

RTOL_MIXED = 2e-3   # tests/test_mixed_wide_gpu.py
BIG_PRESET = dict(geo_feat_dim=30, hidden_dim_semantics=128, num_layers_semantic=3, max_res=4096)
CNB_ERR_UNSUPPORTED = -3


def _preset_cfg(preset, log2_hashmap_size=15):
    big = dict(BIG_PRESET, num_nerf_samples_per_ray=128, num_proposal_samples_per_ray=(512, 256), proposal_weights_anneal_max_num_iters=5000,
               log2_hashmap_size=log2_hashmap_size)
    if preset == "huge":
        big.update(num_nerf_samples_per_ray=64, num_proposal_samples_per_ray=(512, 512), max_res=8192, proposal_net_args_list=[
            {"hidden_dim": 16, "log2_hashmap_size": 13, "num_levels": 5, "max_res": 512, "use_linear": False},
            {"hidden_dim": 16, "log2_hashmap_size": 13, "num_levels": 7, "max_res": 2048, "use_linear": False}])
    return cases.make_config(big)


def _model(dev, preset, table_precision, rounded, training=True, num_images=20, test_mode="val"):
    cfg = _preset_cfg(preset)
    _, state = cases.build_oracle(cfg, num_images, 0, 0.5)
    model = product_model(cfg, state, num_images, dev, training, precision="mixed", test_mode=test_mode)
    if rounded:   # in place: the state dict holds the table under two aliases (mlp_base_grid / mlp_base.0)
        with torch.no_grad():
            t = model.field.mlp_base_grid.hash_table
            t.copy_(t.half().float())
    if table_precision == "fp16":   # the same weights behind an fp16-table field
        from cropnerf_b200.fruit_nerf import FruitModel

        c = model.config
        c.table_precision = "fp16"
        m2 = FruitModel(c, num_train_data=num_images, test_mode=test_mode)
        m2.load_state_dict(model.state_dict())
        model = m2.to(dev)
        model.train(training)
    return model


def _copy_matches(field):
    torch.cuda.synchronize()
    return torch.equal(field.table_half, field.mlp_base_grid.hash_table.detach().half())


# ---- kernels --------------------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("log2_T", [19, 21])
@pytest.mark.parametrize("levels", list(range(1, 17)))
def test_gather_equals_fp32_kernel_on_rounded_table(dev, levels, log2_T):
    g = torch.Generator(device=dev).manual_seed(levels * 100 + log2_T)
    rows = levels << log2_T
    table = (torch.rand((rows, 2), device=dev, generator=g) * 2 - 1) * 0.5
    half = table.half()
    rounded = half.float()   # kept alive: the descriptor holds a raw pointer
    n = 1 << 16
    pos = torch.rand((n, 3), device=dev, generator=g)
    pos[:64] = torch.floor(pos[:64] * 64) / 64   # lattice points: ceil == floor on some axes
    scal = hash_scalings(levels, 16, 4096).tolist()
    grid = L.make_grid(rounded, None, levels, log2_T, scal)
    a, b = torch.empty((n, 2 * levels), device=dev), torch.empty((n, 2 * levels), device=dev)
    ia, ib = torch.empty((n, levels, 8), device=dev, dtype=torch.int32), torch.empty((n, levels, 8), device=dev, dtype=torch.int32)
    st = L.stream_ptr(dev)
    L.check(L.lib().cnb_hashgrid_fwd(C.byref(grid), pos.data_ptr(), n, a.data_ptr(), ia.data_ptr(), st), "fwd")
    grid.table = table.data_ptr()   # the fp32 master must not be read
    L.check(L.lib().cnb_hashgrid_fwd_half(C.byref(grid), half.data_ptr(), pos.data_ptr(), n, b.data_ptr(), ib.data_ptr(), st), "fwd_half")
    assert torch.equal(a, b)
    assert torch.equal(ia, ib)


@pytest.mark.parametrize("log2_T", [19, 21])
@pytest.mark.parametrize("contract", [True, False])
def test_position_gradient_equals_fp32_kernel_on_rounded_table(dev, contract, log2_T):
    levels = 16
    g = torch.Generator(device=dev).manual_seed(7 + log2_T)
    table = (torch.rand((levels << log2_T, 2), device=dev, generator=g) * 2 - 1) * 0.5
    half = table.half()
    rounded = half.float()
    R, S = 512, 32   # one warp per ray: each ray gradient is one atomic add, so the two runs are bit-comparable
    rays = synthetic.make_rays(R, seed=3, num_cameras=4)
    o, d = rays["origins"].to(dev).contiguous(), rays["directions"].to(dev).contiguous()
    edges = torch.sort(torch.rand((R, S + 1), device=dev, generator=g) * 4 + 0.05, dim=1).values.contiguous()
    sm = ops.make_samples(o, d, edges, edges[:, 1:], None, R, S, S + 1)
    warp = L.make_warp(contract, None if contract else [[-2.0, -2.0, -2.0], [2.0, 2.0, 2.0]])
    d_feat = torch.randn((R * S, 2 * levels), device=dev, generator=g)
    scal = hash_scalings(levels, 16, 4096).tolist()
    out = []
    for fp16 in (False, True):
        grid = L.make_grid(table if fp16 else rounded, None, levels, log2_T, scal)
        d_o, d_d = torch.zeros_like(o), torch.zeros_like(d)
        if fp16:
            rc = L.lib().cnb_position_grad_rays_half(C.byref(grid), half.data_ptr(), C.byref(warp), C.byref(sm), d_feat.data_ptr(), d_o.data_ptr(),
                                                     d_d.data_ptr(), L.stream_ptr(dev))
        else:
            rc = L.lib().cnb_position_grad_rays(C.byref(grid), C.byref(warp), C.byref(sm), d_feat.data_ptr(), d_o.data_ptr(), d_d.data_ptr(),
                                                L.stream_ptr(dev))
        L.check(rc, "position_grad_rays")
        out.append((d_o, d_d))
    assert out[0][0].abs().max() > 0
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])


def test_table_to_half_and_fused_update_store(dev):
    g = torch.Generator(device=dev).manual_seed(1)
    n, first, count = 4096, 512, 2048
    p = torch.randn(n, device=dev, generator=g)
    grad = torch.randn(n, device=dev, generator=g)
    m, v = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    half = torch.zeros(count, device=dev, dtype=torch.float16)
    ops.table_to_half(p[first:first + count], half)
    assert torch.equal(half, p[first:first + count].half())
    ref = p.clone()
    ops.adam_step(ref, grad.clone(), m.clone(), v.clone(), 1e-2, 1, zero_grad=True)
    ops.adam_step(p, grad, m, v, 1e-2, 1, zero_grad=True, half=(half, first, count))
    assert torch.equal(p, ref)
    assert torch.equal(half, p[first:first + count].half())
    assert not grad.any()


# ---- whole models ---------------------------------------------------------------------------------------------------------------------


def _step_pair(dev, preset, graph):
    R = 256
    rays = synthetic.make_rays(R, seed=6, num_cameras=20)
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    jit = synthetic.make_jitter(R, 3, seed=2)
    res = []
    for tp in ("fp32", "fp16"):
        model = _model(dev, preset, tp, rounded=True)
        feed = synthetic.JitterFeed(jit)
        model.proposal_sampler.initial_sampler.rand_fn = feed
        model.proposal_sampler.pdf_sampler.rand_fn = feed
        tr = engine.Trainer(model, optimizers=engine.BIG_PRESET_OPTIMIZERS, cuda_graph=graph, force_proposal_update=True)
        grads = {}
        orig = tr.optimizer_step

        def spy(step, tr=tr, grads=grads, orig=orig, **kw):
            for name, gr in tr.groups.items():
                grads[name] = gr.grad.clone()
            orig(step, **kw)

        tr.optimizer_step = spy
        stats = []
        for step in (6000, 6001, 6002):   # eager warm-up, capture, replay (past the 5000 anneal iterations)
            feed.reset()
            st = tr.train_iteration(step, product_bundle(rays, dev), targets)
            stats.append({k: float(v) for k, v in st.items()})
        tr.wait_deferred_update()
        res.append((model, tr, stats, grads))
    return res


@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("preset", ["big", "huge"])
def test_training_step_equals_fp32_table_on_rounded_table(dev, preset, graph):
    (m32, t32, s32, g32), (m16, t16, s16, g16) = _step_pair(dev, preset, graph)
    for a, b in zip(s32, s16):
        for k in ("rgb_loss", "semantics_loss", "interlevel_loss", "distortion", "psnr"):
            assert abs(a[k] - b[k]) <= 1e-5 * abs(a[k]) + 1e-7, (k, a[k], b[k])
    for name in g32:   # the eager path's last gradients (graphed steps update inside the graph: nothing to spy on)
        scale = g32[name].abs().max().item() + 1e-20
        assert (g32[name] - g16[name]).abs().max().item() <= 1e-4 * scale, name
    lr = engine.BIG_PRESET_OPTIMIZERS["fields"].lr
    for name in t32.groups:
        diff = (t32.groups[name].flat - t16.groups[name].flat).abs()
        # a scatter-order difference can flip the first Adam steps of a near-zero gradient: at most a few lr, on few entries
        assert diff.max().item() <= 6 * lr, name
        assert (diff > 1e-6).float().mean().item() < 1e-3, name
    assert _copy_matches(m16.field)


@pytest.mark.parametrize("preset", ["big", "huge"])
def test_render_and_sample_volume_equal_fp32_table_on_rounded_table(dev, preset):
    rays = synthetic.make_rays(777, seed=4, num_cameras=20)
    outs, vols = [], []
    for tp in ("fp32", "fp16"):
        m = _model(dev, preset, tp, rounded=True, training=False)
        with torch.no_grad():
            outs.append(m(product_bundle(rays, dev)))
        m = _model(dev, preset, tp, rounded=True, training=False, test_mode="export")
        m.field.test_mode = "export"
        m.setup_inference(True, 40)
        m.eval()
        vols.append(export.sample_volume(m, ((-0.5, -0.5, -0.5), (0.5, 0.5, 0.5)), 24, num_rays_per_batch=256, semantic_threshold=-1e9,
                                         density_threshold=0.0))
    for k in ("rgb", "accumulation", "depth", "semantics", "semantics_colormap"):
        assert torch.equal(outs[0][k], outs[1][k]), k
    assert vols[0]["density"]["points"].shape[0] > 0
    for cloud in ("semantic_colormap", "semantic", "density"):
        for k in ("points", "colors"):
            assert torch.equal(vols[0][cloud][k], vols[1][cloud][k]), (cloud, k)


@pytest.mark.parametrize("mode", ["eager_adam", "eager_radam", "graphed", "deferred"])
def test_copy_in_step_after_updates(dev, mode):
    R = 256
    model = _model(dev, "big", "fp16", rounded=False)
    rays = synthetic.make_rays(R, seed=6, num_cameras=20)
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    opts = engine.DEFAULT_OPTIMIZERS if mode == "eager_adam" else engine.BIG_PRESET_OPTIMIZERS
    tr = engine.Trainer(model, optimizers=opts, cuda_graph=mode in ("graphed", "deferred"), force_proposal_update=True)
    tr.defer_fields = mode == "deferred"
    before = model.field.mlp_base_grid.hash_table.detach().clone()
    for step in (6000, 6001, 6002, 6003):
        tr.train_iteration(step, product_bundle(rays, dev), targets)
        tr.wait_deferred_update()
        assert _copy_matches(model.field), (mode, step)
    assert not torch.equal(before, model.field.mlp_base_grid.hash_table.detach())
    if mode in ("graphed", "deferred"):
        assert len(tr._graphs) == 1


def test_copy_unchanged_by_grad_scaler_skipped_step(dev):
    R = 256
    model = _model(dev, "big", "fp16", rounded=False)
    rays = synthetic.make_rays(R, seed=6, num_cameras=20)
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    scaler = engine.GradScaler(init_scale=1.0)
    tr = engine.Trainer(model, optimizers=engine.DEFAULT_OPTIMIZERS, grad_scaler=scaler, force_proposal_update=True)
    tr.train_iteration(6000, product_bundle(rays, dev), targets)
    assert scaler.skipped_steps == 0 and _copy_matches(model.field)
    table = model.field.mlp_base_grid.hash_table.detach().clone()
    half = model.field.table_half.clone()
    scaler.scale = float("inf")   # every scaled gradient is non-finite: GradScaler skips the update
    tr.train_iteration(6001, product_bundle(rays, dev), targets)
    torch.cuda.synchronize()
    assert scaler.skipped_steps == 1
    assert torch.equal(table, model.field.mlp_base_grid.hash_table.detach())
    assert torch.equal(half, model.field.table_half) and _copy_matches(model.field)


def test_writes_outside_the_trainer_reach_the_copy(dev):
    model = _model(dev, "big", "fp16", rounded=False, training=False)
    rays = synthetic.make_rays(128, seed=4, num_cameras=20)
    field = model.field
    with torch.no_grad():
        model(product_bundle(rays, dev))
    assert _copy_matches(field)
    # in-place copy_ under no_grad
    with torch.no_grad():
        field.mlp_base_grid.hash_table.copy_(torch.rand_like(field.mlp_base_grid.hash_table) - 0.5)
        model(product_bundle(rays, dev))
    assert _copy_matches(field)
    # load_nerfstudio_checkpoint
    other = _model(dev, "big", "fp32", rounded=False, training=False)
    with torch.no_grad():
        other.field.mlp_base_grid.hash_table.mul_(-3.0)
    state = {"pipeline": {"_model." + k: v.cpu() for k, v in other.state_dict().items()}, "step": 7}
    load_nerfstudio_checkpoint(model, state)
    with torch.no_grad():
        model(product_bundle(rays, dev))
    assert _copy_matches(field)
    # writes through .data bump no version counter: refresh_table_copy() is the documented call
    field.mlp_base_grid.hash_table.data.mul_(0.5)
    field.refresh_table_copy()
    assert _copy_matches(field)


def test_peer_memory_exchange_refuses_fp16_tables(dev):
    model = _model(dev, "big", "fp16", rounded=False)
    with pytest.raises(ValueError, match="fp16"):
        engine.Trainer(model, world_size=2, ddp="p2p")


def test_c_entries_refuse_fp16_tables_outside_the_wide_mixed_path(dev):
    model = product_model(cases.make_config(dict(log2_hashmap_size=12)), cases.build_oracle(cases.make_config(dict(log2_hashmap_size=12)), 4, 0, 0.5)[1],
                          4, dev, False, precision="mixed")
    f = model.field
    cfg = f._cfg(False)
    fs, _ = ops._build_field(cfg, f.kernel_params(), None)
    half = f.mlp_base_grid.hash_table.detach().half()
    o = torch.zeros((1, 3), device=dev)
    e = torch.ones((1, 2), device=dev)
    sm = ops.make_samples(o, o, e, e[:, 1:], None, 1, 1, 2)
    out = torch.empty(8, device=dev)
    for prec in (L.PREC_MIXED, L.PREC_FP32):
        fs.precision = prec
        rc = L.lib().cnb_field_fwd_half(C.byref(fs), half.data_ptr(), C.byref(sm), out.data_ptr(), None, None, None, None, out.data_ptr(), 0,
                                        L.stream_ptr(dev))
        assert rc == CNB_ERR_UNSUPPORTED
        assert "fp16 tables" in L.last_error()


# ---- against the oracle, and a short training run ------------------------------------------------------------------------------------


@pytest.mark.parametrize("preset", ["big", "huge"])
def test_fp16_tables_against_oracle(dev, preset):
    cfg = _preset_cfg(preset)
    num_images, R = 20, 96
    oracle, _ = cases.build_oracle(cfg, num_images, 0, 0.5)
    oracle.train(False)
    model = _model(dev, preset, "fp16", rounded=False, training=False)
    rays = synthetic.make_rays(R, seed=4, num_cameras=num_images)
    with torch.no_grad():
        ref = oracle(cases.oracle_bundle(rays))
        out = model(product_bundle(rays, dev))
    assert_close(out["rgb"], ref["rgb"], RTOL_MIXED, "fp16-table rgb", floor=1e-1)
    assert_close(out["accumulation"], ref["accumulation"], RTOL_MIXED, "fp16-table accumulation", floor=1e-1)
    agree = (out["semantics_colormap"].cpu() == ref["semantics_colormap"]).float().mean().item()
    assert agree >= 0.999, agree


def test_short_training_big_preset_fp16_vs_fp32(dev):
    """300 steps of the big preset on synthetic data, fp16 vs fp32 tables, same seed: finite throughout.  Both loss curves are printed."""
    R = 4096
    curves = {}
    for tp in ("fp32", "fp16"):
        torch.manual_seed(0)
        model = _model(dev, "big", tp, rounded=False)
        tr = engine.Trainer(model, optimizers=engine.BIG_PRESET_OPTIMIZERS, cuda_graph=True)
        losses = []
        for step in range(300):
            rays = synthetic.make_rays(R, seed=1000 + step, num_cameras=20)
            targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=2000 + step).items()}
            st = tr.train_iteration(step, product_bundle(rays, dev), targets)
            losses.append(st["loss"].detach().clone())
        tr.wait_deferred_update()
        curves[tp] = torch.stack(losses).cpu()
        assert torch.isfinite(curves[tp]).all(), tp
        for g in tr.groups.values():
            assert torch.isfinite(g.flat).all()
        if tp == "fp16":
            assert _copy_matches(model.field)
    for tp, c in curves.items():
        print(f"{tp} tables, total loss every 25 steps: {[round(float(x), 5) for x in c[::25]]}  last {float(c[-1]):.5f}")

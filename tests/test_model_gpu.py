"""End-to-end parity of the B200 FruitField / FruitModel against the oracle (fp32 mode: 1e-4 relative; semantic label
agreement >= 99.9 %), against the committed golden fixtures, and gradient parity of one training step."""
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN, assert_close, product_bundle, product_model, rel_err

from cropnerf_b200 import synthetic
from cropnerf_b200.field_components import FieldHeadNames
from cropnerf_b200.rays import ray_layout
from oracle import cases
from oracle import nerfstudio_torch as ns

pytestmark = pytest.mark.gpu

RTOL_FP32 = 1e-4  # north_star: per-ray RGB / depth / accumulation within 1e-4 relative in fp32


def _field_samples(R, S, seed):
    rays = synthetic.make_rays(R, seed=seed, num_cameras=20)
    g = torch.Generator().manual_seed(seed)
    edges = torch.sort(torch.rand((R, S + 1), generator=g) * 3.0, dim=-1).values
    edges[0] = torch.linspace(0, 2000.0, S + 1)  # far samples: contraction branch
    return rays, edges


# the FruitField dimensions the reference's other presets forward (fruit_nerf_config.py:86-98 `fruit_nerf_big`, :141-150 `fruit_nerf_huge`):
# a 128-wide three-layer semantic MLP and geo_feat_dim = 30, i.e. a 78-wide RGB input -- layers above 64 run on csrc/mlp_wide.cu (exact mode)
BIG_PRESET = dict(geo_feat_dim=30, hidden_dim_semantics=128, num_layers_semantic=3, max_res=4096)


@pytest.mark.parametrize("preset", [{}, BIG_PRESET], ids=["base", "big"])
@pytest.mark.parametrize("contraction", [True, False])
@pytest.mark.parametrize("training", [True, False])
def test_field_forward_backward(dev, contraction, training, preset):
    R, S, num_images = 160, 48, 20
    cfg = cases.make_config(dict(log2_hashmap_size=14, disable_scene_contraction=not contraction, **preset))
    oracle, state = cases.build_oracle(cfg, num_images, seed=0, table_scale=0.5)
    oracle.train(training)
    model = product_model(cfg, state, num_images, dev, training)
    rays, edges = _field_samples(R, S, 3)
    rb = cases.oracle_bundle(rays)
    rs = rb.get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    out_ref = oracle.field(rs)
    rbm = product_bundle(rays, dev)
    e = edges.to(dev)
    rsm = rbm.get_ray_samples(e[:, :-1, None], e[:, 1:, None])
    out = model.field(rsm)
    assert_close(out[FieldHeadNames.DENSITY], out_ref["density"], RTOL_FP32, "density", floor=1e-3)
    assert_close(out[FieldHeadNames.RGB], out_ref["rgb"], RTOL_FP32, "rgb")
    assert_close(out[FieldHeadNames.SEMANTICS], out_ref["semantics"], 5e-4, "semantics", floor=1e-2)
    # _sample_locations (BayesRays hook): normalised + masked positions, bit-exact
    assert torch.equal(model.field._sample_locations.cpu(), oracle.field._sample_locations.detach())
    if not training:
        return
    g = torch.Generator().manual_seed(11)
    gd, gr, gs = torch.randn((R, S, 1), generator=g) * 0.01, torch.randn((R, S, 3), generator=g), torch.randn((R, S, 1), generator=g)
    (out_ref["density"] * gd).sum().add((out_ref["rgb"] * gr).sum()).add((out_ref["semantics"] * gs).sum()).backward()
    (out[FieldHeadNames.DENSITY] * gd.to(dev)).sum().add((out[FieldHeadNames.RGB] * gr.to(dev)).sum()).add(
        (out[FieldHeadNames.SEMANTICS] * gs.to(dev)).sum()).backward()
    ref_params = dict(oracle.field.named_parameters())
    for name, p in model.field.named_parameters():
        gr_ = ref_params[name].grad
        assert gr_ is not None and p.grad is not None, name
        scale = gr_.abs().max().item() + 1e-20
        err = (p.grad.cpu() - gr_).abs().max().item() / scale
        assert err < 5e-4, f"field grad {name}: {err:.3e}"


@pytest.mark.parametrize("precision", ["fp32", "mixed"])
def test_density_field_forward_backward(dev, precision):
    """mixed: the forward and the table scatter are the fp32 kernels' (same tolerances); only the MLP parameter gradients are contracted
    with plain bf16 operands on the tensor cores (k_density_bwd_tc<0>): relative L2 <= 2e-2 (8 mantissa bits, fp32 accumulation)."""
    R, S, num_images = 200, 64, 20
    cfg = cases.make_config(dict(log2_hashmap_size=14))
    oracle, state = cases.build_oracle(cfg, num_images, seed=0, table_scale=0.5)
    model = product_model(cfg, state, num_images, dev, True, precision=precision)
    rays, edges = _field_samples(R, S, 4)
    rs = cases.oracle_bundle(rays).get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    e = edges.to(dev)
    rsm = product_bundle(rays, dev).get_ray_samples(e[:, :-1, None], e[:, 1:, None])
    for i in range(2):
        ref_net, net = oracle.proposal_networks[i], model.proposal_networks[i]
        d_ref, _ = ref_net.get_density(rs)
        d, _ = net.get_density(rsm)
        assert_close(d, d_ref, RTOL_FP32, f"proposal {i} density", floor=1e-3)
        # density_fn(positions) path (arbitrary positions, one zero-length frustum per point)
        pos = rs.frustums.get_positions()
        d2 = net.density_fn(pos.to(dev))
        assert_close(d2, ref_net.density_fn(pos), RTOL_FP32, f"proposal {i} density_fn", floor=1e-3)
        g = torch.Generator().manual_seed(i)
        gd = torch.randn(d_ref.shape, generator=g) * 0.1
        (d_ref * gd).sum().backward()
        (d * gd.to(dev)).sum().backward()
        ref_params = dict(ref_net.named_parameters())
        for name, p in net.named_parameters():
            gr_ = ref_params[name].grad
            scale = gr_.abs().max().item() + 1e-20
            err = (p.grad.cpu() - gr_).abs().max().item() / scale
            if precision == "mixed" and "hash_table" not in name:
                l2 = (p.grad.cpu().double() - gr_.double()).norm().item() / (gr_.double().norm().item() + 1e-30)
                assert l2 < 2e-2, f"mixed proposal {i} grad {name}: relative L2 {l2:.3e}"
            else:
                assert err < 5e-4, f"proposal {i} grad {name}: {err:.3e}"


def _run_product(name, dev, spec=None, num_images=20, seed=0):
    spec = spec or cases.CASES[name]
    R = spec["num_rays"]
    cfg = cases.make_config(spec.get("cfg"))
    oracle, state = cases.build_oracle(cfg, num_images, seed, spec["table_scale"])
    model = product_model(cfg, state, num_images, dev, spec["training"])
    rays = synthetic.make_rays(R, seed=1, num_cameras=num_images)
    if spec["training"]:
        feed = synthetic.JitterFeed(synthetic.make_jitter(R, 3, seed=2))
        model.proposal_sampler.initial_sampler.rand_fn = feed
        model.proposal_sampler.pdf_sampler.rand_fn = feed
        for cb in model.get_training_callbacks():
            if "BEFORE_TRAIN_ITERATION" in cb.where_to_run:
                cb.func(500)
    model.proposal_sampler.pdf_sampler.keep_inds = True
    outputs = model(product_bundle(rays, dev))
    return model, outputs


def _check_outputs(outputs, ref, tag):
    # per-ray outputs: within 1e-4 relative for (nearly) every ray; the median depth is a discontinuous pick of one
    # sample, so a last-ulp difference in the cumulative weights may move a few rays by one sample
    assert_close(outputs["rgb"], ref["rgb"], RTOL_FP32, tag + " rgb")
    assert_close(outputs["accumulation"], ref["accumulation"], RTOL_FP32, tag + " accumulation")
    # (measured on the B200: 100 % of the rays, 99.9 % for prop_depth_0 at 1024 rays -- profiles/r1_parity_report_fp32.json)
    assert_close(outputs["depth"], ref["depth"], RTOL_FP32, tag + " depth", frac=0.999)
    assert_close(outputs["prop_depth_0"], ref["prop_depth_0"], RTOL_FP32, tag + " prop_depth_0", frac=0.998)
    assert_close(outputs["prop_depth_1"], ref["prop_depth_1"], RTOL_FP32, tag + " prop_depth_1", frac=0.999)
    assert_close(outputs["semantics"], ref["semantics"], 5e-4, tag + " semantics", floor=1e-2)
    agree = (outputs["semantics_colormap"].cpu().numpy() == ref["semantics_colormap"]).mean()
    assert agree >= 0.999, f"{tag}: semantic label agreement {agree}"


@pytest.mark.parametrize("name", list(cases.CASES))
def test_model_against_golden(dev, name):
    ref = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    model, outputs = _run_product(name, dev)
    _check_outputs(outputs, ref, name)
    inds = model.proposal_sampler.pdf_sampler.last_inds.cpu().numpy()
    same = (inds == ref["pdf_inds_last"]).mean()
    # bit-exact GIVEN an identical cdf (test_pdf_sampler_bit_exact_given_identical_cdf); end to end the cdf may differ in the last ulp (fp32 sum
    # order of the histogram, powf), which can move a tie: at most 2 of the ~4700 bin indices of these cases
    assert same >= 0.9995, f"{name}: resampling bins agree on {same*100:.3f}%"
    assert inds.shape == ref["pdf_inds_last"].shape  # proposal sample counts


def test_training_step_losses_and_gradients(dev):
    name = "tiny_train"
    ref = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    model, outputs = _run_product(name, dev)
    R = cases.CASES[name]["num_rays"]
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    loss_dict = model.get_loss_dict(outputs, targets)
    metrics = model.get_metrics_dict(outputs, targets)
    for k, v in loss_dict.items():
        r = float(ref["loss_" + k])
        assert abs(v.item() - r) <= 2e-4 * abs(r) + 1e-8, f"{k}: {v.item()} vs {r}"
    assert abs(metrics["distortion"].item() - float(ref["metric_distortion"])) <= 1e-3 * abs(float(ref["metric_distortion"]))
    assert abs(metrics["psnr"].item() - float(ref["metric_psnr"])) <= 1e-3
    sum(loss_dict.values()).backward()
    checked = 0
    for pname, p in model.named_parameters():
        key = "gradnorm/" + pname
        if key not in ref:
            continue
        assert p.grad is not None, pname
        gn = p.grad.double().norm().item()
        rn = float(ref[key])
        # end-to-end gradients also see the (rare) resampling-bin flips between the two pipelines, which move whole
        # samples on a 96-ray batch; the per-stage backward tests above/in test_kernels_gpu.py are the tight ones
        assert abs(gn - rn) <= 2e-2 * rn + 1e-12, f"grad norm {pname}: {gn} vs {rn}"
        if "grad/" + pname in ref:
            g_ref = ref["grad/" + pname]
            scale = np.abs(g_ref).max() + 1e-20
            err = np.abs(p.grad.cpu().numpy().reshape(-1) - g_ref).max() / scale
            assert err < 3e-2, f"grad {pname}: {err:.3e}"
        checked += 1
    assert checked >= 20


def test_full_size_config_vs_oracle(dev):
    """The fruit_nerf preset at full table sizes (2^19 x 16 field, 2^17 x 5 proposals), 384 rays, eval mode."""
    spec = dict(num_rays=384, training=False, cfg=dict(), table_scale=0.5)
    cfg = cases.make_config(spec["cfg"], small=False)
    oracle, state = cases.build_oracle(cfg, 20, 0, 0.5)
    oracle.eval()
    rays = synthetic.make_rays(spec["num_rays"], seed=1, num_cameras=20)
    with torch.no_grad():
        ref = oracle(cases.oracle_bundle(rays))
    model = product_model(cfg, state, 20, dev, False)
    with torch.no_grad():
        out = model(product_bundle(rays, dev))
    ref_np = {k: v.numpy() for k, v in ref.items() if isinstance(v, torch.Tensor)}
    _check_outputs(out, ref_np, "full-size")


@pytest.mark.parametrize("preset", ["big", "huge"])
@pytest.mark.parametrize("training", [False, True])
def test_big_preset_model_vs_oracle(dev, training, preset):
    """The models of the reference's `fruit_nerf_big` / `fruit_nerf_huge` presets (fruit_nerf_config.py:86-98, 141-150): 128 / (512, 256) resp.
    64 / (512, 512) samples per ray, three-layer 128-wide semantic MLP, geo_feat_dim 30, 5000 anneal iterations, a 7-level proposal grid --
    through the same fused render / training step in exact fp32 (the wide layers on csrc/mlp_wide.cu), against the oracle: per-ray outputs
    in eval mode; the five losses and every parameter-gradient norm in training.  (Table sizes reduced, as in every small case.)"""
    big = dict(BIG_PRESET, num_nerf_samples_per_ray=128, num_proposal_samples_per_ray=(512, 256), proposal_weights_anneal_max_num_iters=5000,
               log2_hashmap_size=15)
    if preset == "huge":   # fruit_nerf_config.py:141-150: 7-level second proposal grid, (512, 512) + 64 samples, max_res 8192
        big.update(num_nerf_samples_per_ray=64, num_proposal_samples_per_ray=(512, 512), max_res=8192, proposal_net_args_list=[
            {"hidden_dim": 16, "log2_hashmap_size": 13, "num_levels": 5, "max_res": 512, "use_linear": False},
            {"hidden_dim": 16, "log2_hashmap_size": 13, "num_levels": 7, "max_res": 2048, "use_linear": False}])
    cfg = cases.make_config(big)
    num_images, R = 20, 96
    oracle, state = cases.build_oracle(cfg, num_images, 0, 0.5)
    oracle.train(training)
    rays = synthetic.make_rays(R, seed=4, num_cameras=num_images)
    model = product_model(cfg, state, num_images, dev, training)
    if not training:
        with torch.no_grad():
            ref = oracle(cases.oracle_bundle(rays))
            out = model(product_bundle(rays, dev))
        _check_outputs(out, {k: v.numpy() for k, v in ref.items() if isinstance(v, torch.Tensor)}, "big preset")
        return
    jit = synthetic.make_jitter(R, 3, seed=2)
    for mdl in (oracle, model):   # the same uniform draws on both sides (initial sampler + two PDF levels)
        feed = synthetic.JitterFeed(jit)
        mdl.proposal_sampler.initial_sampler.rand_fn = feed
        mdl.proposal_sampler.pdf_sampler.rand_fn = feed
    oracle.set_anneal(2500)   # mid-anneal of the preset's 5000 iterations
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
        assert abs(float(v) - r) <= 5e-4 * abs(r) + 1e-8, f"{k}: {float(v)} vs {r}"
    sum(loss.values()).backward()
    ref_params = dict(oracle.named_parameters())
    checked = 0
    for name, p in model.named_parameters():
        gr = ref_params[name].grad if name in ref_params else None
        if gr is None or p.grad is None:
            continue
        gn, rn = p.grad.double().norm().item(), gr.double().norm().item()
        assert abs(gn - rn) <= 2e-2 * rn + 1e-12, f"grad norm {name}: {gn} vs {rn}"
        checked += 1
    assert checked >= 20


def test_export_mode_and_density_projection(dev):
    """setup_inference (uniform sampler, contraction off) + get_export_outputs, and the opacity-in-front-of-AABB
    path of semantic_projection (get_density_for_camera_ray_bundle with injected near/far)."""
    cfg = cases.make_config(dict(log2_hashmap_size=14))
    oracle, state = cases.build_oracle(cfg, 20, 0, 0.5)
    oracle.eval()
    model = product_model(cfg, state, 20, dev, False)
    rays = synthetic.make_rays(100, seed=5, num_cameras=20)
    with torch.no_grad():
        acc_ref = oracle.get_density_for_ray_bundle(cases.oracle_bundle(rays, with_near_far=(0.0, 0.8)))
        acc = model.get_density_for_camera_ray_bundle(product_bundle(rays, dev, near_far=(0.0, 0.8)))
    assert_close(acc, acc_ref, RTOL_FP32, "opacity in front of box")
    oracle.test_mode = model.test_mode = "export"
    oracle.field.test_mode = model.field.test_mode = "export"
    oracle.setup_inference(True, 200)
    model.setup_inference(True, 200)
    oracle.eval()
    model.eval()
    with torch.no_grad():
        ref = oracle(cases.oracle_bundle(rays, with_near_far=(0.0, 1.5)))
        out = model(product_bundle(rays, dev, near_far=(0.0, 1.5)))
    assert_close(out["density"], ref["density"], RTOL_FP32, "export density", floor=1e-3)
    assert_close(out["rgb"], ref["rgb"], RTOL_FP32, "export rgb")
    assert_close(out["point_location"], ref["point_location"], 1e-6, "export positions")
    assert (out["semantics_colormap"].cpu() == ref["semantics_colormap"]).float().mean() >= 0.999


RTOL_MIXED = 2e-3  # north_star: 2e-3 relative in mixed precision


@pytest.mark.parametrize("training", [False, True])
def test_field_forward_mixed_precision(dev, training):
    """fp16 tensor-core MLPs (fp32 tables, accumulation, exp): within 2e-3 of the fp32 oracle."""
    R, S, num_images = 200, 48, 20
    cfg = cases.make_config(dict(log2_hashmap_size=14))
    oracle, state = cases.build_oracle(cfg, num_images, seed=0, table_scale=0.5)
    oracle.train(training)
    model = product_model(cfg, state, num_images, dev, training, precision="mixed")
    rays, edges = _field_samples(R, S, 3)
    rs = cases.oracle_bundle(rays).get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    with torch.no_grad():
        out_ref = oracle.field(rs)
        e = edges.to(dev)
        out = model.field(product_bundle(rays, dev).get_ray_samples(e[:, :-1, None], e[:, 1:, None]))
    assert_close(out[FieldHeadNames.RGB], out_ref["rgb"], RTOL_MIXED, "mixed rgb", floor=1e-1)
    assert_close(out[FieldHeadNames.DENSITY], out_ref["density"], 1e-2, "mixed density", floor=1e-2, frac=0.999)
    assert_close(out[FieldHeadNames.SEMANTICS], out_ref["semantics"], 1e-2, "mixed semantics", floor=1e-1)
    assert torch.equal(model.field._sample_locations.cpu(), oracle.field._sample_locations.detach())


@pytest.mark.parametrize("precision", ["fp32", "mixed"])
@pytest.mark.parametrize("training", [False, True])
def test_get_density_get_outputs_split(dev, precision, training):
    """The Field interface the reference and BayesRays call as a PAIR (fruit_nerf.py:340,431,480,503; bayesrays/uncertainty.py:109):
    ``density, embedding = field.get_density(rs); heads = field.get_outputs(rs, density_embedding=embedding)`` -- in BOTH precisions.
    The pair must return exactly what ``forward`` returns (same fused operator), the embedding must be the base MLP's geo features
    (oracle, 1e-4 fp32 / 2e-2 absolute for the fp16 tensor-core MLP), and gradients must flow through the pair as through forward."""
    R, S, num_images = 96, 48, 20
    cfg = cases.make_config(dict(log2_hashmap_size=14))
    oracle, state = cases.build_oracle(cfg, num_images, seed=0, table_scale=0.5)
    oracle.train(training)
    model = product_model(cfg, state, num_images, dev, training, precision=precision)
    rays, edges = _field_samples(R, S, 5)
    rs_o = cases.oracle_bundle(rays).get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    e = edges.to(dev)
    rs = product_bundle(rays, dev).get_ray_samples(e[:, :-1, None], e[:, 1:, None])
    with torch.set_grad_enabled(training):
        d_ref, emb_ref = oracle.field.get_density(rs_o)
        density, emb = model.field.get_density(rs)
        heads = model.field.get_outputs(rs, density_embedding=emb)
        full = model.field(rs)
    assert emb.shape == (R, S, 15) and density.shape == (R, S, 1)
    assert torch.equal(density, full[FieldHeadNames.DENSITY]) and torch.equal(heads[FieldHeadNames.RGB], full[FieldHeadNames.RGB])
    assert torch.equal(heads[FieldHeadNames.SEMANTICS], full[FieldHeadNames.SEMANTICS])
    if precision == "fp32":
        assert_close(emb, emb_ref, RTOL_FP32, "geo embedding", floor=1e-2)
    else:
        assert (emb.detach().cpu() - emb_ref.detach()).abs().max().item() <= 2e-2 * max(1.0, emb_ref.detach().abs().max().item())
    assert model.field._density_before_activation.shape == (R, S, 1)   # side effect of fruit_field.py:181-187
    with pytest.raises(RuntimeError, match="get_density"):
        model.field.get_outputs(rs, density_embedding=emb.clone())   # not the pair's embedding: the field is one fused operator
    if training:
        g = torch.Generator().manual_seed(3)
        gd, gr = torch.randn((R, S, 1), generator=g).to(dev) * 0.01, torch.randn((R, S, 3), generator=g).to(dev)
        for p in model.field.parameters():
            p.grad = None
        ((density * gd).sum() + (heads[FieldHeadNames.RGB] * gr).sum()).backward()
        g_pair = {n: p.grad.clone() for n, p in model.field.named_parameters() if p.grad is not None}
        for p in model.field.parameters():
            p.grad = None
        ((full[FieldHeadNames.DENSITY] * gd).sum() + (full[FieldHeadNames.RGB] * gr).sum()).backward()
        assert g_pair and all(float(v.abs().max()) > 0 for k, v in g_pair.items() if "semantic" not in k)
        for n, p in model.field.named_parameters():
            if p.grad is not None:
                scale = float(p.grad.abs().max()) + 1e-20
                assert float((g_pair[n] - p.grad).abs().max()) <= 1e-4 * scale, n   # same kernels; fp32 atomics order only


def test_model_eval_mixed_precision(dev):
    spec = dict(num_rays=512, training=False, cfg=dict(), table_scale=0.5)
    cfg = cases.make_config(spec["cfg"], small=False)
    oracle, state = cases.build_oracle(cfg, 20, 0, 0.5)
    oracle.eval()
    rays = synthetic.make_rays(spec["num_rays"], seed=1, num_cameras=20)
    with torch.no_grad():
        ref = oracle(cases.oracle_bundle(rays))
    model = product_model(cfg, state, 20, dev, False, precision="mixed")
    with torch.no_grad():
        out = model(product_bundle(rays, dev))
    assert_close(out["rgb"], ref["rgb"], RTOL_MIXED, "mixed rgb", floor=1e-1)
    assert_close(out["accumulation"], ref["accumulation"], RTOL_MIXED, "mixed accumulation", floor=1e-1)
    assert_close(out["depth"], ref["depth"], RTOL_MIXED, "mixed depth", frac=0.97)
    agree = (out["semantics_colormap"].cpu() == ref["semantics_colormap"]).float().mean().item()
    assert agree >= 0.999, agree


@pytest.mark.parametrize("R,S", [(160, 48), (37, 21), (9, 5)])
def test_field_backward_mixed_precision(dev, R, S):
    """Fused tensor-core backward (default: the tcgen05 kernel -- bf16 forward recompute with the forward's ReLU flags and fp32 end-layer
    derivatives, bf16 gradient operands, fp32 accumulation in TMEM) against the fp32 oracle's autograd: relative L2 error of every
    parameter gradient <= 4e-2 (measured 0.1-2 %: the fp16 forward it differentiates already differs from the fp32 oracle by up to 1e-2
    in density, and bf16 has 8 mantissa bits; the products are summed over thousands of samples in fp32).  (37, 21): a ragged last
    128-sample batch, warps that straddle three rays (the per-lane path of the appearance-embedding gradient); (9, 5): one partial batch,
    up to seven rays per warp."""
    num_images = 20
    cfg = cases.make_config(dict(log2_hashmap_size=14))
    oracle, state = cases.build_oracle(cfg, num_images, seed=0, table_scale=0.5)
    oracle.train(True)
    model = product_model(cfg, state, num_images, dev, True, precision="mixed")
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
        err = (p.grad.cpu().double() - gr_.double()).norm().item() / (gr_.double().norm().item() + 1e-30)
        worst[name] = err
    tol = 4e-2 if R * S >= 500 else 6e-2   # 45 samples: no averaging over the batch (measured 4.2 % on one bias, identical in every kernel variant)
    bad = {k: v for k, v in worst.items() if not v < tol}
    assert not bad, f"mixed backward relative L2 errors: {bad} (all: {worst})"


# ---------------------------------------------------------------------------------------------------------------------
# row a17: gradients with respect to the rays (what the camera optimizer trains through)


def _leaf_bundles(rays, dev):
    ro = cases.oracle_bundle({k: v.clone() for k, v in rays.items()})  # oracle_bundle may alias the input tensors
    ro.origins.requires_grad_(True)
    ro.directions.requires_grad_(True)
    rp = product_bundle(rays, dev)
    rp.origins.requires_grad_(True)
    rp.directions.requires_grad_(True)
    return ro, rp


def _check_ray_grads(ro, rp, tag, tol=2e-3):
    for name in ("origins", "directions"):
        ref = getattr(ro, name).grad
        got = getattr(rp, name).grad
        assert ref is not None and got is not None, f"{tag}: no gradient for {name}"
        scale = ref.abs().max().item() + 1e-20
        err = (got.cpu() - ref).abs().max().item() / scale
        assert err < tol, f"{tag}: d{name} differs from the oracle autograd by {err:.3e} of max |g| ({scale:.3e})"


@pytest.mark.parametrize("contraction", [True, False])
def test_field_and_proposal_ray_gradients(dev, contraction):
    """dLoss/d(origins, directions) through hash grid -> normalisation / contraction, per-module operators vs torch autograd
    of the oracle (fp32 mode).  Far samples exercise the contraction Jacobian; samples outside the box the selector mask."""
    R, S, num_images = 96, 48, 20
    cfg = cases.make_config(dict(log2_hashmap_size=14, disable_scene_contraction=not contraction))
    oracle, state = cases.build_oracle(cfg, num_images, seed=0, table_scale=0.5)
    oracle.train(True)
    model = product_model(cfg, state, num_images, dev, True)
    rays, edges = _field_samples(R, S, 3)
    ro, rp = _leaf_bundles(rays, dev)
    rs = ro.get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    e = edges.to(dev)
    rsm = rp.get_ray_samples(e[:, :-1, None], e[:, 1:, None])
    g = torch.Generator().manual_seed(5)
    gd, gr, gs = torch.randn((R, S, 1), generator=g) * 0.01, torch.randn((R, S, 3), generator=g), torch.randn((R, S, 1), generator=g)
    out_ref = oracle.field(rs)
    out = model.field(rsm)
    (out_ref["density"] * gd).sum().add((out_ref["rgb"] * gr).sum()).add((out_ref["semantics"] * gs).sum()).backward()
    (out[FieldHeadNames.DENSITY] * gd.to(dev)).sum().add((out[FieldHeadNames.RGB] * gr.to(dev)).sum()).add(
        (out[FieldHeadNames.SEMANTICS] * gs.to(dev)).sum()).backward()
    _check_ray_grads(ro, rp, f"field(contraction={contraction})")
    # proposal network
    ro, rp = _leaf_bundles(rays, dev)
    rs = ro.get_ray_samples(edges[:, :-1, None], edges[:, 1:, None])
    rsm = rp.get_ray_samples(e[:, :-1, None], e[:, 1:, None])
    d_ref, _ = oracle.proposal_networks[0].get_density(rs)
    d, _ = model.proposal_networks[0].get_density(rsm)
    gd = torch.randn(d_ref.shape, generator=g) * 0.1
    (d_ref * gd).sum().backward()
    (d * gd.to(dev)).sum().backward()
    _check_ray_grads(ro, rp, f"proposal(contraction={contraction})")


@pytest.mark.parametrize("precision", ["fp32", "mixed"])
def test_train_step_ray_gradients_and_camera_optimizer(dev, precision):
    """One-call training step with ray gradients: dLoss/d rays against the oracle's autograd through its whole model, then
    the SO3xR3 camera optimizer end to end (pose_adjustment receives a gradient and Adam moves it)."""
    from cropnerf_b200 import engine
    from cropnerf_b200.pipeline import FusedPipeline

    R, num_images = 128, 20
    small = precision == "fp32"
    cfg = cases.make_config({}, small=small)
    oracle, state = cases.build_oracle(cfg, num_images, 0, 0.5)
    oracle.train(True)
    model = product_model(cfg, state, num_images, dev, True, precision=precision)
    rays = synthetic.make_rays(R, seed=6, num_cameras=num_images)
    targets = synthetic.make_targets(R, seed=3)
    jit = synthetic.make_jitter(R, 3, seed=2)
    for mdl in (oracle, model):
        feed = synthetic.JitterFeed(jit)
        mdl.proposal_sampler.initial_sampler.rand_fn = feed
        mdl.proposal_sampler.pdf_sampler.rand_fn = feed
    ro, rp = _leaf_bundles(rays, dev)
    out_ref = oracle(ro)
    sum(oracle.get_loss_dict(out_ref, targets).values()).backward()
    model.collider(rp)
    fp = FusedPipeline(model)
    for p in model.parameters():
        p.grad = torch.zeros_like(p)
    fp.train_step(rp, {k: v.to(dev) for k, v in targets.items()}, update_proposals=True)
    # end to end the two pipelines also differ by the (rare) last-ulp resampling-bin flips, which move whole samples on a
    # 128-ray batch (same allowance as test_training_step_losses_and_gradients); the per-module test above is the tight one
    _check_ray_grads(ro, rp, f"train step ({precision})", tol=3e-2 if precision == "fp32" else 5e-2)
    # camera optimizer end to end
    ccfg = cases.make_config({}, small=small)
    model2 = product_model(ccfg, state, num_images, dev, True, precision=precision)
    from cropnerf_b200.fruit_nerf import CameraOptimizer
    model2.camera_optimizer = CameraOptimizer(num_images, "SO3xR3").to(dev)
    tr = engine.Trainer(model2)
    assert "camera_opt" in tr.groups
    before = tr.groups["camera_opt"].flat.clone()
    tr.train_iteration(3, product_bundle(rays, dev), {k: v.to(dev) for k, v in targets.items()})
    moved = (tr.groups["camera_opt"].flat - before).abs().max().item()
    assert moved > 0, "camera poses did not move"


@pytest.mark.parametrize("precision", ["fp32", "mixed"])
def test_in_step_camera_optimizer_matches_the_autograd_route(dev, precision):
    """Row a17 inside the step (csrc/camera_opt.cu: exp_map_SO3xR3 + apply_to_raybundle before the samplers, dLoss/d rays chained through the
    Rodrigues formula, regulariser gradient) against the plain PyTorch route of the same op (CameraOptimizer.apply_to_raybundle /
    get_loss_dict with autograd around cnb_train_step): same losses, same regulariser, same pose_adjustment gradient -- including a
    camera below the |w|^2 = 1e-4 clamp of the exponential map and one with a zero adjustment (norm subgradient 0)."""
    from cropnerf_b200 import engine
    from cropnerf_b200.fruit_nerf import CameraOptimizer

    R, num_images = 256, 12
    small = precision == "fp32"
    cfg = cases.make_config({}, small=small)
    _, state = cases.build_oracle(cfg, num_images, 0, 0.5)
    rays = synthetic.make_rays(R, seed=6, num_cameras=num_images)
    targets = {k: v.to(dev) for k, v in synthetic.make_targets(R, seed=3).items()}
    jit = synthetic.make_jitter(R, 3, seed=2)
    g = torch.Generator().manual_seed(5)
    pose0 = torch.randn((num_images, 6), generator=g) * 0.02
    pose0[0] = 0.0
    pose0[1, 3:] = torch.tensor([1e-3, -2e-3, 5e-4])       # |w|^2 < 1e-4: the clamped branch
    got = []
    for eager in (True, False):
        model = product_model(cfg, state, num_images, dev, True, precision=precision)
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
    reg = (pose0[:, :3].norm(dim=-1).mean() * 1e-2 + pose0[:, 3:].norm(dim=-1).mean() * 1e-3).item()
    assert abs(sb["camera_opt_regularizer"] - reg) <= 1e-5 * reg
    for name in ("camera_opt", "fields", "proposal_networks"):
        a, b = ga[name].double(), gb[name].double()
        err = (a - b).norm().item() / (a.norm().item() + 1e-30)
        # the two routes evaluate the exponential map with different libraries (torch vs sinf / cosf in the kernel): corrected rays differ
        # in the last ulp, samples move by ~1e-7 and a few cross hash-grid cell faces (measured: 6e-4 fp32, 1.2e-3 mixed)
        assert err <= (2e-3 if precision == "fp32" else 5e-3), (name, err)
        assert a.abs().max().item() > 0
    pg = gb["camera_opt"][: num_images * 6].view(num_images, 6)
    assert float(pg[0, :3].abs().max()) > 0 and torch.isfinite(pg).all()

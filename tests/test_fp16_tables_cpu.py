"""fp16 field tables (FruitField table_precision="fp16"): configuration plumbing and refusals, without a GPU."""
import dataclasses

import pytest
import torch

from cropnerf_b200 import _lib as L
from cropnerf_b200 import method_config
from cropnerf_b200.fruit_field import FruitField
from cropnerf_b200.fruit_nerf import FruitModel, FruitNerfModelConfig

BIG = dict(geo_feat_dim=30, hidden_dim_semantics=128, num_layers_semantic=3, max_res=4096, log2_hashmap_size=8)
AABB = torch.tensor([[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]])


def _field(**kw):
    return FruitField(AABB, num_images=4, use_semantics=True, num_semantic_classes=1, **kw)


def test_default_is_fp32_and_holds_no_copy():
    assert FruitNerfModelConfig().table_precision == "fp32"
    f = _field(log2_hashmap_size=8, precision="mixed")
    assert f.table_precision == "fp32"
    assert "table_half" not in dict(f.named_buffers())
    assert f.table_half_current() is None and not f.table_copy_stale()


def test_config_reaches_the_field_of_the_big_preset():
    model = FruitModel(FruitNerfModelConfig(precision="mixed", table_precision="fp16", **BIG), num_train_data=4)
    f = model.field
    assert f.table_precision == "fp16"
    assert f.table_half.dtype == torch.float16 and f.table_half.shape == f.mlp_base_grid.hash_table.shape
    assert f.table_copy_stale()   # written from the fp32 table before the first forward
    # the proposal networks keep their fp32 tables and no copy
    for net in model.proposal_networks:
        assert not [n for n, _ in net.named_buffers() if "half" in n]


def test_state_dict_is_unchanged_by_the_option():
    torch.manual_seed(0)
    a = FruitModel(FruitNerfModelConfig(precision="mixed", **BIG), num_train_data=4)
    b = FruitModel(FruitNerfModelConfig(precision="mixed", table_precision="fp16", **BIG), num_train_data=4)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb)
    assert all(sa[k].shape == sb[k].shape and sa[k].dtype == sb[k].dtype for k in sa)
    b.load_state_dict(sa)   # a checkpoint of either loads into the other
    a.load_state_dict(b.state_dict())


def test_exact_mode_is_refused_with_the_reason():
    with pytest.raises(ValueError, match="precision='mixed'"):
        FruitModel(FruitNerfModelConfig(precision="fp32", table_precision="fp16", **BIG), num_train_data=4)


def test_base_architecture_is_refused_with_the_reason():
    with pytest.raises(ValueError, match="L2"):
        FruitModel(FruitNerfModelConfig(precision="mixed", table_precision="fp16", log2_hashmap_size=8), num_train_data=4)
    with pytest.raises(ValueError, match="L2"):
        _field(log2_hashmap_size=8, precision="mixed", table_precision="fp16")


def test_unknown_table_precision_is_refused():
    with pytest.raises(ValueError, match="table_precision"):
        _field(log2_hashmap_size=8, precision="mixed", table_precision="bf16")


def test_method_config_carries_the_option():
    if method_config.UNAVAILABLE:
        # without nerfstudio the method config is not defined; the model config field it forwards to is what it copies by name
        assert "table_precision" in FruitNerfModelConfig.__dataclass_fields__
        return
    fields = {f.name: f.default for f in dataclasses.fields(method_config.FruitNerfB200ModelConfig)}
    assert fields["table_precision"] == "fp32"


def test_abi_mirrors_append_after_the_existing_fields():
    import ctypes as C

    class ModelBefore(C.Structure):
        _fields_ = [f for f in L.Model._fields_ if f[0] != "field_table_half"]

    assert L.Model._fields_[-1][0] == "field_table_half" and L.Model.field_table_half.offset == C.sizeof(ModelBefore)
    assert L.TrainCfg._fields_[-1][0] == "opt_half" and L.TrainCfg.opt_half.offset >= L.TrainCfg._pad_camopt.offset + 4
    assert (L.OptHalf.table_half.offset, L.OptHalf.first.offset, L.OptHalf.count.offset, C.sizeof(L.OptHalf)) == (0, 8, 16, 24)

"""CPU tests of the mixed-precision path for MLPs wider than 64 (csrc/mlp_mixed.cu) and the big / huge FruitField built on it: exported
symbols and their ctypes prototypes, and the scratch / ctx sizes, which are host arithmetic."""
import ctypes as C
import os
import re

from helpers import ROOT

from cropnerf_b200 import _lib as L

HEADER = os.path.join(ROOT, "include", "cropnerf_b200.h")
NEW = ("cnb_mlp_mixed_scratch_floats", "cnb_mlp_mixed_fwd", "cnb_mlp_mixed_bwd")


def _prototype(name):
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    m = re.search(r"(\w+)\s+" + name + r"\s*\(([^)]*)\)", src)
    assert m, name
    return m.group(1), [a.strip() for a in m.group(2).split(",")]


def _ctype_of(decl):
    if "*" in decl:
        return "cnb_mlp*" if "cnb_mlp" in decl else "ptr"
    if decl.startswith("cnb_stream_t"):
        return "ptr"
    return decl.split()[0]


def test_new_symbols_exported_and_prototypes_match():
    lib = L.lib()
    to_ctypes = {"ptr": C.c_void_p, "int64_t": C.c_int64, "int32_t": C.c_int32, "int": C.c_int}
    for name in NEW:
        assert hasattr(lib, name), name
        ret, args = _prototype(name)
        res, argtypes = L.SIGNATURES[name]
        assert res is to_ctypes[ret], (name, ret, res)
        assert len(args) == len(argtypes), name
        for decl, t in zip(args, argtypes):
            kind = _ctype_of(decl)
            if kind == "cnb_mlp*":
                assert t is C.POINTER(L.Mlp), (name, decl)
            else:
                assert t is to_ctypes[kind], (name, decl, t)


def _mlp(dims, act=L.ACT_NONE):
    m = L.Mlp()
    m.num_layers = len(dims) - 1
    m.out_activation = act
    for i, d in enumerate(dims):
        m.dims[i] = d
    return m


def _field(geo, sem_hidden, sem_layers, precision):
    f = L.Field()
    f.grid.num_levels = 16
    f.grid.log2_hashmap_size = 21
    f.base = _mlp((32, 64, 1 + geo))
    f.sem = _mlp((geo,) + (sem_hidden,) * (sem_layers - 1) + (64,))
    f.sem_head = _mlp((64, 1))
    f.rgb = _mlp((16 + geo + 32, 64, 64, 3), L.ACT_SIGMOID)
    f.appearance_dim = 32
    f.geo_feat_dim = geo
    f.precision = precision
    return f


def test_operator_scratch_sizes():
    lib = L.lib()
    n = 196608
    sem = _mlp((30, 128, 128, 64))
    tr, inf = lib.cnb_mlp_mixed_scratch_floats(C.byref(sem), n, 1), lib.cnb_mlp_mixed_scratch_floats(C.byref(sem), n, 0)
    # training keeps both 128-wide hidden layers in fp16 (128 halves per row each) plus the backward's work space
    assert tr > inf > 0
    assert tr >= n * 128
    # inference: two fp16 ping-pong buffers of the widest hidden layer
    assert inf == 2 * n * 128 // 2
    assert lib.cnb_mlp_mixed_scratch_floats(C.byref(_mlp((30, 256, 64))), n, 1) == 0   # outside support: no scratch, the calls refuse it
    assert lib.cnb_mlp_mixed_scratch_floats(C.byref(_mlp((78, 64, 64, 3))), 0, 1) == 0


def test_big_preset_mixed_ctx_size():
    lib = L.lib()
    n = 8192 * 128
    big_mixed = _field(30, 128, 3, L.PREC_MIXED)
    tr, inf = lib.cnb_field_ctx_floats(C.byref(big_mixed), n, 1), lib.cnb_field_ctx_floats(C.byref(big_mixed), n, 0)
    assert tr > 0 and inf > 0 and tr >= inf
    # the mixed layout keeps fp16 activations where the exact one keeps fp32: it is the smaller of the two in training
    big_fp32 = _field(30, 128, 3, L.PREC_FP32)
    assert tr < lib.cnb_field_ctx_floats(C.byref(big_fp32), n, 1)
    print(f"big preset ctx bytes per sample: mixed training {4 * tr / n:.1f}, inference {4 * inf / n:.1f}; "
          f"fp32 training {4 * lib.cnb_field_ctx_floats(C.byref(big_fp32), n, 1) / n:.1f}")


def test_base_preset_mixed_ctx_size_unchanged():
    """The base architecture keeps the fused kernels and their ctx layout (field_mixed.cuh ctx_total)."""
    lib = L.lib()
    base = _field(15, 64, 2, L.PREC_MIXED)
    for n in (1, 4096 * 48, 12345):
        part_off = ((n * 19 + 3) & ~3) + n * 32 + n * 4 + n * 8
        assert lib.cnb_field_ctx_floats(C.byref(base), n, 1) == part_off + 16896 * 160 + 16
        assert lib.cnb_field_ctx_floats(C.byref(base), n, 0) == 0   # the fused inference forward needs no scratch

"""No-GPU checks: the exact workspace sizes and score-log lengths the host-side planners report for the ViT-B layer
shapes.  The device workspace is carved into 256-byte aligned slices by the planner, so these numbers pin its layout:
a change of any slice (or of the order they are carved in) shows up here and has to update them on purpose."""
import ctypes

import pytest

_LIN = dict(rows=6304, tokens=197, n_a=1, w_bit=8, a_bit=8, eq_n=100, search_round=3, eq_alpha=0.01, eq_beta=1.2,
            post_gelu=0, has_bias=1, operand=0, kernel=0, init_layerwise=0)
# ViT-B/224 at 32 images, n_V = n_H = 24 (qkv: three row blocks per head group, head: one), as bench.py builds them
LINEAR = {
    "qkv": dict(in_features=768, out_features=2304, n_V=72, n_H=24),
    "proj": dict(in_features=768, out_features=768, n_V=24, n_H=24),
    "fc1": dict(in_features=768, out_features=3072, n_V=24, n_H=24),
    "fc2": dict(in_features=3072, out_features=768, n_V=24, n_H=24, post_gelu=1),
    "head": dict(rows=32, tokens=1, in_features=768, out_features=1000, n_V=1, n_H=24),
}
_MM = dict(batch=32, heads=12, A_bit=8, B_bit=8, eq_n=100, search_round=3, eq_alpha=0.01, eq_beta=1.2, operand=0, kernel=0,
           init_layerwise=0)
MATMUL = {
    "qk": dict(S1=197, S2=64, S3=197, sos=0),
    "sv": dict(S1=197, S2=197, S3=64, sos=1),
}
CONV = dict(images=32, out_channels=768, K=768, positions=196, w_bit=8, eq_n=100, eq_alpha=0.01, eq_beta=1.2, has_bias=1, kernel=0)
OPERANDS = {"auto": 0, "int8": 1, "bf16": 2}


@pytest.fixture(scope="module")
def lib():
    from ptq4vit_b200 import build, _lib
    build.build()
    return _lib.lib()


def _desc(cls, fields):
    d = cls()
    for k, v in fields.items():
        setattr(d, k, v)
    return d


def _query(lib, fn, desc):
    n = ctypes.c_size_t()
    assert getattr(lib, fn)(ctypes.byref(desc), ctypes.byref(n)) == 0, lib.p4v_last_error()
    return n.value


def linear_sizes(lib, layer):
    """{(operand, gram), function: value} for one Linear layer; P4V_GRAM must be set by the caller."""
    from ptq4vit_b200 import _lib
    out = {}
    for op_name, op in OPERANDS.items():
        d = _desc(_lib.LinearDesc, {**_LIN, **LINEAR[layer], "operand": op})
        out[op_name] = (_query(lib, "p4v_linear_workspace_bytes", d), _query(lib, "p4v_linear_quant_forward_workspace_bytes", d),
                        _query(lib, "p4v_linear_score_log_floats", d))
    return out


def matmul_sizes(lib, name):
    from ptq4vit_b200 import _lib
    out = {}
    for op_name, op in OPERANDS.items():
        d = _desc(_lib.MatMulDesc, {**_MM, **MATMUL[name], "operand": op})
        out[op_name] = (_query(lib, "p4v_matmul_workspace_bytes", d), _query(lib, "p4v_matmul_quant_forward_workspace_bytes", d),
                        _query(lib, "p4v_matmul_score_log_floats", d))
    return out


def conv_size(lib):
    from ptq4vit_b200 import _lib
    return _query(lib, "p4v_conv_workspace_bytes", _desc(_lib.ConvDesc, CONV))


# (search workspace, quant_forward workspace, score-log floats) per operand choice
LINEAR_EXPECTED = {
    ("fc1", "0"): {"auto": (1486347264, 16078336, 173100), "bf16": (1486347264, 16078336, 173100),
                   "int8": (751620864, 8803840, 173100)},
    ("fc1", "default"): {"auto": (2137103872, 16078336, 173100), "bf16": (2137103872, 16078336, 173100),
                         "int8": (1402377472, 8803840, 173100)},
    ("fc2", "0"): {"auto": (2247977216, 42099200, 173100), "bf16": (4491687680, 83780864, 173100),
                   "int8": (2247977216, 42099200, 173100)},
    ("fc2", "default"): {"auto": (2247977216, 42099200, 173100), "bf16": (4491687680, 83780864, 173100),
                         "int8": (2247977216, 42099200, 173100)},
    ("head", "0"): {"auto": (179326464, 2267136, 7500), "bf16": (179326464, 2267136, 7500),
                    "int8": (89965824, 1382400, 7500)},
    ("head", "default"): {"auto": (232981504, 2267136, 7500), "bf16": (232981504, 2267136, 7500),
                          "int8": (143620864, 1382400, 7500)},
    ("proj", "0"): {"auto": (1116271872, 11417344, 173100), "bf16": (1116271872, 11417344, 173100),
                    "int8": (560262144, 5912320, 173100)},
    ("proj", "default"): {"auto": (1532177152, 11417344, 173100), "bf16": (1532177152, 11417344, 173100),
                          "int8": (976167424, 5912320, 173100)},
    ("qkv", "0"): {"auto": (1363041280, 14577152, 518700), "bf16": (1363041280, 14577152, 518700),
                   "int8": (687887104, 7892480, 518700)},
    ("qkv", "default"): {"auto": (1935446784, 14577152, 518700), "bf16": (1935446784, 14577152, 518700),
                         "int8": (1260292608, 7892480, 518700)},
}
MATMUL_EXPECTED = {
    "qk": {"auto": (1290555392, 12604160, 7200), "bf16": (2561429504, 25187072, 7200), "int8": (1290555392, 12604160, 7200)},
    "sv": {"auto": (2863026176, 55071488, 3660), "bf16": (3853930752, 102257408, 3660), "int8": (2863026176, 55071488, 3660)},
}
CONV_EXPECTED = 234200576


@pytest.mark.parametrize("gram", ["default", "0"])
@pytest.mark.parametrize("layer", sorted(LINEAR))
def test_linear_plan_sizes(lib, layer, gram, monkeypatch):
    if gram == "default":
        monkeypatch.delenv("P4V_GRAM", raising=False)
    else:
        monkeypatch.setenv("P4V_GRAM", gram)
    assert linear_sizes(lib, layer) == LINEAR_EXPECTED[(layer, gram)]


@pytest.mark.parametrize("name", sorted(MATMUL))
def test_matmul_plan_sizes(lib, name):
    assert matmul_sizes(lib, name) == MATMUL_EXPECTED[name]


def test_conv_plan_size(lib):
    assert conv_size(lib) == CONV_EXPECTED

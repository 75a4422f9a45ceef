"""Integer export (SURVEY.md 8f rank 3): ptq4vit_b200.utils.integer against the reference's utils/integer.py functions
as recorded running on a B200 (tests/golden/ref_integer.npz) and against the oracle's restatement of their formulas."""
import pytest
import torch

from oracle import ptq_oracle as O
from tests import _refgold as G

pytestmark = pytest.mark.gpu


def _lin(cls, K, Oo, **kw):
    m = cls(K, Oo, **kw)
    gen = torch.Generator().manual_seed(5)
    m.weight.data = torch.randn(Oo, K, generator=gen) * 0.05
    return m.cuda()


def test_int8_weight_and_roundtrip():
    from ptq4vit_b200.quant_layers.linear import PTQSLBatchingQuantLinear
    from ptq4vit_b200.utils import integer as I
    m = _lin(PTQSLBatchingQuantLinear, 96, 64, n_V=4, n_H=3)
    wv = m.weight.data.view(4, 16, 3, 32)
    m.w_interval = (wv.abs().amax([1, 3], keepdim=True) / 127.5)
    w_int = I.quantize_int_weight(m)
    ref = O.int_plain(wv, m.w_interval, 128).view(64, 96)
    assert w_int.dtype == torch.int8 and torch.equal(w_int, ref)
    w_sim = I.dequantize_int_weight(m, w_int)
    assert torch.allclose(w_sim, m.quant_weight_bias()[0], rtol=0, atol=0)
    # the reference's own function (valid for one block, integer.py:15)
    m1 = _lin(PTQSLBatchingQuantLinear, 96, 64)
    m1.w_interval = (m1.weight.data.abs().max() / 127.5).view(1, 1, 1, 1)
    ref = torch.from_numpy(G.load("integer")["int8_weight"])
    assert torch.equal(I.quantize_int_weight(m1).cpu().view(-1), ref.view(-1))
    assert set(I.get_model_int_weight({"a": m1, "b": torch.nn.Identity()}).keys()) == {"a"}


def _activation_inputs():
    gen = torch.Generator().manual_seed(9)
    x = torch.randn(8, 197, 256, generator=gen).cuda()
    xg = torch.nn.functional.gelu(torch.randn(8, 197, 256, generator=gen) * 1.5).cuda()
    A = torch.randn(8, 6, 197, 64, generator=gen).cuda(); B = torch.randn(8, 6, 64, 197, generator=gen).cuda()
    S = torch.softmax(torch.randn(8, 6, 197, 197, generator=gen) * 4, -1).cuda(); V = torch.randn(8, 6, 197, 64, generator=gen).cuda()
    return x, xg, A, B, S, V


def activation_layout_modules(ns):
    """{key: (module, inputs)}: a Linear, a PostGelu Linear, a MatMul and a SoS MatMul of the classes in `ns` (this
    package's or the reference's quant_layers) carrying min-max step sizes of seeded inputs."""
    x, xg, A, B, S, V = _activation_inputs()
    lin = _lin(ns.linear.PTQSLBatchingQuantLinear, 256, 64); lin.a_interval = (x.abs().max() / 127.5).view(1, 1)
    gel = _lin(ns.linear.PostGeluPTQSLBatchingQuantLinear, 256, 64); gel.a_interval = (xg.max() / 127.5).view(1, 1)
    mm = ns.matmul.PTQSLBatchingQuantMatMul()
    mm.A_interval = (A.abs().amax((0, 2, 3)) / 127.5).view(1, 6, 1, 1, 1, 1, 1); mm.B_interval = (B.abs().amax((0, 2, 3)) / 127.5).view(1, 6, 1, 1, 1, 1, 1)
    mm._get_padding_parameters(A, B)
    sos = ns.matmul.SoSPTQSLBatchingQuantMatMul()
    sos.split = torch.tensor(2.0 ** -5, device="cuda"); sos.A_interval = sos.split / 127
    sos.B_interval = (V.abs().amax((0, 2, 3)) / 127.5).view(1, 6, 1, 1, 1, 1, 1)
    sos._get_padding_parameters(S, V)
    return {"lin": (lin, (x,)), "gelu": (gel, (xg,)), "mm": (mm, (A, B)), "sos": (sos, (S, V))}


def test_activation_layouts_match_reference_hooks():
    import types
    from ptq4vit_b200.quant_layers import linear, matmul
    from ptq4vit_b200.utils import integer as I
    mods = activation_layout_modules(types.SimpleNamespace(linear=linear, matmul=matmul))
    for mod, inputs in mods.values():
        I.quantize_int_activation(mod, inputs)
    (lin, (x,)), (gel, (xg,)), (mm, (A, B)), (sos, (S, V)) = mods["lin"], mods["gelu"], mods["mm"], mods["sos"]
    # oracle restatements (torch ops on the same device)
    assert torch.equal(lin.int_input[0], O.int_plain(x, lin.a_interval, 128))
    assert torch.equal(gel.int_input[0], O.int_gelu_twin(xg, gel.a_interval, gel.a_neg_interval, 128))
    assert torch.equal(mm.int_input[0], O.int_plain(A, mm.A_interval.view(1, 6, 1, 1), 128))
    assert torch.equal(mm.int_input[1], O.int_plain(B, mm.B_interval.view(1, 6, 1, 1), 128))
    assert torch.equal(sos.int_input[0], O.int_sos_twin(S, sos.split, sos.A_interval, 128))
    assert gel.int_input[0].dtype == torch.uint8 and sos.int_input[0].dtype == torch.uint8 and lin.int_input[0].dtype == torch.int8
    # the reference's pre-forward hook on its own classes carrying the same step sizes
    z = G.load("integer")
    for key, (mod, _) in mods.items():
        for i, t in enumerate(mod.int_input):
            G.assert_sample_equal(z, "act_", f"{key}{i}", t.cpu().numpy(), f"{key} input {i}")

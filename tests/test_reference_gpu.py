"""Full-size parity against the UNMODIFIED reference classes, as recorded running on a B200.

BASELINE.json configs[2] geometry: ViT-B/224, 32 images (M = 6304 tokens), n_H = 24, n_V = 24 (qkv 72, head 1),
n_a = 1, eq_n = 100, hessian metric, W8A8 and W6A6 -- one layer of every type the model has (qkv, proj, fc1,
fc2 twin-uniform, head, matmul1, matmul2 split-of-softmax), one search round.

The reference ran its own eager GPU path (quant_layers/linear.py:536-555 (+ :557-642), quant_layers/matmul.py:565-576,
:633-644) on the same seeded tensors; tests/golden/make_ref_golden.py recorded what is compared here
(tests/golden/ref_*.npz, see tests/_refgold.py for the format).  Compared per search step, in the reference's call
order:
  * the score table: per group the reference's best candidates (the whole table where it is small), max abs
    difference relative to the table's max (bar 2e-4; north_star 1e-3);
  * the argmax per group: a different pick is accepted only as a near-tie of the REFERENCE's own table
    (relative gap < 1e-4) and is counted;
  * the final step sizes (identical when no pick differs) and the quantized layer output on the reference's
    step sizes (1e-3 relative, north_star's bar; observed ~1e-6), on a seeded sample of the output's entries.
"""
import numpy as np
import pytest
import torch

from oracle import ptq_oracle as O
from tests import _refgold as G

pytestmark = pytest.mark.gpu

IMGS, TOK, D, HEADS = 32, 197, 768, 12
SCORE_RTOL = 2e-4
TIE_EPS = 1e-4
FLIP_FRAC = 0.02      # of the (row block, column block) picks of a layer; every one of them a near-tie (TIE_EPS)

LINEAR = {
    # name: (K, O, n_V, post_gelu, tokens)
    "qkv": (D, 3 * D, 72, False, TOK),
    "proj": (D, D, 24, False, TOK),
    "fc1": (D, 4 * D, 24, False, TOK),
    "fc2": (4 * D, D, 24, True, TOK),
    "head": (D, 1000, 1, False, 0),
}


def _compare_steps(name, got_tables, z, prefix, group_independent_until):
    flips, worst, compared, _ = G.compare_steps(name, got_tables, G.unpack_tables(z, prefix), group_independent_until,
                                                SCORE_RTOL, TIE_EPS)
    return flips, worst, compared


def _linear_case(name, bit):
    from ptq4vit_b200.quant_layers.linear import PTQSLBatchingQuantLinear, PostGeluPTQSLBatchingQuantLinear
    K, Oo, n_V, gelu, tok = LINEAR[name]
    x, W, b, y, g = O.make_linear_fixture(100 + bit + len(name), IMGS, tok, K, Oo, post_gelu=gelu)
    mod = dict(n_V=n_V, n_H=24, n_a=1, w_bit=bit, a_bit=bit, search_round=1)
    z = G.load(f"vitb_{name}_w{bit}")
    ref_w, ref_a = torch.from_numpy(z["w_interval"]), torch.from_numpy(z["a_interval"])
    # ---- ours
    cls = PostGeluPTQSLBatchingQuantLinear if gelu else PTQSLBatchingQuantLinear
    m = cls(K, Oo, metric="hessian", eq_alpha=0.01, eq_beta=1.2, eq_n=100, **mod)
    m.weight.data = W.clone(); m.bias.data = b.clone(); m.cuda(); m.keep_scores = True
    xd, yd, gd = x.cuda(), y.cuda(), g.cuda()

    def ours():
        m.raw_input, m.raw_out, m.raw_grad = xd, yd, gd
        with torch.no_grad():
            m.calibration_step2()
    ours(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); ours(); e1.record(); torch.cuda.synchronize()
    our_s = e0.elapsed_time(e1) / 1e3
    got_tables = [s.cpu().numpy() for s in m.last_scores]
    flips, worst, compared = _compare_steps(f"{name}/W{bit}A{bit}", got_tables, z, "s", group_independent_until=24)
    w_err = float((m.w_interval.cpu().reshape(-1) - ref_w.reshape(-1)).abs().max() / ref_w.abs().max())
    a_err = float((m.a_interval.cpu().reshape(-1) - ref_a.reshape(-1)).abs().max() / ref_a.abs().max())
    if flips == 0:
        assert w_err < 1e-6 and a_err < 1e-6, f"{name}: step sizes differ without a differing pick ({w_err:.2e}, {a_err:.2e})"
    else:
        assert flips <= max(1, int(FLIP_FRAC * n_V * 24)), f"{name}: {flips} near-tie picks differ"
    # quantized layer output on the reference's step sizes
    m.w_interval, m.a_interval = ref_w.cuda().view(n_V, 1, 24, 1), ref_a.cuda().view(1, 1)
    m.mode = "quant_forward"
    with torch.no_grad():
        out = m(x[:2].cuda()).cpu()
    o_err = G.sample_rel_err(z, "out_", "out", out)
    assert o_err < 1e-3, f"{name}: quantized layer output differs by {o_err:.3e}"
    print(f"[reference parity] {name} W{bit}A{bit}: flips {flips}/{compared}, worst score err {worst:.2e}, "
          f"dW {w_err:.1e} dX {a_err:.1e} out {o_err:.1e}; ours {our_s * 1e3:.1f} ms")


@pytest.mark.parametrize("bit", [8, 6])
@pytest.mark.parametrize("name", list(LINEAR))
def test_vitb_linear_matches_reference_on_gpu(name, bit):
    _linear_case(name, bit)


@pytest.mark.parametrize("bit", [8, 6])
@pytest.mark.parametrize("sos", [False, True])
def test_vitb_matmul_matches_reference_on_gpu(sos, bit):
    from ptq4vit_b200.quant_layers.matmul import PTQSLBatchingQuantMatMul, SoSPTQSLBatchingQuantMatMul
    name = "matmul2" if sos else "matmul1"
    S2, S3 = (TOK, D // HEADS) if sos else (D // HEADS, TOK)
    A, B, Y, Gr = O.make_matmul_fixture(200 + bit + sos, IMGS, HEADS, TOK, S2, S3, softmax_A=sos)
    mod = dict(A_bit=bit, B_bit=bit, search_round=1)
    z = G.load(f"vitb_{name}_w{bit}")
    ref_A, ref_B = torch.from_numpy(z["A_interval"]), torch.from_numpy(z["B_interval"])
    ref_split = torch.from_numpy(z["split"]) if sos else None
    cls = SoSPTQSLBatchingQuantMatMul if sos else PTQSLBatchingQuantMatMul
    m = cls(metric="hessian", eq_alpha=0.01, eq_beta=1.2, eq_n=100, **mod)
    m.keep_scores = True
    Ad, Bd, Yd, Gd = A.cuda(), B.cuda(), Y.cuda(), Gr.cuda()

    def ours():
        m.raw_input, m.raw_out, m.raw_grad = [Ad, Bd], Yd, Gd
        with torch.no_grad():
            m.calibration_step2()
    ours(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); ours(); e1.record(); torch.cuda.synchronize()
    our_s = e0.elapsed_time(e1) / 1e3
    got_tables = [s.cpu().numpy() for s in m.last_scores]
    # step 0 (A / split) is independent per head (split: one global group); step 1 (B) depends on step 0's pick
    flips, worst, compared = _compare_steps(f"{name}/W{bit}", got_tables, z, "s", group_independent_until=1)
    A_got = torch.as_tensor(m.A_interval).float().cpu().reshape(-1)
    a_err = float((A_got - ref_A.reshape(-1)).abs().max() / ref_A.abs().max())
    b_err = float((m.B_interval.cpu().reshape(-1) - ref_B.reshape(-1)).abs().max() / ref_B.abs().max())
    if flips == 0:
        assert a_err < 1e-6 and b_err < 1e-6, f"{name}: step sizes differ without a differing pick ({a_err:.2e}, {b_err:.2e})"
        if sos:
            assert float(m.split) == float(ref_split)
    else:
        assert flips <= 1, f"{name}: {flips} near-tie picks differ"
    if sos:
        m.split, m.A_interval = ref_split.cuda(), ref_A.cuda().reshape(())
    else:
        m.A_interval = ref_A.cuda().view(1, HEADS, 1, 1, 1, 1, 1)
    m.B_interval = ref_B.cuda().view(1, HEADS, 1, 1, 1, 1, 1)
    with torch.no_grad():
        out = m.quant_forward(A[:2].cuda(), B[:2].cuda()).cpu()
    o_err = G.sample_rel_err(z, "out_", "out", out)
    assert o_err < 1e-3, f"{name}: quantized output differs by {o_err:.3e}"
    print(f"[reference parity] {name} W{bit}: flips {flips}/{compared}, worst score err {worst:.2e}, "
          f"dA {a_err:.1e} dB {b_err:.1e} out {o_err:.1e}; ours {our_s * 1e3:.1f} ms")


def test_init_layerwise_matches_reference_on_gpu():
    """init_layerwise=True (linear.py:382-383, :393-394; matmul.py:430-432): every block / head starts from the
    layer-wise min-max step size, so the candidate grid itself changes."""
    from ptq4vit_b200.quant_layers.linear import PTQSLBatchingQuantLinear
    from ptq4vit_b200.quant_layers.matmul import PTQSLBatchingQuantMatMul
    z = G.load("init_layerwise")
    x, W, b, y, g = O.make_linear_fixture(301, 8, 50, 128, 192)
    mod = dict(n_V=3, n_H=4, n_a=2, w_bit=8, a_bit=8, search_round=2, init_layerwise=True)
    m = PTQSLBatchingQuantLinear(128, 192, metric="hessian", eq_alpha=0.01, eq_beta=1.2, eq_n=100, **mod)
    m.weight.data = W.clone(); m.bias.data = b.clone(); m.cuda(); m.keep_scores = True
    m.raw_input, m.raw_out, m.raw_grad = x.cuda(), y.cuda(), g.cuda()
    with torch.no_grad():
        m.calibration_step2()
    flips, worst, _ = _compare_steps("init_layerwise linear", [s.cpu().numpy() for s in m.last_scores], z, "lin_s", 0)
    assert worst < 1e-5 and flips <= 1            # a pick may only differ as a near-tie of the reference's table (checked above)
    if flips == 0:
        assert np.array_equal(m.w_interval.cpu().numpy().reshape(-1), z["lin_w_interval"].reshape(-1))
        assert np.array_equal(m.a_interval.cpu().numpy().reshape(-1), z["lin_a_interval"].reshape(-1))
    A, B, Y, Gr = O.make_matmul_fixture(302, 4, 3, 50, 32, 50)
    mm = PTQSLBatchingQuantMatMul(metric="hessian", eq_alpha=0.01, eq_beta=1.2, eq_n=100, search_round=2, init_layerwise=True)
    mm.raw_input, mm.raw_out, mm.raw_grad = [A.cuda(), B.cuda()], Y.cuda(), Gr.cuda()
    with torch.no_grad():
        mm.calibration_step2()
    rA, rB = torch.from_numpy(z["mm_A_interval"]).reshape(-1), torch.from_numpy(z["mm_B_interval"]).reshape(-1)
    ra = (mm.A_interval.cpu().reshape(-1) - rA).abs() / rA
    rb = (mm.B_interval.cpu().reshape(-1) - rB).abs() / rB
    assert int((ra > 2e-6).sum()) + int((rb > 2e-6).sum()) <= 1 and float(torch.cat([ra, rb]).max()) < 0.05


@pytest.mark.parametrize("metric", ["L2_norm", "linear_weighted_L2_norm", "square_weighted_L2_norm"])
def test_squared_error_metrics_match_reference_on_gpu(metric):
    """The reference's other squared-error metrics (linear.py:411-416, matmul.py:467-472, conv.py:511-516) through the
    same kernels, against the unmodified reference running that metric itself."""
    from ptq4vit_b200.quant_layers.conv import ChannelwiseBatchingQuantConv2d
    from ptq4vit_b200.quant_layers.linear import PTQSLBatchingQuantLinear
    from ptq4vit_b200.quant_layers.matmul import PTQSLBatchingQuantMatMul
    z = G.load(f"metric_{metric}")
    x, W, b, y, g = O.make_linear_fixture(401, 8, 50, 128, 192)
    mod = dict(n_V=3, n_H=4, n_a=2, w_bit=8, a_bit=8, search_round=2, metric=metric)
    m = PTQSLBatchingQuantLinear(128, 192, eq_alpha=0.01, eq_beta=1.2, eq_n=100, **mod)
    m.weight.data = W.clone(); m.bias.data = b.clone(); m.cuda(); m.keep_scores = True
    m.raw_input, m.raw_out, m.raw_grad = x.cuda(), y.cuda(), None
    with torch.no_grad():
        m.calibration_step2()
    flips, worst, _ = _compare_steps(f"{metric} linear", [s.cpu().numpy() for s in m.last_scores], z, "lin_s", 0)
    assert worst < 1e-5 and flips <= 1
    if flips == 0:
        assert np.array_equal(m.w_interval.cpu().numpy().reshape(-1), z["lin_w_interval"].reshape(-1))
        assert np.array_equal(m.a_interval.cpu().numpy().reshape(-1), z["lin_a_interval"].reshape(-1))
    A, B, Y, _ = O.make_matmul_fixture(402, 4, 3, 50, 32, 50)
    mm = PTQSLBatchingQuantMatMul(metric=metric, eq_alpha=0.01, eq_beta=1.2, eq_n=100, search_round=1)
    mm.keep_scores = True
    mm.raw_input, mm.raw_out, mm.raw_grad = [A.cuda(), B.cuda()], Y.cuda(), None
    with torch.no_grad():
        mm.calibration_step2()
    fl, worst_m, _ = _compare_steps(f"{metric} matmul", [s.cpu().numpy() for s in mm.last_scores], z, "mm_s", 1)
    assert worst_m < 1e-5 and fl <= 1
    if fl == 0:
        assert np.array_equal(mm.A_interval.cpu().numpy().reshape(-1), z["mm_A_interval"].reshape(-1))
        assert np.array_equal(mm.B_interval.cpu().numpy().reshape(-1), z["mm_B_interval"].reshape(-1))
    xc, Wc, bc, yc, gc = O.make_conv_fixture(403, 4, 3, 32, 16, 4)
    cv = ChannelwiseBatchingQuantConv2d(3, 32, (4, 4), stride=4, a_bit=32, metric=metric, eq_alpha=0.01, eq_beta=1.2, eq_n=100)
    cv.weight.data = Wc.clone(); cv.bias.data = bc.clone(); cv.cuda(); cv.keep_scores = True
    cv.raw_input, cv.raw_out, cv.raw_grad = xc.cuda(), yc.cuda(), None
    with torch.no_grad():
        cv.calibration_step2()
    rs = torch.from_numpy(z["conv_scores"]).double(); gs = cv.last_scores[0].cpu().double()
    assert float((gs - rs).abs().max() / rs.abs().max()) < SCORE_RTOL
    differing = int((cv.w_interval.cpu().reshape(-1) != torch.from_numpy(z["conv_w_interval"]).reshape(-1)).sum())
    assert differing <= 1, f"{metric} conv: {differing} channels differ"

"""Channel-wise weight search of the patch-embedding convolution (SURVEY.md 8f rank 2): the CUDA path against
tests/golden/conv_small.npz (reference class on the CPU), the oracle restatement and -- at ViT-B's patch-embedding size
(3 -> 768, 16x16 stride 16, 32 images of 224x224) -- the UNMODIFIED reference class as recorded running on a B200
(quant_layers/conv.py:444-614 with a_bit = 32 as configs/PTQ4ViT.py:54 builds it; tests/golden/ref_patch_embed_w*.npz)."""
import os

import numpy as np
import pytest
import torch

from oracle import ptq_oracle as O
from tests import _refgold as G

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _ours(x, W, b, y, g, stride, **kw):
    from ptq4vit_b200.quant_layers.conv import ChannelwiseBatchingQuantConv2d
    oc, ic, kh, kwid = W.shape
    m = ChannelwiseBatchingQuantConv2d(ic, oc, (kh, kwid), stride=stride, bias=b is not None, a_bit=32, metric="hessian",
                                       eq_alpha=0.01, eq_beta=1.2, eq_n=100, search_round=3, **kw)
    m.weight.data = W.clone()
    if b is not None:
        m.bias.data = b.clone()
    m.cuda(); m.keep_scores = True
    m.raw_input, m.raw_out, m.raw_grad = x.cuda(), y.cuda(), g.cuda()
    with torch.no_grad():
        m.calibration_step2()
    torch.cuda.synchronize()
    return m


def _check(m, ref_w, ref_scores, what):
    got = m.last_scores[0].cpu().numpy().astype(np.float64)
    ref = np.asarray(ref_scores, dtype=np.float64)
    err = np.abs(got - ref).max() / np.abs(ref).max()
    assert err < 2e-4, f"{what}: score table differs by {err:.2e}"
    flips = int((got.argmax(0) != ref.argmax(0)).sum())
    for j in np.nonzero(got.argmax(0) != ref.argmax(0))[0]:
        gap = (ref[ref[:, j].argmax(), j] - ref[got[:, j].argmax(), j]) / abs(ref[ref[:, j].argmax(), j])
        assert gap < 1e-4, f"{what}: channel {j} picked a candidate the reference scores {gap:.2e} worse"
    w = m.w_interval.cpu().reshape(-1).numpy()
    rw = np.asarray(ref_w).reshape(-1)
    if flips == 0:
        assert np.abs(w - rw).max() / np.abs(rw).max() < 1e-6, what
    return err, flips


def test_conv_search_matches_cpu_golden(monkeypatch):
    monkeypatch.setenv("P4V_SCALAR_DIV", "ieee")     # the golden comes from the reference on the CPU (see test_linear_gpu.py)
    z = np.load(os.path.join(GOLD, "conv_small.npz"))
    x, W, b, y, g = O.make_conv_fixture(31, 4, 3, 32, 16, 4)
    m = _ours(x, W, b, y, g, stride=4)
    err, flips = _check(m, z["w_interval"], z["scores_000"], "conv_small")
    assert m.w_interval.shape == (32, 1, 1, 1) and m.calibrated
    # quantized forward on the chosen step sizes (torch ops on the device, conv.py:609-613)
    m.mode = "quant_forward"
    with torch.no_grad():
        out = m(x.cuda())
    w_sim = (W / torch.from_numpy(z["w_interval"])).round_().clamp_(-128, 127).mul_(torch.from_numpy(z["w_interval"]))
    ref_out = torch.nn.functional.conv2d(x, w_sim, b, stride=4)
    if flips == 0:
        assert float((out.cpu() - ref_out).abs().max() / ref_out.abs().max()) < 1e-5


@pytest.mark.parametrize("bit", [8, 6])
def test_vitb_patch_embedding_matches_reference_on_gpu(bit):
    x, W, b, y, g = O.make_conv_fixture(32 + bit, 32, 3, 768, 224, 16)
    z = G.load(f"patch_embed_w{bit}")
    m = _ours(x, W, b, y, g, stride=16, w_bit=bit)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m.raw_input, m.raw_out, m.raw_grad = x.cuda(), y.cuda(), g.cuda()
    e0.record()
    with torch.no_grad():
        m.calibration_step2()
    e1.record(); torch.cuda.synchronize()
    # every differing channel is checked as a near-tie of the reference's own table
    flips, err, _, _ = G.compare_steps(f"patch_embed W{bit}", [m.last_scores[0].cpu().numpy()], G.unpack_tables(z, "s"), 1, 2e-4, 1e-4)
    w, rw = m.w_interval.cpu().reshape(-1).numpy(), z["w_interval"].reshape(-1)
    if flips == 0:
        assert np.abs(w - rw).max() / np.abs(rw).max() < 1e-6
    assert flips <= 8       # 1 % of the channels
    # (the reference's F.conv2d runs through cuDNN, TF32 allowed by default: its scores carry ~1e-6 of noise)
    print(f"[conv parity] patch embedding W{bit}: worst score err {err:.2e}, {flips}/768 channels differ; "
          f"ours {e0.elapsed_time(e1):.1f} ms")

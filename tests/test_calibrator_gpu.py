"""The public calibrator end to end: `HessianQuantCalibrator(net, wrapped, loader, sequential, batch_size)
.batching_quant_calib()` on a 2-block synthetic ViT, against

  * the UNMODIFIED reference calibrator (utils/quant_calib.py:300-378 + utils/net_wrap.py + configs/PTQ4ViT.py) as
    recorded running on a B200 (tests/golden/ref_calib_*.npz): captured x / y / grad tensors (a seeded sample of
    their entries) and every chosen step size;
  * tests/golden/calib_tiny_vit.npz (the same reference run on the CPU).  CPU and GPU capture numerics differ in the
    last bits, so near-tie picks may move by a grid step: the comparison counts differing entries.

Also: single-pass capture == the reference's one-sweep-per-module capture (SURVEY.md 8f rank 1), sequential=True works
(gradients reach the modules behind an already quantized layer), QuantCalibrator.{parallel,sequential}_quant_calib and
the base batching_quant_calib run on the non-batching / L2 configurations.
"""
import importlib
import os

import numpy as np
import pytest
import torch

os.environ.setdefault("TQDM_DISABLE", "1")

from oracle import ref_harness as RH
from tests import _refgold as G

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "calib_tiny_vit.npz")
GRID = (1.2 - 0.01) / 100


TINY_SWIN = dict(img_size=32, patch=4, dim=32, depths=(2, 2), num_heads=(2, 4), window_size=4, num_classes=10)


def _net(kind="vit"):
    from ptq4vit_b200.utils.models import SwinTransformer, VisionTransformer
    net = (SwinTransformer(**TINY_SWIN) if kind == "swin" else VisionTransformer(**RH.TINY_VIT)).cuda().eval()
    RH.add_target_noise(net, 8, 10)
    return net


def _ours(sequential=False, capture="auto", keep=None, wrap_conv=True, kind="vit"):
    from ptq4vit_b200.configs import PTQ4ViT as cfg
    from ptq4vit_b200.utils import quant_calib as Q
    from ptq4vit_b200.utils.net_wrap import wrap_modules_in_net
    importlib.reload(cfg)
    net = _net(kind)
    wrapped = wrap_modules_in_net(net, cfg, wrap_conv=wrap_conv)
    cal = Q.HessianQuantCalibrator(net, wrapped, RH.ListLoader(RH.tiny_images()), sequential=sequential, batch_size=4, capture=capture)
    cal.keep_captured = keep
    cal.batching_quant_calib()
    torch.cuda.synchronize()
    assert all(m.mode == "quant_forward" and m.calibrated for m in wrapped.values())
    return RH.collect_intervals(wrapped), net, wrapped, cal


def _count_diff(got, ref, what, max_frac, max_steps=3):
    """Entries must be identical; a differing entry must be a neighbouring grid point (near-tie).  Returns #differing."""
    n = bad = 0
    for name, d in ref.items():
        if name not in got:
            continue
        for key, rv in d.items():
            if key not in got[name]:
                continue
            gv = got[name][key].reshape(-1).numpy().astype(np.float64); rv = rv.reshape(-1).numpy().astype(np.float64)
            assert gv.shape == rv.shape, f"{what}: {name}.{key} shape {gv.shape} vs {rv.shape}"
            rel = np.abs(gv - rv) / np.abs(rv)
            diff = rel > 2e-6
            n += rv.size; bad += int(diff.sum())
            if diff.any():     # a near-tie moves a pick to a neighbouring candidate (split: the next power of two)
                lim = 0.51 if key == "split" or (name.endswith("matmul2") and key == "A_interval") else 0.1
                assert np.all(rel[diff] < lim), f"{what}: {name}.{key} differs by more than a near-tie: {gv} vs {rv}"
    assert bad <= max(1, int(max_frac * n)), f"{what}: {bad} of {n} step sizes differ"
    return bad, n


def _as_dict(npz, prefix):
    out = {}
    for k in npz.files:
        parts = k.split("|")
        if len(parts) == 3 and parts[0] == prefix:
            out.setdefault(parts[1], {})[parts[2]] = torch.from_numpy(npz[k])
    return out


def test_batching_quant_calib_matches_reference_calibrator_on_gpu():
    snap_ours = {}
    got, net, wrapped, cal = _ours(keep=snap_ours)
    assert cal.timings["single_pass"] and cal.timings["total_s"] > 0
    z = G.load("calib_vit")
    ref = _as_dict(z, "iv")
    # captured tensors: same net, same ops, same kind of device
    worst = 0.0
    for name, d in snap_ours.items():
        for key, t in d.items():
            err = G.sample_rel_err(z, "cap_", f"{name}|{key}", t.cpu())
            worst = max(worst, err)
            assert err < 1e-4, f"captured {name}.{key} differs from the reference's capture: {err:.2e}"
    bad, n = _count_diff(got, ref, "vs reference on GPU", max_frac=0.05)
    print(f"[calibrator parity] {len(snap_ours)} modules, captured tensors worst rel diff {worst:.2e}; {bad}/{n} step sizes differ")
    # the calibrated nets agree on the calibration images
    with torch.no_grad():
        ours_out = net(RH.tiny_images().cuda()[:4])
    assert torch.isfinite(ours_out).all()


def test_swin_windowed_attention_and_reduction_match_reference_calibrator():
    """BASELINE.json configs[4] geometry in small: shifted windows, window attention MatMuls with the batch dimension
    images x windows (reference utils/models.py:28-56) and the `reduction` Linear of patch merging (utils/net_wrap.py:42)."""
    snap_ours = {}
    got, net, wrapped, cal = _ours(keep=snap_ours, kind="swin")
    assert any(n.endswith("downsample.reduction") for n in wrapped) and any("layers.0.blocks.1.attn.matmul1" == n for n in wrapped)
    z = G.load("calib_swin")
    ref = _as_dict(z, "iv")
    assert set(ref) == set(got)
    for name, d in snap_ours.items():
        for key, t in d.items():
            assert G.sample_rel_err(z, "cap_", f"{name}|{key}", t.cpu()) <= 1e-5, f"captured {name}.{key}"
    bad, n = _count_diff(got, ref, "swin vs reference on GPU", max_frac=0.05)
    print(f"[calibrator swin] {len(got)} modules (window attention + patch merging), {bad}/{n} step sizes differ")


def test_batching_quant_calib_matches_cpu_golden():
    got, *_ = _ours()
    ref = _as_dict(np.load(GOLD), "par")
    bad, n = _count_diff(got, ref, "vs CPU golden", max_frac=0.15)
    print(f"[calibrator golden] {bad}/{n} step sizes differ from the CPU reference run")


def test_single_pass_capture_equals_per_module_capture():
    a, b = {}, {}
    got1, *_ = _ours(capture="single_pass", keep=a)
    got2, *_ = _ours(capture="per_module", keep=b)
    for name in a:
        for key, t in a[name].items():
            r = b[name][key]
            assert float((t - r).abs().max()) <= 1e-6 * float(r.abs().max()) + 1e-30, f"{name}.{key}"
    _count_diff(got1, got2, "single-pass vs per-module", max_frac=0.0)


def test_sequential_calibration_runs_and_tracks_reference():
    got, net, wrapped, cal = _ours(sequential=True)
    assert not cal.timings["single_pass"]
    bad, n = _count_diff(got, _as_dict(G.load("calib_vit_sequential"), "iv"), "sequential", max_frac=0.3)
    bad_cpu, _ = _count_diff(got, _as_dict(np.load(GOLD), "seq"), "sequential vs CPU golden", max_frac=0.3)
    print(f"[calibrator sequential] {bad}/{n} step sizes differ from the GPU reference run, {bad_cpu} from the CPU one")


def test_quant_calibrator_parallel_and_sequential_drivers():
    """QuantCalibrator.quant_calib (reference :95-104) with the non-batching classes and the L2 metric."""
    from ptq4vit_b200.quant_layers.linear import PTQSLQuantLinear, PostGeluPTQSLQuantLinear
    from ptq4vit_b200.quant_layers.matmul import PTQSLQuantMatMul, SoSPTQSLQuantMatMul
    from ptq4vit_b200.utils import quant_calib as Q
    from ptq4vit_b200.utils.models import MatMul
    kw = dict(metric="L2_norm", eq_alpha=0.01, eq_beta=1.2, eq_n=100, search_round=1)

    def wrap(net):
        wrapped = {}
        for name, m in list(net.named_modules()):
            parent = net.get_submodule(name.rsplit(".", 1)[0]) if "." in name else net
            leaf = name.rsplit(".", 1)[-1]
            if isinstance(m, torch.nn.Linear):
                cls = PostGeluPTQSLQuantLinear if leaf == "fc2" else PTQSLQuantLinear
                q = cls(m.in_features, m.out_features, **kw)
                q.weight.data = m.weight.data; q.bias = m.bias; q.to(m.weight.device)
            elif isinstance(m, MatMul):
                q = (SoSPTQSLQuantMatMul if leaf == "matmul2" else PTQSLQuantMatMul)(**kw)
            else:
                continue
            setattr(parent, leaf, q); wrapped[name] = q
        return wrapped

    res = {}
    for sequential in (False, True):
        net = _net()
        wrapped = wrap(net)
        cal = Q.QuantCalibrator(net, wrapped, RH.ListLoader(RH.tiny_images()), sequential=sequential)
        cal.quant_calib()
        torch.cuda.synchronize()
        assert cal.calibrated and all(m.mode == "quant_forward" and m.calibrated for m in wrapped.values())
        res[sequential] = RH.collect_intervals(wrapped)
        with torch.no_grad():
            assert torch.isfinite(net(RH.tiny_images().cuda())).all()
    # the first module sees the same FP32 input in both modes
    first = next(iter(res[False]))
    assert torch.equal(res[False][first]["w_interval"], res[True][first]["w_interval"])


def test_base_batching_quant_calib_l2():
    """QuantCalibrator.batching_quant_calib (reference :106-171): forward-only capture, gradient-free metric."""
    from ptq4vit_b200.configs import PTQ4ViT as cfg
    from ptq4vit_b200.utils import quant_calib as Q
    from ptq4vit_b200.utils.net_wrap import wrap_modules_in_net
    importlib.reload(cfg)
    for d in (cfg.ptqsl_linear_kwargs, cfg.ptqsl_matmul_kwargs, cfg.ptqsl_conv2d_kwargs):
        d["metric"] = "L2_norm"; d["search_round"] = 1
    net = _net()
    wrapped = wrap_modules_in_net(net, cfg, wrap_conv=True)
    cal = Q.QuantCalibrator(net, wrapped, RH.ListLoader(RH.tiny_images()), sequential=False)
    cal.batch_size = 4
    cal.batching_quant_calib()
    torch.cuda.synchronize()
    assert all(m.calibrated for m in wrapped.values())
    importlib.reload(cfg)


def wrap_non_batching(net, lin, gelu, mm, sos, matmul_type):
    """Replace every Linear / MatMul of `net` by the given non-batching classes (hessian metric, two rounds)."""
    kw = dict(metric="hessian", eq_alpha=0.01, eq_beta=1.2, eq_n=100, search_round=2)
    wrapped = {}
    for name, m in list(net.named_modules()):
        parent = net.get_submodule(name.rsplit(".", 1)[0]) if "." in name else net
        leaf = name.rsplit(".", 1)[-1]
        if isinstance(m, torch.nn.Linear):
            q = (gelu if leaf == "fc2" else lin)(m.in_features, m.out_features, n_V=3 if leaf == "qkv" else 1, **kw)
            q.weight.data = m.weight.data; q.bias = m.bias; q.to(m.weight.device)
        elif isinstance(m, matmul_type):
            q = (sos if leaf == "matmul2" else mm)(**kw)
        else:
            continue
        setattr(parent, leaf, q); wrapped[name] = q
    return wrapped


def test_hessian_quant_calib_non_batching_driver_matches_reference():
    """HessianQuantCalibrator.quant_calib (reference :216-298): the non-batching driver -- per module one forward+backward
    sweep, then `calibration_step2(x)` / `(A, B)` of the NON-batching classes with the hessian metric -- against the
    reference's same driver on its own non-batching classes (Linear and MatMul modules; both nets wrapped by hand)."""
    from ptq4vit_b200.quant_layers import linear as L, matmul as M
    from ptq4vit_b200.utils import quant_calib as Q
    from ptq4vit_b200.utils.models import MatMul
    net = _net()
    ours = wrap_non_batching(net, L.PTQSLQuantLinear, L.PostGeluPTQSLQuantLinear, M.PTQSLQuantMatMul, M.SoSPTQSLQuantMatMul, MatMul)
    Q.HessianQuantCalibrator(net, ours, RH.ListLoader(RH.tiny_images()), sequential=False, batch_size=4).quant_calib()
    torch.cuda.synchronize()
    assert all(m.calibrated and m.mode == "quant_forward" for m in ours.values())
    ref = _as_dict(G.load("calib_non_batching"), "iv")
    assert set(ref) == set(ours)
    bad, n = _count_diff(RH.collect_intervals(ours), ref, "non-batching hessian driver", max_frac=0.1)
    print(f"[calibrator non-batching] {len(ours)} modules, {bad}/{n} step sizes differ")

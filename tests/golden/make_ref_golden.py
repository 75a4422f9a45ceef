"""Record the unmodified reference's outputs that the parity tests compare against (tests/golden/ref_*.npz).

Needs the reference tree (staged under oracle/_ref by `PTQ4VIT_REFERENCE=<tree> python oracle/stage_ref.py`, or
named by $PTQ4VIT_REFERENCE).  The GPU cases run the reference's own eager path on a B200, the same tensors and
settings the tests use; the CPU cases run it on the host, as the CPU tests do:

    python tests/golden/make_ref_golden.py gpu [OUT_DIR]      # on the GPU machine
    python tests/golden/make_ref_golden.py cpu [OUT_DIR]      # anywhere, no GPU needed

Fixtures are regenerated from seeds (oracle.ptq_oracle.make_*_fixture, torch CPU RNG) and are not stored.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
os.environ.setdefault("TQDM_DISABLE", "1")

from oracle import ptq_oracle as O  # noqa: E402
from oracle import ref_harness as RH  # noqa: E402
from tests import _refgold as G  # noqa: E402

METRICS = ["L2_norm", "linear_weighted_L2_norm", "square_weighted_L2_norm"]


def pack_intervals(prefix, res):
    return {f"{prefix}{name}|{key}": v.numpy() for name, d in res.items() for key, v in d.items()}


def gpu_cases(out):
    from tests import test_calibrator_gpu as TC
    from tests import test_integer_gpu as TI
    from tests import test_reference_gpu as TR
    # ---- full-size layers (test_reference_gpu.py)
    for name, (K, Oo, n_V, gelu, tok) in TR.LINEAR.items():
        for bit in (8, 6):
            x, W, b, y, g = O.make_linear_fixture(100 + bit + len(name), TR.IMGS, tok, K, Oo, post_gelu=gelu)
            ref = RH.run_linear(x, W, b, y, g, post_gelu=gelu, quant_forward=True, n_V=n_V, n_H=24, n_a=1, w_bit=bit,
                                a_bit=bit, search_round=1)
            out(f"vitb_{name}_w{bit}", **G.pack_tables("s", [s.numpy() for s in ref["scores"]]),
                w_interval=ref["w_interval"].numpy(), a_interval=ref["a_interval"].numpy(), **G.pack_samples("out_", {"out": ref["out"].numpy()}))
    for sos in (False, True):
        for bit in (8, 6):
            S2, S3 = (TR.TOK, TR.D // TR.HEADS) if sos else (TR.D // TR.HEADS, TR.TOK)
            A, B, Y, Gr = O.make_matmul_fixture(200 + bit + sos, TR.IMGS, TR.HEADS, TR.TOK, S2, S3, softmax_A=sos)
            ref = RH.run_matmul(A, B, Y, Gr, sos=sos, A_bit=bit, B_bit=bit, search_round=1)
            extra = {"split": ref["split"].numpy()} if sos else {}
            out(f"vitb_matmul{2 if sos else 1}_w{bit}", **G.pack_tables("s", [s.numpy() for s in ref["scores"]]),
                A_interval=ref["A_interval"].numpy(), B_interval=ref["B_interval"].numpy(), **extra,
                **G.pack_samples("out_", {"out": ref["out"].numpy()}))
    # ---- init_layerwise and the squared-error metrics (test_reference_gpu.py)
    x, W, b, y, g = O.make_linear_fixture(301, 8, 50, 128, 192)
    ref = RH.run_linear(x, W, b, y, g, quant_forward=False, n_V=3, n_H=4, n_a=2, w_bit=8, a_bit=8, search_round=2, init_layerwise=True)
    A, B, Y, Gr = O.make_matmul_fixture(302, 4, 3, 50, 32, 50)
    refm = RH.run_matmul(A, B, Y, Gr, quant_forward=False, search_round=2, init_layerwise=True)
    out("init_layerwise", **G.pack_tables("lin_s", [s.numpy() for s in ref["scores"]]), lin_w_interval=ref["w_interval"].numpy(),
        lin_a_interval=ref["a_interval"].numpy(), mm_A_interval=refm["A_interval"].numpy(), mm_B_interval=refm["B_interval"].numpy())
    for metric in METRICS:
        x, W, b, y, g = O.make_linear_fixture(401, 8, 50, 128, 192)
        ref = RH.run_linear(x, W, b, y, g, quant_forward=False, n_V=3, n_H=4, n_a=2, w_bit=8, a_bit=8, search_round=2, metric=metric)
        A, B, Y, Gr = O.make_matmul_fixture(402, 4, 3, 50, 32, 50)
        refm = RH.run_matmul(A, B, Y, Gr, quant_forward=False, search_round=1, metric=metric)
        xc, Wc, bc, yc, gc = O.make_conv_fixture(403, 4, 3, 32, 16, 4)
        refc = RH.run_conv(xc, Wc, bc, yc, gc, stride=4, metric=metric)
        out(f"metric_{metric}", **G.pack_tables("lin_s", [s.numpy() for s in ref["scores"]]), lin_w_interval=ref["w_interval"].numpy(),
            lin_a_interval=ref["a_interval"].numpy(), **G.pack_tables("mm_s", [s.numpy() for s in refm["scores"]]),
            mm_A_interval=refm["A_interval"].numpy(), mm_B_interval=refm["B_interval"].numpy(),
            conv_scores=refc["scores"][0].reshape(100, -1).numpy(), conv_w_interval=refc["w_interval"].numpy())
    # ---- ViT-B patch embedding (test_conv_gpu.py)
    for bit in (8, 6):
        x, W, b, y, g = O.make_conv_fixture(32 + bit, 32, 3, 768, 224, 16)
        ref = RH.run_conv(x, W, b, y, g, stride=16, search_round=1, w_bit=bit)
        out(f"patch_embed_w{bit}", **G.pack_tables("s", [ref["scores"][0].reshape(100, -1).numpy()]), w_interval=ref["w_interval"].numpy())
    # ---- integer export (test_integer_gpu.py)
    R = RH.load()
    from ptq4vit_b200.quant_layers.linear import PTQSLBatchingQuantLinear
    m1 = TI._lin(PTQSLBatchingQuantLinear, 96, 64)
    r = R.linear.PTQSLBatchingQuantLinear(96, 64).cuda()
    r.weight.data = m1.weight.data.clone(); r.w_interval = (m1.weight.data.abs().max() / 127.5).view(1, 1, 1, 1)
    w_int = R.integer.quantize_int_weight(r).cpu().numpy()
    layouts = TI.activation_layout_modules(R)
    acts = {}
    for key, (mod, inputs) in layouts.items():
        R.integer.quantize_int_activation(mod, inputs)
        for i, t in enumerate(mod.int_input):
            acts[f"{key}{i}"] = t.cpu().numpy()
    out("integer", int8_weight=w_int, **G.pack_samples("act_", acts))
    # ---- the calibrator on the tiny ViT / Swin (test_calibrator_gpu.py)
    for kind in ("vit", "swin"):
        snap = {}
        res, _, _ = RH.run_reference_calibrator(TC._net(kind), RH.tiny_images(), batch_size=4, sequential=False, snapshot=snap)
        caps = {f"{name}|{key}": t.cpu().numpy() for name, d in snap.items() for key, t in d.items() if t is not None}
        out(f"calib_{kind}", **pack_intervals("iv|", res), **G.pack_samples("cap_", caps, n=64))
    res, _, _ = RH.run_reference_calibrator(TC._net(), RH.tiny_images(), batch_size=4, sequential=True)
    out("calib_vit_sequential", **pack_intervals("iv|", res))
    net_r = TC._net()
    for mod in net_r.modules():
        for leaf in ("matmul1", "matmul2"):
            if hasattr(mod, leaf):
                setattr(mod, leaf, R.models.MatMul())
    refs = TC.wrap_non_batching(net_r, R.linear.PTQSLQuantLinear, R.linear.PostGeluPTQSLQuantLinear, R.matmul.PTQSLQuantMatMul,
                                R.matmul.SoSPTQSLQuantMatMul, R.models.MatMul)
    R.quant_calib.HessianQuantCalibrator(net_r, refs, RH.ListLoader(RH.tiny_images()), sequential=False, batch_size=4).quant_calib()
    torch.cuda.synchronize()
    out("calib_non_batching", **pack_intervals("iv|", RH.collect_intervals(refs)))


def cpu_cases(out):
    from tests import test_reference_harness_cpu as TH
    R = RH.load()
    # ---- utils/integer.py on the host (test_integer_oracle_matches_reference_functions)
    W, x, xg, S, V = TH.integer_inputs()
    lin = R.linear.PTQSLBatchingQuantLinear(64, 32)
    lin.weight.data = W.clone(); lin.w_interval = (W.abs().max() / 127.5).view(1, 1, 1, 1)
    w_int = R.integer.quantize_int_weight(lin).view(32, 64)
    lin.a_interval = (x.abs().max() / 127.5).view(1, 1)
    R.integer.quantize_int_activation(lin, (x,))
    gel = R.linear.PostGeluPTQSLBatchingQuantLinear(64, 32)
    gel.a_interval = (xg.max() / 127.5).view(1, 1)
    R.integer.quantize_int_activation(gel, (xg,))
    sos = R.matmul.SoSPTQSLBatchingQuantMatMul()
    sos.split = torch.tensor(2.0 ** -4); sos.A_interval = sos.split / 127
    sos.B_interval = (V.abs().amax((0, 2, 3)) / 127.5).view(1, 3, 1, 1, 1, 1, 1)
    sos._get_padding_parameters(S, V)
    R.integer.quantize_int_activation(sos, (S, V))
    out("integer_functions", w_int=w_int.numpy(), x_int=lin.int_input[0].numpy(), gelu_int=gel.int_input[0].numpy(),
        gelu_a_neg_interval=np.float64(float(gel.a_neg_interval)), sos_A_int=sos.int_input[0].numpy(), sos_B_int=sos.int_input[1].numpy())
    # ---- the squared-error metrics run by the reference itself (test_weighted_l2_metrics_are_hessian_with_a_surrogate_weight)
    for metric in METRICS:
        x, W, b, y, g = O.make_linear_fixture(41, 4, 20, 32, 48)
        d = RH.run_linear(x, W, b, y, g, quant_forward=False, metric=metric, **TH.METRIC_LINEAR)
        A, B, Y, Gr = O.make_matmul_fixture(42, 2, 3, 12, 8, 12)
        dm = RH.run_matmul(A, B, Y, Gr, quant_forward=False, metric=metric, search_round=1, eq_n=25)
        xc, Wc, bc, yc, gc = O.make_conv_fixture(43, 2, 3, 8, 8, 4)
        dc = RH.run_conv(xc, Wc, bc, yc, gc, stride=4, metric=metric, eq_n=25)
        out(f"metric_cpu_{metric}", **G.pack_tables("lin_s", [s.numpy() for s in d["scores"]]), lin_w_interval=d["w_interval"].numpy(),
            lin_a_interval=d["a_interval"].numpy(), mm_A_interval=dm["A_interval"].numpy(), mm_B_interval=dm["B_interval"].numpy(),
            conv_w_interval=dc["w_interval"].numpy())


def main():
    mode = sys.argv[1]
    dest = sys.argv[2] if len(sys.argv) > 2 else HERE
    os.makedirs(dest, exist_ok=True)
    assert RH.available(), "reference tree not found: set PTQ4VIT_REFERENCE or stage it under oracle/_ref"

    def out(name, **arrays):
        path = os.path.join(dest, f"ref_{name}.npz")
        np.savez_compressed(path, **arrays)
        print(f"{name}: {os.path.getsize(path)} bytes", flush=True)

    if mode == "gpu":
        assert torch.cuda.is_available(), "the GPU cases run the reference on the GPU"
        gpu_cases(out)
    else:
        cpu_cases(out)


if __name__ == "__main__":
    main()

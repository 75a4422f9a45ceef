"""Checks of the test / baseline infrastructure itself on the CPU: the oracle's restatements of utils/integer.py
against the reference's functions and the squared-error metrics against the reference running them (both as recorded
in tests/golden/ref_*.npz by tests/golden/make_ref_golden.py), the reference timing helpers bench.py uses (on stand-ins
for the reference's classes), and bench.py's unit / extrapolation arithmetic."""
import argparse
import types

import numpy as np
import pytest
import torch

from oracle import ptq_oracle as O
from oracle import ref_harness as RH
from tests import _refgold as G

METRIC_LINEAR = dict(n_V=3, n_H=2, n_a=2, search_round=2, eq_n=25)


def integer_inputs():
    gen = torch.Generator().manual_seed(2)
    W = torch.randn(32, 64, generator=gen) * 0.1
    x = torch.randn(4, 9, 64, generator=gen)
    xg = torch.nn.functional.gelu(x * 1.5)
    S = torch.softmax(torch.randn(2, 3, 10, 10, generator=gen) * 4, -1); V = torch.randn(2, 3, 10, 8, generator=gen)
    return W, x, xg, S, V


def test_integer_oracle_matches_reference_functions():
    z = G.load("integer_functions")
    W, x, xg, S, V = integer_inputs()
    assert torch.equal(torch.from_numpy(z["w_int"]), O.int_plain(W, (W.abs().max() / 127.5).view(1, 1), 128))
    assert torch.equal(torch.from_numpy(z["x_int"]), O.int_plain(x, (x.abs().max() / 127.5).view(1, 1), 128))
    assert float(z["gelu_a_neg_interval"]) == O.GELU_MIN_NEG / 128
    assert torch.equal(torch.from_numpy(z["gelu_int"]), O.int_gelu_twin(xg, (xg.max() / 127.5).view(1, 1), float(z["gelu_a_neg_interval"]), 128))
    split = torch.tensor(2.0 ** -4)
    B_interval = (V.abs().amax((0, 2, 3)) / 127.5).view(1, 3, 1, 1)
    assert torch.equal(torch.from_numpy(z["sos_A_int"]), O.int_sos_twin(S, split, split / 127, 128))
    assert torch.equal(torch.from_numpy(z["sos_B_int"]), O.int_plain(V, B_interval, 128))


class _SearchStandIn(torch.nn.Module):
    """The part of the reference's Batching classes the timing helpers drive (quant_layers/linear.py:536-555,
    matmul.py:565-576): every search step ends in one argmax over its score table.  Records the steps it ran."""

    def __init__(self, *shape, bias=True, n_V=1, n_H=1, n_a=1, search_round=3, eq_n=100, eq_alpha=0.01, eq_beta=1.2, **kw):
        super().__init__()
        self.n_V, self.n_H, self.n_a, self.search_round = n_V, n_H, n_a, search_round
        self.eq_n, self.eq_alpha, self.eq_beta = eq_n, eq_alpha, eq_beta
        if shape:
            self.weight = torch.nn.Parameter(torch.zeros(shape[1], shape[0]))
            self.bias = torch.nn.Parameter(torch.zeros(shape[1])) if bias else None
        self.steps = []

    def _step(self, kind, groups):
        self.steps.append(kind)
        torch.zeros(self.eq_n + 1, groups).argmax(dim=0)

    def _initialize_calib_parameters(self):
        pass

    def _initialize_intervals(self):
        self.w_interval, self.a_interval = torch.ones(self.n_V, 1, self.n_H, 1), torch.ones(self.n_a, 1)

    def _search_best_w_interval(self, w_cands):
        for _ in range(self.n_H):
            self._step("w", self.n_V)

    def _search_best_a_interval(self, a_cands):
        for _ in range(self.n_a):
            self._step("a", 1)

    def calibration_step2(self):
        self._initialize_calib_parameters()
        self._initialize_intervals()
        for _ in range(self.search_round):
            if self.n_V:
                self._search_best_w_interval(None)
            self._search_best_a_interval(None)


def test_reference_timing_helpers_count_units(monkeypatch):
    """RH.time_linear / time_matmul: the bounded CPU sample interrupts the weight search after w_blocks column blocks
    and still runs the activation search; the unit counts are the ones bench.py extrapolates with."""
    made = []

    def cls(*a, **k):
        m = _SearchStandIn(*a, **k)
        made.append(m)
        return m
    ns = types.SimpleNamespace(linear=types.SimpleNamespace(PTQSLBatchingQuantLinear=cls, PostGeluPTQSLBatchingQuantLinear=cls),
                               matmul=types.SimpleNamespace(PTQSLBatchingQuantMatMul=cls, SoSPTQSLBatchingQuantMatMul=cls))
    monkeypatch.setattr(RH, "load", lambda: ns)
    monkeypatch.setattr(RH, "_dev", lambda: "cpu")
    x, W, b, y, g = O.make_linear_fixture(1, 4, 20, 32, 48)
    s, units = RH.time_linear(x, W, b, y, g, False, eq_n=4, w_blocks=1, n_V=3, n_H=2, n_a=1, search_round=1)
    assert units == 8 and s > 0                      # one column block + one activation step, 4 candidates each
    assert made[-1].steps == ["w", "a"]
    s, units = RH.time_linear(x, W, b, y, g, False, eq_n=4, w_blocks=None, n_V=3, n_H=2, n_a=1, search_round=2)
    assert units == 2 * (2 + 1) * 4 and made[-1].steps == ["w", "w", "a"] * 2
    A, B, Y, Gr = O.make_matmul_fixture(2, 2, 3, 12, 8, 12)
    assert RH.time_matmul(A, B, Y, Gr, False, eq_n=4, search_round=1)[1] == 8
    As, Bs, Ys, Gs = O.make_matmul_fixture(3, 2, 3, 12, 12, 8, softmax_A=True)
    assert RH.time_matmul(As, Bs, Ys, Gs, True, eq_n=4, search_round=1)[1] == 24


def test_bench_unit_accounting_and_extrapolation():
    import bench
    a = argparse.Namespace(model="vit_base_patch16_224", images=32, blocks=24, rounds=3, bit=8)
    types = bench.layer_types(a)
    assert types["qkv"][2]["n_V"] == 72 and types["head"][2]["n_V"] == 1 and types["fc2"][1][2] is True
    total = sum(count * per for (_, _, _, count, per) in types.values())
    assert total == 49 * 7500 + 12 * 600 + 12 * 360        # SURVEY 8d: 367 500 Linear units + MatMul units
    v, job_s, rates = bench.extrapolate(a, {k: (1.0, 10.0) for k in types})
    assert abs(job_s - total / 10.0) < 1e-6 and abs(v - 10.0) < 1e-9
    assert bench.is_default_workload(a) and "n_V=n_H=24" in bench.workload_name(a)


def test_module_cost_uses_probed_shapes():
    from ptq4vit_b200.quant_layers import linear as L, matmul as M
    from ptq4vit_b200.utils import quant_calib as Q
    lin = L.PTQSLBatchingQuantLinear(128, 384, n_V=3, search_round=3)
    c1 = Q.module_cost(lin, 32, {"x": (1, 144, 128)}) - 3 * Q._ROUND_OVERHEAD_S
    c64 = Q.module_cost(lin, 32, {"x": (64, 144, 128)}) - 3 * Q._ROUND_OVERHEAD_S       # Swin: 64 windows per image fold into the leading dim
    assert abs(c64 / c1 - 64.0) < 1e-6
    mm = M.PTQSLBatchingQuantMatMul(search_round=3)
    cm = Q.module_cost(mm, 32, {"A": (64, 4, 144, 32), "B": (64, 4, 32, 144)})
    assert abs(cm - 3 * (Q._ROUND_OVERHEAD_S + 2 * 100 * 2.0 * 32 * 64 * 4 * 144 * 32 * 144 / Q._MATMUL_RATE)) < 1e-9
    # ViT-B/224 x 32 images at n_V = n_H = 24: the model reproduces the measured per-round times within 20 %
    qkv = L.PTQSLBatchingQuantLinear(768, 2304, n_V=72, n_H=24, search_round=1)
    qk = M.PTQSLBatchingQuantMatMul(search_round=1)
    assert abs(Q.module_cost(qkv, 32, {"x": (1, 197, 768)}) / 11.4e-3 - 1) < 0.2
    assert abs(Q.module_cost(qk, 32, {"A": (1, 12, 197, 64), "B": (1, 12, 64, 197)}) / 6.0e-3 - 1) < 0.2


@pytest.mark.parametrize("metric", ["L2_norm", "linear_weighted_L2_norm", "square_weighted_L2_norm"])
def test_weighted_l2_metrics_are_hessian_with_a_surrogate_weight(metric):
    """The product evaluates the reference's squared-error metrics (linear.py:411-416, matmul.py:467-472,
    conv.py:511-516) as the Hessian metric with a surrogate per-element weight (quant_layers/_metric.py).  The search
    with that weight (the oracle's restatement of the reference's Hessian search) must pick what the reference picks
    running the metric itself."""
    from ptq4vit_b200.quant_layers._metric import metric_weight
    z = G.load(f"metric_cpu_{metric}")
    x, W, b, y, g = O.make_linear_fixture(41, 4, 20, 32, 48)
    sp = O.LinearSpec(32, 48, eq_n=25, **{k: v for k, v in METRIC_LINEAR.items() if k != "eq_n"})
    w_int, a_int, log = O.linear_calibrate(sp, W, b, x, y, metric_weight(metric, y, None, "test").clone(), return_scores=True)
    assert np.array_equal(w_int.numpy().reshape(-1), z["lin_w_interval"].reshape(-1))
    assert np.array_equal(a_int.numpy().reshape(-1), z["lin_a_interval"].reshape(-1))
    ref = G.unpack_tables(z, "lin_s")
    mine = [t.numpy() for sw, sa in log for t in list(sw) + list(sa)]
    assert len(mine) == len(ref)
    for sd, (rows, scale, idx, val, best) in zip(mine, ref):
        assert float(np.abs(sd.reshape(rows, -1).astype(np.float64) - val).max() / scale) < 1e-5
    A, B, Y, Gr = O.make_matmul_fixture(42, 2, 3, 12, 8, 12)
    A_int, B_int, _ = O.matmul_calibrate(O.MatMulSpec(eq_n=25, search_round=1), A, B, Y, metric_weight(metric, Y, None, "test").clone())
    assert np.array_equal(torch.as_tensor(A_int).numpy().reshape(-1), z["mm_A_interval"].reshape(-1))
    assert np.array_equal(B_int.numpy().reshape(-1), z["mm_B_interval"].reshape(-1))
    xc, Wc, bc, yc, gc = O.make_conv_fixture(43, 2, 3, 8, 8, 4)
    wc, _ = O.conv_calibrate(Wc, bc, xc, yc, metric_weight(metric, yc, None, "test").clone(), stride=4, eq_n=25)
    assert np.array_equal(wc.numpy().reshape(-1), z["conv_w_interval"].reshape(-1))


def test_unsupported_metrics_raise_like_the_reference():
    from ptq4vit_b200.quant_layers._metric import metric_weight
    y = torch.ones(2, 3)
    for metric in ("cosine", "L1_norm", "pearson", "nonsense"):
        with pytest.raises(NotImplementedError):
            metric_weight(metric, y, None, "test")
    with pytest.raises(AssertionError):
        metric_weight("hessian", y, None, "test")

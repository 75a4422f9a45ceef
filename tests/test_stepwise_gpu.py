"""GPU: the step-wise Linear ABI (p4v_linear_begin, then per round p4v_linear_search_w over every column block and
p4v_linear_search_a over every activation chunk) computes exactly what the one-shot p4v_linear_calibrate computes: the
same step sizes and the same score log, bit for bit.  Both run the same search steps; the only difference is where the
scale tables of a step are built (by the select of the step before it, or at the start of a range), and both places
build them with the same code."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

ROUNDS, EQ_N = 2, 16


def _desc(post_gelu, M, tokens, K, O, n_V, n_H, n_a):
    from ptq4vit_b200 import _lib
    d = _lib.LinearDesc()
    fields = dict(rows=M, tokens=tokens, in_features=K, out_features=O, n_V=n_V, n_H=n_H, n_a=n_a, w_bit=8, a_bit=8,
                  eq_n=EQ_N, search_round=ROUNDS, eq_alpha=0.01, eq_beta=1.2, post_gelu=post_gelu, has_bias=1, operand=0,
                  kernel=0, init_layerwise=0)
    for k, v in fields.items():
        setattr(d, k, v)
    return d


def _sizes(lib, d):
    nbytes, nlog = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.p4v_linear_workspace_bytes(ctypes.byref(d), ctypes.byref(nbytes)) == 0, lib.p4v_last_error()
    assert lib.p4v_linear_score_log_floats(ctypes.byref(d), ctypes.byref(nlog)) == 0, lib.p4v_last_error()
    return nbytes.value, nlog.value


@pytest.mark.parametrize("post_gelu", [1, 0], ids=["post_gelu", "plain_slab_wsearch"])
def test_stepwise_matches_calibrate(post_gelu, monkeypatch):
    from ptq4vit_b200 import build, _lib
    build.build()
    if not post_gelu:
        monkeypatch.setenv("P4V_GRAM", "0")   # the step-wise W search runs the slab sweep; so must the one-shot call
    lib = _lib.lib()
    P = _lib.ptr
    M, tokens, K, O, n_V, n_H, n_a = 4 * 49, 49, 256, 128, 2, 4, 2
    d = _desc(post_gelu, M, tokens, K, O, n_V, n_H, n_a)
    gen = torch.Generator().manual_seed(7)
    x = torch.randn(M, K, generator=gen)
    if post_gelu:
        x = torch.nn.functional.gelu(x)
    W = torch.randn(O, K, generator=gen) / K ** 0.5
    b = 0.1 * torch.randn(O, generator=gen)
    y = x @ W.t() + b
    g = torch.randn(M, O, generator=gen) * 1e-3
    x, W, b, y, g = (t.cuda().contiguous() for t in (x, W, b, y, g))
    nbytes, nlog = _sizes(lib, d)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    w_one, a_one = torch.empty(n_V * n_H, device="cuda"), torch.empty(n_a, device="cuda")
    log_one = torch.full((nlog,), float("nan"), device="cuda")
    _lib.check(lib.p4v_linear_calibrate(ctypes.byref(d), P(x), P(W), P(b), P(y), P(g), P(ws), nbytes, P(w_one), P(a_one),
                                        P(log_one), st), "calibrate")

    ws2 = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    w_step, a_step = torch.empty(n_V * n_H, device="cuda"), torch.empty(n_a, device="cuda")
    log_step = torch.full((nlog,), float("nan"), device="cuda")
    _lib.check(lib.p4v_linear_begin(ctypes.byref(d), P(x), P(W), P(b), P(y), P(g), P(ws2), nbytes, st), "begin")
    per_w, per_round = n_H * EQ_N * n_V, n_H * EQ_N * n_V + n_a * EQ_N
    for e in range(ROUNDS):
        _lib.check(lib.p4v_linear_search_w(ctypes.byref(d), P(b), P(y), P(g), P(ws2), 0, n_H, P(log_step[e * per_round:]), st),
                   "search_w")
        _lib.check(lib.p4v_linear_search_a(ctypes.byref(d), P(b), P(y), P(g), P(ws2), 0, n_a,
                                           P(log_step[e * per_round + per_w:]), st), "search_a")
    _lib.check(lib.p4v_linear_intervals(ctypes.byref(d), P(ws2), P(w_step), P(a_step), st), "intervals")
    torch.cuda.synchronize()

    assert nlog == ROUNDS * per_round
    assert not torch.isnan(log_one).any() and not torch.isnan(log_step).any()
    assert torch.equal(w_step, w_one), (w_step, w_one)
    assert torch.equal(a_step, a_one), (a_step, a_one)
    assert torch.equal(log_step, log_one)
    assert log_one.unique().numel() > EQ_N      # real score tables, not a constant fill

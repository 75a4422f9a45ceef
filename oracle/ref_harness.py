"""Run the UNMODIFIED reference classes (TEST / BASELINE INFRASTRUCTURE ONLY).

Imports the reference's `quant_layers`, `utils.quant_calib`, `utils.net_wrap`, `configs.PTQ4ViT` from
oracle/_ref (staged by oracle/stage_ref.py) or straight from the tree named by $PTQ4VIT_REFERENCE.  `timm` is not installed offline: a stub module tree provides the two class names
`utils/models.py` imports.  On a machine without a GPU the reference's hard-coded `.cuda()` calls
(quant_layers/linear.py:391, :461-464; quant_layers/matmul.py:428, :493-498) are made the identity by a
harness-only shim; on a GPU the reference runs unmodified.

Score tables are captured by spying on argmax: every search step of the reference calls it exactly once on its
similarity table (linear.py:493, :531; matmul.py:520, :561, :626).

Only bench.py's reference legs, tests/golden/make_*.py and tests that need no reference tree import this file.
"""
import contextlib
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGED = os.path.join(ROOT, "oracle", "_ref")
_ref = None


def reference_path():
    if os.path.isdir(os.path.join(STAGED, "quant_layers")):
        return STAGED
    src = os.environ.get("PTQ4VIT_REFERENCE", "")
    if src and os.path.isdir(os.path.join(src, "quant_layers")):
        return src
    return None


def available():
    return reference_path() is not None


def _stub_timm():
    if "timm" in sys.modules:
        return
    timm = types.ModuleType("timm")
    models = types.ModuleType("timm.models")
    vt = types.ModuleType("timm.models.vision_transformer")
    st = types.ModuleType("timm.models.swin_transformer")

    class Attention(torch.nn.Module):          # placeholder types for the isinstance checks of utils/models.py:79-88
        pass

    class WindowAttention(torch.nn.Module):
        pass

    vt.Attention = Attention
    st.WindowAttention = WindowAttention
    models.vision_transformer = vt
    models.swin_transformer = st
    timm.models = models

    def create_model(*a, **k):
        raise RuntimeError("timm is a stub here (no network, no pretrained weights)")

    timm.create_model = create_model
    sys.modules.update({"timm": timm, "timm.models": models, "timm.models.vision_transformer": vt,
                        "timm.models.swin_transformer": st})


def cpu_shim():
    """No GPU: make the reference's `.cuda()` calls the identity (harness only)."""
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self
    torch.cuda.empty_cache = lambda: None


def load():
    """Returns a namespace with the reference modules: linear, matmul, conv, quant_calib, net_wrap, models, cfg, integer."""
    global _ref
    if _ref is not None:
        return _ref
    path = reference_path()
    if path is None:
        raise RuntimeError("reference tree not found: set $PTQ4VIT_REFERENCE or stage it with `python oracle/stage_ref.py`")
    if not torch.cuda.is_available():
        cpu_shim()
    _stub_timm()
    if path not in sys.path:
        sys.path.insert(0, path)
    # the reference's top-level package names are generic: make sure no foreign `utils` / `configs` shadows them
    for name in ("utils", "configs", "quant_layers"):
        m = sys.modules.get(name)
        if m is not None and not getattr(m, "__file__", "").startswith(path) and not any(
                p.startswith(path) for p in getattr(m, "__path__", [])):
            del sys.modules[name]
    import importlib
    ns = types.SimpleNamespace(path=path)
    ns.linear = importlib.import_module("quant_layers.linear")
    ns.matmul = importlib.import_module("quant_layers.matmul")
    ns.conv = importlib.import_module("quant_layers.conv")
    ns.quant_calib = importlib.import_module("utils.quant_calib")
    ns.models = importlib.import_module("utils.models")
    ns.net_wrap = importlib.import_module("utils.net_wrap")
    ns.integer = importlib.import_module("utils.integer")
    ns.cfg = importlib.import_module("configs.PTQ4ViT")
    ns.cfg_base = importlib.import_module("configs.BasePTQ")
    _ref = ns
    return ns


@contextlib.contextmanager
def capture_argmax(store):
    """Append every tensor an argmax is taken of (method and function form) to `store` (as CPU fp32)."""
    orig_m, orig_f = torch.Tensor.argmax, torch.argmax

    def spy_m(self, *a, **k):
        store.append(self.detach().float().cpu().clone())
        return orig_m(self, *a, **k)

    def spy_f(inp, *a, **k):
        store.append(inp.detach().float().cpu().clone())
        return orig_f(inp, *a, **k)

    torch.Tensor.argmax, torch.argmax = spy_m, spy_f
    try:
        yield store
    finally:
        torch.Tensor.argmax, torch.argmax = orig_m, orig_f


COMMON = dict(metric="hessian", eq_alpha=0.01, eq_beta=1.2, eq_n=100)


def _dev():
    return "cuda" if torch.cuda.is_available() else "cpu"


def run_linear(x, W, b, y, g, post_gelu=False, quant_forward=True, **mod):
    """PTQSLBatchingQuantLinear / PostGelu variant, calibration_step2() on the cached tensors (CPU tensors, as the
    reference's hooks leave them).  Returns dict(w_interval, a_interval, scores=[...], seconds, out)."""
    import time
    R = load()
    cls = R.linear.PostGeluPTQSLBatchingQuantLinear if post_gelu else R.linear.PTQSLBatchingQuantLinear
    kw = dict(COMMON); kw.update(mod)
    m = cls(W.shape[1], W.shape[0], bias=b is not None, **kw)
    m.weight.data = W.clone()
    if b is not None:
        m.bias.data = b.clone()
    m.to(_dev())
    m.raw_input, m.raw_out, m.raw_grad = x.cpu().clone(), y.cpu().clone(), g.cpu().clone()
    scores = []
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    t0 = time.time()
    with torch.no_grad(), capture_argmax(scores):
        m.calibration_step2()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    dt = time.time() - t0
    out = None
    if quant_forward:
        m.mode = "quant_forward"
        with torch.no_grad():
            out = m(x[:2].to(_dev())).float().cpu()
    return dict(w_interval=m.w_interval.detach().float().cpu(), a_interval=m.a_interval.detach().float().cpu(),
                scores=scores, seconds=dt, out=out, module=m)


def run_matmul(A, B, Y, G, sos=False, quant_forward=True, **mod):
    import time
    R = load()
    cls = R.matmul.SoSPTQSLBatchingQuantMatMul if sos else R.matmul.PTQSLBatchingQuantMatMul
    kw = dict(COMMON); kw.update(mod)
    m = cls(**kw)
    m.raw_input, m.raw_out, m.raw_grad = [A.cpu().clone(), B.cpu().clone()], Y.cpu().clone(), G.cpu().clone()
    scores = []
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    t0 = time.time()
    with torch.no_grad(), capture_argmax(scores):
        m.calibration_step2()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    dt = time.time() - t0
    out = None
    if quant_forward:
        m.mode = "quant_forward"
        with torch.no_grad():
            out = m(A[:2].to(_dev()), B[:2].to(_dev())).float().cpu()
    res = dict(A_interval=torch.as_tensor(m.A_interval).detach().float().cpu(), B_interval=m.B_interval.detach().float().cpu(),
               scores=scores, seconds=dt, out=out, module=m)
    if sos:
        res["split"] = torch.as_tensor(m.split).detach().float().cpu()
    return res


class ListLoader:
    """The minimum of a DataLoader the reference's calibrators touch: iteration and `.batch_size`
    (utils/quant_calib.py:131, :254, :333)."""

    def __init__(self, images, targets=None):
        self.images = images
        self.targets = targets if targets is not None else torch.zeros(images.shape[0], dtype=torch.long)
        self.batch_size = images.shape[0]

    def __iter__(self):
        yield self.images, self.targets

    def __len__(self):
        return 1


# ---------------------------------------------------------------- whole-calibrator harness (tiny synthetic ViT)
TINY_VIT = dict(img_size=32, patch=8, dim=64, depth=2, num_heads=2, num_classes=10)


def tiny_images(n=8, size=32, seed=3):
    return torch.randn(n, 3, size, size, generator=torch.Generator().manual_seed(seed))


def add_target_noise(net, n_img, n_cls, scale=1.0, seed=1234):
    """Harness-only: the reference computes its KL target from the FP32 net itself (utils/quant_calib.py:308-313), so
    on synthetic nets the loss gradient is pure round-off noise (SURVEY.md 8a).  A forward hook that perturbs the
    logits of the no-grad target pass -- and nothing else -- gives both implementations the same O(1e-2) gradients
    without touching the reference's code."""
    noise = torch.randn(n_img, n_cls, generator=torch.Generator().manual_seed(seed)) * scale

    def hook(mod, inp, out):
        if not torch.is_grad_enabled() and out.shape[0] == n_img:
            return out + noise.to(out.device)
        return None
    return net.register_forward_hook(hook)


def reference_wrapped_copy(net):
    """Deep copy of a ptq4vit_b200.utils.models net whose MatMul modules are the reference's class, wrapped by the
    reference's own utils/net_wrap.py with its configs/PTQ4ViT.py."""
    import copy
    import importlib
    R = load()
    net_r = copy.deepcopy(net)
    for mod in net_r.modules():
        for leaf in ("matmul1", "matmul2"):
            if hasattr(mod, leaf):
                setattr(mod, leaf, R.models.MatMul())
    importlib.reload(R.cfg)
    wrapped = R.net_wrap.wrap_modules_in_net(net_r, R.cfg)
    return net_r, wrapped


def run_reference_calibrator(net, images, batch_size=4, sequential=False, snapshot=None, cfg_edit=None):
    """HessianQuantCalibrator(...).batching_quant_calib() of the reference on a copy of `net`.
    Returns {name: {w_interval, a_interval | A_interval, B_interval, split}} (CPU tensors)."""
    R = load()
    if cfg_edit is not None:
        import importlib
        importlib.reload(R.cfg)
        cfg_edit(R.cfg)
        import copy
        net_r = copy.deepcopy(net)
        for mod in net_r.modules():
            for leaf in ("matmul1", "matmul2"):
                if hasattr(mod, leaf):
                    setattr(mod, leaf, R.models.MatMul())
        wrapped = R.net_wrap.wrap_modules_in_net(net_r, R.cfg)
    else:
        net_r, wrapped = reference_wrapped_copy(net)
    net_r.to(_dev()).eval()
    if snapshot is not None:
        for name, m in wrapped.items():
            orig = m.calibration_step2

            def spy(*a, _orig=orig, _m=m, _name=name, **k):
                d = {}
                if isinstance(_m.raw_input, (list, tuple)):
                    d["A"], d["B"] = _m.raw_input[0].clone(), _m.raw_input[1].clone()
                else:
                    d["x"] = _m.raw_input.clone()
                d["y"] = _m.raw_out.clone()
                d["g"] = _m.raw_grad.clone() if _m.raw_grad is not None else None
                snapshot[_name] = d
                return _orig(*a, **k)
            m.calibration_step2 = spy
    cal = R.quant_calib.HessianQuantCalibrator(net_r, wrapped, ListLoader(images), sequential=sequential, batch_size=batch_size)
    cal.batching_quant_calib()
    return collect_intervals(wrapped), net_r, wrapped


def collect_intervals(wrapped):
    out = {}
    for name, m in wrapped.items():
        d = {}
        for key in ("w_interval", "a_interval", "A_interval", "B_interval", "split"):
            v = getattr(m, key, None)
            if v is None:
                continue
            if isinstance(v, (list, tuple)):
                v = v[0]
            d[key] = torch.as_tensor(v).detach().float().cpu().reshape(-1).clone()
        out[name] = d
    return out


# ---------------------------------------------------------------- timing the reference (bench.py's reference legs)
class _StopSearch(Exception):
    pass


@contextlib.contextmanager
def _stop_after_argmax(n):
    """Interrupt the reference's greedy loop after its n-th argmax (= after n search steps)."""
    orig = torch.Tensor.argmax
    seen = [0]

    def spy(self, *a, **k):
        r = orig(self, *a, **k)
        seen[0] += 1
        if seen[0] >= n:
            raise _StopSearch()
        return r
    torch.Tensor.argmax = spy
    try:
        yield
    finally:
        torch.Tensor.argmax = orig


def _sync():
    if torch.cuda.is_available():
        torch.cuda.synchronize()


def time_linear(x, W, b, y, g, post_gelu, eq_n, w_blocks=None, **mod):
    """Seconds and candidate-GEMM units of the reference's Linear search on the given tensors (CPU tensors in, as its
    hooks leave them).  w_blocks=None: the whole `calibration_step2()` (search_round rounds); w_blocks=k: the unmodified
    `_search_best_w_interval` interrupted after k column blocks plus one full `_search_best_a_interval`
    (bounded sample for the CPU arm; the per-candidate work is the same in every column block)."""
    import time
    R = load()
    cls = R.linear.PostGeluPTQSLBatchingQuantLinear if post_gelu else R.linear.PTQSLBatchingQuantLinear
    kw = dict(COMMON); kw.update(mod); kw["eq_n"] = eq_n
    m = cls(W.shape[1], W.shape[0], bias=b is not None, **kw)
    m.weight.data = W.clone()
    if b is not None:
        m.bias.data = b.clone()
    m.to(_dev())
    m.raw_input, m.raw_out, m.raw_grad = x, y, g
    _sync(); t0 = time.perf_counter()
    with torch.no_grad():
        if w_blocks is None:
            m.calibration_step2()
            units = m.search_round * (m.n_H + m.n_a) * eq_n
        else:
            m._initialize_calib_parameters()
            m._initialize_intervals()
            f = torch.tensor([m.eq_alpha + i * (m.eq_beta - m.eq_alpha) / m.eq_n for i in range(m.eq_n + 1)]).to(m.w_interval.device)
            wc = f.view(-1, 1, 1, 1, 1) * m.w_interval.unsqueeze(0)          # linear.py:544
            ac = f.view(1, 1, -1) * m.a_interval.unsqueeze(-1)               # linear.py:545
            try:
                with _stop_after_argmax(w_blocks):
                    m._search_best_w_interval(wc)
            except _StopSearch:
                pass
            m._search_best_a_interval(ac)
            units = (min(w_blocks, m.n_H) + m.n_a) * eq_n
    _sync()
    return time.perf_counter() - t0, units


def time_matmul(A, B, Y, G, sos, eq_n, **mod):
    import time
    R = load()
    cls = R.matmul.SoSPTQSLBatchingQuantMatMul if sos else R.matmul.PTQSLBatchingQuantMatMul
    kw = dict(COMMON); kw.update(mod); kw["eq_n"] = eq_n
    m = cls(**kw)
    m.raw_input, m.raw_out, m.raw_grad = [A, B], Y, G
    _sync(); t0 = time.perf_counter()
    with torch.no_grad():
        m.calibration_step2()
    _sync()
    return time.perf_counter() - t0, m.search_round * ((20 if sos else eq_n) + eq_n)


def run_conv(x, W, b, y, g, stride, **mod):
    """ChannelwiseBatchingQuantConv2d(..., a_bit=32).calibration_step2() of the reference (conv.py:444-614)."""
    import time
    R = load()
    kw = dict(COMMON); kw.update(mod)
    oc, ic, kh, kwid = W.shape
    m = R.conv.ChannelwiseBatchingQuantConv2d(ic, oc, (kh, kwid), stride=stride, bias=b is not None, a_bit=32, **kw)
    m.weight.data = W.clone()
    if b is not None:
        m.bias.data = b.clone()
    m.to(_dev())
    m.raw_input, m.raw_out, m.raw_grad = x.cpu().clone(), y.cpu().clone(), g.cpu().clone()
    scores = []
    _sync(); t0 = time.perf_counter()
    with torch.no_grad(), capture_argmax(scores):
        m.calibration_step2()
    _sync()
    return dict(w_interval=m.w_interval.detach().float().cpu(), scores=scores, seconds=time.perf_counter() - t0, module=m)

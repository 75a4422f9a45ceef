#!/usr/bin/env python
"""bench.py -- candidate-GEMMs/s of the PTQ4ViT scale-factor search on B200.

A "step" = the full `calibration_step2` search of every wrapped Linear / MatMul of the workload
(default: ViT-B/224, 32 synthetic images, W8A8, n_V=n_H=24 (qkv 72, head 1), n_a=1, eq_n=100, 3 rounds, hessian
metric = BASELINE.json configs[2] at one bit width) over tensors already resident in HBM.
`value`   = candidate-GEMM units of ALL ranks / max-over-ranks device time.
`e2e`     = the same through the reference-facing call (`module.calibration_step2()`) with pinned HOST tensors,
            host<->device copies inside the timing.
`calib_wallclock` = the public `HessianQuantCalibrator(...).batching_quant_calib()` (capture + search + gather), the
            equivalent of what example/test_all.py:31-34 times.
`reference_gpu` = the UNMODIFIED reference classes (oracle/_ref) on the same GPU, one layer per type, one round.
`cpu_baseline` / `--impl reference` = the reference classes on the host cores (bounded sample, see below).

  python bench.py --gpus 1 --steps 3 --warmup 3
  torchrun ... bench.py --gpus N ...          (layer-sharded, one all_gather of the step sizes per step)
  python bench.py --impl reference            (reference on the host cores)
  python bench.py ... --dump-outputs DIR      (the step sizes of the last timed step as DIR/<module>.<name>.npy)
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                 # the tree may be read-only: nothing is written there
os.environ.setdefault("TQDM_DISABLE", "1")
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "NONE"          # keep stdout to the one JSON line (NCCL prints its version banner there)

import torch  # noqa: E402

UNIT = "cand-GEMM/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="vit_base_patch16_224")
    ap.add_argument("--images", type=int, default=32)
    ap.add_argument("--blocks", type=int, default=24, help="n_V = n_H of the Linear layers (BASELINE: 24; 1 = the reference's default)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--bit", type=int, default=8)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true")
    ap.add_argument("--no-wallclock", action="store_true")
    ap.add_argument("--cpu-eq-n", type=int, default=20, help="candidates per search step of the CPU reference sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the step sizes the last timed step chose, one float32 "
                    "DIR/<module>.<name>.npy per array, to compare two builds output for output")
    return ap.parse_args()


def metric_name(a):
    return f"candidate-GEMMs/s (scale-factor search, {a.model} {a.images}-img W{a.bit}A{a.bit})"


def workload_name(a):
    return (f"{a.model} {a.images} synthetic imgs W{a.bit}A{a.bit} n_V=n_H={a.blocks} (qkv x3, head 1) n_a=1 "
            f"eq_n=100 rounds={a.rounds} hessian")


def is_default_workload(a):
    return (a.model, a.images, a.blocks, a.rounds, a.bit) == ("vit_base_patch16_224", 32, 24, 3, 8)


# ------------------------------------------------------------------ unit accounting (SURVEY.md 8d)
def units_of(module):
    from ptq4vit_b200.quant_layers.conv import MinMaxQuantConv2d
    from ptq4vit_b200.quant_layers.linear import MinMaxQuantLinear
    if isinstance(module, MinMaxQuantConv2d):
        return module.eq_n            # the weight-only search is the same in every round: evaluated (and counted) once
    if isinstance(module, MinMaxQuantLinear):
        return module.search_round * (module.n_H + module.n_a) * module.eq_n
    return module.search_round * ((20 if module.sos else module.eq_n) + module.eq_n)


def model_dims(a):
    from ptq4vit_b200.utils.models import _ZOO
    z = _ZOO[a.model]
    tok = (z["img_size"] // z["patch"]) ** 2 + 1
    return z["dim"], z["num_heads"], tok, z["depth"]


# ------------------------------------------------------------------ workload construction
def build_workload(a, device, rank, world):
    """Synthetic ViT + one fwd/bwd capture sweep; returns the net, the wrapped modules and THIS rank's shard."""
    import importlib
    from ptq4vit_b200.configs import PTQ4ViT as cfg
    from ptq4vit_b200.utils import quant_calib as Q
    from ptq4vit_b200.utils.models import get_net
    from ptq4vit_b200.utils.net_wrap import wrap_modules_in_net
    importlib.reload(cfg)
    for d in (cfg.w_bit, cfg.a_bit, cfg.A_bit, cfg.B_bit):
        for k in d:
            d[k] = a.bit
    cfg.ptqsl_linear_kwargs.update(n_V=a.blocks, n_H=a.blocks, n_a=1, search_round=a.rounds)
    cfg.ptqsl_matmul_kwargs.update(search_round=a.rounds)
    net = get_net(a.model, device=device, seed=0)
    wrapped = wrap_modules_in_net(net, cfg)
    gen = torch.Generator().manual_seed(3)               # mirrors calib_loader(seed=3), utils/datasets.py:88
    size = 384 if "384" in a.model else 224
    images = torch.randn(a.images, 3, size, size, generator=gen).pin_memory()
    loader = [(images, None)]
    dist = None
    if world > 1:
        import torch.distributed as dist
    cal = Q.HessianQuantCalibrator(net, wrapped, loader, sequential=False, batch_size=4, target_noise=1.0, distributed=dist)
    names = list(wrapped.keys())
    mine, owner = cal._my_modules()
    if owner is None:
        owner = {n: 0 for n in names}
    raw = cal._raw_pred_softmax()
    hooks = []
    for n in mine:
        hooks += cal._hooks_for(wrapped[n])
    cal._fwd_bwd(raw)
    for h in hooks:
        h.remove()
    net.zero_grad(set_to_none=True)
    work = {}
    for n in mine:
        m = wrapped[n]
        Q._cat_captured(m)
        if isinstance(m.raw_input, list):
            t = dict(A=m.raw_input[0].contiguous(), B=m.raw_input[1].contiguous(), y=m.raw_out.contiguous(), g=m.raw_grad.contiguous())
        else:
            t = dict(x=m.raw_input.contiguous(), y=m.raw_out.contiguous(), g=m.raw_grad.contiguous())
        m.raw_input = m.raw_out = m.raw_grad = None
        work[n] = (m, t)
    torch.cuda.empty_cache()
    return net, wrapped, work, owner, names, cal


def dump_outputs(wrapped, out_dir):
    """The arrays calibration_step2() leaves on every wrapped module (w_interval, a_interval, A_interval, B_interval,
    split) as float32 .npy files."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, m in wrapped.items():
        for key in ("w_interval", "a_interval", "A_interval", "B_interval", "split"):
            v = getattr(m, key, None)
            if v is not None:
                arr = torch.as_tensor(v).detach().float().cpu().numpy()
                np.save(os.path.join(out_dir, f"{name}.{key}.npy"), arr)


def run_module(m, t):
    """One module's search through the reference-facing call, tensors already on the device."""
    if "x" in t:
        m.raw_input, m.raw_out, m.raw_grad = t["x"], t["y"], t["g"]
    else:
        m.raw_input, m.raw_out, m.raw_grad = [t["A"], t["B"]], t["y"], t["g"]
    with torch.no_grad():
        m.calibration_step2()


class ClockSampler:
    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------ the reference, timed (CPU arm and GPU comparator)
def layer_types(a):
    """One layer of every type of the workload: name -> (kind, shape spec, module kwargs, count in the model, units per layer)."""
    D, H, tok, depth = model_dims(a)
    nb = a.blocks
    lin = dict(n_H=nb, n_a=1, w_bit=a.bit, a_bit=a.bit)
    per_lin = a.rounds * (nb + 1) * 100
    types = {
        "qkv": ("linear", (D, 3 * D, False, tok), dict(lin, n_V=3 * nb), depth, per_lin),
        "proj": ("linear", (D, D, False, tok), dict(lin, n_V=nb), depth, per_lin),
        "fc1": ("linear", (D, 4 * D, False, tok), dict(lin, n_V=nb), depth, per_lin),
        "fc2": ("linear", (4 * D, D, True, tok), dict(lin, n_V=nb), depth, per_lin),
        "head": ("linear", (D, 1000, False, 0), dict(lin, n_V=1), 1, per_lin),
        "matmul1": ("matmul", (H, tok, D // H, tok, False), dict(A_bit=a.bit, B_bit=a.bit), depth, a.rounds * 200),
        "matmul2": ("matmul", (H, tok, tok, D // H, True), dict(A_bit=a.bit, B_bit=a.bit), depth, a.rounds * 120),
    }
    return types


def reference_rates(a, on_gpu, eq_n, only=None):
    """Times the reference classes (oracle/ref_harness -> oracle/_ref; falls back to the oracle port) on one seeded
    synthetic layer of every type at the workload's sizes.  GPU: the whole calibration_step2() of one round, eq_n=100,
    the reference's own H2D copies included.  CPU: eq_n candidates per search step, the weight search of a Linear layer
    interrupted after one column block (+ one activation step).  Returns {type: (seconds, units)} and the kind."""
    from oracle import ptq_oracle as O
    from oracle import ref_harness as RH
    kind = "reference" if RH.available() else "port"
    out = {}
    for i, (name, (k, shape, mod, count, per_layer)) in enumerate(layer_types(a).items()):
        if only and name not in only:
            continue
        if k == "linear":
            K, Oo, gelu, tok = shape
            x, W, b, y, g = O.make_linear_fixture(40 + i, a.images, tok, K, Oo, post_gelu=gelu)
            if kind == "reference":
                out[name] = RH.time_linear(x, W, b, y, g, gelu, eq_n, w_blocks=None if on_gpu else 1, search_round=1, **mod)
            else:
                out[name] = _port_linear(O, x, W, b, y, g, gelu, eq_n, on_gpu, mod)
        else:
            H, S1, S2, S3, sos = shape
            A, B, Y, G = O.make_matmul_fixture(60 + i, a.images, H, S1, S2, S3, softmax_A=sos)
            if kind == "reference":
                out[name] = RH.time_matmul(A, B, Y, G, sos, eq_n, search_round=1, **mod)
            else:
                out[name] = _port_matmul(O, A, B, Y, G, sos, eq_n, on_gpu, mod)
    return out, kind


def _port_linear(O, x, W, b, y, g, gelu, eq_n, on_gpu, mod):
    dev = "cuda" if on_gpu else "cpu"
    sp = O.LinearSpec(W.shape[1], W.shape[0], n_V=mod["n_V"], n_H=mod["n_H"], n_a=1, w_bit=mod["w_bit"], a_bit=mod["a_bit"],
                      eq_n=eq_n, search_round=1, post_gelu=gelu)
    x, W, b, y, g = [t.to(dev) for t in (x, W, b, y, g)]
    t0 = time.perf_counter()
    w_int, a_int = O.linear_initial_intervals(sp, W, x)
    f = O.candidate_factors(0.01, 1.2, eq_n).to(dev)
    wc = f.view(-1, 1, 1, 1, 1) * w_int.unsqueeze(0); ac = f.view(1, 1, -1) * a_int.unsqueeze(-1)
    hl = None if on_gpu else [0]
    O.linear_search_w(sp, W, b, x, y, g, w_int, a_int, wc, h_list=hl)
    O.linear_search_a(sp, W, b, x, y, g, w_int, a_int, ac)
    if on_gpu:
        torch.cuda.synchronize()
    return time.perf_counter() - t0, ((sp.n_H if on_gpu else 1) + 1) * eq_n


def _port_matmul(O, A, B, Y, G, sos, eq_n, on_gpu, mod):
    dev = "cuda" if on_gpu else "cpu"
    sp = O.MatMulSpec(A_bit=mod["A_bit"], B_bit=mod["B_bit"], eq_n=eq_n, search_round=1, sos=sos)
    A, B, Y, G = [t.to(dev) for t in (A, B, Y, G)]
    t0 = time.perf_counter()
    O.matmul_calibrate(sp, A, B, Y, G)
    if on_gpu:
        torch.cuda.synchronize()
    return time.perf_counter() - t0, (20 if sos else eq_n) + eq_n


def extrapolate(a, samples):
    """samples {type: (seconds, units)} -> (cand-GEMM/s of the whole job, job seconds, per-type rate)."""
    types = layer_types(a)
    total_units = total_s = 0.0
    rates = {}
    for name, (sec, units) in samples.items():
        k, shape, mod, count, per_layer = types[name]
        rates[name] = units / sec
        total_units += count * per_layer
        total_s += count * per_layer / rates[name]
    return total_units / total_s, total_s, rates


def physical_cores():
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def reference_cpu_main(a):
    """`--impl reference`: the reference's own classes on the host cores (harness-only `.cuda()` no-op shim so that
    the hard-coded device moves of the Batching classes stay on the CPU)."""
    from oracle import ref_harness as RH
    t_start = time.time()
    cores = physical_cores()
    torch.set_num_threads(cores)
    RH.cpu_shim()
    if hasattr(torch.cuda, "synchronize"):
        torch.cuda.is_available = lambda: False
    vals, per_step = [], []
    for i in range(a.warmup + a.steps):
        eq_n = 4 if i < a.warmup else a.cpu_eq_n           # warm-up: thread pools, allocator, first-touch of the fixtures
        samples, kind = reference_rates(a, on_gpu=False, eq_n=eq_n)
        v, job_s, rates = extrapolate(a, samples)
        if i >= a.warmup:
            vals.append(v)
            per_step.append({"value": round(v, 3), "job_s": round(job_s, 1), "sample_s": round(sum(s for s, _ in samples.values()), 2),
                             "rates": {k: round(r, 3) for k, r in rates.items()}})
    value = statistics.median(vals)
    sample = (f"{'unmodified reference classes (oracle/_ref)' if kind == 'reference' else 'oracle port'} on {cores} threads "
              f"(physical cores, torch.set_num_threads): one seeded synthetic layer per type (qkv, proj, fc1, fc2, head, matmul1, matmul2) at "
              f"the workload's sizes; Linear: one column block of the weight search + the activation search, {a.cpu_eq_n} candidates "
              f"each; MatMul: calibration_step2 with eq_n={a.cpu_eq_n}, one round; extrapolated by unit counts to the whole job; "
              f"median of {a.steps} step(s), spread {min(vals):.3f}..{max(vals):.3f}")
    out = {"impl": "reference", "metric": metric_name(a), "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
           "warmup": a.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": {"workload": workload_name(a)},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample,
                            "spread": [min(vals), max(vals)], "per_step": per_step},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": round(time.time() - t_start, 1)}
    print(json.dumps(out))


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if a.impl == "reference":
        if rank == 0:
            reference_cpu_main(a)
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist_.init_process_group("nccl", device_id=device)
        dist = dist_
    from ptq4vit_b200 import _lib
    lib = _lib.lib()

    net, wrapped, work, owner, names, cal = build_workload(a, device, rank, world)
    my_units = sum(units_of(m) for m, _ in work.values())
    units_t = torch.tensor([float(my_units)], device=device)
    if dist:
        dist.all_reduce(units_t)
    total_units = float(units_t.item())

    def gather():
        if dist:
            cal._gather(owner)

    def step():
        for m, t in work.values():
            run_module(m, t)
        gather()

    def sync_all():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        step()
    sync_all()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.p4v_profile_enable(1)
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(a.steps):
        step()
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    lib.p4v_profile_enable(0)
    prof = (ctypes.c_double * 12)()
    lib.p4v_profile_collect_kinds(prof, 12)
    launches = _lib.launch_count() - n0
    clocks = sampler.stop() if rank == 0 else None
    tmax = torch.tensor([ms], device=device)
    if dist:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax.item())
    value = total_units * a.steps / (ms / 1e3)
    if a.dump_outputs and rank == 0:
        dump_outputs(wrapped, a.dump_outputs)          # after the gather every rank holds every module's step sizes

    # ---- the public calibrator: capture + search + gather (what example/test_all.py:31-34 times)
    wallclock = None
    if not a.no_wallclock:
        runs = []
        for _ in range(2):
            for m in wrapped.values():
                if hasattr(m, "calibrated"):
                    del m.calibrated
                m.mode = "raw"
                m.raw_input = m.raw_out = m.raw_grad = None      # calibration_step2 deletes them (linear.py:554)
            sync_all()
            cal.batching_quant_calib()
            t = cal.timings
            tt = torch.tensor([t["total_s"], t["capture_s"], t["search_s"], t["gather_s"]], device=device, dtype=torch.float64)
            if dist:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            runs.append([float(v) for v in tt.tolist()])
        total_s, capture_s, search_s, gather_s = runs[-1]
        wallclock = {"total_s": total_s, "capture_s": capture_s, "search_s": search_s, "gather_s": gather_s,
                     "first_run_total_s": runs[0][0],
                     "what": "HessianQuantCalibrator(net, wrapped, loader, sequential=False, batch_size=4).batching_quant_calib(): "
                             "KL target pass, one forward+backward sweep with hooks on this rank's modules, search, all_gather; "
                             "max over ranks; images start in pinned host memory"}

    # ---- end to end through the public call with HOST (pinned) tensors
    e2e = None
    if not a.no_e2e:
        host = {}
        h2d = 0
        for n, (m, t) in work.items():
            host[n] = {k: v.cpu().pin_memory() for k, v in t.items()}
            h2d += sum(v.numel() * 4 for v in t.values())
        for n in work:
            work[n] = (work[n][0], None)
        torch.cuda.empty_cache()
        d2h = 0

        from ptq4vit_b200.utils.quant_calib import search_from_host
        items = [(m, host[n]) for n, (m, _) in work.items()]

        def e2e_step():
            # pinned host tensors -> (copy stream, one module ahead) -> search -> step sizes back to pinned host memory
            nonlocal d2h
            _, d2h = search_from_host(items, device)
            gather()

        e2e_step()
        sync_all()
        k_e2e = max(1, min(a.steps, 2))
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler2 = ClockSampler(local)
        if rank == 0:
            sampler2.start()
        f0.record()
        for _ in range(k_e2e):
            e2e_step()
        f1.record()
        sync_all()
        e2e_clocks = sampler2.stop() if rank == 0 else None
        ems = f0.elapsed_time(f1)
        et = torch.tensor([ems], device=device)
        hb = torch.tensor([float(h2d), float(d2h)], device=device)
        if dist:
            dist.all_reduce(et, op=dist.ReduceOp.MAX); dist.all_reduce(hb)
        e2e = {"value": total_units * k_e2e / (float(et.item()) / 1e3), "unit": UNIT,
               "h2d_bytes_per_step": int(hb[0].item()), "d2h_bytes_per_step": int(hb[1].item()), "steps": k_e2e,
               "ms_per_step": float(et.item()) / k_e2e, "clocks": e2e_clocks}
        del host, items

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    # ---- roofline: per launch kind against its own peak
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    bf16_peak = peaks.get("bf16_tflops_sustained") or 1400.0
    bf16_burst = peaks.get("bf16_tflops") or 1700.0
    peak_src = "MEASURED_PEAKS.json (cuBLAS bf16: sustained inside a long step, burst for a launch alone)" if peaks else \
        "fallback 1.4 / 1.7 PFLOP/s (B200_PROFILING.md)"
    kinds = ["sweep_bf16", "sweep_int8", "gram_gemm"]
    kernels = {"sweep_bf16": "sweep_tc_kernel<f32 accumulators>", "sweep_int8": "sweep_tc_kernel<s32 accumulators>", "gram_gemm": "gram_gemm_kernel"}
    by_kind = {}
    for i, k in enumerate(kinds):
        t_ms, ops, n = prof[i], prof[3 + i], int(prof[6 + i])
        if n == 0:
            continue
        pk = bf16_peak * (2.0 if k == "sweep_int8" else 1.0)
        ach = ops / (t_ms / 1e3) / 1e12
        by_kind[k] = {"kernel": kernels[k], "ms": t_ms, "launches": n, "avg_launch_ms": t_ms / n, "share_of_step": t_ms / ms,
                      "achieved": ach, "peak": pk, "frac": ach / pk, "unit": "TOP/s" if k == "sweep_int8" else "TFLOP/s"}
    dom = max(by_kind, key=lambda k: by_kind[k]["ms"])
    top_kind = kinds[int(prof[11])]
    top_peak = bf16_burst * (2.0 if top_kind == "sweep_int8" else 1.0)
    top_ach = prof[10] / (prof[9] / 1e3) / 1e12 if prof[9] > 0 else 0.0
    # DRAM bytes (read + write) of the longest launch from this round's `ncu --set full` capture (profiles/): a measured
    # constant of the DEFAULT workload, omitted for any other arguments
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if is_default_workload(a):
            traffic = tr.get("dominant_launch_dram_bytes")
    except Exception:
        tr = {}
    roofline = {"bound": "tensor", "kernel": by_kind[dom]["kernel"], "achieved": by_kind[dom]["achieved"], "peak": by_kind[dom]["peak"],
                "unit": by_kind[dom]["unit"], "frac": by_kind[dom]["frac"], "traffic": traffic,
                "traffic_note": tr.get("note") if traffic is not None else "ncu DRAM bytes are recorded for the default workload only",
                "by_kind": by_kind,
                "longest_launch": {"kind": top_kind, "ms": prof[9], "achieved": top_ach, "peak": top_peak, "frac": top_ach / top_peak,
                                   "peak_is": "burst (a launch timed alone)",
                                   "traffic": tr.get("longest_launch_dram_bytes") if traffic is not None else None},
                "note": "achieved = EXECUTED tensor-core operations (slab-incremental search: only the K segment a candidate changes is "
                        "multiplied; Gram GEMM: three bf16 term products) / CUDA-event time of the launches of that kind on this rank; "
                        "peak = " + peak_src + "; int8 launches are held against 2x the measured bf16 rate (stated, not measured: "
                        "MEASURED_PEAKS.json has no int8 figure)"}
    out = {"metric": metric_name(a), "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
           "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "int8/bf16-int operands, s32/f32 accumulate, f32 error", "data": "synthetic",
           "config": {"workload": workload_name(a), "parallelism": f"layer-sharded x{world}", "units_per_step": total_units,
                      "l2": "inputs (the staged tensors of a step, 9.5 GB for the default workload) are larger than L2; no explicit flush"},
           "calib_search_wallclock_s": ms / a.steps / 1e3,
           "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline}
    if wallclock:
        out["calib_wallclock_s"] = wallclock["total_s"]
        out["calib_wallclock"] = wallclock
    if e2e:
        out["e2e"] = e2e
    if dist:
        dist.destroy_process_group()
    del work
    torch.cuda.empty_cache()
    from ptq4vit_b200.utils.models import _ZOO
    if a.model not in _ZOO:          # the reference legs below are laid out for the ViT / DeiT layer types
        a.no_ref_gpu = a.no_cpu = True
    if world == 1 and not a.no_ref_gpu:
        try:
            samples, kind = reference_rates(a, on_gpu=True, eq_n=100)
            samples, kind = reference_rates(a, on_gpu=True, eq_n=100)          # second pass: warm allocator / cuBLAS handles
            v, job_s, rates = extrapolate(a, samples)
            out["reference_gpu"] = {"value": v, "unit": UNIT, "kind": kind, "extrapolated_full_job_s": job_s,
                                    "per_type_units_per_s": {k: round(r, 1) for k, r in rates.items()},
                                    "per_type_s_one_round": {k: round(s, 3) for k, (s, _) in samples.items()},
                                    "sample": "the reference's own eager GPU path (calibration_step2 of the unmodified classes, CPU-resident "
                                              "captured tensors as its hooks leave them) on this GPU: one seeded synthetic layer per type at the "
                                              "workload's sizes, one search round, eq_n=100; extrapolated by unit counts",
                                    "speedup_device": value / v, "speedup_e2e": (e2e["value"] / v) if e2e else None}
        except Exception as exc:   # the comparator must never take the bench line down
            out["reference_gpu"] = {"unavailable": repr(exc)[:200]}
    if world == 1 and not a.no_cpu:
        try:
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1",
                   "--model", a.model, "--images", str(a.images), "--blocks", str(a.blocks), "--rounds", str(a.rounds),
                   "--bit", str(a.bit), "--cpu-eq-n", str(a.cpu_eq_n)]
            env = dict(os.environ); env["CUDA_VISIBLE_DEVICES"] = ""
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
            out["cpu_baseline"] = json.loads(line)["cpu_baseline"]
        except Exception as exc:
            out["cpu_baseline"] = {"unavailable": repr(exc)[:200]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()

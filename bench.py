#!/usr/bin/env python
"""bench.py — RK4 sample-steps/sec of the closed-loop rollout (BASELINE.json metric) on N B200s of one box.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload swarm50|swap12|singlequad|...] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one OCflow call (mean mode) over one batch of synthetic initial states drawn from the problem's initial
distribution (SURVEY.md 8d).  The DEFAULT workload is the north_star's target shape, BASELINE.json configs[3]: the swarm50
pretrained checkpoint (d = 150, m = 512), nt = 80, fp32 — on a 2^22-sample sub-batch of its 2^24 samples (one step of the
full batch takes ~24 s on one GPU; the sub-sampling is stated in `config.workload`).  With --gpus N (torchrun) the SAME
total batch is row-sharded over the ranks — strong scaling, as configs[3] shards its 16M samples over 1/2/4/8 GPUs — and a
step ends with the single all-reduce of the 8-double cost vector; `weak` in the JSON line is the second figure (fixed samples
per GPU).  Other workloads (`--workload`) keep per-GPU sizes (weak scaling).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput of the whole job; `e2e` = the same metric through the
public API with HOST (pinned) buffers, copies inside the timed region; `roofline` = the rollout kernel of one launch against
its roof (tensor kernels: executed MMA flops / MEASURED_PEAKS.json bf16 peak, with the algorithmic fp32 rate / live-measured
FMA peak alongside; FMA kernels: algorithmic flops / live-measured FMA peak); `cpu_baseline` = the CPU oracle port (torch CPU,
all host threads) on a bounded sample of the same workload; `extra` = the full-size configs[1] (swap12, 2^20) and configs[2]
(singlequad, 2^22) lines and two training-iteration lines (`--train`), N = 1 only.
`--impl reference` times only the CPU arm (the reference is pure Python/torch and cannot travel to the GPU box;
oracle/ocflow_oracle.py is its restatement, pinned against the reference's outputs in tests/).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402
import torch         # noqa: E402

DEFAULT_WORKLOAD = "swarm50"
# n = samples per GPU (weak) or in total (strong); flops/sample-step = 4 (4 m D + 4 m^2 (nTh-1) + min(2 D^2, 4 r D))
WORKLOADS = {
    "softcorridor": dict(ckpt="softcorridor", n=1 << 20, nt=50, dtype="f32", n_cpu=65536, scaling="weak"),
    "swap2": dict(ckpt="swap2", n=1 << 20, nt=50, dtype="f32", n_cpu=65536, scaling="weak"),
    "swap12": dict(ckpt="swap12", n=1 << 20, nt=50, dtype="f32", n_cpu=65536, scaling="weak"),
    "singlequad": dict(ckpt="singlequad", n=1 << 22, nt=50, dtype="f32", n_cpu=32768, scaling="weak"),
    # configs[3]: 2^24 samples sharded over the GPUs; the bench steps over a 2^22-sample sub-batch of it (strong scaling)
    "swarm50": dict(ckpt="swarm50", n=1 << 22, nt=80, dtype="f32", n_cpu=256, scaling="strong", full_n=1 << 24),
    "config5": dict(ckpt=None, n=1 << 20, nt=50, dtype="f64", n_cpu=256, scaling="weak"),
}


def load_ckpt(name):
    """state_dict + run arguments of a pretrained checkpoint from the committed fixtures (tests/golden/ckpt/*.npz, written from
    the reference's .pth files by tests/golden/make_golden.py; /root/reference does not exist on the GPU box)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "ckpt", name + ".npz"))
    meta = json.loads(str(z["meta_json"]))
    sd = {k: torch.from_numpy(z[k]) for k in z.files if k != "meta_json"}
    return sd, meta


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def dram_bytes_per_sample(workload, path):
    """DRAM bytes per sample of the rollout kernel from this round's `ncu --set full` captures (profiles/r02_dram_traffic.json,
    written by scripts/ncu_traffic.py from the .ncu-rep files: dram__bytes_read.sum + dram__bytes_write.sum / samples)."""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "r02_dram_traffic.json")))
        e = tab.get("%s:%s" % (workload, path))
        return (float(e["bytes_per_sample"]), e.get("source")) if e else (None, None)
    except Exception:
        return None, None


def tensor_flops_per_sample_step(workload, d, m):
    """16-bit tensor-core flops the tcgen05 kernels EXECUTE per sample-step, and what they are.
    noc_tc_rollout.cuh (m <= 128): 4 evaluations x 3 split products (fp16 x 2) x 2 flops x the padded GEMM volumes
    KS*mp + 2*mp*mp + mp*KS + KS*KS (KS = d+2 rounded up to 16; mp = m padded to 64 for the quadcopter shape, 16 otherwise).
    noc_ts_rollout.cuh (swarm50): 4 evaluations x 3 split products (fp16 x 2) x 2 flops x (2*KS*512 + 2*512*512 + KS*KS), KS = 160."""
    if d == 150:
        ks, mp = 160, 512
        return 4 * 3 * 2 * (2 * ks * mp + 2 * mp * mp + ks * ks), "rollout_ts_kernel (tcgen05 cta_group::2, fp16 x 2 split: 3 MMAs per fp32 product, TMA-streamed weights)"
    ks = -(-(d + 2) // 16) * 16
    pad = 64 if workload == "singlequad" else 16
    mp = -(-m // pad) * pad
    return 4 * 3 * 2 * (ks * mp + 2 * mp * mp + mp * ks + ks * ks), "rollout_tc_kernel (tcgen05, fp16 x 2 split: 3 MMAs per fp32 product)"


def flops_per_sample_step(d, m, nTh, r):
    D = d + 1
    return 4 * (4 * m * D + 4 * m * m * (nTh - 1) + min(2 * D * D, 4 * r * D))


def roofline(workload, W, d, meta, n, nt, fl, step_s, fma_peak, path, clocks):
    """Roofline of the rollout kernel of ONE launch (n = samples of this GPU's launch).  Tensor-core kernels: the 16-bit MMA
    flops they execute against MEASURED_PEAKS.json's dense bf16 figure — the burst figure when the step ran at full SM clocks,
    the sustained one when the clocks sagged under the power cap — with the algorithmic fp32-equivalent rate and its ratio to the
    FP32 FMA peak (measured live) alongside.  FMA kernels: algorithmic flops against the live FMA peak."""
    alg = n * nt * fl / step_s / 1e12
    bps, src = dram_bytes_per_sample(workload, path)
    traffic = bps * n if bps is not None else None
    note = ("DRAM bytes per launch = bytes per sample of this round's ncu capture (%s) x samples; algorithmic = %d bytes "
            "(4 d per sample: the initial state is read once, mean mode writes nothing per sample)" % (src, 4 * d * n))
    if path == "tensor":
        peaks = measured_peaks()
        full_clock = bool(clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and clocks["sm_mhz"] >= 0.95 * clocks["sm_max_mhz"])
        key = "bf16_tflops" if full_clock else "bf16_tflops_sustained"
        tpeak = float(peaks.get(key, 0) or 0)
        psrc = "MEASURED_PEAKS.json %s (%s)" % (key, "SM clocks at max during the timed steps" if full_clock else "SM clocks below max during the timed steps")
        if not tpeak:
            tpeak, psrc = 1590.0, "B200_PROFILING.md fallback 1.59 PFLOP/s (MEASURED_PEAKS.json absent)"
        ex, kern = tensor_flops_per_sample_step(workload, d, meta["m"])
        ach = n * nt * ex / step_s / 1e12
        return {"bound": "tensor", "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak, "traffic": traffic,
                "traffic_note": note, "peak_source": psrc, "kernel": kern, "executed_flops_per_sample_step": ex,
                "algorithmic_fp32_tflops": alg, "fp32_fma_peak_tflops": fma_peak, "algorithmic_over_fma_peak": alg / fma_peak}
    return {"bound": "fp32_fma" if W["dtype"] == "f32" else "fp64_fma", "achieved": alg, "peak": fma_peak, "unit": "TFLOP/s",
            "frac": alg / fma_peak, "traffic": traffic, "traffic_note": note, "kernel": "rollout_kernel (FMA sample tiles)",
            "peak_source": "measured live: register-resident FMA micro-benchmark on all SMs (noc_measure_fma_peak); "
                           "MEASURED_PEAKS.json has no FP32/FP64 FMA figure"}


def build_case(workload, device, dtype):
    """-> net, prob, xInit (on device), meta — from committed fixtures only (no /root/reference, no test helpers)."""
    import neuraloc_b200 as nb
    w = WORKLOADS[workload]
    cvt = lambda v: v.to(dtype).to(device)
    if w["ckpt"] is None:       # BASELINE.json configs[4]: random-init swarm50-shape Phi
        alph = [1800.0, 1e7, 25000.0, 2.0, 1.0, 3.0]
        torch.manual_seed(0)
        net = nb.Phi(nTh=2, m=512, d=150, alph=alph)
        meta = dict(data="swarm50", alph=alph, var0=0.1, m=512, nTh=2)
    else:
        sd, meta = load_ckpt(w["ckpt"])
        net = None
    prob, x0, _, xinit = nb.initProb(meta["data"], 2, 2, var0=1.0, alph=meta["alph"], cvt=cvt)
    prob.eval()
    if net is None:
        net = nb.Phi(nTh=meta["nTh"], m=meta["m"], d=x0.shape[1], alph=meta["alph"])
        net.load_state_dict(sd)
    net = net.to(dtype).to(device)
    net.eval()
    return net, prob, xinit, meta


def sample_x(workload, xinit, var0, n, seed, device, dtype):
    """x ~ rho_0 of the problem (SURVEY.md 8d): xInit + var0 N(0,I); singlequad perturbs the position only."""
    g = torch.Generator(device=device).manual_seed(seed)
    d = xinit.shape[1]
    if workload == "singlequad":
        x = torch.zeros(n, d, device=device, dtype=dtype)
        x[:, :3] = -1.5 + var0 * torch.randn(n, 3, generator=g, device=device, dtype=dtype)
        return x
    x = torch.randn(n, d, generator=g, device=device, dtype=dtype)
    x.mul_(var0).add_(xinit.to(device))
    return x


def cpu_rate(workload, n_cpu, nt, dtype, threads):
    """sample-steps/s of the CPU oracle port on a bounded sample (one small warm-up call, one timed call)."""
    from oracle import ocflow_oracle as orc
    w = WORKLOADS[workload]
    torch.set_num_threads(threads)
    if w["ckpt"] is None:
        import neuraloc_b200 as nb
        alph = [1800.0, 1e7, 25000.0, 2.0, 1.0, 3.0]
        torch.manual_seed(0)
        sd = nb.Phi(nTh=2, m=512, d=150, alph=alph).state_dict()
        meta = dict(data="swarm50", alph=alph, var0=0.1)
    else:
        sd, meta = load_ckpt(w["ckpt"])
    P = orc.params_from_state_dict(sd, dtype)
    D, xinit = orc.make_problem(meta["data"], meta["alph"], dtype)
    x = sample_x(workload, xinit, meta["var0"], n_cpu, 1234, "cpu", dtype)
    with torch.no_grad():
        orc.ocflow(x[: max(1, n_cpu // 16)], P, D, [0.0, 1.0], nt, "rk4", meta["alph"])
        t0 = time.perf_counter()
        orc.ocflow(x, P, D, [0.0, 1.0], nt, "rk4", meta["alph"])
        dt = time.perf_counter() - t0
    return n_cpu * nt / dt, dt


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU while the timed region runs (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin, t_end):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, pw, reasons = [], None, [], set()
        for t, line in self.rows:
            f = [v.strip() for v in line.split(",")]
            if len(f) < 7:
                continue
            try:
                clk, mx = float(f[0]), float(f[1])
            except ValueError:
                continue
            smax = mx
            if t_begin - 0.05 <= t <= t_end + 0.05:
                sm.append(clk)
                try:
                    pw.append(float(f[2]))
                except ValueError:
                    pass
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:       # region shorter than the sampling period: use whatever was seen
            sm = [float(l.split(",")[0]) for _, l in self.rows if l and l.split(",")[0].strip().replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(pw) if pw else None}


def latency_mode(workload, W, dtype, threads):
    """Batch-1 rollout latency: ONE OCflow(xInit) call, wall clock, CPU tensors in and out — the protocol of
    timeDeployment/timeOC.py:76-81 (nt = 50; 80 for swarm50 as in README.md:85) — beside the CPU oracle port timed on
    one thread (the published numbers were taken under `taskset -c 0`, README.md:152-155)."""
    import neuraloc_b200 as nb
    from oracle import ocflow_oracle as orc
    nb._cabi.lib()
    torch.cuda.set_device(0)
    nt = W["nt"]
    net, prob, xinit, meta = build_case(workload, torch.device("cpu"), dtype)      # CPU tensors, like timeOC.py
    alph = meta["alph"]
    with torch.no_grad():
        for _ in range(5):
            nb.OCflow(xinit, net, prob, [0.0, 1.0], nt, "rk4", alph)
        wall = []
        for _ in range(200):
            t0 = time.perf_counter()
            Jc, cs = nb.OCflow(xinit, net, prob, [0.0, 1.0], nt, "rk4", alph)        # H2D + rollout + D2H + sync inside
            wall.append(time.perf_counter() - t0)
        xd = xinit.cuda()
        netd = net.cuda()
        ev = []
        for _ in range(100):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); nb.ocflow_sums(xd, netd, prob, [0.0, 1.0], nt, "rk4", alph); e1.record()
            ev.append((e0, e1))
        torch.cuda.synchronize()
        dev_ms = statistics.median(a.elapsed_time(b) for a, b in ev)
        # CPU oracle port, one thread
        torch.set_num_threads(1)
        if W["ckpt"] is None:
            sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        else:
            sd, _ = load_ckpt(W["ckpt"])
        P = orc.params_from_state_dict(sd, dtype)
        D, xi = orc.make_problem(meta["data"], alph, dtype)
        orc.ocflow(xi, P, D, [0.0, 1.0], nt, "rk4", alph)
        cpu = []
        for _ in range(5):
            t0 = time.perf_counter()
            Jr, _ = orc.ocflow(xi, P, D, [0.0, 1.0], nt, "rk4", alph)
            cpu.append(time.perf_counter() - t0)
        torch.set_num_threads(threads)
    line = {"metric": "batch1_rollout_latency", "value": statistics.median(wall) * 1e3, "unit": "ms", "n_gpus": 1,
            "higher_is_better": False, "dtype": W["dtype"], "data": "xInit of the problem",
            "config": {"workload": "%s, one OCflow(xInit) call, nt=%d, CPU tensors in/out (timeOC.py:76-81)" % (workload, nt)},
            "host_wall_ms": {"median": statistics.median(wall) * 1e3, "p10": sorted(wall)[20] * 1e3, "p90": sorted(wall)[180] * 1e3},
            "device_ms_median": dev_ms, "ms_per_rk4_step": statistics.median(wall) * 1e3 / nt,
            "cpu_baseline": {"value": statistics.median(cpu) * 1e3, "unit": "ms", "cores": 1, "kind": "port",
                             "sample": "median of 5 warm calls of the torch-CPU oracle port, 1 thread"},
            "Jc": float(Jc), "Jc_cpu": float(Jr)}
    return line


def intermediates_mode(args, W, dtype):
    """OCflow(..., intermediates=True) on a device-resident batch: zFull [n,d+4,nt+1] and ctrlFull [n,nCtrl,nt+1] are written
    to HBM (5 grad-Phi evaluations per step instead of 4).  Reports sample-steps/s and the output bandwidth against the measured
    HBM copy bandwidth."""
    import neuraloc_b200 as nb
    nb._cabi.lib()
    torch.cuda.set_device(0)
    device = torch.device("cuda", 0)
    n, nt = (args.n or min(W["n"], 1 << 16 if args.workload == "swarm50" else 1 << 18)), W["nt"]
    net, prob, xinit, meta = build_case(args.workload, device, dtype)
    x = sample_x(args.workload, xinit, meta["var0"], n, 1234, device, dtype)
    with torch.no_grad():
        for _ in range(max(1, args.warmup)):
            zf, cf = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            zf, cf = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
    out_bytes = (zf.numel() + cf.numel()) * zf.element_size()
    t = statistics.mean(ms) * 1e-3
    hbm = float(measured_peaks().get("hbm_gbs", 0) or 6650.0)
    return {"metric": "rk4_sample_steps_per_sec_intermediates", "value": n * nt / t, "unit": "sample-steps/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": statistics.mean(ms), "dtype": W["dtype"],
            "config": {"workload": "%s, intermediates=True, %d samples, nt=%d, kernel path %s" % (args.workload, n, nt, nb._cabi.last_path())},
            "output_bytes": out_bytes, "output_GBps": out_bytes / t / 1e9,
            "roofline": {"bound": "hbm", "achieved": out_bytes / t / 1e9, "peak": hbm, "unit": "GB/s", "frac": out_bytes / t / 1e9 / hbm,
                         "note": "peak = MEASURED_PEAKS.json hbm_gbs (copy: read + write); algorithmic bytes = the two output tensors, written once"}}


# the reference's own training commands (README.md:103-123): batch size and time steps of one trainOC.py iteration
TRAIN = {"softcorridor": (1024, 20), "swap2": (1024, 20), "swap12": (2048, 20), "swarm50": (1024, 26), "singlequad": (1024, 26),
         "config5": (1024, 26)}


def train_mode(args, W, dtype, threads):
    """One training evaluation, trainOC.py:169-173: Jc, cs = OCflow(x0, net, prob, ...) in train mode, then Jc.backward() —
    here ONE fused kernel (forward sweep + discrete adjoint, noc_ocflow_grad) behind the same two Python calls.  Batch size and
    nt are those of the reference's README training commands.  CPU arm: autograd through the oracle port on all host threads."""
    import neuraloc_b200 as nb
    nb._cabi.lib()
    torch.cuda.set_device(0)
    device = torch.device("cuda", 0)
    n, nt = TRAIN[args.workload]
    n = args.n or n
    net, prob, xinit, meta = build_case(args.workload, device, dtype)
    prob.train(); net.train()
    x = sample_x(args.workload, xinit, meta["var0"], n, 1234, device, dtype)
    params = list(net.parameters())

    def iteration():
        for p in params:
            p.grad = None
        Jc, cs = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"])
        Jc.backward()
        return Jc
    for _ in range(max(3, args.warmup)):
        Jc = iteration()
    torch.cuda.synchronize()
    before = nb._cabi.launch_count()
    ms = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        Jc = iteration()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    launches = nb._cabi.launch_count() - before
    t = statistics.mean(ms) * 1e-3
    gnorm = float(torch.sqrt(sum((p.grad.double() ** 2).sum() for p in params)))
    # forward flops (SURVEY 8d) x (1 forward + 4 stages re-evaluated with 8 instead of 4 contractions + 4 rank-TS updates)
    d, m = x.shape[1], meta["m"]
    fl = flops_per_sample_step(d, m, 2, min(10, d + 1))
    import ctypes
    pk = ctypes.c_double(0.0)
    nb._cabi.check(nb._cabi.lib().noc_measure_fma_peak(0 if W["dtype"] == "f32" else 1, ctypes.byref(pk)))
    line = {"metric": "train_sample_steps_per_sec", "value": n * nt / t, "unit": "sample-steps/s (forward + backward)", "n_gpus": 1,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": statistics.mean(ms), "higher_is_better": True,
            "dtype": W["dtype"], "data": "synthetic",
            "config": {"workload": "%s, one trainOC.py iteration (OCflow in train mode + Jc.backward()), n_train=%d, nt=%d "
                                   "(README.md:103-123), x ~ xInit + var0*N(0,I)" % (args.workload, n, nt),
                       "Jc": float(Jc.detach()), "grad_norm": gnorm},
            "gpu_launches": launches,
            "roofline": {"bound": "fp32_fma" if W["dtype"] == "f32" else "fp64_fma", "unit": "TFLOP/s",
                         "achieved": 4.0 * fl * n * nt / t / 1e12, "peak": pk.value, "frac": 4.0 * fl * n * nt / t / 1e12 / pk.value,
                         "kernel": "rollout_grad_kernel (FMA panels, one launch per iteration)",
                         "peak_source": "measured live: register-resident FMA micro-benchmark on all SMs (noc_measure_fma_peak)",
                         "note": "algorithmic flops of forward + adjoint = 4 x the forward's (8 instead of 4 contractions per "
                                 "re-evaluated stage + the parameter-gradient outer products) / time; FMA kernel"}}
    if not args.no_cpu_baseline:
        from oracle import ocflow_oracle as orc
        import dataclasses
        torch.set_num_threads(threads)
        sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        P = orc.params_from_state_dict(sd, dtype)
        D, _ = orc.make_problem(meta["data"], meta["alph"], dtype)
        D = dataclasses.replace(D, training=True)
        leaves = [t.clone().requires_grad_(True) for t in (P.A, P.c_w, P.c_b, P.w, P.K[0], P.K[1], P.b[0], P.b[1])]
        Pg = orc.PhiParams(leaves[0], leaves[1], leaves[2], leaves[3], [leaves[4], leaves[5]], [leaves[6], leaves[7]], P.h)
        xc = x.cpu()
        best, Jr = 1e30, None
        for _ in range(2):
            for t_ in leaves:
                t_.grad = None
            t0 = time.perf_counter()
            Jr, _ = orc.ocflow(xc, Pg, D, [0.0, 1.0], nt, "rk4", meta["alph"])
            Jr.backward()
            best = min(best, time.perf_counter() - t0)
        gn = float(torch.sqrt(sum((t_.grad.double() ** 2).sum() for t_ in leaves)))
        line["cpu_baseline"] = {"value": n * nt / best, "unit": "sample-steps/s (forward + backward)", "cores": threads, "kind": "port",
                                "ms_per_iteration": best * 1e3, "Jc": float(Jr.detach()), "grad_norm": gn,
                                "sample": "the same batch (n=%d, nt=%d), torch autograd through the oracle port, best of 2" % (n, nt)}
    return line


def measure(workload, n, steps, warmup, device, dtype, dist, rank, world, seed_rank, want_clocks, e2e_steps):
    """Device-timed rollout steps over this rank's n samples (+ the e2e leg with host buffers).  Returns a dict of raw numbers."""
    import neuraloc_b200 as nb
    W = WORKLOADS[workload]
    nt = W["nt"]
    net, prob, xinit, meta = build_case(workload, device, dtype)
    d = xinit.shape[1]
    x = sample_x(workload, xinit, meta["var0"], n, 1234 + seed_rank, device, dtype)
    alph = meta["alph"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)      # > L2 (126 MB)

    def step(xx):
        sums = nb.ocflow_sums(xx, net, prob, [0.0, 1.0], nt, "rk4", alph)
        if dist is not None:
            dist.all_reduce(sums)
        return sums

    with torch.no_grad():
        # the clock sampler starts before the warm-up: nvidia-smi needs a few hundred ms before its first row, longer than
        # a short timed region; rows are filtered by timestamp to the timed region afterwards
        sampler = ClockSampler(device.index) if (want_clocks and rank == 0) else None
        for _ in range(warmup):
            sums = step(x)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = nb._cabi.launch_count()
        t_begin = time.perf_counter()
        for e0, e1 in ev:
            flush.zero_()                 # L2 flush between timed iterations (not timed)
            e0.record()
            sums = step(x)
            e1.record()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t_end = time.perf_counter()
        launches = nb._cabi.launch_count() - l0
        clocks = sampler.stop(t_begin, t_end) if sampler else None
    step_ms = [e0.elapsed_time(e1) for e0, e1 in ev]
    tot_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(tot_ms, op=dist.ReduceOp.MAX)
    path = nb._cabi.last_path()
    out = dict(W=W, meta=meta, d=d, nt=nt, n=n, step_ms=step_ms, tot_s=float(tot_ms) * 1e-3, sums=sums, path=path, launches=int(launches),
               clocks=clocks, alph=alph)
    # ---- e2e: public API with HOST buffers (H2D of the step's inputs + D2H of its result inside the timed region)
    if e2e_steps > 0:
        xh = x.cpu().pin_memory()
        del x
        with torch.no_grad():
            for _ in range(2):
                nb.ocflow_sums(xh, net, prob, [0.0, 1.0], nt, "rk4", alph)
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                sh = nb.ocflow_sums(xh, net, prob, [0.0, 1.0], nt, "rk4", alph)     # noc_ocflow_host: H2D + rollout + D2H + sync
                if dist is not None:
                    sd_ = sh.to(device)
                    dist.all_reduce(sd_)
                    sh = sd_.cpu()
            torch.cuda.synchronize()
            e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=device)
        if dist is not None:
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        out.update(e2e_s=float(e2e_s), e2e_steps=e2e_steps, e2e_sums=sh, h2d=int(xh.numel() * xh.element_size()))
    return out


def dump_outputs(out_dir, sums, Jc, cs):
    """What the last timed step returned, so that two builds can be compared output for output on the same seeded inputs:
    sums.npy = the float64 vector [sum L, G, HJt, HJfin, HJgrad, Q, W, row count] of ocflow_sums (after the all-reduce), and
    costs.npy = [Jc, L, G, HJt, HJfin, HJgrad, Q, W], the objective and mean costs OCflow returns, in the workload's precision."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "sums.npy"), sums.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "costs.npy"), torch.stack([Jc] + list(cs)).cpu().numpy())


def shard(total, world, rank):
    """rows [lo, hi) of rank `rank`: contiguous blocks of ceil(total / world) rows (neuraloc_b200.sharded.shard_rows)."""
    per = -(-total // world)
    lo = min(total, rank * per)
    return lo, min(total, lo + per)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--samples", dest="n", type=int, default=0, help="samples (total for strong-scaled workloads, per GPU otherwise)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the swap12 / singlequad full-size extra lines")
    ap.add_argument("--latency", action="store_true", help="batch-1 rollout latency (timeDeployment/timeOC.py protocol) instead of throughput")
    ap.add_argument("--train", action="store_true", help="time one training evaluation: OCflow in train mode + Jc.backward() (SURVEY.md 8f N1)")
    ap.add_argument("--intermediates", action="store_true", help="time OCflow(..., intermediates=True): trajectories + controls written to HBM (SURVEY.md 8f N2)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (throughput measurement)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.latency or args.intermediates or args.train):
        ap.error("--dump-outputs applies to the throughput measurement only")
    W = WORKLOADS[args.workload]
    nt = W["nt"]
    dtype = torch.float32 if W["dtype"] == "f32" else torch.float64
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    threads = os.cpu_count() or 1
    total = args.n or W["n"]

    # ------------------------------------------------------------------ reference arm: CPU oracle port on host cores
    if args.impl == "reference":
        if rank != 0:
            return
        rates = []
        for _ in range(max(1, args.steps)):
            r, dt = cpu_rate(args.workload, W["n_cpu"], nt, dtype, threads)
            rates.append((r, dt))
        rate = W["n_cpu"] * nt * len(rates) / sum(dt for _, dt in rates)
        sample = "%d samples x nt=%d per step (a bounded sample of the workload's %d), torch CPU %s, %d threads" % (W["n_cpu"], nt, total, torch.__version__, threads)
        line = {"impl": "reference", "metric": "rk4_sample_steps_per_sec", "value": rate, "unit": "sample-steps/s",
                "n_gpus": args.gpus, "steps": len(rates), "warmup": 1, "ms_per_step": 1e3 * sum(dt for _, dt in rates) / len(rates),
                "higher_is_better": True, "scaling": W["scaling"], "vs_baseline": None, "dtype": W["dtype"], "data": "synthetic",
                "config": {"workload": "%s pretrained checkpoint, nt=%d, x ~ xInit + var0*N(0,I)" % (args.workload, nt),
                           "samples_per_step": W["n_cpu"]},
                "cpu_baseline": {"value": rate, "unit": "sample-steps/s", "cores": threads, "kind": "port", "sample": sample},
                "e2e": {"value": rate, "unit": "sample-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    if args.latency:
        print(json.dumps(latency_mode(args.workload, W, dtype, threads)))
        return
    if args.intermediates:
        print(json.dumps(intermediates_mode(args, W, dtype)))
        return
    if args.train:
        print(json.dumps(train_mode(args, W, dtype, threads)))
        return

    # ------------------------------------------------------------------ our arm
    import neuraloc_b200 as nb
    lib = nb._cabi.lib()      # raises if the CUDA library is missing: no fallback
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)

    strong = W["scaling"] == "strong"
    if strong:
        lo, hi = shard(total, world, rank)
        n_local, job = hi - lo, total
    else:
        n_local, job = total, total * world
    m = measure(args.workload, n_local, args.steps, args.warmup, device, dtype, dist, rank, world, rank, True, max(3, args.steps // 2))
    value = job * nt * args.steps / m["tot_s"]
    e2e_val = job * nt * m["e2e_steps"] / m["e2e_s"]
    # second figure for strong-scaled workloads: weak scaling at the N = 8 shard size per GPU
    weak = None
    if strong:
        n_w = max(1, total // 8)
        mw = measure(args.workload, n_w, 3, 1, device, dtype, dist, rank, world, rank, False, 0)
        weak = {"value": world * n_w * nt * 3 / mw["tot_s"], "unit": "sample-steps/s", "samples_per_gpu": n_w, "steps": 3,
                "note": "weak scaling: fixed samples per GPU (= the 8-GPU shard of the strong-scaled batch)"}

    if rank == 0:
        import ctypes
        d, meta = m["d"], m["meta"]
        fl = flops_per_sample_step(d, meta["m"], meta["nTh"], min(10, d + 1))
        pk = ctypes.c_double(0.0)
        nb._cabi.check(lib.noc_measure_fma_peak(0 if W["dtype"] == "f32" else 1, pk))
        peak = pk.value
        Jc, cs = nb.costs_from_sums(m["sums"], m["alph"], dtype)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, m["sums"], Jc, cs)
        e2e_Jc = float(nb.costs_from_sums(m["e2e_sums"], m["alph"], dtype)[0])
        sub = ""
        if W.get("full_n") and total != W["full_n"]:
            sub = " (a %d-sample sub-batch of configs[3]'s %d: one step of the full batch is ~%.0f s on one GPU)" % (
                total, W["full_n"], W["full_n"] * nt / max(value / world, 1.0))
        line = {
            "metric": "rk4_sample_steps_per_sec", "value": value, "unit": "sample-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["tot_s"] * 1e3 / args.steps,
            "higher_is_better": True, "scaling": W["scaling"], "vs_baseline": None, "dtype": W["dtype"], "data": "synthetic",
            "config": {"workload": "%s %s, nt=%d, %d samples %s%s, x ~ xInit + var0*N(0,I) seed 1234+rank, eval mode"
                                   % (args.workload, "pretrained checkpoint" if W["ckpt"] else "random-init swarm50-shape Phi", nt, total,
                                      "in total, row-sharded over the GPUs" if strong else "per GPU", sub),
                       "samples_total": job, "samples_this_gpu": n_local, "nt": nt, "d": d, "m": meta["m"], "nTh": meta["nTh"],
                       "parallelism": "dp%d (row shards, one all-reduce of 8 doubles)" % world,
                       "l2": "flushed between timed steps (256 MiB write, untimed)", "flops_per_sample_step": fl,
                       "kernel_path": m["path"], "Jc": float(Jc), "Jc_e2e": e2e_Jc},
            "clocks": m["clocks"],
            "e2e": {"value": e2e_val, "unit": "sample-steps/s", "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": 64, "steps": m["e2e_steps"]},
            "gpu_launches": m["launches"],
            "roofline": roofline(args.workload, W, d, meta, n_local, nt, fl, statistics.mean(m["step_ms"]) * 1e-3, peak, m["path"], m["clocks"]),
        }
        if weak:
            line["weak"] = weak
        if world == 1 and not args.no_cpu_baseline:
            lat = latency_mode(args.workload, W, dtype, threads)     # the other half of BASELINE.json's metric
            line["batch1_latency"] = {"value": lat["value"], "unit": "ms", "device_ms": lat["device_ms_median"],
                                      "ms_per_rk4_step": lat["ms_per_rk4_step"], "protocol": lat["config"]["workload"],
                                      "cpu_port_1thread_ms": lat["cpu_baseline"]["value"]}
            r, dt = cpu_rate(args.workload, W["n_cpu"], nt, dtype, threads)
            line["cpu_baseline"] = {"value": r, "unit": "sample-steps/s", "cores": threads, "kind": "port",
                                    "sample": "%d of the %d samples, nt=%d, one call, %.1f s; torch CPU %s oracle port (the Python reference cannot travel)"
                                              % (W["n_cpu"], total, nt, dt, torch.__version__)}
        if world == 1 and args.workload == DEFAULT_WORKLOAD and not args.no_extra:
            # configs[1] and configs[2] at their full sizes (5 timed steps each): the other two GPU lines of BASELINE.json
            extra = {}
            for wl in ("swap12", "singlequad"):
                We = WORKLOADS[wl]
                dte = torch.float32
                me = measure(wl, We["n"], 5, 3, device, dte, None, 0, 1, 0, True, 3)
                fle = flops_per_sample_step(me["d"], me["meta"]["m"], me["meta"]["nTh"], min(10, me["d"] + 1))
                Je = float(nb.costs_from_sums(me["sums"], me["alph"], dte)[0])
                extra[wl] = {"value": We["n"] * We["nt"] * 5 / me["tot_s"], "unit": "sample-steps/s", "steps": 5, "warmup": 3,
                             "ms_per_step": me["tot_s"] * 1e3 / 5, "samples": We["n"], "nt": We["nt"], "kernel_path": me["path"],
                             "e2e": {"value": We["n"] * We["nt"] * me["e2e_steps"] / me["e2e_s"], "unit": "sample-steps/s",
                                     "h2d_bytes_per_step": me["h2d"], "d2h_bytes_per_step": 64},
                             "clocks": me["clocks"], "Jc": Je,
                             "roofline": roofline(wl, We, me["d"], me["meta"], We["n"], We["nt"], fle, statistics.mean(me["step_ms"]) * 1e-3,
                                                  peak, me["path"], me["clocks"])}
            # one trainOC.py iteration (forward + backward, SURVEY.md 8f N1) at the reference's training shapes
            class _A:
                pass
            for wl in ("swarm50", "softcorridor"):
                ta = _A()
                ta.workload, ta.n, ta.steps, ta.warmup, ta.no_cpu_baseline = wl, 0, 5, 3, (wl != "swarm50")
                tl = train_mode(ta, WORKLOADS[wl], torch.float32, threads)
                extra["train_" + wl] = {k: tl[k] for k in ("metric", "value", "unit", "ms_per_step", "config", "gpu_launches", "roofline", "cpu_baseline") if k in tl}
            line["extra"] = extra
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Device time of the reverse-mode product of Phi (noc_phi_vjp) against the forward evaluation (noc_phi_eval) on the same rows.

For swarm50 (m = 512, n = 65 536) and softcorridor (m = 32, n = 2^20), fp32 and fp64, from the shipped checkpoints: rows
s = [x, t] with x ~ xInit + var0 N(0, I), t ~ U(0, 1), random seeds a and B.  noc_phi_eval writes Phi and grad Phi;
noc_phi_vjp writes the summed parameter gradient and d psi / d s for psi_i = a_i Phi(s_i) + B_i . grad Phi(s_i).  Each figure is
the mean over `--reps` back-to-back calls between two CUDA events (device time per call, allocation of the outputs included),
after `--warmup` calls; L2 is not flushed between calls.  Prints the card name and power limit with the figures, one JSON line
per case.

    python scripts/phi_vjp_bench.py [--reps 20] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CASES = (("swarm50", 1 << 16), ("softcorridor", 1 << 20))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    name, _, limit = q.stdout.strip().partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": limit.strip() or "unknown"}


def device_ms(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("phi_vjp_bench.py needs a CUDA device")
    import neuraloc_b200 as nb
    from neuraloc_b200.ocflow import phi_eval, phi_vjp
    from helpers import product_setup
    info = card()
    print("card: %s, power limit %s" % (info["name"], info["power_limit"]))
    for name, n in CASES:
        for dtype in (torch.float32, torch.float64):
            net, _, xinit, meta = product_setup(name, dtype)
            g = torch.Generator().manual_seed(5)
            d = xinit.shape[-1]
            x = xinit.reshape(1, d).double().cpu() + meta["var0"] * torch.randn(n, d, generator=g, dtype=torch.float64)
            s = torch.cat((x, torch.rand(n, 1, generator=g, dtype=torch.float64)), 1).to(dtype).cuda()
            a = torch.randn(n, generator=g, dtype=torch.float64).to(dtype).cuda()
            B = torch.randn(n, d + 1, generator=g, dtype=torch.float64).to(dtype).cuda()
            t_eval = device_ms(lambda: phi_eval(net, s, True, True), args.reps, args.warmup)
            t_vjp = device_ms(lambda: phi_vjp(net, s, a, B), args.reps, args.warmup)
            line = {"workload": name, "m": meta["m"], "d": d, "n": n, "dtype": str(dtype).split(".")[-1],
                    "phi_eval_ms": round(t_eval, 4), "phi_vjp_ms": round(t_vjp, 4), "ratio": round(t_vjp / t_eval, 2),
                    "card": info["name"], "power_limit": info["power_limit"], "reps": args.reps}
            print(json.dumps(line))
            del net, s, a, B
            nb.invalidate_cache()
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

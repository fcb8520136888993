"""More GPU coverage: randomized problem functors against the oracle (all thread decompositions), the drop-in import hook
driving an evalOC-style script end to end, intermediates at a size that spans many tiles, and size-independent properties
at benchmark-scale batches."""
import json
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from helpers import QW, ROOT, check_costs, load_cases, product_setup, rel_err, rel_state_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nb():
    import neuraloc_b200
    neuraloc_b200._cabi.lib()
    return neuraloc_b200


@pytest.mark.parametrize("cfg", [None, 2, 3, 5, 6])
@pytest.mark.parametrize("name", ["softcorridor", "swap2", "swap12", "midcross4", "swarm50", "swarm", "singlequad"])
def test_randomized_functors_vs_oracle(nb, name, cfg, monkeypatch):
    """calcLHQW / calcGradpH / calcCtrls on 300 random (x, p) rows, eval and train mode, through the one-thread-per-sample
    decomposition (default) and the split-across-threads ones (forced mid / large tiles)."""
    from oracle import ocflow_oracle as orc
    dtype = torch.float64 if cfg in (5, 6) else torch.float32
    if cfg is not None:
        monkeypatch.setenv("NOC_FORCE_CFG", str(cfg))
    alph = [300.0, 2.5, 7.0, 1.0, 1.0, 1.0] if name != "singlequad" else [5000.0, 0.0, 0.0, 0.1, 0.0, 0.0]
    prob, _, _, xinit = nb.initProb(name, 2, 2, 1.0, alph, lambda v: v.to(dtype).cuda())
    D, _ = orc.make_problem(name, alph, torch.float64)
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    n, d = 300, xinit.shape[1]
    x = xinit.cpu() + 0.7 * torch.randn(n, d, generator=g, dtype=dtype)
    p = 1.5 * torch.randn(n, d, generator=g, dtype=dtype)
    if prob.nAgents >= 2 and name != "singlequad":       # squeeze some agents together so that W is exercised
        A, dim = prob.nAgents, prob.agentDim
        xa = x.view(n, A, dim).clone()
        xa[: n // 3, 1] = xa[: n // 3, 0] + prob.r * torch.rand(n // 3, dim, generator=g, dtype=dtype) * 1.5
        x = xa.reshape(n, d)
    tol = 2e-5 if dtype == torch.float32 else 1e-11
    for mode in ("eval", "train"):
        getattr(prob, mode)()
        D.training = (mode == "train")
        try:
            L, H, Q, W = prob.calcLHQW(x.cuda(), p.cuda())
        except nb._cabi.NocError as e:               # e.g. d = 150 does not fit the forced 2-warp-wide tiling: loud
            assert cfg is not None and "noc error -4" in str(e)
            pytest.skip("problem does not fit forced configuration %s" % cfg)
        Lr, Hr, Qr, Wr = orc.lhqw(D, x.double(), p.double())
        for got, ref, nm in ((L, Lr, "L"), (H, Hr, "H"), (Q, Qr, "Q"), (W, Wr, "W")):
            ref = ref.reshape(-1).numpy() if torch.is_tensor(ref) else np.zeros(n)
            got = got.reshape(-1).cpu().numpy()
            # a pair (or an agent) within rounding of a cut-off can land on either side in fp32: allow two such rows
            err = np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)
            assert (err > tol).sum() <= (2 if dtype == torch.float32 else 0), (name, mode, nm, cfg, err.max())
        assert rel_err(prob.calcGradpH(x.cuda(), p.cuda()).cpu().numpy(),
                       orc.grad_p_hamiltonian(D, x.double(), p.double()).numpy(), floor=1.0) <= tol
        assert rel_err(prob.calcCtrls(x.cuda(), p.cuda()).cpu().numpy(),
                       orc.controls(D, x.double(), p.double()).numpy(), floor=1.0) <= tol


def test_dropin_hook_runs_an_evalOC_style_script(nb, tmp_path):
    """INTEGRATION.md §1 without the reference checkout (absent on the GPU box): a stand-in `src` package whose OCflow
    must never run, the sitecustomize hook first on PYTHONPATH, and a script written like evalOC.py:51-85."""
    src = tmp_path / "src"
    src.mkdir()
    (src / "__init__.py").write_text("")
    (src / "OCflow.py").write_text(textwrap.dedent("""
        def OCflow(*a, **k):
            raise AssertionError("the stand-in reference OCflow ran: the drop-in hook did not rebind it")
        stepRK4 = stepRK1 = ocOdefun = OCflow
        def ocG(z, xtarget):
            return z[:, :xtarget.shape[0]] - xtarget
    """))
    script = tmp_path / "eval_like.py"
    script.write_text(textwrap.dedent("""
        import sys, json, torch
        sys.path.insert(0, %r)
        from src.OCflow import OCflow                 # what evalOC.py:9 does
        from helpers import load_ckpt
        import neuraloc_b200 as nb
        sd, meta = load_ckpt("softcorridor")
        cvt = lambda v: v.type(torch.float32).to("cpu")          # evalOC.py is CPU-only (F2)
        prob, x0, _, xInit = nb.initProb(meta["data"], 10, 11, var0=1.0, alph=meta["alph"], cvt=cvt)
        prob.eval()
        net = nb.Phi(nTh=meta["nTh"], m=meta["m"], d=x0.size(1), alph=meta["alph"])
        net.load_state_dict(sd)
        with torch.no_grad():
            Jc, cs = OCflow(xInit, net, prob, tspan=[0.0, 1.0], nt=50, stepper="rk4", alph=net.alph)
            zFull, ctrlFull = OCflow(xInit, net, prob, tspan=[0.0, 1.0], nt=50, stepper="rk4", alph=net.alph, intermediates=True)
        print('{:12.4e} {:11.3e}'.format(cs[0] + meta["alph"][0] * cs[1], cs[0]))
        print("RESULT " + json.dumps([float(Jc)] + [float(c) for c in cs] + [float(zFull[0, :4, -1].norm()), float(ctrlFull[0, :, -1].norm())]))
    """ % os.path.join(ROOT, "tests")))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "neuraloc_b200", "dropin"), ROOT, str(tmp_path)]))
    env.pop("NOC_FORCE_PATH", None)
    out = subprocess.run([sys.executable, str(script)], env=env, capture_output=True, text=True, cwd=str(tmp_path), timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    vals = json.loads([l for l in out.stdout.splitlines() if l.startswith("RESULT ")][0][7:])
    c = load_cases("softcorridor")
    check_costs(vals[:8], c["xinit_mean_f32"], 2e-3, 2e-4, "evalOC-style run through the hook", floor_mask=QW)
    # SURVEY.md §8c known answers: |x(T)| = 3.95163, |u(T)| = 5.23089
    assert abs(vals[8] - 3.95163178) < 1e-4 and abs(vals[9] - 5.23088646) < 1e-3


def test_dropin_hook_runs_a_trainOC_style_script(nb, tmp_path):
    """trainOC.py:150-210 through the hook without the reference checkout: Adam iterations with `Jc.backward()`, validation under
    no_grad in eval mode, resampling, and the `{args, state_dict}` checkpoint it saves (trainOC.py:204-207) reloaded evalOC-style."""
    src = tmp_path / "src"
    src.mkdir()
    (src / "__init__.py").write_text("")
    (src / "OCflow.py").write_text(textwrap.dedent("""
        def OCflow(*a, **k):
            raise AssertionError("the stand-in reference OCflow ran: the drop-in hook did not rebind it")
        stepRK4 = stepRK1 = ocOdefun = OCflow
    """))
    script = tmp_path / "train_like.py"
    script.write_text(textwrap.dedent("""
        import sys, json, argparse, os, torch
        sys.path.insert(0, %r)
        from src.OCflow import OCflow                 # what trainOC.py:13 does
        import neuraloc_b200 as nb
        args = argparse.Namespace(data="softcorridor", m=32, nTh=2, nt=10, nt_val=16, n_train=512, var0=1.0, lr=0.01,
                                  alph=[100.0, 10000.0, 300.0, 0.02, 0.02, 0.02], niters=30, val_freq=10, sample_freq=15)
        device = torch.device("cuda:0")
        cvt = lambda x: x.type(torch.float32).to(device, non_blocking=True)
        torch.manual_seed(0)
        prob, x0, x0v, xInit = nb.initProb(args.data, args.n_train, 256, var0=args.var0, alph=args.alph, cvt=cvt)
        net = nb.Phi(nTh=args.nTh, m=args.m, d=x0.size(1), alph=args.alph).to(torch.float32).to(device)
        optim = torch.optim.Adam(net.parameters(), lr=args.lr)
        net.train(); prob.train()
        hist, val = [], []
        best = float("inf")
        for itr in range(1, args.niters + 1):
            optim.zero_grad()
            Jc, cs = OCflow(x0, net, prob, tspan=[0.0, 1.0], nt=args.nt, stepper="rk4", alph=net.alph)
            Jc.backward()
            optim.step()
            hist.append(float(Jc.detach()))
            line = '{:05d} {:9.3e}  {:8.2e}  {:8.2e}'.format(itr, Jc, cs[0], cs[1])      # the reference formats the tensors directly
            if itr %% args.val_freq == 0:
                with torch.no_grad():
                    net.eval(); prob.eval()
                    tl, tcs = OCflow(x0v, net, prob, tspan=[0.0, 1.0], nt=args.nt_val, stepper="rk4", alph=net.alph)
                    val.append(float(tl))
                    if tl.item() < best:
                        best = tl.item()
                        torch.save({"args": args, "state_dict": net.state_dict()}, "ckpt.pth")
                    net.train(); prob.train()
            if itr %% args.sample_freq == 0:
                x0 = nb.resample(x0, xInit, args.var0, cvt)
        ck = torch.load("ckpt.pth", map_location=lambda storage, loc: storage, weights_only=False)
        net2 = nb.Phi(nTh=ck["args"].nTh, m=ck["args"].m, d=4, alph=ck["args"].alph)
        net2.load_state_dict(ck["state_dict"])
        with torch.no_grad():
            prob.eval()
            J2, _ = OCflow(x0v.cpu(), net2, prob, tspan=[0.0, 1.0], nt=args.nt_val, stepper="rk4", alph=net2.alph)
        print("RESULT " + json.dumps({"hist": hist, "val": val, "best": best, "reloaded": float(J2)}))
    """ % os.path.join(ROOT, "tests")))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "neuraloc_b200", "dropin"), ROOT, str(tmp_path)]))
    for k in ("NOC_FORCE_PATH", "NOC_NO_LAT"):
        env.pop(k, None)
    out = subprocess.run([sys.executable, str(script)], env=env, capture_output=True, text=True, cwd=str(tmp_path), timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    r = json.loads([l for l in out.stdout.splitlines() if l.startswith("RESULT ")][0][7:])
    assert len(r["hist"]) == 30 and len(r["val"]) == 3 and all(np.isfinite(r["hist"]))
    assert r["hist"][-1] < 0.6 * r["hist"][0]                         # the loss goes down
    assert abs(r["reloaded"] - r["best"]) <= 1e-3 * abs(r["best"])    # the saved checkpoint reproduces its validation loss (CPU tensors: host entry)


@pytest.mark.parametrize("name", ["softcorridor", "swarm50"])
def test_real_pth_checkpoint_evalOC_and_timeOC_flow(nb, tmp_path, name):
    """A real checkpoint FILE in the reference's layout — torch.save({'args': argparse.Namespace, 'state_dict': ...}) as
    trainOC.py:204-207 writes it — loaded exactly the way evalOC.py:51-64 / timeOC.py:45-64 load it (torch.load with the
    map_location lambda, args.m / nTh / alph / data from the pickled Namespace, load_state_dict, .to(prec).to(device)), on the
    box, through the sitecustomize hook, with CPU tensors as both scripts use; then evalOC's two OCflow calls (:81,:83) and
    timeOC's timed call (:76-81).  The reference checkout itself cannot travel: a stand-in `src` package provides only what
    the hook replaces."""
    import argparse
    from helpers import load_ckpt
    sd, meta = load_ckpt(name)
    ns = argparse.Namespace(data=meta["data"], m=meta["m"], nTh=meta["nTh"], alph=meta["alph"], var0=meta["var0"], nt=meta.get("nt", 50),
                            prec="single", resume=None, gpu=0, lr=0.01, niters=6000)
    ckpt = tmp_path / ("%s_alph_checkpt.pth" % name)
    torch.save({"args": ns, "state_dict": sd}, str(ckpt))
    src = tmp_path / "src"
    src.mkdir()
    (src / "__init__.py").write_text("")
    (src / "OCflow.py").write_text(textwrap.dedent("""
        def OCflow(*a, **k):
            raise AssertionError("the stand-in reference OCflow ran: the drop-in hook did not rebind it")
        stepRK4 = stepRK1 = ocOdefun = OCflow
        def ocG(z, xtarget):
            return z[:, :xtarget.shape[0]] - xtarget
    """))
    nt = 80 if name == "swarm50" else 50
    script = tmp_path / "eval_pth.py"
    script.write_text(textwrap.dedent("""
        import argparse, json, os, sys, time, torch
        from src.OCflow import OCflow                             # evalOC.py:9 / timeOC.py:9
        from neuraloc_b200 import Phi, initProb                  # stand-ins for src.Phi / src.initProb (same interface)
        argPrec = torch.float32
        device = torch.device('cpu')                              # evalOC.py:38: only support cpu
        torch.set_default_dtype(argPrec)
        cvt = lambda x: x.type(argPrec).to(device, non_blocking=True)
        checkpt = torch.load(%r, map_location=lambda storage, loc: storage)
        m = checkpt['args'].m
        alph = checkpt['args'].alph
        nTh = checkpt['args'].nTh
        data = checkpt['args'].data
        prob, x0, _, xInit = initProb(data, 10, 11, var0=1.0, alph=alph, cvt=cvt)
        prob.eval()
        d = x0.size(1)
        net = Phi(nTh=nTh, m=m, d=d, alph=alph)
        net.load_state_dict(checkpt["state_dict"])
        net = net.to(argPrec).to(device)
        nt = %d
        with torch.no_grad():
            net.eval()
            Jc, cs = OCflow(xInit, net, prob, tspan=[0.0, 1.0], nt=nt, stepper="rk4", alph=net.alph)
            zFull, ctrlFull = OCflow(xInit, net, prob, tspan=[0.0, 1.0], nt=nt, stepper="rk4", alph=net.alph, intermediates=True)
            line = '         {:12.4e} {:11.3e} {:11.3e} {:11.3e} {:11.3e} {:11.3e} {:11.3e} {:11.3e}'.format(
                cs[0] + alph[0]*cs[1], cs[0], alph[0]*cs[1], alph[3]*cs[2], alph[4]*cs[3], alph[5]*cs[4], cs[5], cs[6])
            start = time.time()                                   # timeOC.py:76-81
            Jc2, cs2 = OCflow(xInit, net, prob, tspan=[0.0, 1.0], nt=nt, stepper="rk4", alph=net.alph)
            end = time.time()
        assert isinstance(Jc, torch.Tensor) and Jc.dim() == 0 and Jc.device.type == 'cpu'
        print(line)
        print("RESULT " + json.dumps([float(Jc)] + [float(c) for c in cs] + [float(zFull[0, :d, -1].norm()), float(ctrlFull[0, :, -1].norm()),
                                     end - start, float(Jc2)]))
    """ % (str(ckpt), nt)))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "neuraloc_b200", "dropin"), ROOT, str(tmp_path)]),
               TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD="1")      # SURVEY.md F7(a): the pickled Namespace needs weights_only=False on torch >= 2.6
    env.pop("NOC_FORCE_PATH", None)
    out = subprocess.run([sys.executable, str(script)], env=env, capture_output=True, text=True, cwd=str(tmp_path), timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    vals = json.loads([l for l in out.stdout.splitlines() if l.startswith("RESULT ")][0][7:])
    c = load_cases(name)
    check_costs(vals[:8], c["xinit_mean_f64"], 1e-4, 2e-4, "evalOC flow from a real .pth (%s)" % name, floor_mask=QW,
                ref_noise=c["xinit_mean_f32"].astype(np.float64) - c["xinit_mean_f64"])
    d = c["xinit_z_f64"].shape[1] - 4
    assert abs(vals[8] - np.linalg.norm(c["xinit_z_f64"][0, :d, -1])) <= 1e-5 * np.linalg.norm(c["xinit_z_f64"][0, :d, -1])
    assert abs(vals[9] - np.linalg.norm(c["xinit_ctrl_f64"][0, :, -1])) <= 1e-4 * np.linalg.norm(c["xinit_ctrl_f64"][0, :, -1])
    assert vals[11] == vals[0] and vals[10] < 5.0             # the timed call repeats the result; seconds, not minutes


def test_two_problems_with_cpu_targets_do_not_share_a_target(nb):
    """ADVICE r1: the device copy of prob.xtarget must follow the problem, not a recycled host address: roll the SAME net out
    against two problems whose (CPU) targets differ; G must differ accordingly."""
    net, prob, xinit, meta = product_setup("softcorridor", torch.float32, device="cpu")
    x = xinit.clone()
    with torch.no_grad():
        g1 = float(nb.OCflow(x, net, prob, [0.0, 1.0], 20, "rk4", meta["alph"])[1][1])
        import copy
        prob2 = copy.copy(prob)
        prob2.xtarget = (prob.xtarget.clone() + 0.5)
        g2 = float(nb.OCflow(x, net, prob2, [0.0, 1.0], 20, "rk4", meta["alph"])[1][1])
        del prob2
        g1b = float(nb.OCflow(x, net, prob, [0.0, 1.0], 20, "rk4", meta["alph"])[1][1])
    assert g1 == g1b and abs(g2 - g1) > 1e-3 * max(abs(g1), 1e-6)


@pytest.mark.parametrize("name", ["swap12", "singlequad"])
def test_intermediates_across_many_tiles(nb, name, monkeypatch):
    """intermediates=True on 3000 samples (several tiles per CTA, ragged last tile): trajectories agree with the small-batch
    kernel sample by sample, zFull's last column agrees with the noMean costs, controls at step 0 are zero."""
    net, prob, xinit, meta = product_setup(name, torch.float32)
    d = xinit.shape[1]
    g = torch.Generator().manual_seed(4)
    x = (xinit.cpu() + 0.3 * torch.randn(3000, d, generator=g)).cuda()
    if name == "singlequad":
        x[:, 3:] = 0
    nt = 12
    with torch.no_grad():
        monkeypatch.setenv("NOC_FORCE_PATH", "tile")
        zf, cf = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
        Jn, cn = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], noMean=True)
        monkeypatch.setenv("NOC_FORCE_PATH", "vec")
        idx = torch.tensor([0, 1, 479, 480, 481, 1500, 2879, 2880, 2999], device="cuda")
        zv, cv = nb.OCflow(x[idx].contiguous(), net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
    assert zf.shape == (3000, d + 4, nt + 1) and not cf[:, :, 0].any()
    assert rel_state_err(zf[idx].cpu().numpy(), zv.cpu().numpy(), d) <= 2e-6
    assert (cf[idx] - cv).abs().max() <= 1e-4 * max(1.0, float(cv.abs().max()))
    assert torch.allclose(zf[:, d, -1:], cn[0], rtol=1e-6, atol=1e-6)          # accumulated L
    assert torch.allclose(zf[:, d + 1, -1:], cn[2], rtol=1e-6, atol=1e-6)      # accumulated HJt


@pytest.mark.parametrize("name,n,nt", [("softcorridor", 4096, 50), ("swap2", 4096, 50), ("swap12", 4096, 50),
                                       ("singlequad", 4096, 50), ("swarm50", 512, 80)])
def test_parity_gate_4096_samples(nb, name, n, nt, monkeypatch):
    """SURVEY.md 8(d) parity gate at its stated size: 4 096 samples per problem from the benchmark distribution (512 for
    swarm50), the documented nt, the kernel the library picks by itself (tensor cores where they apply): per-step state
    <= 1e-5 relative against the fp32 oracle and against the fp64 oracle, mean cost terms <= 1e-4 relative (fp64 oracle)."""
    from oracle import ocflow_oracle as orc
    from helpers import oracle_setup, mean_vec
    monkeypatch.delenv("NOC_FORCE_PATH", raising=False)
    net, prob, xinit, meta = product_setup(name, torch.float32)
    P32, D32, _, _ = oracle_setup(name, torch.float32)
    P64, D64, _, _ = oracle_setup(name, torch.float64)
    d = xinit.shape[1]
    g = torch.Generator().manual_seed(1234)
    if name == "singlequad":
        x = torch.zeros(n, d)
        x[:, :3] = -1.5 + meta["var0"] * torch.randn(n, 3, generator=g)
    else:
        x = xinit.cpu() + meta["var0"] * torch.randn(n, d, generator=g)
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        zg, _ = nb.OCflow(x.cuda(), net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
        mg = mean_vec(nb.OCflow(x.cuda(), net, prob, [0.0, 1.0], nt, "rk4", meta["alph"]))
        z32, _ = orc.ocflow(x, P32, D32, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
        z64, _ = orc.ocflow(x.double(), P64, D64, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
        m64 = mean_vec(orc.ocflow(x.double(), P64, D64, [0.0, 1.0], nt, "rk4", meta["alph"]))
    zg = zg.cpu().numpy()
    e32, e64, ref = rel_state_err(zg, z32.numpy(), d), rel_state_err(zg, z64.numpy(), d), rel_state_err(z32.numpy(), z64.numpy(), d)
    assert e32 <= 1e-5, "%s: state vs fp32 oracle %.2e" % (name, e32)
    assert e64 <= max(1e-5, 2 * ref), "%s: state vs fp64 oracle %.2e (fp32 oracle itself: %.2e)" % (name, e64, ref)
    check_costs(mg, m64, 1e-4, 2e-4, name + " mean costs vs fp64 oracle, %d samples" % n, floor_mask=QW)


def test_benchmark_scale_properties(nb, monkeypatch):
    """Size-independent properties at benchmark-like batch sizes (the oracle cannot run there): permutation invariance of
    the means, additivity of the cost sums over row shards, determinism, and mean == mean of noMean."""
    monkeypatch.delenv("NOC_FORCE_PATH", raising=False)
    net, prob, xinit, meta = product_setup("swap12", torch.float32)
    g = torch.Generator(device="cuda").manual_seed(1)
    n = 200_000
    x = xinit + torch.randn(n, 24, generator=g, device="cuda")
    with torch.no_grad():
        s_all = nb.ocflow_sums(x, net, prob, [0.0, 1.0], 10, "rk4", meta["alph"])
        s_again = nb.ocflow_sums(x, net, prob, [0.0, 1.0], 10, "rk4", meta["alph"])
        perm = torch.randperm(n, generator=g, device="cuda")
        s_perm = nb.ocflow_sums(x[perm].contiguous(), net, prob, [0.0, 1.0], 10, "rk4", meta["alph"])
        lo = nb.ocflow_sums(x[:77_777].contiguous(), net, prob, [0.0, 1.0], 10, "rk4", meta["alph"])
        hi = nb.ocflow_sums(x[77_777:].contiguous(), net, prob, [0.0, 1.0], 10, "rk4", meta["alph"])
        Jn, cn = nb.OCflow(x, net, prob, [0.0, 1.0], 10, "rk4", meta["alph"], noMean=True)
    assert torch.equal(s_all, s_again)                                           # fixed reduction order
    assert float(s_all[7]) == n
    assert torch.allclose(s_all, s_perm, rtol=1e-9, atol=1e-6)                   # per-sample results do not depend on the tile
    assert torch.allclose(s_all, lo + hi, rtol=1e-9, atol=1e-6)                  # shards add (the multi-GPU contract)
    means = (s_all[:7] / n).cpu().numpy()
    nm = torch.cat(list(cn), 1).double().mean(0).cpu().numpy()
    check_costs(means, nm, 1e-6, 1e-7, "mean mode vs mean of noMean", floor_mask=QW[1:])


def test_batched_shock_restart(nb, monkeypatch):
    """plotter.py:815-823 for a batch: the two legs of OCflow_shock against the oracle's two calls (fp64), with the reference's
    minor and major softcorridor shocks (evalOC.py:115-118) applied per row."""
    from oracle import ocflow_oracle as orc
    from helpers import oracle_setup
    monkeypatch.delenv("NOC_FORCE_PATH", raising=False)
    net, prob, xinit, meta = product_setup("softcorridor", torch.float32)
    P64, D64, _, _ = oracle_setup("softcorridor", torch.float64)
    g = torch.Generator().manual_seed(21)
    n, nt = 700, 50
    x = xinit.cpu() + 0.3 * torch.randn(n, 4, generator=g)
    shock = torch.where(torch.arange(n).view(-1, 1) % 2 == 0, torch.tensor([[-0.2, -0.7, -0.0, -0.6]]), torch.tensor([[-1.4, -1.0, -5.2, -2.8]]))
    with torch.no_grad():
        t1, c1, t2, c2 = nb.OCflow_shock(x.cuda(), net, prob, nt, [0.1, shock], "rk4", meta["alph"])
        r1, _ = orc.ocflow(x.double(), P64, D64, [0.0, 0.1], 5, "rk4", meta["alph"], intermediates=True)
        xs = r1[:, :4, -1] + shock.double()
        r2, rc2 = orc.ocflow(xs, P64, D64, [0.1, 1.0], 46, "rk4", meta["alph"], intermediates=True)
    assert t1.shape == (n, 8, 6) and t2.shape == (n, 8, 47) and t1.is_cuda
    assert rel_state_err(t1.cpu().numpy(), r1.numpy(), 4) <= 1e-5 and rel_state_err(t2.cpu().numpy(), r2.numpy(), 4) <= 1e-5
    assert (c2.cpu().double() - rc2).abs().max() <= 2e-4 * max(1.0, float(rc2.abs().max()))
    with torch.no_grad():
        one = nb.OCflow_shock(x[:3].cuda(), net, prob, nt, [0.1, shock[:1]], "rk4", meta["alph"])  # a [1,d] shock row broadcasts
    assert one[2].shape == (3, 8, 47)


def test_bench_dump_outputs_are_the_timed_steps_results(nb, tmp_path):
    """bench.py --dump-outputs: two runs with different --steps time that many steps (launches scale with it) and dump the same
    arrays, which are what ocflow_sums returns for the bench's seeded batch and what OCflow derives from them."""
    import importlib.util
    runs = {}
    for steps in (2, 5):
        out = tmp_path / ("s%d" % steps)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "swap12", "--samples", "8192",
                            "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, cwd=str(tmp_path), timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads(p.stdout.strip().splitlines()[-1])
        runs[steps] = (line, np.load(out / "sums.npy"), np.load(out / "costs.npy"))
    (l2, s2, c2), (l5, s5, c5) = runs[2], runs[5]
    assert (l2["steps"], l5["steps"]) == (2, 5) and l2["gpu_launches"] > 0 and 2 * l5["gpu_launches"] == 5 * l2["gpu_launches"]
    assert s2.dtype == np.float64 and s2.shape == (8,) and c2.dtype == np.float32 and c2.shape == (8,)
    assert np.array_equal(s2, s5) and np.array_equal(c2, c5) and s2[7] == 8192
    assert float(c2[0]) == l2["config"]["Jc"]
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    device = torch.device("cuda", 0)
    net, prob, xinit, meta = b.build_case("swap12", device, torch.float32)
    x = b.sample_x("swap12", xinit, meta["var0"], 8192, 1234, device, torch.float32)
    with torch.no_grad():
        sums = nb.ocflow_sums(x, net, prob, [0.0, 1.0], b.WORKLOADS["swap12"]["nt"], "rk4", meta["alph"])
    Jc, cs = nb.costs_from_sums(sums, meta["alph"], torch.float32)
    assert np.array_equal(sums.cpu().numpy(), s2)
    assert np.array_equal(torch.stack([Jc] + cs).cpu().numpy(), c2)

"""GPU: Phi.forward / Phi.getGrad under autograd — the reverse-mode product noc_phi_vjp (the training kernel's second-order sweep on
one evaluation per row) against torch.autograd of the CPU oracle's phi_forward / phi_grad (src/Phi.py:91-138), and the autograd
wiring of neuraloc_b200.Phi on top of it."""
import ctypes as C
import copy
import dataclasses

import numpy as np
import pytest
import torch

from helpers import DT, GOLDEN, PROBLEMS, load_ckpt, oracle_setup, product_setup, rel_err
from oracle import ocflow_oracle as orc

pytestmark = pytest.mark.gpu

ORDER = ["A", "c_w", "c_b", "w", "K0", "K1", "b0", "b1"]          # split_param_grads order


def _leaves(P):
    return [t.clone().requires_grad_(True) for t in (P.A, P.c_w, P.c_b, P.w, P.K[0], P.K[1], P.b[0], P.b[1])]


def _params(leaves, h):
    return orc.PhiParams(leaves[0], leaves[1], leaves[2], leaves[3], [leaves[4], leaves[5]], [leaves[6], leaves[7]], h)


def oracle_vjp(P, s, a, B):
    """({name: sum_i d psi_i / d theta}, d psi_i / d s_i) for psi_i = a_i Phi(s_i) + B_i . grad Phi(s_i), autograd of the oracle
    in the dtype of its arguments; a or B may be None (zero)."""
    leaves = _leaves(P)
    Pg = _params(leaves, P.h)
    sg = s.clone().requires_grad_(True)
    psi = s.new_zeros(())
    if a is not None:
        psi = psi + (a.reshape(-1, 1) * orc.phi_forward(Pg, sg)).sum()
    if B is not None:
        psi = psi + (B * orc.phi_grad(Pg, sg)).sum()
    g = torch.autograd.grad(psi, leaves + [sg], allow_unused=True)          # without a, c.bias does not enter psi
    g = [torch.zeros_like(v) if u is None else u for u, v in zip(g, leaves + [sg])]
    return dict(zip(ORDER, g[:8])), g[8]


def kernel_vjp(net, s, a, B):
    import neuraloc_b200 as nb
    gp, gs = nb.ocflow.phi_vjp(net, s.cuda(), None if a is None else a.cuda(), None if B is None else B.cuda())
    return {k: v.double().cpu() for k, v in zip(ORDER, nb.split_param_grads(net, gp))}, gs.double().cpu()


def _worst(got, ref):
    """largest entry error of each tensor relative to the tensor's largest entry"""
    out = {k: float((got[k].reshape(ref[k].shape) - ref[k]).abs().max()) / max(float(ref[k].abs().max()), 1e-300) for k in ref}
    return out


def random_net(m, d, seed, dtype):
    """an nTh = 2 net with every parameter random (c and w included, which the reference initialises to constants)"""
    import neuraloc_b200 as nb
    torch.manual_seed(seed)
    net = nb.Phi(nTh=2, m=m, d=d)
    with torch.no_grad():
        net.c.weight.normal_(0.0, 0.5)
        net.c.bias.normal_(0.0, 0.5)
        net.w.weight.normal_(1.0, 0.3)
        net.A.mul_(2.0)
    P = orc.params_from_state_dict({k: v.detach().clone() for k, v in net.state_dict().items()}, torch.float64)
    return net.to(dtype).cuda(), P


def rows(xinit, var0, n, seed, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    d = xinit.shape[-1]
    x = xinit.reshape(1, d).double().cpu() + var0 * torch.randn(n, d, generator=g, dtype=torch.float64)
    t = torch.rand(n, 1, generator=g, dtype=torch.float64)
    t[0] = 1.0
    return torch.cat((x, t), 1).to(dtype)


def seeds(n, D, seed, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, generator=g, dtype=torch.float64).to(dtype), torch.randn(n, D, generator=g, dtype=torch.float64).to(dtype)


def _cases():
    """(label, builder) for the five shipped checkpoints and random nets whose widths are not tile multiples"""
    out = [(name, name) for name in PROBLEMS]
    out += [("random_m%d" % m, (m, d)) for m, d in ((24, 6), (96, 15), (320, 40))]
    return out


def _build(spec, dtype):
    if isinstance(spec, str):
        net, prob, xinit, meta = product_setup(spec, dtype)
        P, _, _, _ = oracle_setup(spec, torch.float64)
        return net, P, xinit, meta["var0"]
    m, d = spec
    net, P = random_net(m, d, 7 + m, dtype)
    return net, P, torch.zeros(d, dtype=torch.float64), 1.0


# ---------------------------------------------------------------------------------------------------------------------------
# 1. random seeds, fp64
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("label,spec", _cases(), ids=[c[0] for c in _cases()])
def test_vjp_fp64_matches_oracle_autograd(label, spec):
    net, P, xinit, var0 = _build(spec, torch.float64)
    n = 37
    s = rows(xinit, var0, n, 11)
    a, B = seeds(n, s.shape[1], 12)
    Gr, sr = oracle_vjp(P, s, a, B)
    Gk, sk = kernel_vjp(net, s, a, B)
    worst = _worst(Gk, Gr)
    assert max(worst.values()) <= 1e-10, (label, worst)
    serr = float((sk - sr).abs().max()) / float(sr.abs().max())
    assert serr <= 1e-10, (label, serr)


# ---------------------------------------------------------------------------------------------------------------------------
# 2. fp32 against the fp64 reference, gated by torch's own fp32 distance on the same rows
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("label,spec", _cases(), ids=[c[0] for c in _cases()])
def test_vjp_fp32_within_fp32_rounding(label, spec):
    net, P64, xinit, var0 = _build(spec, torch.float32)
    P32 = P64.to(torch.float32)
    P64 = P32.to(torch.float64)                      # the fp32 weights, exactly: only the arithmetic differs
    n = 37
    s32 = rows(xinit, var0, n, 21, torch.float32)
    a32, B32 = seeds(n, s32.shape[1], 22, torch.float32)
    Gr, sr = oracle_vjp(P64, s32.double(), a32.double(), B32.double())
    Gt, st = oracle_vjp(P32, s32, a32, B32)           # torch's fp32 autograd on the same rows
    Gk, sk = kernel_vjp(net, s32, a32, B32)
    torch_dist = _worst({k: v.double() for k, v in Gt.items()}, Gr)
    torch_dist["s"] = float((st.double() - sr).abs().max()) / float(sr.abs().max())
    got = _worst(Gk, Gr)
    got["s"] = float((sk - sr).abs().max()) / float(sr.abs().max())
    # of the order of torch's distance: 10x, and never below 1e-5 of the tensor's largest entry (a few hundred fp32 ulps: sums of
    # 37 rows through atomics, where torch's own distance can happen to be a single rounding)
    bad = {k: (got[k], torch_dist[k]) for k in got if got[k] > max(10.0 * torch_dist[k], 1e-5)}
    assert not bad, (label, bad)


# ---------------------------------------------------------------------------------------------------------------------------
# 3. tiling: every tile width, ragged tiles, more tiles than one wave of CTAs
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,ts", [("softcorridor", 2), ("softcorridor", 4), ("softcorridor", 8), ("singlequad", 4),
                                     ("singlequad", 8), ("swarm50", 4), ("swarm50", 8)])
def test_vjp_tile_widths(name, ts, monkeypatch):
    monkeypatch.setenv("NOC_GRAD_TS", str(ts))
    import neuraloc_b200 as nb
    sm = C.c_int32()
    nb._cabi.check(nb._cabi.lib().noc_device_info(C.byref(sm), None, None, None))
    dtype = torch.float32 if (name == "swarm50" and ts == 8) else torch.float64   # 8-sample fp64 panels of m = 512 do not fit
    net, P, xinit, var0 = _build(name, dtype)
    # one CTA per SM for the m = 512 net; the narrow nets run many CTAs per SM: 64 tiles per SM is more than one wave for them
    big = (sm.value + 1) * ts + 1 if name == "swarm50" else 64 * sm.value * ts + 3
    sizes = [1, ts - 1, ts, ts + 1, big] if ts > 2 else [1, 2, 3, big]
    s_all = rows(xinit, var0, big, 31)
    a_all, B_all = seeds(big, s_all.shape[1], 32)
    for n in sizes:
        s, a, B = s_all[:n].to(dtype), a_all[:n].to(dtype), B_all[:n].to(dtype)
        Gk, sk = kernel_vjp(net, s, a, B)
        Pr = P.to(dtype).to(torch.float64)
        Gr, sr = oracle_vjp(Pr, s.double(), a.double(), B.double())
        worst = _worst(Gk, Gr)
        serr = float((sk - sr).abs().max()) / float(sr.abs().max())
        tol = 1e-10 if dtype == torch.float64 else 2e-3
        assert max(worst.values()) <= tol and serr <= tol, (name, ts, n, worst, serr)
        if n == big and dtype == torch.float64:
            monkeypatch.delenv("NOC_GRAD_TS")                 # the host's own choice of tiling on the same rows
            Gd, sd = kernel_vjp(net, s, a, B)
            monkeypatch.setenv("NOC_GRAD_TS", str(ts))
            assert float((sd - sk).abs().max()) <= 1e-13 * float(sk.abs().max())        # per-row arithmetic: tiling-independent
            assert max(_worst(Gd, Gk).values()) <= 1e-12                                  # sums: atomics order only


# ---------------------------------------------------------------------------------------------------------------------------
# 4. NULL seeds and outputs through the C ABI
# ---------------------------------------------------------------------------------------------------------------------------
def test_vjp_null_seeds_and_outputs():
    import neuraloc_b200 as nb
    from neuraloc_b200.ocflow import _phi_struct, _grad_len
    L = nb._cabi.lib()
    # a random net, not a trained one: without the seed on Phi the gradient of N.layers.1.bias is h w (1 - tanh^2) times the tangent,
    # and on the saturated units of the checkpoints the oracle's autograd forms 1 - tanh^2 with cancellation (DESIGN.md 3.6)
    net, P, xinit, var0 = _build((24, 6), torch.float64)
    n = 29
    s = rows(xinit, var0, n, 41).cuda()
    a, B = [t.cuda() for t in seeds(n, s.shape[1], 42)]
    dev = s.device
    phi = _phi_struct(net, dev, torch.float64)
    stream = torch.cuda.current_stream(dev).cuda_stream
    gp = torch.full((_grad_len(phi),), float("nan"), dtype=torch.float64, device=dev)
    gs = torch.full_like(s, float("nan"))

    def call(a_, B_, gp_, gs_):
        p = lambda t: None if t is None else t.data_ptr()
        return L.noc_phi_vjp(C.byref(phi), s.data_ptr(), n, p(a_), p(B_), nb._cabi.F64, p(gp_), p(gs_), stream)

    # a only: grad_s = a * getGrad(s); no parameter output
    nb._cabi.check(call(a, None, None, gs))
    with torch.no_grad():
        g = net.getGrad(s)
    ref = a.reshape(-1, 1) * g
    assert float((gs - ref).abs().max()) <= 1e-11 * float(ref.abs().max())
    assert torch.isnan(gp).all()                                    # NULL output: not written
    # B only: the beta (Phi itself) terms are left out
    nb._cabi.check(call(None, B, gp, gs))
    Gr, sr = oracle_vjp(P, s.cpu(), None, B.cpu())
    Gk = {k: v.cpu() for k, v in zip(ORDER, nb.split_param_grads(net, gp))}
    assert max(_worst(Gk, Gr).values()) <= 1e-10
    assert float((gs.cpu() - sr).abs().max()) <= 1e-10 * float(sr.abs().max())
    gs0 = gs.clone()
    nb._cabi.check(call(torch.zeros_like(a), B, gp, gs))                  # NULL means zero
    assert max(_worst({k: v.cpu() for k, v in zip(ORDER, nb.split_param_grads(net, gp))}, Gk).values()) <= 1e-14
    assert torch.equal(gs, gs0)
    # both seeds NULL: zero gradients; both outputs NULL: nothing to do
    nb._cabi.check(call(None, None, gp, gs))
    assert not gp.any() and not gs.any()
    assert call(a, B, None, None) == 0
    # nTh = 3: unsupported, with a message
    net3 = nb.Phi(nTh=3, m=8, d=4).double().cuda()
    phi3 = _phi_struct(net3, dev, torch.float64)
    s3 = torch.zeros(3, 5, dtype=torch.float64, device=dev)
    rc = L.noc_phi_vjp(C.byref(phi3), s3.data_ptr(), 3, None, None, nb._cabi.F64, None, s3.data_ptr(), stream)
    assert rc == -2 and b"nTh = 3" in L.noc_last_error()


# ---------------------------------------------------------------------------------------------------------------------------
# 5. composition with the training rollout, and a short training run against CPU autograd
# ---------------------------------------------------------------------------------------------------------------------------
LAM, MU = 1e-4, 0.01


def _setup_training():
    import neuraloc_b200 as nb
    _, meta0 = load_ckpt("softcorridor")
    alph = meta0["alph"]
    torch.manual_seed(3)
    net_gpu = nb.Phi(nTh=2, m=32, d=4, alph=alph).double()
    net_cpu = copy.deepcopy(net_gpu)
    net_gpu = net_gpu.cuda()
    prob, _, _, _ = nb.initProb("softcorridor", 2, 2, var0=1.0, alph=alph, cvt=lambda v: v.double().cuda())
    prob.train()
    D, xi = orc.make_problem("softcorridor", alph, torch.float64)
    D = dataclasses.replace(D, training=True)
    g = torch.Generator().manual_seed(9)
    x = xi + torch.randn(128, 4, generator=g, dtype=torch.float64)
    sc = torch.cat((x, torch.rand(128, 1, generator=g, dtype=torch.float64)), 1)      # collocation points for the gradient penalty
    return net_gpu, net_cpu, prob, D, x, sc, alph


def _loss_gpu(net, prob, x, sc, alph, nt):
    import neuraloc_b200 as nb
    xc, scc = x.cuda(), sc.cuda()
    Jc, _ = nb.OCflow(xc, net, prob, tspan=[0.0, 1.0], nt=nt, stepper="rk4", alph=alph)
    s1 = torch.cat((xc, torch.ones(xc.shape[0], 1, dtype=xc.dtype, device=xc.device)), 1)
    G = 0.5 * ((xc - prob.xtarget.reshape(1, -1)) ** 2).sum(1, keepdim=True)
    term = LAM * ((net(s1) - alph[0] * G) ** 2).mean()
    pen = MU * (net.getGrad(scc) ** 2).sum(1).mean()
    return Jc + term + pen


def _loss_cpu(net, D, x, sc, alph, nt):
    Pg = orc.PhiParams(net.A, net.c.weight, net.c.bias, net.w.weight, [l.weight for l in net.N.layers],
                       [l.bias for l in net.N.layers], net.N.h)
    Jc, _ = orc.ocflow(x, Pg, D, [0.0, 1.0], nt, "rk4", alph)
    s1 = torch.cat((x, torch.ones(x.shape[0], 1, dtype=x.dtype)), 1)
    G = 0.5 * ((x - D.xtarget.reshape(1, -1)) ** 2).sum(1, keepdim=True)
    term = LAM * ((orc.phi_forward(Pg, s1) - alph[0] * G) ** 2).mean()
    pen = MU * (orc.phi_grad(Pg, sc) ** 2).sum(1).mean()
    return Jc + term + pen


def test_phi_terms_compose_with_training_rollout():
    """Jc of a training OCflow call + a terminal-condition fit on Phi + a penalty on getGrad: one backward() accumulates all three
    into .grad, equal to CPU autograd of the same loss; the Phi terms do contribute."""
    net_gpu, net_cpu, prob, D, x, sc, alph = _setup_training()
    nt = 8
    loss = _loss_gpu(net_gpu, prob, x, sc, alph, nt)
    loss.backward()
    ref = _loss_cpu(net_cpu, D, x, sc, alph, nt)
    ref.backward()
    assert abs(float(loss.detach()) - float(ref.detach())) <= 1e-10 * abs(float(ref.detach()))
    import neuraloc_b200 as nb
    Jc, _ = nb.OCflow(x.cuda(), net_gpu, prob, tspan=[0.0, 1.0], nt=nt, stepper="rk4", alph=alph)
    only_jc = torch.autograd.grad(Jc, list(net_gpu.parameters()))
    for pg, pc, gj in zip(net_gpu.parameters(), net_cpu.parameters(), only_jc):
        scale = max(float(pc.grad.abs().max()), 1e-30)
        assert float((pg.grad.cpu() - pc.grad).abs().max()) <= 1e-9 * scale
    assert any(float((pg.grad - gj).abs().max()) > 1e-6 * max(float(pg.grad.abs().max()), 1e-30)
               for pg, gj in zip(net_gpu.parameters(), only_jc))


def test_short_training_run_with_phi_terms_matches_cpu_autograd():
    """20 Adam iterations of Jc + terminal fit + gradient penalty on the GPU and on the CPU (oracle autograd), fp64, from the same
    initialisation: the loss histories and the final weights agree."""
    net_gpu, net_cpu, prob, D, x, sc, alph = _setup_training()
    nt, iters = 8, 20
    hist = {}
    for tag, net in (("gpu", net_gpu), ("cpu", net_cpu)):
        optim = torch.optim.Adam(net.parameters(), lr=0.01)
        losses = []
        for _ in range(iters):
            optim.zero_grad()
            loss = _loss_gpu(net, prob, x, sc, alph, nt) if tag == "gpu" else _loss_cpu(net, D, x, sc, alph, nt)
            loss.backward()
            optim.step()
            losses.append(float(loss.detach()))
        hist[tag] = losses
    a, b = np.array(hist["gpu"]), np.array(hist["cpu"])
    assert b[-1] < b[0]
    assert np.abs(a - b).max() <= 1e-7 * np.abs(b).max(), (a, b)
    for pg, pc in zip(net_gpu.parameters(), net_cpu.parameters()):
        assert float((pg.detach().cpu() - pc.detach()).abs().max()) <= 1e-7 * max(float(pc.detach().abs().max()), 1e-30)


def test_input_gradient_and_cpu_inputs():
    """d/ds through net(s) and net.getGrad(s) with s on the CPU in fp64 and the parameters fp32 on the GPU (the computation runs in
    s.dtype, as the forward does): every gradient comes back on its own tensor's device and in its dtype"""
    net, P, xinit, var0 = _build("softcorridor", torch.float32)
    s = rows(xinit, var0, 9, 51).requires_grad_(True)
    B = seeds(9, 5, 52)[1]
    y = (net(s) * 2.0).sum() + (net.getGrad(s) * B).sum()
    y.backward()
    assert s.grad.device.type == "cpu" and s.grad.dtype == torch.float64
    P64 = P.to(torch.float32).to(torch.float64)
    Gr, sr = oracle_vjp(P64, s.detach(), torch.full((9,), 2.0, dtype=torch.float64), B)
    assert float((s.grad - sr).abs().max()) <= 1e-10 * float(sr.abs().max())
    for k, p in zip(ORDER, [net.A, net.c.weight, net.c.bias, net.w.weight, net.N.layers[0].weight, net.N.layers[1].weight,
                            net.N.layers[0].bias, net.N.layers[1].bias]):
        assert p.grad is not None and p.grad.device.type == "cuda" and p.grad.dtype == torch.float32
        ref = Gr[k].reshape(p.shape)
        assert float((p.grad.double().cpu() - ref).abs().max()) <= 1e-6 * max(float(ref.abs().max()), 1e-30), k


# ---------------------------------------------------------------------------------------------------------------------------
# 6. loud failures
# ---------------------------------------------------------------------------------------------------------------------------
def test_double_backward_raises():
    net, P, xinit, var0 = _build("softcorridor", torch.float64)
    s = rows(xinit, var0, 5, 61).cuda().requires_grad_(True)
    gs, = torch.autograd.grad(net(s).sum(), s, create_graph=True)
    with pytest.raises(RuntimeError):
        gs.sum().backward()
    gp = torch.autograd.grad(net.getGrad(s).sum(), list(net.parameters()), create_graph=True)
    with pytest.raises(RuntimeError):
        sum(g.sum() for g in gp).backward()


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_deeper_net_raises_under_autograd_and_evaluates_under_no_grad(tag):
    import neuraloc_b200 as nb
    z = np.load(GOLDEN + "/phi_random.npz")
    pre = "net1_"
    nTh, m, d = [int(v) for v in z[pre + "dims"]]
    assert nTh == 3
    net = nb.Phi(nTh=nTh, m=m, d=d)
    net.load_state_dict({k[len(pre):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(pre) and ("." in k or k == pre + "A")})
    net = net.to(DT[tag]).cuda()
    x = torch.from_numpy(z[pre + "x"]).to(DT[tag]).cuda()
    with pytest.raises(RuntimeError, match="nTh = 2"):
        net(x)
    with pytest.raises(RuntimeError, match="nTh = 2"):
        net.getGrad(x.clone().requires_grad_(True))
    with torch.no_grad():
        f, g = net(x), net.getGrad(x)
    tol = 5e-6 if tag == "f32" else 1e-12
    assert rel_err(f.cpu().numpy(), z[pre + "fwd_" + tag], floor=1.0) <= tol
    assert rel_err(g.cpu().numpy(), z[pre + "grad_" + tag], floor=1.0) <= tol


def test_problem_evaluators_refuse_gradients():
    import neuraloc_b200 as nb
    net, prob, xinit, meta = product_setup("softcorridor", torch.float64)
    g = torch.Generator().manual_seed(71)
    x = (xinit.cpu() + torch.randn(6, 4, generator=g, dtype=torch.float64)).cuda()
    p = torch.randn(6, 4, generator=g, dtype=torch.float64).cuda()
    z = torch.cat((x, torch.zeros(6, 4, dtype=torch.float64, device=x.device)), 1)
    with torch.no_grad():
        lhqw0, f0 = prob.calcLHQW(x, p), nb.ocOdefun(z, 0.3, net, prob)
    with pytest.raises(RuntimeError, match="forward-only"):
        prob.calcLHQW(x, p.clone().requires_grad_(True))
    with pytest.raises(RuntimeError, match="forward-only"):
        prob.calcGradpH(x.clone().requires_grad_(True), p)
    with pytest.raises(RuntimeError, match="forward-only"):
        prob.calcLHQW(x, net.getGrad(torch.cat((x, torch.ones(6, 1, dtype=x.dtype, device=x.device)), 1))[:, :4])
    with pytest.raises(RuntimeError, match="forward-only"):
        nb.ocOdefun(z, 0.3, net, prob)                                   # the net's parameters require grad
    with pytest.raises(RuntimeError, match="forward-only"):
        nb.ocOdefun(z.clone().requires_grad_(True), 0.3, net.requires_grad_(False), prob)
    # plain tensors with grad mode on: as before
    lhqw1 = prob.calcLHQW(x, p)
    f1 = nb.ocOdefun(z, 0.3, net, prob)                                  # parameters no longer require grad
    assert all(torch.equal(u, v) for u, v in zip(lhqw1, lhqw0)) and torch.equal(f1, f0)

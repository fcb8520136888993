"""The small-batch rollout kernels at every cluster size and on the problem shapes no checkpoint reaches.

Batches up to NOC_VEC_MAX samples (the batch-1 calls of evalOC.py / timeOC.py among them) run one thread-block cluster per sample
(noc_lat.cu) or, where the cluster kernel does not apply, one CTA per sample (noc_vec.cu).  Here both run on randomly initialised
value nets whose widths leave padded units and padded gradient components in the cluster slices (whole CTAs of padding included),
on midcross2, midcross20, midcross30, the 32-agent swarm and two quadcopters (the nAgents == 2 interaction term), in eval and
train mode, and are compared with the fp64 CPU oracle, with each other and with the FMA tile kernel.  Every case proves which
kernel ran: the cluster size from the NOC_DEBUG line of noc_lat.cu, its absence where noc_vec.cu must take the call, and
noc_last_path() for the tile kernel."""
import copy
import dataclasses
import re

import numpy as np
import pytest
import torch

from helpers import QW, check_costs, rel_state_err
from oracle import ocflow_oracle as orc

pytestmark = pytest.mark.gpu

ALPH = [300.0, 2.5, 7.0, 1.0, 1.0, 1.0]       # non-zero Q and W weights
N = 160                                      # > 148 one-CTA clusters: every cluster loops over several samples
NT = 6
DT = {"f32": torch.float32, "f64": torch.float64}
TOL = {"f32": dict(state=1e-5, cost=1e-4, floor=2e-4, ctrl=2e-4, rows=1e-4, flips=2),
       "f64": dict(state=1e-11, cost=1e-9, floor=1e-10, ctrl=1e-9, rows=1e-9, flips=0)}
SHAPES = {"midcross2": ("Cross2D", 4), "midcross20": ("Cross2D", 40), "midcross30": ("Cross2D", 60),
          "swarm": ("SwarmTraj", 96), "quad2": ("Quadcopter", 24)}
MODES = ("eval", "train")

# Variants: "ncK" = the cluster kernel pinned to K CTAs (NOC_LAT_NC), "lat" = the cluster kernel choosing its own size (a
# multi-CTA one is expected), "vec" = noc_vec.cu (NOC_NO_LAT), "fallback" = the library's own choice, which must fall through
# from the cluster kernel to noc_vec.cu, "tile" = the FMA tile kernel.
ALL = ["nc1", "nc2", "nc4", "nc8", "nc16", "vec", "tile"]
NO1 = ALL[1:]
WIDE = ["lat", "nc8", "nc16", "vec", "tile"]
# shape -> [(m, nTh, n, {tag: variants})].  Cluster slices hold mc = align_up(ceil(m / NC), 4 (fp32) | 2 (fp64)) units:
#   m = 90: padded units at every NC > 1 and the last rank owns real units at NC = 4 and 8 (72..89 and 84..89); fp64 only fits
#           one CTA for d <= 24.
#   m = 20: at NC = 16 the fp32 ranks 5..15 and the fp64 ranks 10..15 hold nothing but padding.
#   m = 256 (fp32) / 128 (fp64) on the wide shapes: no single CTA holds the slices, the kernel picks a cluster of 4.
#   m = 1000: no cluster fits; noc_vec.cu with weights read from L2, 1024 threads of which 24 idle.
#   nTh = 3: only noc_vec.cu and the tile kernel take it (3 and 4 warps, the last one ragged).
CASES = {
    "midcross2": [(90, 2, N, {"f32": ALL, "f64": ALL}), (20, 2, N, {"f32": ALL, "f64": ALL})],
    "midcross20": [(90, 2, N, {"f32": ALL, "f64": NO1}), (20, 2, N, {"f32": ALL, "f64": ALL})],
    "midcross30": [(90, 2, N, {"f32": ALL, "f64": NO1}), (256, 2, N, {"f32": WIDE}), (128, 2, N, {"f64": WIDE}),
                   (70, 3, N, {"f32": ["fallback", "vec", "tile"], "f64": ["fallback", "vec", "tile"]})],
    "swarm": [(90, 2, N, {"f32": ALL, "f64": NO1}), (20, 2, N, {"f32": ALL, "f64": ALL}), (256, 2, N, {"f32": WIDE}),
              (128, 2, N, {"f64": WIDE}), (70, 3, N, {"f32": ["fallback", "vec", "tile"], "f64": ["fallback", "vec", "tile"]}),
              (1000, 2, 24, {"f32": ["fallback", "vec"], "f64": ["fallback", "vec"]})],
    "quad2": [(90, 2, N, {"f32": ALL, "f64": ALL}), (20, 2, N, {"f32": ALL, "f64": ALL})],
}
LAT_LINE = re.compile(r"\[noc\] latency kernel: cluster of (\d+), (\d+) units \+ (\d+) components per CTA, smem \d+ B, (\d+) clusters")
RAN = []              # (tag, shape, mode, NC, units per CTA, m): what the cluster kernel reported, for the coverage summary
_ORACLE = {}          # oracle results, shared by every kernel variant and both precisions of a case


@pytest.fixture(scope="module")
def nb():
    import neuraloc_b200
    neuraloc_b200._cabi.lib()
    assert torch.cuda.is_available()
    return neuraloc_b200


def quad2_target():
    return torch.tensor([2.0, 2.0, 2.0] + [0.0] * 9 + [2.0, -2.0, 2.0] + [0.0] * 9, dtype=torch.float64)


def make_problem(nb, name, dtype, mode):
    """-> (product problem on the GPU in `dtype`, fp64 oracle ProbDesc), both in `mode`."""
    cvt = lambda v: v.to(dtype).cuda()
    if name == "quad2":
        prob = nb.Quadcopter(cvt(quad2_target()), alph_Q=0.0, alph_W=ALPH[2], r=1.0)
        D = orc.ProbDesc("Quadcopter", quad2_target(), None, 0.0, ALPH[2], 1.0, nAgents=2, agentDim=12)
    else:
        prob = nb.initProb(name, 2, 2, 1.0, ALPH, cvt)[0]
        D = orc.make_problem(name, ALPH, torch.float64)[0]
    getattr(prob, mode)()
    return prob, dataclasses.replace(D, training=(mode == "train"))


def quad2_near_rows(n):
    return torch.arange(n) % 2 == 0


def initial_states(name, n, seed=7):
    """fp32-representable rows (the fp64 oracle then sees exactly what both precisions roll out).  Some agent pairs are squeezed
    inside the interaction cut-off; for two quadcopters every other row starts with both within 2r = 2 of each other."""
    g = torch.Generator().manual_seed(seed)
    if name == "quad2":
        x = 0.1 * torch.randn(n, 24, generator=g, dtype=torch.float64)
        x[:, 0:3] = -1.5 + 0.5 * torch.randn(n, 3, generator=g, dtype=torch.float64)
        x[:, 12:15] = 1.5 + 0.5 * torch.randn(n, 3, generator=g, dtype=torch.float64)
        near = quad2_near_rows(n)
        off = torch.randn(int(near.sum()), 3, generator=g, dtype=torch.float64)
        off *= (0.2 + 1.4 * torch.rand(off.shape[0], 1, generator=g, dtype=torch.float64)) / off.norm(dim=1, keepdim=True)
        x[near, 12:15] = x[near, 0:3] + off
        return x.float()
    D, xi = orc.make_problem(name, ALPH, torch.float64)
    x = xi + 0.3 * torch.randn(n, xi.shape[1], generator=g, dtype=torch.float64)
    A, dim = D.nAgents, D.agentDim
    xa = x.view(n, A, dim)
    for k in range(min(3, A // 2)):
        xa[: n // 3, 2 * k + 1] = xa[: n // 3, 2 * k] + D.r * 1.5 * torch.rand(n // 3, dim, generator=g, dtype=torch.float64)
    return x.float()


def make_net(nb, d, m, nTh):
    """Random Phi (fp32 weights) with modest hidden weights, std 0.2 (scaled down beyond 90 units so that grad Phi stays O(1))."""
    torch.manual_seed(1000 * nTh + m + d)
    net = nb.Phi(nTh=nTh, m=m, d=d, alph=ALPH)
    s = min(1.0, (90.0 / m) ** 0.5)
    with torch.no_grad():
        for lay in net.N.layers[1:]:
            lay.weight.normal_(std=0.2 * s)
            lay.bias.normal_()
        net.w.weight.normal_(std=s)
        net.c.weight.normal_()
        net.c.bias.normal_()
    return net


def oracle(key, x, net, D, prec, tspan, nt, stepper):
    """(per-sample table [n, 8], zFull, ctrlFull) of the CPU oracle in `prec`, as float64 arrays; computed once per case."""
    key = key + (prec, tuple(tspan), nt, stepper)
    if key not in _ORACLE:
        P = orc.params_from_state_dict(net.state_dict(), prec)
        Dp = D.to(prec)
        xp = x.to(prec)
        with torch.no_grad():
            J, cs = orc.ocflow(xp, P, Dp, tspan, nt, stepper, ALPH, noMean=True)
            z, c = orc.ocflow(xp, P, Dp, tspan, nt, stepper, ALPH, intermediates=True)
        _ORACLE[key] = (torch.cat([J] + cs, 1).double().numpy(), z.double().numpy(), c.double().numpy())
    return _ORACLE[key]


def run_variant(nb, monkeypatch, capfd, variant, x, net, prob, tspan, nt, stepper):
    """All three return modes through one kernel variant -> ((mean, noMean table, zFull, ctrlFull), cluster report or None)."""
    for k in ("NOC_FORCE_PATH", "NOC_LAT_NC", "NOC_NO_LAT", "NOC_VEC_MAX", "NOC_TC", "NOC_FORCE_CFG"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("NOC_DEBUG", "1")
    if variant == "tile":
        monkeypatch.setenv("NOC_FORCE_PATH", "tile")
    elif variant != "fallback":
        monkeypatch.setenv("NOC_FORCE_PATH", "vec")
    if variant == "vec":
        monkeypatch.setenv("NOC_NO_LAT", "1")
    if variant.startswith("nc"):
        monkeypatch.setenv("NOC_LAT_NC", variant[2:])
    capfd.readouterr()
    with torch.no_grad():
        Jc, cs = nb.OCflow(x, net, prob, tspan, nt, stepper, ALPH)
        path = nb._cabi.last_path()
        Jn, cn = nb.OCflow(x, net, prob, tspan, nt, stepper, ALPH, noMean=True)
        zf, cf = nb.OCflow(x, net, prob, tspan, nt, stepper, ALPH, intermediates=True)
    lines = LAT_LINE.findall(capfd.readouterr().err)
    got = (np.array([float(Jc)] + [float(c) for c in cs]), torch.cat([Jn] + list(cn), 1).double().cpu().numpy(),
           zf.double().cpu().numpy(), cf.double().cpu().numpy())
    assert path == ("tile" if variant == "tile" else "sample"), (variant, path)
    if variant in ("tile", "vec", "fallback"):
        assert not lines, "%s: the cluster kernel ran: %s" % (variant, lines)
        return got, None
    assert len(lines) == 3, "%s: expected one cluster-kernel line per call, got %s" % (variant, lines)
    rep = [tuple(int(v) for v in ln) for ln in lines]
    assert len(set(rep)) == 1, rep
    nc, mc, dc, ncl = rep[0]
    if variant == "lat":
        assert nc >= 2, "the cluster kernel picked %d CTA(s) for a net that does not fit one" % nc
    else:
        assert nc == int(variant[2:]), "asked for a cluster of %s CTAs, the kernel ran %d" % (variant[2:], nc)
    assert x.shape[0] > ncl, "%d samples on %d clusters: no cluster loops over samples" % (x.shape[0], ncl)
    return got, (nc, mc, dc, ncl)


def bad_rows(tag, table, ref, noise=None):
    """Rows of a per-sample cost table [n, 8] off `ref` by more than the row tolerance, relative to the column's largest entry
    (at least 1), or 3x the fp32 oracle's own distance from the fp64 oracle in that column (fp32 runs)."""
    sc = np.maximum(np.abs(ref).max(axis=0), 1.0)
    lim = np.full(ref.shape[1], TOL[tag]["rows"])
    if noise is not None:
        lim = np.maximum(lim, 3.0 * (np.abs(noise - ref) / sc).max(axis=0))
    return ((np.abs(table - ref) / sc) > lim).any(axis=1)


def path_cost_rows(tag, z, zref, d, znoise=None):
    """The same for the cost integrals along the path (zFull rows d..d+3, every step)."""
    a, r = z[:, d:, :], zref[:, d:, :]
    sc = np.maximum(np.abs(r).max(axis=(0, 2)), 1.0)[None, :, None]
    lim = np.full((1, 4, 1), TOL[tag]["rows"])
    if znoise is not None:
        lim = np.maximum(lim, 3.0 * (np.abs(znoise[:, d:, :] - r) / sc).max(axis=(0, 2))[None, :, None])
    return ((np.abs(a - r) / sc) > lim).any(axis=(1, 2))


def check_vs_oracle(tag, d, got, truth, noise, what):
    """fp64: state 1e-11, controls / per-sample costs / means 1e-9 relative.  fp32: state within max(1e-5, 2x the fp32 oracle's own
    distance), costs 1e-4 relative with an absolute floor for Q and W only, at most two rows off (a pair within rounding of a
    cut-off lands on either side)."""
    tol = TOL[tag]
    mean, table, zf, cf = got
    tn, tz, tc = truth
    assert zf.shape == tz.shape and cf.shape == tc.shape, what
    stol, ctol = tol["state"], tol["ctrl"]
    if noise is not None:
        stol = max(stol, 2 * rel_state_err(noise[1], tz, d))
        ctol = max(ctol, 2 * np.abs(noise[2] - tc).max() / max(np.abs(tc).max(), 1.0))
    serr = rel_state_err(zf, tz, d)
    assert serr <= stol, "%s: per-step state rel err %.3e (limit %.3e)" % (what, serr, stol)
    assert not cf[:, :, 0].any(), what
    cerr = np.abs(cf - tc).max() / max(np.abs(tc).max(), 1.0)
    assert cerr <= ctol, "%s: controls rel err %.3e (limit %.3e)" % (what, cerr, ctol)
    bad = bad_rows(tag, table, tn, None if noise is None else noise[0]) | \
        path_cost_rows(tag, zf, tz, d, None if noise is None else noise[1])
    assert bad.sum() <= tol["flips"], "%s: per-sample costs off on rows %s: got %s, oracle %s" % (
        what, np.nonzero(bad)[0][:8], table[bad][:2], tn[bad][:2])
    ref = tn.copy()
    ref[bad] = table[bad]                  # a flipped row counts as the kernel has it in the mean as well
    check_costs(mean, ref.mean(axis=0), tol["cost"], tol["floor"], what + ": mean costs", floor_mask=QW,
                ref_noise=None if noise is None else noise[0].mean(axis=0) - tn.mean(axis=0))
    return bad


def check_across(tag, tables, noise_tab, truth_tab, what):
    """Per-sample tables of every variant agree with each other to the row tolerance."""
    names = list(tables)
    for v in names[1:]:
        noise = None if noise_tab is None else tables[names[0]] + (noise_tab - truth_tab)
        bad = bad_rows(tag, tables[v], tables[names[0]], noise)
        assert bad.sum() <= TOL[tag]["flips"], "%s: %s and %s disagree on rows %s" % (what, v, names[0], np.nonzero(bad)[0][:8])


def run_case(nb, monkeypatch, capfd, shape, tag, mode, m, nTh, n, variants, tspan=(0.0, 1.0), nt=NT, stepper="rk4"):
    tspan = list(tspan)
    kind, d = SHAPES[shape]
    x = initial_states(shape, n)
    net = make_net(nb, d, m, nTh)
    prob, D = make_problem(nb, shape, DT[tag], mode)
    key = (shape, m, nTh, n, mode)
    truth = oracle(key, x, net, D, torch.float64, tspan, nt, stepper)
    noise = oracle(key, x, net, D, torch.float32, tspan, nt, stepper) if tag == "f32" else None
    live_w = shape == "quad2" and stepper != "none"      # the interaction term is live on the rows that start close
    if live_w:
        assert (truth[0][quad2_near_rows(n).numpy(), 7] > 0).all()
    netd = copy.deepcopy(net).to(DT[tag]).cuda()
    xd = x.to(DT[tag]).cuda()
    tables = {}
    for v in variants:
        what = "%s %s %s m=%d nTh=%d %s [%s nt=%d %s]" % (shape, tag, mode, m, nTh, v, stepper, nt, tspan)
        got, rep = run_variant(nb, monkeypatch, capfd, v, xd, netd, prob, tspan, nt, stepper)
        check_vs_oracle(tag, d, got, truth, noise, what)
        if live_w:
            assert (got[1][quad2_near_rows(n).numpy(), 7] > 0).all(), what + ": W is zero on rows with both quadcopters close"
        if rep is not None:
            RAN.append((tag, shape, mode, rep[0], rep[1], m))
        tables[v] = got[1]
    check_across(tag, tables, None if noise is None else noise[0], truth[0], "%s %s %s m=%d nTh=%d" % (shape, tag, mode, m, nTh))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("tag", ["f32", "f64"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_small_batch_rollouts_vs_oracle(nb, monkeypatch, capfd, shape, tag, mode):
    """Every net of CASES[shape] through every listed variant, three return modes, against the oracle and each other."""
    for m, nTh, n, per_tag in CASES[shape]:
        if tag in per_tag:
            run_case(nb, monkeypatch, capfd, shape, tag, mode, m, nTh, n, per_tag[tag])


# (stepper, nt, tspan): Euler, no stepper, one step, and a late start with an odd step count
STEPPINGS = [("rk1", 5, (0.0, 1.0)), ("none", 3, (0.0, 1.0)), ("rk4", 1, (0.0, 1.0)), ("rk4", 7, (0.3, 1.0))]
PIN = {"midcross2": "nc2", "midcross20": "nc4", "midcross30": "nc8", "swarm": "nc16", "quad2": "nc4"}


@pytest.mark.parametrize("tag", ["f32", "f64"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_small_batch_steppers_and_time_spans(nb, monkeypatch, capfd, shape, tag):
    """rk1, no stepper, nt = 1 and tspan = [0.3, 1] through a pinned cluster, noc_vec.cu and the tile kernel (m = 90, train mode)."""
    for stepper, nt, tspan in STEPPINGS:
        run_case(nb, monkeypatch, capfd, shape, tag, "train", 90, 2, N, [PIN[shape], "vec", "tile"], tspan, nt, stepper)


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_widths_without_a_kernel_fail_loudly(nb, monkeypatch, tag):
    """No tile configuration holds more than 512 hidden units (the widest ones stream PB = 512 outputs per pass), so a wide net
    that the batch size or m > 1024 sends to the tile kernel must raise NocError -4, not return numbers."""
    for k in ("NOC_FORCE_PATH", "NOC_LAT_NC", "NOC_NO_LAT", "NOC_VEC_MAX", "NOC_TC", "NOC_FORCE_CFG"):
        monkeypatch.delenv(k, raising=False)
    prob, _ = make_problem(nb, "swarm", DT[tag], "eval")
    net = make_net(nb, 96, 1000, 2).to(DT[tag]).cuda()
    x = initial_states("swarm", 300).to(DT[tag]).cuda()          # > NOC_VEC_MAX (256): the tile kernel
    for kw in ({}, {"noMean": True}, {"intermediates": True}):
        with torch.no_grad(), pytest.raises(nb._cabi.NocError, match="noc error -4"):
            nb.OCflow(x, net, prob, [0.0, 1.0], 2, "rk4", ALPH, **kw)
    monkeypatch.setenv("NOC_FORCE_PATH", "vec")                  # m > 1024: one CTA per sample cannot hold a thread per unit
    prob, _ = make_problem(nb, "midcross2", DT[tag], "eval")
    net = make_net(nb, 4, 1100, 2).to(DT[tag]).cuda()
    x = initial_states("midcross2", 3).to(DT[tag]).cuda()
    for kw in ({}, {"noMean": True}, {"intermediates": True}):
        with torch.no_grad(), pytest.raises(nb._cabi.NocError, match="noc error -4"):
            nb.OCflow(x, net, prob, [0.0, 1.0], 2, "rk4", ALPH, **kw)


@pytest.mark.parametrize("tag", ["f32", "f64"])
@pytest.mark.parametrize("name", ["midcross20", "midcross30", "quad2"])
def test_functors_on_the_new_shapes(nb, name, tag):
    """calcLHQW / calcGradpH / calcCtrls (noc_prob_eval) against the oracle on 300 random (x, p) rows, eval and train mode."""
    dtype = DT[tag]
    n, d = 300, SHAPES[name][1]
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    if name == "quad2":
        x = initial_states(name, n).double()
    else:
        _, xi = orc.make_problem(name, ALPH, torch.float64)
        x = xi + 0.7 * torch.randn(n, d, generator=g, dtype=torch.float64)
        D0 = orc.make_problem(name, ALPH, torch.float64)[0]
        xa = x.view(n, D0.nAgents, 2)
        xa[: n // 3, 1] = xa[: n // 3, 0] + D0.r * 1.5 * torch.rand(n // 3, 2, generator=g, dtype=torch.float64)
    p = 1.5 * torch.randn(n, d, generator=g, dtype=torch.float64)
    x, p = x.to(dtype), p.to(dtype)
    tol = 2e-5 if tag == "f32" else 1e-11
    for mode in MODES:
        prob, D = make_problem(nb, name, dtype, mode)
        L, H, Q, W = prob.calcLHQW(x.cuda(), p.cuda())
        Lr, Hr, Qr, Wr = orc.lhqw(D, x.double(), p.double())
        for got, ref, nm in ((L, Lr, "L"), (H, Hr, "H"), (Q, Qr, "Q"), (W, Wr, "W")):
            ref = ref.reshape(-1).numpy() if torch.is_tensor(ref) else np.zeros(n)
            got = got.reshape(-1).double().cpu().numpy()
            err = np.abs(got - ref) / np.maximum(np.abs(ref), 1.0)
            assert (err > tol).sum() <= (2 if tag == "f32" else 0), (name, mode, nm, err.max())
            if nm == "W":
                assert (ref > 0).sum() >= n // 4 and (got > 0).sum() >= n // 4, (name, mode, "W is rarely live")
        gr =orc.grad_p_hamiltonian(D, x.double(), p.double()).numpy()
        gg = prob.calcGradpH(x.cuda(), p.cuda()).double().cpu().numpy()
        assert (np.abs(gg - gr) / np.maximum(np.abs(gr), 1.0)).max() <= tol, (name, mode, "grad_p H")
        cr = orc.controls(D, x.double(), p.double()).numpy()
        cg = prob.calcCtrls(x.cuda(), p.cuda()).double().cpu().numpy()
        assert (np.abs(cg - cr) / np.maximum(np.abs(cr), 1.0)).max() <= tol, (name, mode, "controls")


def test_every_cluster_size_ran_in_both_precisions():
    """Summary of what the cluster kernel reported in this session; with the whole rollout test run, every cluster size must have
    run in both precisions on a Cross2D and a SwarmTraj shape, at NC = 4 and 8 with real units on the last rank, at NC = 16
    with CTAs that hold only padding, and the two quadcopters on a multi-CTA cluster."""
    if len({(t, s, md) for t, s, md, *_ in RAN}) < 2 * len(SHAPES) * len(MODES):
        pytest.skip("the rollout tests did not all run in this session")
    for tag in ("f32", "f64"):
        for nc in (1, 2, 4, 8, 16):
            runs = [(s, m, mc) for t, s, _, k, mc, m in RAN if t == tag and k == nc]
            kinds = sorted({SHAPES[s][0] for s, _, _ in runs})
            print("%s NC=%-2d  %s" % (tag, nc, ", ".join(sorted({"%s m=%d (%d units/CTA)" % r for r in runs}))))
            assert {"Cross2D", "SwarmTraj"} <= set(kinds), (tag, nc, kinds)
            if nc in (4, 8):
                assert any((nc - 1) * mc < m for _, m, mc in runs), (tag, nc, "no run with real units on the last rank")
        assert any(s == "quad2" and k >= 2 for t, s, _, k, _, _ in RAN if t == tag), tag
    assert any(k == 16 and -(-m // mc) < 16 for t, s, _, k, mc, m in RAN if t == "f32"), "no fp32 CTA of pure padding"

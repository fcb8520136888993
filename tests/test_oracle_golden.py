"""Pin the CPU oracle (oracle/ocflow_oracle.py) against outputs of the unmodified reference.

The reference has no tests or golden vectors of its own (SURVEY.md §4); the fixtures under
tests/golden/ were produced by tests/golden/make_golden.py importing /root/reference."""
import json

import numpy as np
import pytest
import torch

from oracle import ocflow_oracle as orc
from helpers import DT, GOLDEN, PROBLEMS, load_cases, load_ckpt, oracle_setup, rel_err, rel_state_err

TOL = {"f32": dict(state=2e-6, cost=2e-5, abs=2e-5), "f64": dict(state=1e-12, cost=1e-10, abs=1e-11)}


def _mean_vec(out):
    Jc, cs = out
    return np.array([float(Jc)] + [float(c) for c in cs])


def _fp32_noise(c, key, tag, axes=()):
    """Twice the reference's own fp32 rounding on fixture `key`: 2 |fp32 run - fp64 run| per entry, or its maximum over
    `axes` (e.g. over the samples and control components of one time step); zeros for fp64.  fp32 sums round differently
    with the host's BLAS kernels and thread count, so the oracle's fp32 run on another machine differs from the stored
    fp32 run by rounding of that size."""
    r32, r64 = np.asarray(c[key + "f32"], dtype=np.float64), np.asarray(c[key + "f64"], dtype=np.float64)
    d = 2 * np.abs(r32 - r64) if tag == "f32" else np.zeros_like(r64)
    return d.max(axis=axes, keepdims=True) if axes != () else d


def _truth(c, key, tag, sl=np.s_[...]):
    """The reference's fp64 run of fixture `key` for fp32 checks (see _entry_err); None for fp64."""
    return c[key + "f64"][sl] if tag == "f32" else None


def _check_costs(got, ref, tol, what, noise):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-30)
    ok = (err <= tol["cost"]) | (np.abs(got - ref) <= np.maximum(tol["abs"], noise))
    assert ok.all(), "%s: got %s ref %s relerr %s" % (what, got, ref, err)


def _state_ok(z, c, key, tag, tol, d):
    """Within the state tolerance of the stored run in the same precision; in fp32, alternatively within twice the
    reference's own fp32 distance from its fp64 run, of either of its runs (fp32 rounding follows the host, see _fp32_noise)."""
    if rel_state_err(z, c[key + tag], d) <= tol["state"]:
        return True
    if tag != "f32":
        return False
    noise = 2 * rel_state_err(c[key + "f32"], c[key + "f64"], d)
    return min(rel_state_err(z, c[key + "f32"], d), rel_state_err(z, c[key + "f64"], d)) <= noise


def _entry_err(got, ref, rel, floor, noise=0.0, truth=None):
    """max over entries of |got - ref| / max(rel * max(|ref|, floor), noise): the check passes at <= 1.  With the reference's
    fp64 run as `truth` (fp32 checks), an entry may instead be within `noise` of that run, as for the states (_state_ok)."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref) / np.maximum(rel * np.maximum(np.abs(ref), floor), np.maximum(noise, 1e-300))
    if truth is not None:
        err = np.minimum(err, np.abs(got - np.asarray(truth, dtype=np.float64)) / np.maximum(noise, 1e-300))
    return float(err.max())


@pytest.mark.parametrize("tag", ["f32", "f64"])
@pytest.mark.parametrize("name", PROBLEMS)
def test_rollout_at_xinit(name, tag):
    c = load_cases(name)
    P, D, xinit, meta = oracle_setup(name, DT[tag])
    nt, tol = int(c["nt"]), TOL[tag]
    assert np.array_equal(xinit.double().numpy(), c["xinit"])
    with torch.no_grad():
        mean = _mean_vec(orc.ocflow(xinit, P, D, [0.0, 1.0], nt, "rk4", meta["alph"]))
        zf, cf = orc.ocflow(xinit, P, D, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
    _check_costs(mean, c["xinit_mean_" + tag], tol, "mean costs", _fp32_noise(c, "xinit_mean_", tag))
    d = xinit.shape[1]
    assert _state_ok(zf.numpy(), c, "xinit_z_", tag, tol, d)
    assert zf.shape == c["xinit_z_" + tag].shape and cf.shape == c["xinit_ctrl_" + tag].shape
    assert _entry_err(cf.numpy()[:, :, 1:], c["xinit_ctrl_" + tag][:, :, 1:], 50 * tol["state"], 1e-3,
                      _fp32_noise(c, "xinit_ctrl_", tag, axes=(0, 1))[:, :, 1:], _truth(c, "xinit_ctrl_", tag, np.s_[:, :, 1:])) <= 1
    assert not cf.numpy()[:, :, 0].any()


@pytest.mark.parametrize("tag", ["f32", "f64"])
@pytest.mark.parametrize("name", PROBLEMS)
def test_rollout_batch_three_modes(name, tag):
    c = load_cases(name)
    P, D, _, meta = oracle_setup(name, DT[tag])
    x = torch.from_numpy(c["xb"]).to(DT[tag])
    nt, tol, d = int(c["nt_batch"]), TOL[tag], x.shape[1]
    with torch.no_grad():
        mean = _mean_vec(orc.ocflow(x, P, D, [0.0, 1.0], nt, "rk4", meta["alph"]))
        Jn, cn = orc.ocflow(x, P, D, [0.0, 1.0], nt, "rk4", meta["alph"], noMean=True)
        zf, cf = orc.ocflow(x, P, D, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
    _check_costs(mean, c["b_mean_" + tag], tol, "batch mean", _fp32_noise(c, "b_mean_", tag))
    nomean = np.concatenate([Jn.numpy()] + [v.numpy() for v in cn], axis=1)
    ref = c["b_nomean_" + tag]
    scale = np.maximum(np.abs(ref).max(axis=0, keepdims=True), 1e-30)
    noise = _fp32_noise(c, "b_nomean_", tag, axes=0)
    assert (np.abs(nomean - ref) / np.maximum(10 * tol["cost"] * scale, np.maximum(noise, 1e-300))).max() <= 1
    assert _state_ok(zf.numpy(), c, "b_z_", tag, tol, d)
    assert _entry_err(cf.numpy(), c["b_ctrl_" + tag], 100 * tol["state"], 1e-2, _fp32_noise(c, "b_ctrl_", tag, axes=(0, 1)), _truth(c, "b_ctrl_", tag)) <= 1


@pytest.mark.parametrize("tag", ["f32", "f64"])
@pytest.mark.parametrize("name", PROBLEMS)
def test_rk1_and_unknown_stepper(name, tag):
    c = load_cases(name)
    P, D, _, meta = oracle_setup(name, DT[tag])
    x = torch.from_numpy(c["xb"]).to(DT[tag])
    tol, d = TOL[tag], x.shape[1]
    with torch.no_grad():
        mean = _mean_vec(orc.ocflow(x[:4], P, D, [0.0, 1.0], 8, "rk1", meta["alph"]))
        zf, _ = orc.ocflow(x[:4], P, D, [0.0, 1.0], 8, "rk1", meta["alph"], intermediates=True)
        mean0 = _mean_vec(orc.ocflow(x[:2], P, D, [0.0, 1.0], 3, "none", meta["alph"]))
        z0, c0 = orc.ocflow(x[:2], P, D, [0.0, 1.0], 3, "none", meta["alph"], intermediates=True)
    _check_costs(mean, c["rk1_mean_" + tag], tol, "rk1 mean", _fp32_noise(c, "rk1_mean_", tag))
    assert _state_ok(zf.numpy(), c, "rk1_z_", tag, tol, d)
    _check_costs(mean0, c["nostep_mean_" + tag], tol, "no-stepper mean", _fp32_noise(c, "nostep_mean_", tag))
    assert _state_ok(z0.numpy(), c, "nostep_z_", tag, tol, d)
    assert _entry_err(c0.numpy(), c["nostep_ctrl_" + tag], 100 * tol["state"], 1e-2, _fp32_noise(c, "nostep_ctrl_", tag, axes=(0, 1)), _truth(c, "nostep_ctrl_", tag)) <= 1


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_shock_restart_tspan(tag):
    """tspan != [0,1] (plotter.py:817-823): [0,0.1] with int(0.1 nt) steps, then [0.1,1] with 1+nt-nShock."""
    c = load_cases("softcorridor")
    P, D, xinit, meta = oracle_setup("softcorridor", DT[tag])
    nt, tol = int(c["nt"]), TOL[tag]
    nS = int(0.1 * nt)
    with torch.no_grad():
        z1, _ = orc.ocflow(xinit, P, D, [0.0, 0.1], nS, "rk4", meta["alph"], intermediates=True)
        xs = torch.from_numpy(c["shock2_x_" + tag]).to(DT[tag])
        m2 = _mean_vec(orc.ocflow(xs, P, D, [0.1, 1.0], 1 + nt - nS, "rk4", meta["alph"]))
        z2, c2 = orc.ocflow(xs, P, D, [0.1, 1.0], 1 + nt - nS, "rk4", meta["alph"], intermediates=True)
    assert _state_ok(z1.numpy(), c, "shock1_z_", tag, tol, 4)
    assert _state_ok(z2.numpy(), c, "shock2_z_", tag, tol, 4)
    _check_costs(m2, c["shock2_mean_" + tag], tol, "shock2 mean", _fp32_noise(c, "shock2_mean_", tag))
    assert _entry_err(c2.numpy(), c["shock2_ctrl_" + tag], 100 * tol["state"], 1e-2, _fp32_noise(c, "shock2_ctrl_", tag, axes=(0, 1)), _truth(c, "shock2_ctrl_", tag)) <= 1


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_problem_functors(tag):
    z = np.load(GOLDEN + "/functors.npz")
    names = sorted({k[: -len("_%s_meta" % tag)] for k in z.files if k.endswith("_%s_meta" % tag)})
    assert len(names) == 8
    tol = 3e-6 if tag == "f32" else 1e-12
    for name in names:
        key = "%s_%s" % (name, tag)
        meta = json.loads(str(z[key + "_meta"]))
        x, p = torch.from_numpy(z[key + "_x"]), torch.from_numpy(z[key + "_p"])
        for mode in ("eval", "train"):
            D = orc.ProbDesc(meta["cls"], torch.from_numpy(z[key + "_xtarget"]), meta["obstacle"], meta["alph_Q"],
                             meta["alph_W"], meta["r"], meta["nAgents"], meta["agentDim"], meta["mass"], meta["grav"],
                             training=(mode == "train"))
            L, H, Q, W = orc.lhqw(D, x, p)
            got = np.stack([np.asarray(v).reshape(-1) for v in (L, H, Q, W)], axis=1)
            ref = lambda k: z["%s_%s_%s" % (key, mode, k)]
            noise = lambda k: _fp32_noise({t: z["%s_%s_%s_%s" % (name, t, mode, k)] for t in ("f32", "f64")}, "", tag)
            truth = lambda k: z["%s_f64_%s_%s" % (name, mode, k)] if tag == "f32" else None
            assert _entry_err(got, ref("LHQW"), tol, 1.0, noise("LHQW"), truth("LHQW")) <= 1, (name, mode)
            assert _entry_err(orc.grad_p_hamiltonian(D, x, p).numpy(), ref("gradpH"), tol, 1.0, noise("gradpH"), truth("gradpH")) <= 1
            assert _entry_err(orc.controls(D, x, p).numpy(), ref("ctrls"), tol, 1.0, noise("ctrls"), truth("ctrls")) <= 1


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_phi_random_nets(tag):
    z = np.load(GOLDEN + "/phi_random.npz")
    tol = 3e-6 if tag == "f32" else 1e-12
    for idx in range(5):
        pre = "net%d_" % idx
        sd = {k[len(pre):]: z[k] for k in z.files if k.startswith(pre) and ("." in k or k == pre + "A")}
        P = orc.params_from_state_dict(sd, DT[tag])
        assert P.nTh == int(z[pre + "dims"][0])
        x = torch.from_numpy(z[pre + "x"]).to(DT[tag])
        assert rel_err(orc.phi_forward(P, x).numpy(), z[pre + "fwd_" + tag], floor=1.0) <= tol
        assert rel_err(orc.phi_grad(P, x).numpy(), z[pre + "grad_" + tag], floor=1.0) <= tol


def test_phi_grad_is_gradient_of_forward():
    """free analytic cross-check (SURVEY.md §4 item 1): getGrad == autograd(forward), incl. nTh = 4."""
    z = np.load(GOLDEN + "/phi_random.npz")
    for idx in range(5):
        pre = "net%d_" % idx
        sd = {k[len(pre):]: z[k] for k in z.files if k.startswith(pre) and ("." in k or k == pre + "A")}
        P = orc.params_from_state_dict(sd, torch.float64)
        x = torch.from_numpy(z[pre + "x"]).double().requires_grad_(True)
        (g,) = torch.autograd.grad(orc.phi_forward(P, x).sum(), x)
        assert rel_err(orc.phi_grad(P, x.detach()).numpy(), g.numpy(), floor=1.0) <= 1e-12


def test_problem_table_matches_reference_initprob():
    z = np.load(GOLDEN + "/initprob.npz")
    names = sorted(k[:-6] for k in z.files if k.endswith("_xinit"))
    assert len(names) == 15
    for name in names:
        meta = json.loads(str(z[name + "_meta"]))
        D, xi = orc.make_problem(name, [1.0, 2.0, 3.0, 1.0, 1.0, 1.0], torch.float64)
        assert np.allclose(D.xtarget.numpy(), z[name + "_xtarget"], rtol=0, atol=1e-6), name
        assert np.allclose(xi.numpy(), z[name + "_xinit"], rtol=0, atol=1e-6), name
        assert (D.kind, D.obstacle, D.nAgents, D.agentDim) == (meta["cls"], meta["obstacle"], meta["nAgents"], meta["agentDim"])
        assert (D.alph_Q, D.alph_W, D.r) == (meta["alph_Q"], meta["alph_W"], meta["r"]), name


def test_known_answer_table_of_the_survey():
    """SURVEY.md §8c known answers (fp64 reference at xInit) — detects an oracle that silently changed."""
    known = {"softcorridor": (50, 6.4450996960e+01), "swap2": (50, 7.5607575177e+02), "swap12": (50, 5.4430337230e+03),
             "swarm50": (80, 1.5968817566e+03), "singlequad": (50, 2.2499753119e+03)}
    for name, (nt, jc) in known.items():
        P, D, xinit, meta = oracle_setup(name, torch.float64)
        with torch.no_grad():
            Jc, _ = orc.ocflow(xinit, P, D, [0.0, 1.0], nt, "rk4", meta["alph"])
        assert abs(float(Jc) - jc) / jc < 2e-10, name


def test_stage_time_table_replays_python_double_arithmetic():
    rows = orc.stage_time_table(0.0, 1.0, 50)
    tk, h = 0.0, 1.0 / 50
    for r in rows:
        hh = (tk + h) - tk
        assert r[0] == tk and r[1] == tk + hh / 2 and r[2] == tk + hh
        tk += h
        assert r[3] == tk - h

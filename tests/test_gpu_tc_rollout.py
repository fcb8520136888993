"""GPU parity of the tensor-core rollout kernel (neuraloc_b200/csrc/noc_tc_rollout.cuh; tcgen05 MMAs on 3-way bf16 splits of
the fp32 operands) against the unmodified reference's outputs, at the same tolerances as the FMA kernels (1e-5 relative
per-step state, 1e-4 relative final cost terms), plus agreement with the FMA tile kernel sample by sample."""
import numpy as np
import pytest
import torch

from helpers import DT, QW, check_costs, load_cases, mean_vec, product_setup, rel_state_err
from test_gpu_parity import _compare, _three_modes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nb():
    import neuraloc_b200
    neuraloc_b200._cabi.lib()
    return neuraloc_b200


@pytest.fixture(autouse=True)
def tc_path(monkeypatch):
    monkeypatch.setenv("NOC_FORCE_PATH", "tc")


TC_PROBLEMS = ["softcorridor", "swap2", "swap12", "singlequad"]


@pytest.mark.parametrize("name", TC_PROBLEMS)
def test_tc_rollout_golden(nb, name):
    c = load_cases(name)
    net, prob, xinit, meta = product_setup(name, DT["f32"])
    d = xinit.shape[1]
    got = _three_modes(nb, xinit, net, prob, [0.0, 1.0], int(c["nt"]), "rk4", meta["alph"])
    _compare("f32", d, got, (c["xinit_mean_f32"], None, c["xinit_z_f32"], c["xinit_ctrl_f32"]), "tc %s xInit" % name,
             truth=(c["xinit_mean_f64"], None))
    xb = torch.from_numpy(c["xb"]).float().cuda()
    got = _three_modes(nb, xb, net, prob, [0.0, 1.0], int(c["nt_batch"]), "rk4", meta["alph"])
    _compare("f32", d, got, (c["b_mean_f32"], c["b_nomean_f32"], c["b_z_f32"], c["b_ctrl_f32"]), "tc %s batch" % name,
             truth=(c["b_mean_f64"], c["b_nomean_f64"]))


@pytest.mark.parametrize("name", TC_PROBLEMS)
def test_tc_rk1_and_unknown_stepper_golden(nb, name):
    c = load_cases(name)
    net, prob, xinit, meta = product_setup(name, DT["f32"])
    d = xinit.shape[1]
    xb = torch.from_numpy(c["xb"]).float().cuda()
    got = _three_modes(nb, xb[:4], net, prob, [0.0, 1.0], 8, "rk1", meta["alph"])
    # Euler with 8 steps on the adversarial rows is ill-conditioned in fp32: the reference's own fp32 run is up to 1.05e-5
    # from its fp64 run (swap12).  Gate against the fp64 trajectories, at 1e-5 or twice the reference's own fp32 error.
    ref_err = rel_state_err(c["rk1_z_f32"], c["rk1_z_f64"], d)
    _compare("f32", d, got, (c["rk1_mean_f64"], None, c["rk1_z_f64"], c["rk1_ctrl_f64"]), "tc rk1", state_tol=max(1e-5, 2 * ref_err))
    got = _three_modes(nb, xb[:2], net, prob, [0.0, 1.0], 3, "none", meta["alph"])
    _compare("f32", d, got, (c["nostep_mean_f32"], None, c["nostep_z_f32"], c["nostep_ctrl_f32"]), "tc no stepper")


def test_tc_shock_restart_golden(nb):
    """tspan != [0,1] (plotter.py:817-823) through the tensor-core kernel."""
    c = load_cases("softcorridor")
    net, prob, xinit, meta = product_setup("softcorridor", DT["f32"])
    nt = int(c["nt"])
    nS = int(0.1 * nt)
    got = _three_modes(nb, xinit, net, prob, [0.0, 0.1], nS, "rk4", meta["alph"])
    _compare("f32", 4, got, (c["shock1_mean_f32"], None, c["shock1_z_f32"], c["shock1_ctrl_f32"]), "tc shock leg 1")
    xs = torch.from_numpy(c["shock2_x_f32"]).float().cuda()
    got = _three_modes(nb, xs, net, prob, [0.1, 1.0], 1 + nt - nS, "rk4", meta["alph"])
    _compare("f32", 4, got, (c["shock2_mean_f32"], None, c["shock2_z_f32"], c["shock2_ctrl_f32"]), "tc shock leg 2")


def _vs_tile(nb, monkeypatch, net, prob, x, alph, nt, d, full):
    with torch.no_grad():
        Jt, ct = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", alph, noMean=True)
        mt = mean_vec(nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", alph))
        if full:
            zt, ut = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", alph, intermediates=True)
        monkeypatch.setenv("NOC_FORCE_PATH", "tile")
        Jf, cf = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", alph, noMean=True)
        if full:
            zf, uf = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", alph, intermediates=True)
    tt, tf = torch.cat([Jt] + list(ct), 1).double().cpu().numpy(), torch.cat([Jf] + list(cf), 1).double().cpu().numpy()
    sc = np.maximum(np.abs(tf).max(axis=0, keepdims=True), 1.0)
    # a pair within rounding of the interaction cut-off can land on either side in the two kernels: allow two such rows
    # (one sample alone: G and HJgrad are pure cancellation, gated at 20x like test_gpu_parity._compare does)
    bad = ((np.abs(tt - tf) / sc).max(axis=1) > (2e-3 if len(tt) == 1 else 1e-4)).sum()
    assert bad <= (2 if len(tt) >= 1000 else 0), "per-sample costs tc vs fma: %d rows differ" % bad
    check_costs(mt, tt.mean(axis=0), 1e-6, 1e-7, "tc mean vs mean of tc noMean", floor_mask=QW)
    if full:
        assert rel_state_err(zt.cpu().numpy(), zf.cpu().numpy(), d) <= 1e-5      # two fp32 kernels, each 3-5e-6 from fp64 on singlequad
        assert (ut - uf).abs().max() <= 1e-4 * max(1.0, float(uf.abs().max()))


@pytest.mark.parametrize("n", [1, 127, 128, 129, 1000, 40_000])
@pytest.mark.parametrize("name", TC_PROBLEMS)
def test_tc_matches_fma_tile_kernel(nb, name, n, monkeypatch):
    """Ragged tile counts (one CTA runs several tiles at n = 40000): per-sample costs and trajectories agree with the
    FMA tile kernel to fp32 rounding, and the mean is the mean of the per-sample table."""
    net, prob, xinit, meta = product_setup(name, torch.float32)
    d = xinit.shape[1]
    g = torch.Generator().manual_seed(n)
    x = xinit.cpu() + 0.4 * torch.randn(n, d, generator=g)
    if name == "singlequad":
        x[:, 3:] = 0 if n % 2 else x[:, 3:] * 0.2
    _vs_tile(nb, monkeypatch, net, prob, x.cuda(), meta["alph"], 20, d, n <= 1000)


@pytest.mark.parametrize("m", [8, 20, 48, 100, 128])
@pytest.mark.parametrize("data", ["midcross4", "swap2", "swap12", "singlequad", "swap12_3pair", "swap12_4pair", "swap12_5pair"])
def test_tc_random_nets_any_width(nb, data, m, monkeypatch):
    """Randomly initialised value nets of widths that are not multiples of the MMA tile (zero-padded units), the 4-agent
    shape and the hard obstacle, train and eval mode of the problem."""
    alph = [100.0, 50.0, 30.0, 1.0, 1.0, 1.0]
    prob, x0, _, xinit = nb.initProb(data, 10, 11, 1.0, alph, lambda v: v.float().cuda())
    d = xinit.shape[1]
    torch.manual_seed(m)
    net = nb.Phi(nTh=2, m=m, d=d, alph=alph)
    with torch.no_grad():
        net.N.layers[1].weight.normal_(std=0.2); net.N.layers[1].bias.normal_()
        net.w.weight.normal_(); net.c.weight.normal_(); net.c.bias.normal_()
    net = net.float().cuda()
    g = torch.Generator().manual_seed(m + d)
    x = (xinit.cpu() + 0.5 * torch.randn(300, d, generator=g))
    if data == "singlequad":
        x[:, 3:] *= 0.1
    for mode in ("eval", "train"):
        getattr(prob, mode)()
        monkeypatch.setenv("NOC_FORCE_PATH", "tc")
        _vs_tile(nb, monkeypatch, net, prob, x.cuda(), alph, 6, d, True)


@pytest.mark.parametrize("name,n", [("swap12", 70_000), ("singlequad", 25_000)])
def test_tc_several_tiles_per_cta(nb, name, n, monkeypatch):
    """More tiles than resident CTAs (444 x 128 samples for swap12, 148 x 128 for singlequad), ragged last tile: every CTA
    loops over tiles; intermediates go through the tile-major staging buffer and the transpose kernel.  Trajectories,
    controls and per-sample costs agree with the FMA tile kernel on rows from the first, a middle and the last tile."""
    net, prob, xinit, meta = product_setup(name, torch.float32)
    d = xinit.shape[1]
    g = torch.Generator(device="cuda").manual_seed(n)
    x = xinit + 0.3 * torch.randn(n, d, generator=g, device="cuda")
    if name == "singlequad":
        x[:, 3:] *= 0.1
    nt = 20        # (a handful of RK4 steps over [0,1] is ill-conditioned in fp32: the two kernels' rounding noise is amplified)
    idx = torch.tensor([0, 1, 127, 128, n // 2, n // 2 + 77, n - 130, n - 2, n - 1], device="cuda")
    with torch.no_grad():
        zt, ut = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
        assert nb._cabi.last_path() == "tensor"
        Jt, ct = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], noMean=True)
        mt = mean_vec(nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"]))
        monkeypatch.setenv("NOC_FORCE_PATH", "tile")
        zf, uf = nb.OCflow(x[idx].contiguous(), net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
        Jf, cf = nb.OCflow(x[idx].contiguous(), net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], noMean=True)
    assert zt.shape == (n, d + 4, nt + 1) and not ut[:, :, 0].any()
    assert rel_state_err(zt[idx].cpu().numpy(), zf.cpu().numpy(), d) <= 5e-6
    assert (ut[idx] - uf).abs().max() <= 1e-4 * max(1.0, float(uf.abs().max()))
    tt = torch.cat([Jt] + list(ct), 1).double()
    tf = torch.cat([Jf] + list(cf), 1).double()
    sc = torch.clamp(tf.abs().max(dim=0, keepdim=True).values, min=1.0)
    assert float(((tt[idx] - tf).abs() / sc).max()) <= 1e-4
    assert torch.allclose(zt[:, d, -1:], ct[0], rtol=1e-6, atol=1e-6)            # accumulated L column == noMean L
    check_costs(mt, tt.mean(dim=0).cpu().numpy(), 1e-6, 1e-7, "mean vs mean of noMean across many tiles", floor_mask=QW)


def test_path_selection(nb, monkeypatch):
    """Default choice by shape and batch size (noc_last_path): tensor-core kernel for the shapes it is written for at
    batch sizes above the small-batch threshold, NOC_TC=0 keeps the FMA tile kernel, other shapes are unaffected, and
    NOC_FORCE_PATH=tc on a shape the kernel is not written for falls back to the normal choice (still CUDA)."""
    monkeypatch.delenv("NOC_FORCE_PATH", raising=False)
    net, prob, xinit, meta = product_setup("swap12", torch.float32)
    x = xinit + 0.1 * torch.randn(1000, 24, device="cuda")
    with torch.no_grad():
        nb.OCflow(x, net, prob, [0.0, 1.0], 4, "rk4", meta["alph"])
        assert nb._cabi.last_path() == "tensor"
        nb.OCflow(x[:8].contiguous(), net, prob, [0.0, 1.0], 4, "rk4", meta["alph"])
        assert nb._cabi.last_path() == "sample"
        monkeypatch.setenv("NOC_TC", "0")
        nb.OCflow(x, net, prob, [0.0, 1.0], 4, "rk4", meta["alph"])
        assert nb._cabi.last_path() == "tile"
        monkeypatch.delenv("NOC_TC")
        nb.OCflow(x.double(), net.double(), product_setup("swap12", torch.float64)[1], [0.0, 1.0], 4, "rk4", meta["alph"])
        assert nb._cabi.last_path() == "tile"                      # fp64 has no tensor-core kernel
        for n, env, want in [(8, {"NOC_FORCE_PATH": "tc"}, "tensor"),
                             (1000, {"NOC_TC": "0", "NOC_FORCE_PATH": "tc"}, "tensor"),      # forcing wins over NOC_TC=0
                             (1000, {"NOC_FORCE_PATH": "vec"}, "sample"),
                             (8, {"NOC_FORCE_PATH": "tile"}, "tile")]:
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            nb.OCflow(x[:n].contiguous(), net, prob, [0.0, 1.0], 4, "rk4", meta["alph"])
            assert nb._cabi.last_path() == want, (n, env)
            for k in env:
                monkeypatch.delenv(k)
        net5, prob5, xinit5, meta5 = product_setup("swarm50", torch.float32)
        for n, env, want in [(100, {}, "tensor"),                       # swarm50's small-batch threshold is 64, not 256
                             (64, {}, "sample"),
                             (100, {"NOC_VEC_MAX": "256"}, "sample")]:   # an explicit threshold replaces the 64
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            nb.OCflow(xinit5.repeat(n, 1), net5, prob5, [0.0, 1.0], 4, "rk4", meta5["alph"])
            assert nb._cabi.last_path() == want, (n, env)
            for k in env:
                monkeypatch.delenv(k)
        Jc, cs = nb.OCflow(xinit5.repeat(300, 1), net5, prob5, [0.0, 1.0], 4, "rk4", meta5["alph"])
        assert nb._cabi.last_path() == "tensor" and np.isfinite(float(Jc))      # the streamed CTA-pair kernel (m = 512)
        monkeypatch.setenv("NOC_TC", "0")
        nb.OCflow(xinit5.repeat(300, 1), net5, prob5, [0.0, 1.0], 4, "rk4", meta5["alph"])
        assert nb._cabi.last_path() == "tile"
        monkeypatch.delenv("NOC_TC")
        monkeypatch.setenv("NOC_FORCE_PATH", "tc")
        net6, prob6, xinit6, meta6 = product_setup("swarm50", torch.float64)     # a shape / dtype without a tensor kernel
        Jc, cs = nb.OCflow(xinit6.repeat(300, 1), net6, prob6, [0.0, 1.0], 4, "rk4", meta6["alph"])
        assert nb._cabi.last_path() == "tile" and np.isfinite(float(Jc))


@pytest.mark.parametrize("name,n", [("swap12", 1 << 20), ("singlequad", 1 << 22)])
def test_tc_bench_size_subsampled_oracle(nb, name, n, monkeypatch):
    """The benchmark batches themselves (BASELINE.json configs[1] / configs[2] sizes) through the kernel the library picks:
    2 000 rows sub-sampled from the batch are checked per sample against the fp64 oracle, and their means at 1e-4 (G included)."""
    import os
    from oracle import ocflow_oracle as orc
    from helpers import oracle_setup
    monkeypatch.delenv("NOC_FORCE_PATH", raising=False)
    net, prob, xinit, meta = product_setup(name, torch.float32)
    P64, D64, _, _ = oracle_setup(name, torch.float64)
    d = xinit.shape[1]
    g = torch.Generator(device="cuda").manual_seed(1234)
    if name == "singlequad":
        x = torch.zeros(n, d, device="cuda")
        x[:, :3] = -1.5 + meta["var0"] * torch.randn(n, 3, generator=g, device="cuda")
    else:
        x = xinit + meta["var0"] * torch.randn(n, d, generator=g, device="cuda")
    nt = 50
    with torch.no_grad():
        J, cs = nb.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"], noMean=True)
        assert nb._cabi.last_path() == "tensor"
        sums = nb.ocflow_sums(x, net, prob, [0.0, 1.0], nt, "rk4", meta["alph"])
    idx = torch.linspace(0, n - 1, 2000).long()
    got = torch.cat([J] + list(cs), 1)[idx.cuda()].double().cpu().numpy()
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        J64, cs64 = orc.ocflow(x[idx.cuda()].cpu().double(), P64, D64, [0.0, 1.0], nt, "rk4", meta["alph"], noMean=True)
    n64 = torch.cat([J64] + list(cs64), 1).numpy()
    sc = np.maximum(np.abs(n64).max(axis=0, keepdims=True), 1e-30)
    perr = (np.abs(got - n64) / sc).max(axis=0)
    assert (perr[[0, 1, 3, 4]] <= 1e-4).all() and perr[2] <= 3e-3 and perr[5] <= 3e-3, "per-sample costs vs fp64 oracle: %s" % perr
    check_costs(got.mean(axis=0)[:6], n64.mean(axis=0)[:6], 1e-4, 0.0, "%s: means over 2 000 sub-sampled rows vs fp64 oracle" % name)
    # the whole batch's means agree with the sub-sample's to sampling noise (a gross error anywhere in the batch would show)
    full = (sums[:7] / sums[7]).cpu().numpy()
    assert np.all(np.abs(full[[0, 2, 3]] - n64.mean(axis=0)[[1, 3, 4]]) <= 0.05 * np.abs(n64.mean(axis=0)[[1, 3, 4]]))

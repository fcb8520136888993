"""CPU-only tests of the host side: C-ABI exports, descriptor flattening, time table, problem factory, Phi mirror."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import neuraloc_b200 as nb
from neuraloc_b200 import _cabi, ocflow
from helpers import GOLDEN, ROOT, load_ckpt
from oracle import ocflow_oracle as orc


def test_library_loads_and_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "noc_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(noc_[a-z_0-9]+)\s*\(", hdr)))
    assert declared == sorted(_cabi.SYMBOLS)
    lib = _cabi.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.noc_version() == 1
    nm = subprocess.run(["nm", "-D", "--defined-only", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(set(re.findall(r" T (noc_[a-z_0-9]+)$", nm, flags=re.M)))
    assert exported == declared       # exactly the header's entry points, nothing torch-typed


def test_no_gpu_means_loud_failure_not_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    prob, x0, _, xinit = nb.initProb("softcorridor", 4, 4, 1.0, [1.0] * 6, lambda v: v.float())
    net = nb.Phi(2, 8, 4)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        nb.OCflow(xinit, net, prob, [0.0, 1.0], 4)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        net.getGrad(torch.zeros(2, 5))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        prob.calcLHQW(x0, x0)


def test_stage_time_table_matches_library_and_oracle():
    lib = _cabi.lib()
    for t0, t1, nt in ((0.0, 1.0, 50), (0.0, 1.0, 80), (0.0, 0.1, 5), (0.1, 1.0, 46), (0.3, 0.7, 7)):
        tab = ocflow.stage_times(t0, t1, nt)
        ctab = (C.c_double * (5 * nt))()
        assert lib.noc_stage_times(t0, t1, nt, ctab) == 0
        rows = orc.stage_time_table(t0, t1, nt)
        for k in range(nt):
            assert list(tab[5 * k:5 * k + 4]) == list(rows[k])          # bit-identical doubles
            assert list(ctab[5 * k:5 * k + 5]) == list(tab[5 * k:5 * k + 5])
            assert tab[5 * k + 4] == (rows[k][2] - rows[k][0]) or abs(tab[5 * k + 4] - (t1 - t0) / nt) < 1e-15


def test_problem_factory_matches_reference_tables():
    z = np.load(GOLDEN + "/initprob.npz")
    names = sorted(k[:-6] for k in z.files if k.endswith("_xinit"))
    for name in names:
        meta = json.loads(str(z[name + "_meta"]))
        torch.manual_seed(0)
        prob, x0, x0v, xinit = nb.initProb(name, 6, 5, 0.5, [1.0, 2.0, 3.0, 1.0, 1.0, 1.0], lambda v: v.double())
        assert type(prob).__name__ == meta["cls"] and prob.obstacle == meta["obstacle"]
        assert (prob.nAgents, prob.agentDim, prob.r) == (meta["nAgents"], meta["agentDim"], meta["r"]), name
        assert (prob.alph_Q, prob.alph_W) == (meta["alph_Q"], meta["alph_W"]), name
        assert np.allclose(prob.xtarget.numpy(), z[name + "_xtarget"], atol=1e-6) and prob.training
        assert np.allclose(xinit.numpy(), z[name + "_xinit"], atol=1e-6) and xinit.shape == (1, prob.d)
        assert x0.shape[1] == prob.d and x0.shape[0] in (6, 2 * (6 // 2))
    with pytest.raises(ValueError):
        nb.initProb("nope", 1, 1, 1.0, [1.0] * 6, lambda v: v)


def test_phi_mirror_has_reference_layout_and_rng_order():
    sd, meta = load_ckpt("swap12")
    net = nb.Phi(nTh=meta["nTh"], m=meta["m"], d=24, alph=meta["alph"])
    assert list(net.state_dict().keys()) == list(sd.keys())
    net.load_state_dict(sd)
    z = np.load(GOLDEN + "/config5.npz")
    torch.manual_seed(0)
    net5 = nb.Phi(nTh=2, m=512, d=150)
    for k, v in net5.state_dict().items():          # same random draws as the reference constructor
        chk = z["chk_" + k]
        assert abs(float(v.double().sum()) - chk[0]) <= 1e-9 * max(1.0, abs(chk[1])), k
    assert net5.N.h == 1.0 and nb.Phi(4, 8, 3).N.h == 1.0 / 3
    with pytest.raises(ValueError):
        nb.Phi(1, 8, 3)


def test_descriptor_flattening_and_guards():
    prob, x0, _, xinit = nb.initProb("swap2", 4, 4, 1.0, [300.0, 1e6, 1e5, 1.0, 1.0, 3.0], lambda v: v.float())
    prob.eval()
    st, keep = ocflow._prob_struct(prob, torch.device("cpu"), torch.float32)
    assert (st.kind, st.obstacle, st.training, st.nAgents, st.agentDim) == (0, 2, 0, 2, 2)
    assert (st.alph_Q, st.alph_W, st.r) == (1e6, 1e5, 1.0) and st.xtarget == keep.data_ptr()
    net = nb.Phi(3, 8, 4)
    ph = ocflow._phi_struct(net, torch.device("cpu"), torch.float64)
    assert (ph.d, ph.m, ph.nTh, ph.r, ph.h) == (4, 8, 3, 5, 0.5)
    assert ocflow._phi_struct(net, torch.device("cpu"), torch.float64) is ph          # cached
    with torch.no_grad():
        net.w.weight.add_(1.0)
    assert ocflow._phi_struct(net, torch.device("cpu"), torch.float64) is not ph      # invalidated by a parameter update
    with pytest.raises(RuntimeError, match="forward-only"):          # noMean / intermediates / rk1 are not differentiable: loud
        nb.OCflow(xinit, net, prob, [0.0, 1.0], 4, noMean=True)
    with pytest.raises(RuntimeError, match="forward-only"):
        nb.OCflow(xinit, net, prob, [0.0, 1.0], 4, "rk1")
    if not torch.cuda.is_available():                                # the training path needs the GPU like everything else
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            nb.OCflow(xinit, net, prob, [0.0, 1.0], 4)
    class Weird:
        pass
    with pytest.raises(ValueError):
        ocflow._prob_struct(Weird(), torch.device("cpu"), torch.float32)
    assert nb.shard_rows(10, 4, 0) == (0, 3) and nb.shard_rows(10, 4, 3) == (9, 10) and nb.shard_rows(2, 4, 3) == (2, 2)
    sums = torch.tensor([10.0, 2.0, 4.0, 6.0, 8.0, 1.0, 3.0, 2.0], dtype=torch.float64)
    Jc, cs = nb.costs_from_sums(sums, [2.0, 0, 0, 3.0, 4.0, 5.0], torch.float32)
    assert [float(c) for c in cs] == [5.0, 1.0, 2.0, 3.0, 4.0, 0.5, 1.5] and float(Jc) == 5 + 2 * 1 + 3 * 2 + 4 * 3 + 5 * 4


def test_dropin_hook_rebinds_reference_module(tmp_path):
    """PYTHONPATH=dropin:repo:reference -> `from src.OCflow import OCflow` is the B200 implementation (INTEGRATION.md §1).
    The reference checkout is not part of this repository: a stand-in `src` package with the reference's module and entry-point
    names takes its place, so the hook is exercised the way the reference scripts import."""
    src = tmp_path / "src"
    src.mkdir()
    (src / "__init__.py").write_text("")
    (src / "OCflow.py").write_text(
        "def OCflow(*a, **k):\n    raise AssertionError('the stand-in reference OCflow ran')\n"
        "stepRK4 = stepRK1 = ocOdefun = OCflow\n"
        "def ocG(z, xtarget):\n    return z[:, :xtarget.shape[0]] - xtarget\n")
    (src / "Phi.py").write_text("class Phi:\n    pass\n")
    (src / "initProb.py").write_text("def initProb(*a, **k):\n    raise NotImplementedError\n")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "neuraloc_b200", "dropin"), ROOT, str(tmp_path)]))
    code = ("from src.OCflow import OCflow, stepRK4, ocG; import src.OCflow as m, neuraloc_b200 as nb;"
            "assert OCflow is nb.OCflow and stepRK4 is nb.stepRK4; assert m._reference_OCflow is not None;"
            "assert m.stepRK1 is nb.stepRK1 and m.ocOdefun is nb.ocOdefun and m._reference_OCflow.__module__ == 'src.OCflow';"
            "from src.Phi import Phi; from src.initProb import initProb; print('hooked')")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=str(tmp_path))
    assert out.returncode == 0 and "hooked" in out.stdout, out.stderr


def test_bench_flop_accounting():
    """bench.py's roofline numerators: SURVEY.md 8(d)'s algorithmic flops per sample-step, and the bf16 flops the tensor-core
    kernel executes (6 split products over the padded GEMM volumes)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    want = {"softcorridor": (4, 32, 19144), "swap2": (4, 16, 5576), "swap12": (24, 32, 33184), "singlequad": (12, 128, 290120),
            "swarm50": (150, 512, 5455456)}
    for name, (d, m, f) in want.items():
        assert b.flops_per_sample_step(d, m, 2, min(10, d + 1)) == f, name
    assert b.tensor_flops_per_sample_step("swap12", 24, 32)[0] == 4 * 3 * 2 * (32 * 32 + 2 * 32 * 32 + 32 * 32 + 32 * 32)
    assert b.tensor_flops_per_sample_step("singlequad", 12, 128)[0] == 4 * 3 * 2 * (16 * 128 + 2 * 128 * 128 + 128 * 16 + 16 * 16)
    assert b.tensor_flops_per_sample_step("swap2", 4, 16)[0] == 4 * 3 * 2 * (16 * 16 * 5)
    assert b.tensor_flops_per_sample_step("singlequad", 12, 100)[0] == b.tensor_flops_per_sample_step("singlequad", 12, 128)[0]   # width padded to 64s
    # streamed swarm kernel: 3 split products (fp16 x 2), KS = 160, m = 512
    assert b.tensor_flops_per_sample_step("swarm50", 150, 512)[0] == 4 * 3 * 2 * (2 * 160 * 512 + 2 * 512 * 512 + 160 * 160)
    # the default workload is the north_star target shape, strong-scaled; shards cover the batch exactly
    assert b.DEFAULT_WORKLOAD == "swarm50" and b.WORKLOADS["swarm50"]["scaling"] == "strong"
    for world in (1, 2, 3, 8):
        rows = [b.shard(1000003, world, r) for r in range(world)]
        assert rows[0][0] == 0 and rows[-1][1] == 1000003 and all(rows[i][1] == rows[i + 1][0] for i in range(world - 1))


def test_bench_dump_outputs_format_and_argument_checks(tmp_path):
    """bench.py --dump-outputs writes the cost sums (float64) and [Jc, cs] in the workload's precision; it refuses the modes it
    does not cover and a step count below one before touching the GPU."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    sums = torch.tensor([10.0, 2.0, 4.0, 6.0, 8.0, 1.0, 3.0, 2.0], dtype=torch.float64)
    for dtype, npt in ((torch.float32, np.float32), (torch.float64, np.float64)):
        Jc, cs = nb.costs_from_sums(sums, [2.0, 0, 0, 3.0, 4.0, 5.0], dtype)
        b.dump_outputs(str(tmp_path / "out"), sums, Jc, cs)
        s, c = np.load(tmp_path / "out" / "sums.npy"), np.load(tmp_path / "out" / "costs.npy")
        assert s.dtype == np.float64 and np.array_equal(s, sums.numpy())
        assert c.dtype == npt and c.tolist() == [45.0, 5.0, 1.0, 2.0, 3.0, 4.0, 0.5, 1.5]
    for extra in (["--latency"], ["--train"], ["--intermediates"], ["--impl", "reference"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path / "x")] + extra,
                           capture_output=True, text=True, cwd=str(tmp_path))
        assert p.returncode == 2 and "--dump-outputs" in p.stderr, (extra, p.stderr[-500:])
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, cwd=str(tmp_path))
    assert p.returncode == 2 and "--steps" in p.stderr
    assert not (tmp_path / "x").exists()


def test_bench_does_not_import_test_helpers_or_oracle_at_import():
    """bench.py's GPU arm must not depend on tests/ or on the oracle (only the cpu_baseline / reference legs import oracle/)."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert "from helpers import" not in src and "import helpers" not in src
    head = src.split("def cpu_rate")[0]
    assert "oracle" not in head.replace("oracle/ocflow_oracle.py", "").replace("CPU oracle port", "").replace("the oracle", "")

"""Oracle vs the LIVE reference: runs only where the environment variable NOC_REFERENCE names a checkout of the original
NeuralOC project (the directory holding its `src/`); skipped otherwise.  No such checkout was available when the suite was
made self-contained, so the fresh-seed outputs this test compares against could not be stored as golden data.  Its main
comparison, the reference's outputs on seeded batches in both precisions for all five problems, is kept everywhere by the
stored tests/golden/cases_*.npz in tests/test_oracle_golden.py.

With a checkout it adds: fresh seeds, larger batches, every problem name of initProb."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import ocflow_oracle as orc
from helpers import PROBLEMS, load_ckpt

REF = os.environ.get("NOC_REFERENCE", "")
pytestmark = [pytest.mark.reference,
              pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "src"))),
                                 reason="NOC_REFERENCE does not name a checkout of the original NeuralOC project")]


@pytest.fixture(scope="module")
def ref():
    sys.path.insert(0, REF)
    import src.OCflow as O
    import src.Phi as PH
    import src.initProb as IP
    yield O, PH, IP
    sys.path.remove(REF)
    for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
        del sys.modules[k]


@pytest.mark.parametrize("prec", [torch.float32, torch.float64])
@pytest.mark.parametrize("name", PROBLEMS)
def test_fresh_batch_matches_reference(ref, name, prec):
    O, PH, IP = ref
    sd, meta = load_ckpt(name)
    old = torch.get_default_dtype()
    torch.set_default_dtype(prec)
    try:
        prob, _, _, xInit = IP.initProb(meta["data"], 4, 4, var0=1.0, alph=meta["alph"], cvt=lambda v: v.type(prec))
        prob.eval()
        net = PH.Phi(nTh=meta["nTh"], m=meta["m"], d=xInit.shape[1], alph=meta["alph"])
        net.load_state_dict(sd)
        net = net.to(prec)
        n = 5 if name == "swarm50" else 64
        g = torch.Generator().manual_seed(99)
        x = xInit + meta["var0"] * torch.randn(n, xInit.shape[1], generator=g, dtype=prec)
        nt = 6
        with torch.no_grad():
            Jr, cr = O.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", net.alph)
            zr, ur = O.OCflow(x, net, prob, [0.0, 1.0], nt, "rk4", net.alph, intermediates=True)
        P = orc.params_from_state_dict(sd, prec)
        D, xi = orc.make_problem(meta["data"], meta["alph"], prec)
        with torch.no_grad():
            Jo, co = orc.ocflow(x, P, D, [0.0, 1.0], nt, "rk4", meta["alph"])
            zo, uo = orc.ocflow(x, P, D, [0.0, 1.0], nt, "rk4", meta["alph"], intermediates=True)
    finally:
        torch.set_default_dtype(old)
    tol = 5e-6 if prec == torch.float32 else 1e-12
    assert torch.equal(xi, xInit)
    assert abs(float(Jo) - float(Jr)) <= 10 * tol * abs(float(Jr))
    for a, b in zip(co, cr):
        assert abs(float(a) - float(b)) <= 10 * tol * max(abs(float(b)), 1e-3)
    assert (zo - zr).abs().max() <= tol * zr.abs().max()
    assert (uo - ur).abs().max() <= 20 * tol * max(float(ur.abs().max()), 1.0)

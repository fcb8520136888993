"""CPU: the autograd guards around Phi and the problem evaluators refuse before any device work (no GPU needed)."""
import pytest
import torch

import neuraloc_b200 as nb


def test_deeper_net_refuses_autograd_before_launching():
    net = nb.Phi(nTh=3, m=8, d=4)
    s = torch.zeros(2, 5)
    with pytest.raises(RuntimeError, match="differentiable for nTh = 2"):
        net(s)
    with pytest.raises(RuntimeError, match="differentiable for nTh = 2"):
        net.requires_grad_(False).getGrad(s.requires_grad_(True))


def test_problem_evaluators_refuse_gradient_requests():
    prob, x0, _, _ = nb.initProb("softcorridor", 4, 4, 1.0, [1.0] * 6, lambda v: v.float())
    p = torch.zeros_like(x0, requires_grad=True)
    for fn in (prob.calcLHQW, prob.calcGradpH, prob.calcCtrls):
        with pytest.raises(RuntimeError, match="forward-only"):
            fn(x0, p)
        with pytest.raises(RuntimeError, match="forward-only"):
            fn(x0.clone().requires_grad_(True), p.detach())

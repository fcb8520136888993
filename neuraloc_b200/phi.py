"""Host-side mirror of the reference value network (src/Phi.py) — parameters and checkpoint layout only.

`Phi` / `ResNN` keep the reference's constructor signature, attribute names (`A, c, w, N.layers, N.h,
N.nTh, alph, m, d`) and state_dict keys (src/Phi.py:77-87, 32-36), so the pretrained `.pth` files load
unchanged, and the same initialisation calls in the same order, so `torch.manual_seed(s); Phi(...)`
yields the reference's random weights.  `forward` and `getGrad` run on the GPU through
noc_phi_eval (they are device functions of the rollout kernel); there is no torch arithmetic here.
Under autograd (nTh = 2) both are differentiable with respect to s and the parameters: the backward
pass is one noc_phi_vjp call.
"""
import copy

import torch
import torch.nn as nn


class ResNN(nn.Module):
    """Parameter container of the ResNet part N(s) (src/Phi.py:15-52)."""

    def __init__(self, d, m, nTh=2):
        super().__init__()
        if nTh < 2:
            raise ValueError("nTh must be an integer >= 2")   # the reference prints and exit(1)s (Phi.py:25-27)
        self.d, self.m, self.nTh = d, m, nTh
        self.layers = nn.ModuleList([nn.Linear(d + 1, m, bias=True), nn.Linear(m, m, bias=True)])
        for _ in range(nTh - 2):
            self.layers.append(copy.deepcopy(self.layers[1]))
        self.h = 1.0 / (self.nTh - 1)


class Phi(nn.Module):
    """Phi(s) = w'N(s) + 0.5 s'A'A s + c's + b  (src/Phi.py:56-138)."""

    def __init__(self, nTh, m, d, r=10, alph=[1.0] * 6):
        super().__init__()
        self.m, self.nTh, self.d, self.alph = m, nTh, d, alph
        r = min(r, d + 1)
        self.A = nn.Parameter(torch.zeros(r, d + 1), requires_grad=True)
        self.A = nn.init.xavier_uniform_(self.A)
        self.c = nn.Linear(d + 1, 1, bias=True)
        self.w = nn.Linear(m, 1, bias=False)
        self.N = ResNN(d, m, nTh=nTh)
        self.w.weight.data = torch.ones(self.w.weight.data.shape)
        self.c.weight.data = torch.zeros(self.c.weight.data.shape)
        self.c.bias.data = torch.zeros(self.c.bias.data.shape)

    def forward(self, x):
        """Phi(s) for rows s = [x, t] of shape [n, d+1] -> [n, 1]  (src/Phi.py:91-96), on the GPU."""
        from .ocflow import phi_apply
        return phi_apply(self, x, False)

    def getGrad(self, x):
        """grad_s Phi -> [n, d+1]  (src/Phi.py:99-138), on the GPU."""
        from .ocflow import phi_apply
        return phi_apply(self, x, True)

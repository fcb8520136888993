"""OCflow — drop-in for the reference's closed-loop rollout (src/OCflow.py:7-95) on a B200.

Same signature, same return conventions, same quirks:

    OCflow(x, Phi, prob, tspan, nt, stepper="rk4", alph=[1.0]*6, intermediates=False, noMean=False)

`Phi` is any module with the reference's layout (src/Phi.py:56-138: `A, c, w, N.layers, N.h, N.nTh`)
— the reference's own class or neuraloc_b200.Phi; `prob` is any object with the duck-typed problem
attributes (class name Cross2D / SwarmTraj / Quadcopter).  The host side only flattens those two
objects into the C structs of include/noc_b200.h and launches; all arithmetic is in libnoc_b200.so.

Deviations from the reference (documented in DESIGN.md):
  * training (trainOC.py:172-173): with autograd enabled and parameters (or x) requiring grad, the default (mean) return mode
    with stepper 'rk4' and nTh = 2 runs the fused rollout + discrete-adjoint kernel (noc_ocflow_grad) and `Jc.backward()` works;
    the gradient flows through Jc only (the entries of cs are detached).  Every other combination raises instead of silently
    returning a non-differentiable result;
  * Phi.forward / Phi.getGrad (phi_apply): with autograd enabled and s or a parameter requiring grad, nTh = 2 nets are
    differentiated by one noc_phi_vjp call per backward; other depths raise.  The problem evaluators (prob_eval, behind
    calcLHQW / calcGradpH / calcCtrls and ocOdefun) are forward-only and raise when asked for a gradient;
  * errors raise (ValueError / RuntimeError) instead of print + exit(1).
"""
import ctypes as C
import weakref

import torch
from torch.autograd.function import once_differentiable

from . import _cabi

_PACK_CACHE = weakref.WeakKeyDictionary()     # Phi module -> {(device, dtype): (signature, tensors, PhiT, keepalive)}


def _require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("neuraloc_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def _dtype_code(dt):
    if dt == torch.float32:
        return _cabi.F32
    if dt == torch.float64:
        return _cabi.F64
    raise ValueError("OCflow supports float32 and float64 tensors (--prec single|double), got %s" % dt)


def invalidate_cache(Phi=None):
    """Drop the cached device copies of a module's weights (all modules if None).  The cache key is (data_ptr, _version, dtype,
    device) of every parameter: load_state_dict, optimizers and in-place ops on the parameters are seen; in-place edits made
    through `p.data` are NOT (Tensor.data has its own version counter) — call this after such edits."""
    if Phi is None:
        _PACK_CACHE.clear()
    else:
        _PACK_CACHE.pop(Phi, None)


def _phi_struct(Phi, device, dtype):
    """Flatten the live module into noc_phi_t (device copies in `dtype`; cached until a parameter changes, see
    invalidate_cache)."""
    layers = list(Phi.N.layers)
    tensors = _phi_tensors(Phi)
    sig = tuple((t.data_ptr(), t._version, t.dtype, str(t.device)) for t in tensors)
    per = _PACK_CACHE.setdefault(Phi, {})
    hit = per.get((str(device), dtype))
    if hit is not None and hit[0] == sig:
        return hit[2]
    nTh = len(layers)
    if nTh < 2:
        raise ValueError("nTh must be an integer >= 2")
    m, D = layers[0].weight.shape
    dev = [t.detach().to(device=device, dtype=dtype).contiguous() for t in tensors]
    K = (C.c_void_p * nTh)(*[t.data_ptr() for t in dev[4:4 + nTh]])
    b = (C.c_void_p * nTh)(*[t.data_ptr() for t in dev[4 + nTh:4 + 2 * nTh]])
    st = _cabi.PhiT(d=D - 1, m=m, nTh=nTh, r=Phi.A.shape[0], h=float(getattr(Phi.N, "h", 1.0 / (nTh - 1))),
                    A=dev[0].data_ptr(), c_w=dev[1].data_ptr(), c_b=dev[2].data_ptr(), w=dev[3].data_ptr(),
                    K=C.cast(K, C.POINTER(C.c_void_p)), b=C.cast(b, C.POINTER(C.c_void_p)))
    per[(str(device), dtype)] = (sig, dev, st, (K, b))
    return st


def _prob_struct(prob, device, dtype):
    name = type(prob).__name__
    if name not in _cabi.PROB_KINDS:
        raise ValueError("unsupported problem class %r (expected Cross2D, SwarmTraj or Quadcopter)" % name)
    obstacle = getattr(prob, "obstacle", None)
    if obstacle not in _cabi.OBSTACLES:
        if name == "Quadcopter":
            obstacle = None        # Quadcopter.calcObstacle ignores unknown obstacles (Quadcopter.py:115-122)
        else:
            raise ValueError("unsupported obstacle %r" % (obstacle,))
    # xtarget is d numbers: upload it on every call when it is not already a device tensor of the rollout dtype (a cache keyed
    # on the source's address could hand back another problem's target after the allocator reuses the address)
    xdev = prob.xtarget.detach().reshape(-1).to(device=device, dtype=dtype).contiguous()
    st = _cabi.ProbT(kind=_cabi.PROB_KINDS[name], obstacle=_cabi.OBSTACLES[obstacle], training=int(bool(prob.training)),
                     nAgents=int(prob.nAgents), agentDim=int(prob.agentDim), alph_Q=float(prob.alph_Q),
                     alph_W=float(prob.alph_W), r=float(prob.r), mass=float(getattr(prob, "mass", 1.0)),
                     grav=float(getattr(prob, "grav", 9.81)), xtarget=xdev.data_ptr())
    return st, xdev


def stage_times(t0, t1, nt):
    """nt x 5 table (t_a, t_a+h'/2, t_a+h', t_ctrl, h') in Python doubles — the reference's own arithmetic
    (OCflow.py:25,35,47,50,53; stepRK4's `h = t1 - t0`, :169), handed to the kernel verbatim."""
    h = (t1 - t0) / nt
    tk = t0
    tab = (C.c_double * (5 * nt))()
    for k in range(nt):
        ta, tb = tk, tk + h
        hh = tb - ta
        tk += h
        tab[5 * k:5 * k + 5] = [ta, ta + (hh / 2), ta + hh, tk - h, hh]
    return tab


def _wants_grad(x, Phi):
    return torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in Phi.parameters()))


def _check_forward_only(x, Phi):
    if _wants_grad(x, Phi):
        raise RuntimeError("neuraloc_b200: this call is forward-only — run it under torch.no_grad() (as evalOC.py / timeOC.py / "
                           "validation do). Differentiation is implemented for OCflow's default return mode with stepper='rk4' "
                           "(trainOC.py:172) and is never silently approximated elsewhere.")


def _phi_tensors(Phi):
    layers = list(Phi.N.layers)
    return [Phi.A, Phi.c.weight, Phi.c.bias, Phi.w.weight] + [l.weight for l in layers] + [l.bias for l in layers]


def ocflow_grad_sums(x, Phi, prob, tspan, nt, alph=(1.0,) * 6, want_xgrad=False):
    """Training evaluation through noc_ocflow_grad: (sums, grad, grad_x) on the CUDA device —
    sums   float64 [8] = sums over the rows of x of [L, G, HJt, HJfin, HJgrad, Q, W] and the row count (as ocflow_sums),
    grad   [P] in x.dtype: SUMS over the rows of d(per-sample objective)/d(parameter), concatenated in state_dict order
           (A, c.weight, c.bias, w.weight, N.layers.0.weight, N.layers.0.bias, N.layers.1.weight, N.layers.1.bias),
    grad_x [n, d] or None.  Sums, so that the shards of a multi-GPU batch add (one all-reduce of the two vectors)."""
    _require_cuda()
    L = _cabi.lib()
    if x.dim() != 2:
        raise ValueError("x must be nex-by-d")
    code = _dtype_code(x.dtype)
    n, d = x.shape
    nt = int(nt)
    device = x.device if x.is_cuda else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(device):
        phi = _phi_struct(Phi, device, x.dtype)
        if phi.d != d:
            raise ValueError("x has %d columns but Phi expects d = %d" % (d, phi.d))
        if phi.nTh != 2:
            raise RuntimeError("differentiating the rollout is implemented for nTh = 2 (got %d)" % phi.nTh)
        pst, _keep = _prob_struct(prob, device, x.dtype)
        tab = stage_times(float(tspan[0]), float(tspan[1]), nt)
        al = (C.c_double * 6)(*[float(a) for a in alph])
        xin = x.detach().to(device).contiguous()
        sums = torch.empty(8, dtype=torch.float64, device=device)
        grad = torch.empty(_grad_len(phi), dtype=x.dtype, device=device)
        gx = torch.empty(n, d, dtype=x.dtype, device=device) if want_xgrad else None
        rc = L.noc_ocflow_grad(C.byref(phi), C.byref(pst), xin.data_ptr(), n, tab, float(tspan[0]), float(tspan[1]), nt, al, code,
                               sums.data_ptr(), grad.data_ptr(), None if gx is None else gx.data_ptr(),
                               torch.cuda.current_stream(device).cuda_stream)
        _cabi.check(rc)
    return sums, grad, gx


def _grad_len(phi):
    """P, the length of the flat parameter gradient of noc_ocflow_grad / noc_phi_vjp for a noc_phi_t with nTh = 2."""
    D, m, r = phi.d + 1, phi.m, phi.r
    return r * D + D + 1 + m + m * D + m + m * m + m


def split_param_grads(Phi, grad):
    """The flat gradient of ocflow_grad_sums as tensors shaped like (and ordered as) _phi_tensors(Phi):
    [A, c.weight, c.bias, w.weight, N.layers.0.weight, N.layers.1.weight, N.layers.0.bias, N.layers.1.bias]."""
    A, cw, cb, w, K0, K1, b0, b1 = _phi_tensors(Phi)
    out, off = {}, 0
    for name, t in (("A", A), ("cw", cw), ("cb", cb), ("w", w), ("K0", K0), ("b0", b0), ("K1", K1), ("b1", b1)):
        out[name] = grad[off:off + t.numel()].reshape(t.shape)
        off += t.numel()
    return [out[k] for k in ("A", "cw", "cb", "w", "K0", "K1", "b0", "b1")]


class _RolloutWithAdjoint(torch.autograd.Function):
    """Jc (differentiable) and the 7 mean cost terms (detached) of one training evaluation; the backward pass only scales the
    gradient the fused kernel already produced (trainOC.py:172-173)."""

    @staticmethod
    def forward(ctx, x, Phi, prob, tspan, nt, alph, *params):
        sums, grad, gx = ocflow_grad_sums(x, Phi, prob, tspan, nt, alph, want_xgrad=x.requires_grad)
        means = (sums[:7] / sums[7]).to(x.dtype)
        Jc = means[0] + alph[0] * means[1] + alph[3] * means[2] + alph[4] * means[3] + alph[5] * means[4]
        inv = (1.0 / sums[7]).to(x.dtype)
        ctx.flat = grad * inv                      # ONE scaling of the flat gradient; the per-parameter tensors are views of it
        ctx.Phi = Phi
        ctx.gx = None if gx is None else (gx * inv).to(x.device)
        ctx.like = [(p.device, p.dtype, p.requires_grad) for p in params]
        Jc, means = Jc.to(x.device), means.to(x.device)
        ctx.mark_non_differentiable(means)
        return Jc, means

    @staticmethod
    @once_differentiable          # the kernels produce first derivatives only: a double backward raises instead of returning zeros
    def backward(ctx, gJ, _gmeans):
        flat = ctx.flat * gJ.to(ctx.flat.device)
        pg = [g.to(device=dev, dtype=dt) if need else None for g, (dev, dt, need) in zip(split_param_grads(ctx.Phi, flat), ctx.like)]
        gx = None if ctx.gx is None else ctx.gx * gJ.to(ctx.gx.device)
        return (gx, None, None, None, None, None, *pg)


def _launch(x, Phi, prob, tspan, nt, stepper, alph, mode):
    """Runs the C-ABI rollout. Returns (out, zFull, ctrlFull) on x.device; `out` is the 8-double sum vector in
    mean mode (CUDA x: a device tensor, no host sync), the [n,8] table in noMean mode."""
    _require_cuda()
    L = _cabi.lib()
    if x.dim() != 2:
        raise ValueError("x must be nex-by-d")
    code = _dtype_code(x.dtype)
    n, d = x.shape
    nt = int(nt)
    on_cuda = x.is_cuda
    device = x.device if on_cuda else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(device):
        phi = _phi_struct(Phi, device, x.dtype)
        if phi.d != d:
            raise ValueError("x has %d columns but Phi expects d = %d" % (d, phi.d))
        pst, _keep = _prob_struct(prob, device, x.dtype)
        tab = stage_times(float(tspan[0]), float(tspan[1]), nt)
        al = (C.c_double * 6)(*[float(a) for a in alph])
        step = _cabi.STEPPERS.get(stepper, 0)
        nctrl = L.noc_ctrl_dim(C.byref(pst), d)
        if nctrl < 0:
            _cabi.check(nctrl)
        odev = x.device
        xin = x.detach().contiguous()
        out = zf = cf = None
        if mode == _cabi.MODE_MEAN:
            out = torch.empty(8, dtype=torch.float64, device=odev)
        elif mode == _cabi.MODE_NOMEAN:
            out = torch.empty(n, 8, dtype=x.dtype, device=odev)
        else:
            zf = torch.empty(n, d + 4, nt + 1, dtype=x.dtype, device=odev)
            cf = torch.empty(n, nctrl, nt + 1, dtype=x.dtype, device=odev)
        ptr = lambda t: None if t is None else t.data_ptr()
        stream = torch.cuda.current_stream(device).cuda_stream
        fn = L.noc_ocflow if on_cuda else L.noc_ocflow_host
        rc = fn(C.byref(phi), C.byref(pst), xin.data_ptr(), n, tab, float(tspan[0]), float(tspan[1]), nt, step, al,
                mode, code, ptr(out), ptr(zf), ptr(cf), stream)
        _cabi.check(rc)
    return out, zf, cf


def costs_from_sums(sums, alph, dtype):
    """means + objective from the 8-vector [sum L, G, HJt, HJfin, HJgrad, Q, W, count] (OCflow.py:80-90)."""
    means = (sums[:7] / sums[7]).to(dtype)
    cs = [means[i] for i in range(7)]
    Jc = cs[0] + alph[0] * cs[1] + alph[3] * cs[2] + alph[4] * cs[3] + alph[5] * cs[4]
    return Jc, cs


def ocflow_sums(x, Phi, prob, tspan, nt, stepper="rk4", alph=(1.0,) * 6):
    """Cost SUMS over the rows of x plus the row count, as a float64 8-vector on x.device.  This is what a
    shard contributes to the all-reduce in the multi-GPU path (neuraloc_b200.sharded)."""
    _check_forward_only(x, Phi)
    return _launch(x, Phi, prob, tspan, nt, stepper, alph, _cabi.MODE_MEAN)[0]


def OCflow(x, Phi, prob, tspan, nt, stepper="rk4", alph=[1.0, 1.0, 1.0, 1.0, 1.0, 1.0], intermediates=False, noMean=False):
    """Closed-loop rollout + objective; see src/OCflow.py:7-22 for the argument meaning.

    returns  Jc, cs                       0-dim tensors, cs = [L, G, HJt, HJfin, HJgrad, Q, W] (means over samples)
             Jc [n,1], cs 7 x [n,1]       with noMean=True (tested first, quirk 4)
             zFull [n,d+4,nt+1], ctrlFull [n,nCtrl,nt+1]   with intermediates=True
    """
    alph = [float(a) for a in alph]
    if _wants_grad(x, Phi) and not noMean and not intermediates and stepper == "rk4":
        Jc, means = _RolloutWithAdjoint.apply(x, Phi, prob, [float(tspan[0]), float(tspan[1])], int(nt), alph, *_phi_tensors(Phi))
        return Jc, [means[i] for i in range(7)]
    _check_forward_only(x, Phi)
    if noMean:
        out = _launch(x, Phi, prob, tspan, nt, stepper, alph, _cabi.MODE_NOMEAN)[0]
        return out[:, 0:1], [out[:, i:i + 1] for i in range(1, 8)]
    if intermediates:
        _, zf, cf = _launch(x, Phi, prob, tspan, nt, stepper, alph, _cabi.MODE_INTERMEDIATES)
        return zf, cf
    sums = _launch(x, Phi, prob, tspan, nt, stepper, alph, _cabi.MODE_MEAN)[0]
    return costs_from_sums(sums, alph, x.dtype)


def phi_eval(Phi, s, want_phi=True, want_grad=True):
    """Phi.forward / Phi.getGrad on rows s = [x,t] (src/Phi.py:91-138) through noc_phi_eval."""
    _require_cuda()
    L = _cabi.lib()
    code = _dtype_code(s.dtype)
    device = s.device if s.is_cuda else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(device):
        phi = _phi_struct(Phi, device, s.dtype)
        n, D = s.shape
        if D != phi.d + 1:
            raise ValueError("s has %d columns but Phi expects d+1 = %d" % (D, phi.d + 1))
        sd = s.detach().to(device).contiguous()
        op = torch.empty(n, 1, dtype=s.dtype, device=device) if want_phi else None
        og = torch.empty(n, D, dtype=s.dtype, device=device) if want_grad else None
        rc = L.noc_phi_eval(C.byref(phi), sd.data_ptr(), n, code, None if op is None else op.data_ptr(),
                            None if og is None else og.data_ptr(), torch.cuda.current_stream(device).cuda_stream)
        _cabi.check(rc)
    back = (lambda t: None if t is None else t.to(s.device))
    return back(op), back(og)


def phi_vjp(Phi, s, seed_phi=None, seed_grad=None, want_params=True, want_s=True):
    """Reverse-mode product of Phi.forward / Phi.getGrad through noc_phi_vjp.  For psi_i = a_i Phi(s_i) + B_i . grad Phi(s_i), with
    a = seed_phi ([n] or [n,1]) and B = seed_grad ([n, d+1]), None meaning zero, returns on the CUDA device in s.dtype
    grad_params [P]    SUMS over the rows of d psi_i / d parameter, flat in split_param_grads' order (None unless want_params),
    grad_s [n, d+1]    d psi_i / d s_i = a_i grad Phi(s_i) + Hess Phi(s_i) B_i (None unless want_s).  nTh = 2 only."""
    _require_cuda()
    L = _cabi.lib()
    code = _dtype_code(s.dtype)
    device = s.device if s.is_cuda else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(device):
        phi = _phi_struct(Phi, device, s.dtype)
        n, D = s.shape
        if D != phi.d + 1:
            raise ValueError("s has %d columns but Phi expects d+1 = %d" % (D, phi.d + 1))
        if phi.nTh != 2:
            raise RuntimeError("the reverse-mode product of Phi is implemented for nTh = 2 (got %d)" % phi.nTh)
        dev = lambda t, shape: None if t is None else t.detach().reshape(shape).to(device=device, dtype=s.dtype).contiguous()
        sd, a, B = dev(s, (n, D)), dev(seed_phi, (n,)), dev(seed_grad, (n, D))
        gp = torch.empty(_grad_len(phi), dtype=s.dtype, device=device) if want_params else None
        gs = torch.empty(n, D, dtype=s.dtype, device=device) if want_s else None
        ptr = lambda t: None if t is None else t.data_ptr()
        rc = L.noc_phi_vjp(C.byref(phi), sd.data_ptr(), n, ptr(a), ptr(B), code, ptr(gp), ptr(gs),
                           torch.cuda.current_stream(device).cuda_stream)
        _cabi.check(rc)
    return gp, gs


class _PhiWithVJP(torch.autograd.Function):
    """Phi(s) [n,1] (want_grad False) or grad_s Phi(s) [n, d+1] (want_grad True) by noc_phi_eval — the values of the no-grad
    path — differentiated with respect to s and every parameter by one noc_phi_vjp call."""

    @staticmethod
    def forward(ctx, s, Phi, want_grad, *params):
        out = phi_eval(Phi, s, not want_grad, want_grad)[1 if want_grad else 0]
        ctx.save_for_backward(s, *params)          # in-place edits of s or of a parameter before backward() raise, as in torch
        ctx.Phi, ctx.want_grad = Phi, want_grad
        return out

    @staticmethod
    @once_differentiable          # the kernel produces first derivatives only: a double backward raises instead of returning zeros
    def backward(ctx, gout):
        s, *params = ctx.saved_tensors
        need_s, need_p = ctx.needs_input_grad[0], ctx.needs_input_grad[3:]
        gp, gs = phi_vjp(ctx.Phi, s, None if ctx.want_grad else gout, gout if ctx.want_grad else None,
                         want_params=any(need_p), want_s=need_s)
        pg = [None] * len(params)
        if gp is not None:
            pg = [g.to(device=p.device, dtype=p.dtype) if need else None
                  for g, p, need in zip(split_param_grads(ctx.Phi, gp), params, need_p)]
        return (None if gs is None else gs.to(s.device), None, None, *pg)


def phi_apply(Phi, s, want_grad):
    """Phi.forward (want_grad False: [n,1]) or Phi.getGrad (want_grad True: [n, d+1]) on rows s = [x,t].  Differentiable when
    autograd is enabled and s or a parameter requires grad (nTh = 2); a plain noc_phi_eval call otherwise."""
    if _wants_grad(s, Phi):
        nTh = len(Phi.N.layers)
        if nTh != 2:
            raise RuntimeError("neuraloc_b200: Phi.forward / Phi.getGrad are differentiable for nTh = 2 (this net has nTh = %d); "
                               "evaluate deeper nets under torch.no_grad()" % nTh)
        return _PhiWithVJP.apply(s, Phi, want_grad, *_phi_tensors(Phi))
    return phi_eval(Phi, s, not want_grad, want_grad)[1 if want_grad else 0]


def prob_eval(prob, x, p):
    """(LHQW [n,4], gradpH [n,d], ctrls [n,nCtrl]) through noc_prob_eval.  Forward-only: the results carry no gradient, so a
    request for one raises."""
    if torch.is_grad_enabled() and (x.requires_grad or p.requires_grad):
        raise RuntimeError("neuraloc_b200: calcLHQW / calcGradpH / calcCtrls (and ocOdefun, which calls them) are forward-only — "
                           "their results would carry no gradient to x or p. Call them under torch.no_grad() or on detached tensors.")
    _require_cuda()
    L = _cabi.lib()
    code = _dtype_code(x.dtype)
    device = x.device if x.is_cuda else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(device):
        n, d = x.shape
        pst, _keep = _prob_struct(prob, device, x.dtype)
        nctrl = L.noc_ctrl_dim(C.byref(pst), d)
        xd = x.detach().to(device).contiguous()
        pd = p.detach().to(device=device, dtype=x.dtype).contiguous()
        o1 = torch.empty(n, 4, dtype=x.dtype, device=device)
        o2 = torch.empty(n, d, dtype=x.dtype, device=device)
        o3 = torch.empty(n, nctrl, dtype=x.dtype, device=device)
        rc = L.noc_prob_eval(C.byref(pst), xd.data_ptr(), pd.data_ptr(), n, d, code, o1.data_ptr(), o2.data_ptr(),
                             o3.data_ptr(), torch.cuda.current_stream(device).cuda_stream)
        _cabi.check(rc)
    return o1.to(x.device), o2.to(x.device), o3.to(x.device)


def OCflow_shock(x, Phi, prob, nt, shockspec, stepper="rk4", alph=[1.0, 1.0, 1.0, 1.0, 1.0, 1.0]):
    """The shock / re-planning experiment of src/plotter.py:815-823 (evalOC.py:113-120) for a whole batch, device-resident:
    roll out to t_s = shockspec[0] with nShock = int(t_s * nt) steps, displace every state by shockspec[1] (a [1,d] row, as in
    evalOC.py, or one row per sample [n,d]), and let the closed loop recover over [t_s, 1] with 1 + nt - nShock steps.

    returns  traj1 [n,d+4,nShock+1], ctrl1, traj2 [n,d+4,nt-nShock+2], ctrl2   (the reference concatenates traj1[:, :d] and
             traj2[:, :d] along time; the four cost integrals of each leg start at 0, as in the reference's two calls)
    Both legs run on x's device; nothing but the two launches happens in between (no host round trip of the trajectories)."""
    prec, shock = float(shockspec[0]), shockspec[1]
    nt = int(nt)
    nShock = int(prec * nt)
    if nShock < 1 or nShock > nt:
        raise ValueError("shock time %g leaves no step on one side of it for nt = %d" % (prec, nt))
    d = x.shape[1]
    traj1, ctrl1 = OCflow(x, Phi, prob, [0.0, prec], nShock, stepper, alph, intermediates=True)
    xs = traj1[:, :d, -1] + torch.as_tensor(shock, dtype=x.dtype, device=traj1.device).reshape(-1, d)
    traj2, ctrl2 = OCflow(xs.contiguous(), Phi, prob, [prec, 1.0], 1 + nt - nShock, stepper, alph, intermediates=True)
    return traj1, ctrl1, traj2, ctrl2


# ---- names other reference scripts import from src.OCflow (compareCorridor.py:18, baseline2D.py:9) ----------
def ocG(z, xtarget):
    """G residual x - xtarget (src/OCflow.py:97-101); trivial host-side helper kept for importers."""
    d = xtarget.shape[0]
    return z[:, 0:d] - xtarget


def ocOdefun(x, t, net, prob, alph=None):
    """RHS of the augmented ODE for z = [x, L, HJt, Q, W] rows (src/OCflow.py:104-140), assembled from the two
    device evaluators (noc_phi_eval, noc_prob_eval); the rollout itself never calls this."""
    d = x.shape[1] - 4
    s = torch.nn.functional.pad(x[:, :d], (0, 1, 0, 0), value=t)
    g = phi_apply(net, s, True)
    lhqw, gph, _ = prob_eval(prob, s[:, :d], g[:, :d])
    hj = torch.abs(g[:, d:d + 1] - lhqw[:, 1:2])
    return torch.cat((-gph, lhqw[:, 0:1], hj, lhqw[:, 2:3], lhqw[:, 3:4]), 1)


def _one_step(z, Phi, prob, alph, t0, t1, stepper):
    d = z.shape[1] - 4
    zf = _launch(z[:, :d], Phi, prob, [t0, t1], 1, stepper, [1.0] * 6 if alph is None else alph, _cabi.MODE_INTERMEDIATES)[1]
    out = zf[:, :, 1].clone()
    out[:, d:] += z[:, d:]          # the four cost integrals are additive in their initial value
    return out


def stepRK4(odefun, z, Phi, prob, alph, t0, t1):
    """One classical RK4 step of the augmented state (src/OCflow.py:157-184) = a 1-step fused rollout.
    `odefun` is accepted for signature parity; the fused kernel always integrates ocOdefun."""
    return _one_step(z, Phi, prob, alph, t0, t1, "rk4")


def stepRK1(odefun, z, Phi, prob, alph, t0, t1):
    """One forward-Euler step (src/OCflow.py:143-155)."""
    return _one_step(z, Phi, prob, alph, t0, t1, "rk1")

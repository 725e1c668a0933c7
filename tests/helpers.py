"""Parity metric of SURVEY.md section 8(d): fp32 tensors must satisfy BOTH
   rel = ||a - b||_inf / ||b||_inf <= tol   and   allclose(a, b, rtol=tol, atol=tol * ||b||_inf)
with tol = 1e-5 (north_star: "fp32 node outputs and gradients within 1e-5 relative")."""
import torch

TOL = 1e-5


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    denom = b.abs().max().item()
    return (a - b).abs().max().item() / (denom if denom > 0 else 1.0)


def assert_close(a, b, tol=TOL, what=""):
    a_, b_ = a.detach().float().cpu(), b.detach().float().cpu()
    assert a_.shape == b_.shape, f"{what}: shape {tuple(a_.shape)} vs {tuple(b_.shape)}"
    scale = b_.abs().max().item()
    r = rel_err(a_, b_)
    assert r <= tol, f"{what}: rel err {r:.3e} > {tol}"
    assert torch.allclose(a_, b_, rtol=tol, atol=tol * max(scale, 1e-30)), f"{what}: allclose failed (rel {r:.3e})"
    return r


def canonical(edge_index):
    ei = edge_index.detach().cpu()
    n = int(ei.max()) + 1 if ei.numel() else 1
    key = ei[1] * n + ei[0]
    return ei[:, torch.sort(key, stable=True).indices]


def assert_close_arbiter(a, ref32, ref64, tol=TOL, what=""):
    """fp64 arbiter (SURVEY.md 8c item 6): where the fp32 oracle itself is ill-conditioned
    (||oracle_fp32 - fp64|| > tol, e.g. softmax-gradient cancellation), the CUDA result must be
    as close to the fp64 evaluation as the fp32 oracle is (factor 2), else the plain 1e-5 bar."""
    r = rel_err(a, ref32)
    if r <= tol:
        return r
    e_ours, e_ref = rel_err(a, ref64), rel_err(ref32, ref64)
    assert e_ours <= max(tol, 2.0 * e_ref), (f"{what}: rel err vs fp32 oracle {r:.3e}; vs fp64 arbiter ours {e_ours:.3e}, "
                                             f"fp32 oracle {e_ref:.3e}")
    return e_ours


def gradient_conditioning(model64, loss_fn, eps=1e-6, samples=3, seed=0):
    """How far the fp64 gradients of ``model64`` move when every weight is perturbed by a relative ``eps`` (the size of an
    fp32 rounding error after a few layers): {parameter name: max over ``samples`` of ||g' - g||_inf / ||g||_inf}.

    The train step is not smooth: ReLU masks (models/model.py:71,77,88) and the sign of the L1 loss (train.py:52) are
    discontinuous, so two correct fp32 evaluations whose activations differ by 1e-6 can flip a unit that sits at zero and
    move a weight gradient by ~1 / (number of nodes) — 1e-4 at BASELINE C1's 8000 nodes, far above any rounding error, and
    which units flip is luck (the fp32 oracle itself is 6e-5 from fp64 on one decoder weight at C1).  This measures that
    sensitivity on the fp64 oracle itself, per parameter; ``assert_close_conditioned`` widens the tolerance by exactly that
    much and no more.  ``loss_fn(model) -> loss`` must rebuild the graph from the model's current weights."""
    import copy
    base = copy.deepcopy(model64)
    base.zero_grad()
    loss_fn(base).backward()
    g0 = {k: p.grad.clone() for k, p in base.named_parameters()}
    gen = torch.Generator().manual_seed(seed)
    out = {k: 0.0 for k in g0}
    for _ in range(samples):
        m = copy.deepcopy(model64)
        with torch.no_grad():
            for p in m.parameters():
                p.mul_(1.0 + eps * torch.randn(p.shape, generator=gen, dtype=p.dtype).to(p.device))
        m.zero_grad()
        loss_fn(m).backward()
        for k, p in m.named_parameters():
            out[k] = max(out[k], rel_err(p.grad, g0[k]))
    return out


def assert_close_conditioned(a, ref32, ref64, cond, tol=TOL, what=""):
    """``assert_close_arbiter`` for a non-smooth problem: within ``tol`` of the fp32 oracle, or as close to the fp64 evaluation
    as the fp32 oracle is (x2), or within twice the movement a 1e-6 perturbation of the weights causes in fp64 (``cond``,
    from ``gradient_conditioning``) — whichever is largest."""
    r = rel_err(a, ref32)
    if r <= tol:
        return r
    e_ours, e_ref = rel_err(a, ref64), rel_err(ref32, ref64)
    assert e_ours <= max(tol, 2.0 * e_ref, 2.0 * cond), (f"{what}: rel err vs fp32 oracle {r:.3e}; vs fp64 arbiter ours {e_ours:.3e}, "
                                                        f"fp32 oracle {e_ref:.3e}, fp64 under a 1e-6 weight perturbation {cond:.3e}")
    return e_ours

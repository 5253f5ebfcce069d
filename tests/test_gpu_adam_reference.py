"""gh_adam_step (through FusedAdam) against torch.optim.Adam's arithmetic written out in float64.

Every step is checked from the kernel's own float32 state before it: the float64 step is applied to that state and
the kernel's update p_new - p_old, exp_avg and exp_avg_sq are compared with it, each relative to its own magnitude.
The parameters are initialised at the scale of their learning rate, so that the rounding of p_new to float32 stays
far below the size of the update and the comparison sees the update's own arithmetic.

What separates the kernel from float64, by reading the code: sqrt.approx and rcp.approx (about 1 ulp each), and
1 - beta1, 1 - beta2 formed in float32 from the float32 betas (0.999f is 0.99900001, so 1 - beta2 is 1.3e-5 below
0.001, which moves exp_avg_sq on the first step by 1.3e-5 relative and the update by half that).  The bounds are
1e-4 relative.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

BETAS = (0.9, 0.999)
EPS = 1e-15
TOL = 1e-4
SIZES = [1, 2, 3, 5, 1023, 4097, 300001, 65536 * 3]     # 8 groups: GH_ADAM_MAX_GROUPS
LRS = [1.6e-4, 2.5e-3, 1.25e-4, 0.05, 0.0025, 0.005, 0.001, 0.01]


def adam_step_f64(p, g, m, v, lr, step):
    """torch.optim.Adam (single-tensor path) in float64 for one step; returns (p, m, v)."""
    b1, b2 = BETAS
    p, g, m, v = (t.double() for t in (p, g, m, v))
    m = m + (g - m) * (1 - b1)                       # exp_avg.lerp_(grad, 1 - beta1)
    v = v * b2 + g * g * (1 - b2)                    # exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    denom = v.sqrt() / bc2 ** 0.5 + EPS
    return p - (lr / bc1) * m / denom, m, v


def rel(a, b):
    """(norm-relative error, max element error over max|b|) of a against b."""
    d = (a.double() - b).flatten()
    nb, mb = float(b.norm()), float(b.abs().max())
    if nb == 0.0:
        return (0.0, 0.0) if float(d.abs().max()) == 0.0 else (float("inf"), float("inf"))
    return float(d.norm()) / nb, float(d.abs().max()) / mb


def make_params(device, misaligned=False, seed=0):
    g = torch.Generator().manual_seed(seed)
    ps = []
    for n, lr in zip(SIZES, LRS):
        init = (torch.randn(n, generator=g) * lr).to(device)
        if misaligned:                               # contiguous, but 4 bytes past a 16-byte boundary
            buf = torch.zeros(n + 1, device=device)
            buf[1:].copy_(init)
            p = torch.nn.Parameter(buf[1:n + 1])
            assert p.data_ptr() % 16 == 4 and p.is_contiguous()
        else:
            p = torch.nn.Parameter(init)
        ps.append(p)
    return ps


def run_and_check(device, ps, misaligned=False, empty=None):
    from gaussianhaircut_b200.optim import FusedAdam
    groups = [{"params": [p], "lr": lr, "name": f"g{k}"} for k, (p, lr) in enumerate(zip(ps, LRS))]
    if empty is not None:
        groups.append({"params": [empty], "lr": 0.01, "name": "empty"})
    opt = FusedAdam(groups, betas=BETAS, eps=EPS)
    gen = torch.Generator().manual_seed(42)
    worst = {"update": 0.0, "exp_avg": 0.0, "exp_avg_sq": 0.0}
    for it in range(6):
        grads = [torch.randn(p.shape, generator=gen).to(device) * (10.0 ** (it - 3)) for p in ps]
        poisoned = it == 3
        if poisoned:
            grads[5][17] = float("nan")
        if misaligned:
            bufs = [torch.zeros(gr.numel() + 1, device=device) for gr in grads]
            for b, gr in zip(bufs, grads):
                b[1:].copy_(gr)
            grads = [b[1:] for b in bufs]
        for p, gr in zip(ps, grads):
            p.grad = gr
        if empty is not None:
            empty.grad = torch.zeros_like(empty)
        before = [(p.detach().clone(), opt._state_for(p)["exp_avg"].clone(), opt._state_for(p)["exp_avg_sq"].clone())
                  for p in ps]
        step_dev = opt.step_count                  # the count held on the device: this step is number step_dev + 1
        opt.step()
        torch.cuda.synchronize()
        assert bool(opt.nan_flag.item() != 0) == poisoned
        assert opt.step_count == step_dev + (0 if poisoned else 1)
        for k, (p, (p0, m0, v0)) in enumerate(zip(ps, before)):
            st = opt.state[p]
            if poisoned:
                assert torch.equal(p.detach(), p0) and torch.equal(st["exp_avg"], m0) and torch.equal(st["exp_avg_sq"], v0), \
                    f"group {k} changed on a skipped step"
                continue
            p_ref, m_ref, v_ref = adam_step_f64(p0, grads[k], m0, v0, LRS[k], step_dev + 1)
            upd, upd_ref = p.detach().double() - p0.double(), p_ref - p0.double()
            for name, got, ref in (("update", upd, upd_ref), ("exp_avg", st["exp_avg"], m_ref),
                                   ("exp_avg_sq", st["exp_avg_sq"], v_ref)):
                e_norm, e_max = rel(got, ref)
                worst[name] = max(worst[name], e_norm, e_max)
                assert e_norm <= TOL and e_max <= TOL, \
                    f"step {it}, group {k} ({SIZES[k]} elements, lr {LRS[k]}): {name} off by {e_norm:.3g} (norm) / {e_max:.3g} (max)"
    assert opt.step_count == 5
    print(f"FusedAdam vs float64 Adam, worst relative error: {worst}")
    return opt


def test_adam_matches_float64(cuda_device):
    """Eight groups (the maximum) of 1, 2, 3, 5, 1023, 4097 elements (vector body plus scalar tail, or the tail only)
    next to large ones, over 6 steps with one NaN-skipped step."""
    run_and_check(cuda_device, make_params(cuda_device))


def test_adam_misaligned_matches_float64(cuda_device):
    """Parameters and gradients that are contiguous but not 16-byte aligned take the scalar path for the whole group."""
    run_and_check(cuda_device, make_params(cuda_device, misaligned=True, seed=1), misaligned=True)


def test_adam_empty_group_is_skipped(cuda_device):
    """A parameter with zero elements (its data_ptr is NULL) is stepped over, as torch.optim.Adam does; the other
    groups are updated as usual."""
    ps = make_params(cuda_device, seed=2)
    empty = torch.nn.Parameter(torch.zeros(0, 3, device=cuda_device))
    assert empty.data_ptr() == 0
    # seven groups checked against float64, the empty one as the eighth
    opt = run_and_check(cuda_device, ps[:7], empty=empty)
    assert empty.shape == (0, 3) and opt.state[empty]["exp_avg"].shape == (0, 3)

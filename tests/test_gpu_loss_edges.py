"""gh_image_loss against the training loss evaluated in float64, at the image sizes and pixels where the kernel's
hand-written parts could go wrong: images smaller than the 11-tap window or one pixel past a 32-pixel loss tile,
and orientation pixels on the branches of the derivative (zero-norm direction, -0.0, the 0.5 / 0.5 split of
torch.minimum's gradient on a tie, the clamp at |y| = 1 - 1e-3), plus degenerate masks, confidences and lambdas.

The reference is oracle/loss_oracle.py run in float64 on the CPU with autograd.  It keeps the reference's float32
window taps (cast to double), because those taps define the operation.  The tolerance is calibrated per case: the
kernel's error against float64 may be at most four times the error of the same restatement run in float32 (which
is how far float32 arithmetic alone is from float64 on these inputs), and never less than a floor of 1e-6 relative
for the loss values and, for each of the 10 gradient channels, 1e-5 norm-relative and 1e-4 * max|ref| element-wise.
"""
import math
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import loss_oracle  # noqa: E402

LAMBDAS = (0.8, 0.2, 0.1, 0.3)
PARTS = ("Ll1", "Lssim", "Lmask", "Lorient")
F32 = np.float32


def _unit_c5(c6: float) -> float:
    """A float32 c5 > 0 for which sqrt(c5^2 + c6^2) rounds to exactly 1 in float32 with or without a fused
    multiply-add, so that y = c6 / |(c5, c6)| == c6 exactly."""
    c6 = F32(c6)
    c5 = F32(math.sqrt(1.0 - float(c6) ** 2))
    for k in range(400):
        x = F32(c5 + F32(k - 200) * np.spacing(c5))
        sums = (F32(F32(x * x) + F32(c6 * c6)), F32(float(x) * float(x) + float(F32(c6 * c6))),
                F32(float(c6) * float(c6) + float(F32(x * x))))
        if all(F32(np.sqrt(s)) == F32(1.0) for s in sums):
            return float(x)
    raise AssertionError("no float32 c5 gives a unit norm")


HI = F32(1.0) - F32(1e-3)                      # the clamp edge as float32 computes it
LO = F32(-1.0) + F32(1e-3)
PAST = np.nextafter(HI, F32(2.0))


def clamp_flips(render):
    """Pixels whose orientation y = normalize(out[5:7]).y falls inside the clamp [-1 + 1e-3, 1 - 1e-3] in float32 but
    not in float64, or the other way round.  The edge itself lies 1.3e-8 apart in the two (0.999f is 0.99900001), so
    at such a pixel the float64 gradient of channels 5 and 6 belongs to the other side of the clamp."""
    y32 = F.normalize(render[5:7].float(), dim=0)[1]
    y64 = F.normalize(render[5:7].double(), dim=0)[1]
    return ((y32 >= float(LO)) & (y32 <= float(HI))) != ((y64 >= -1 + 1e-3) & (y64 <= 1 - 1e-3))


def degenerate_pixels():
    """(name, channel 5, channel 6, gt_angle or None) of the orientation pixels placed on purpose."""
    return [
        ("zero norm", 0.0, 0.0, None),
        ("-0.0 x", -0.0, 0.7, None),
        ("-0.0 x, zero norm", -0.0, 0.0, None),
        ("tie, gt 0", 0.6, 0.0, 0.0),            # angle = acos(0) / pi = 0.5 exactly: |d0| == |d0 - 1|
        ("tie, gt 1", 0.6, 0.0, 1.0),            # |d0| == |d0 + 1|
        ("tie, mirrored", -0.6, 0.0, 0.0),
        ("on clamp", _unit_c5(HI), float(HI), None),
        ("on -clamp", _unit_c5(HI), -float(HI), None),
        ("past clamp", _unit_c5(PAST), float(PAST), None),
        ("past -clamp, mirrored", -_unit_c5(PAST), -float(PAST), None),
        ("y = 1", 0.0, 0.5, None),
    ]


def make_case(W, H, seed, degenerate=True):
    ins = loss_oracle.synthetic_case(W, H, seed)
    if degenerate:
        render, gt_mask, gt_angle, gt_conf = ins[0], ins[2], ins[3], ins[4]
        for k, (_, c5, c6, ga) in enumerate(degenerate_pixels()):
            y, x = divmod((7 * k + 3) % (W * H), W)
            render[5, y, x] = c5
            render[6, y, x] = c6
            if ga is not None:
                gt_angle[0, y, x] = ga
            gt_mask[0, y, x] = 0.8          # the orientation term counts at this pixel
            gt_conf[0, y, x] = 0.7
    return ins


def _loss_and_grad(ins, lambdas, dtype):
    r = ins[0].to(dtype).clone().requires_grad_(True)
    loss, parts = loss_oracle.training_loss(r, *[t.to(dtype) for t in ins[1:]], *lambdas)
    loss.backward()
    vals = {"loss": float(loss.detach())}
    vals.update({k: float(parts[k].detach()) for k in PARTS})
    return vals, r.grad.double()


def check_against_float64(device, ins, lambdas=LAMBDAS):
    """Kernel vs float64 with the calibrated tolerance.  Returns the kernel's gradient, the float64 one, the float32
    restatement's and the kernel's loss values."""
    from gaussianhaircut_b200.losses import hair_image_loss
    ref, g_ref = _loss_and_grad(ins, lambdas, torch.float64)
    o32, g_32 = _loss_and_grad(ins, lambdas, torch.float32)
    r = ins[0].to(device).clone().requires_grad_(True)
    loss, parts = hair_image_loss(r, *[t.to(device) for t in ins[1:]], *lambdas)
    loss.backward()
    got = {"loss": float(loss.detach())}
    got.update({k: float(parts[k]) for k in PARTS})
    g = r.grad.double().cpu()
    assert bool(torch.isfinite(g).all()), "non-finite gradient"
    for k in ("loss",) + PARTS:
        assert math.isfinite(got[k]), f"{k} is {got[k]}"
        err, err32 = abs(got[k] - ref[k]), abs(o32[k] - ref[k])
        bound = max(4 * err32, 1e-6 * max(abs(ref[k]), 0.1))
        assert err <= bound, f"{k}: {got[k]!r} vs float64 {ref[k]!r} (error {err:.3g}, bound {bound:.3g})"
    # a zero-norm direction pixel takes the F.normalize eps branch: its channel-6 gradient is 1e12 times the others
    # and is checked on its own, relative to itself, so that it does not set the scale of the whole channel
    zn = ((ins[0][5] == 0) & (ins[0][6] == 0)).double()
    # pixels on different sides of the orientation clamp in float32 and float64: their channel 5 / 6 gradients are
    # left out of the channel-wide comparison and checked against the float32 restatement, which decides the clamp
    # in the precision that defines the operation, as the kernel does
    flips = clamp_flips(ins[0]).double()
    for ch in range(10):
        d, d32 = g[ch] - g_ref[ch], g_32[ch] - g_ref[ch]
        for y, x in zn.nonzero().tolist():
            e, e32 = abs(float(d[y, x])), abs(float(d32[y, x]))
            assert e <= max(4 * e32, 1e-5 * abs(float(g_ref[ch, y, x]))), \
                f"channel {ch}, zero-norm pixel ({y}, {x}): {float(g[ch, y, x])!r} vs float64 {float(g_ref[ch, y, x])!r}"
        own = zn + (flips if ch in (5, 6) else 0.0) * (1 - zn)
        d, d32, gr = d * (1 - own), d32 * (1 - own), g_ref[ch] * (1 - own)
        amax = float(gr.abs().max())
        if ch in (5, 6):
            for y, x in (flips * (1 - zn)).nonzero().tolist():
                a, b = float(g[ch, y, x]), float(g_32[ch, y, x])
                assert abs(a - b) <= 1e-4 * abs(b) + 1e-6 * amax, \
                    f"channel {ch}, pixel ({y}, {x}) at the orientation clamp: {a!r} vs float32 restatement {b!r}"
        worst, bound = float(d.abs().max()), max(4 * float(d32.abs().max()), 1e-4 * amax)
        where = np.unravel_index(int(d.abs().argmax()), tuple(d.shape))
        assert worst <= bound, f"channel {ch}: pixel (y, x) = {where} off by {worst:.3g} (bound {bound:.3g}, max|ref| {amax:.3g})"
        if amax > 0:
            e, e32 = float(d.norm() / gr.norm()), float(d32.norm() / gr.norm())
            assert e <= max(4 * e32, 1e-5), f"channel {ch}: norm-relative error {e:.3g} (float32 restatement: {e32:.3g})"
    return g, g_ref, g_32, got


SIZES = [(1, 1), (1, 45), (45, 1), (5, 3), (10, 10), (11, 11), (12, 7), (31, 32), (32, 32), (33, 33), (64, 65)]


@pytest.mark.parametrize("W,H", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_loss_sizes_against_float64(cuda_device, W, H):
    """Images narrower than the window (every tap but the centre falls on the zero padding), one pixel wide, and one
    pixel past a loss tile, with the degenerate orientation pixels placed wherever they fit."""
    check_against_float64(cuda_device, make_case(W, H, seed=W * 100 + H))


def test_loss_degenerate_orientation_pixels(cuda_device):
    """Each degenerate pixel gets the gradient float64 autograd gives it (channels 5, 6 and 8 at that pixel)."""
    W, H = 33, 31
    ins = make_case(W, H, seed=5)
    # the placed pixels are what they claim to be, in the float32 the kernel computes in
    for k, (name, c5, c6, ga) in enumerate(degenerate_pixels()):
        y, x = divmod((7 * k + 3) % (W * H), W)
        a, b = F32(ins[0][5, y, x]), F32(ins[0][6, y, x])
        nrm = F32(np.sqrt(F32(a * a + b * b)))
        diry = F32(b / max(nrm, F32(1e-12)))
        if name.startswith("tie"):
            assert diry == 0 and F32(np.arccos(F32(0.0))) / F32(np.pi) == F32(0.5) and float(ins[3][0, y, x]) == ga
        if "clamp" in name:
            assert abs(diry) == (HI if name.startswith("on") else PAST), name
        if name.startswith("-0.0"):
            assert np.signbit(a) and a == 0
        assert float(ins[2][0, y, x]) > 0 and float(ins[4][0, y, x]) > 0, f"{name}: the orientation term is masked out"
    flips = clamp_flips(ins[0])
    zn = (ins[0][5] == 0) & (ins[0][6] == 0)
    g, g_ref, g_32, _ = check_against_float64(cuda_device, ins)
    for k, (name, *_rest) in enumerate(degenerate_pixels()):
        y, x = divmod((7 * k + 3) % (W * H), W)
        # on the clamp edge float32 lets the gradient through and float64 does not: the float32 restatement is the
        # reference there (and its gradient is not zero, so a kernel that clamps at the edge fails)
        on_edge = name.startswith("on")
        assert bool(flips[y, x]) == on_edge, f"{name}: float32 / float64 clamp decisions"
        for ch in (5, 6, 8):
            ref = g_32 if on_edge and ch != 8 else g_ref
            a, b = float(g[ch, y, x]), float(ref[ch, y, x])
            if zn[y, x]:
                scale = abs(b)
            else:                          # the channel's scale, without the 1e12 gradients of zero-norm pixels
                scale = max(abs(b), float((ref[ch] * ~zn).abs().max()))
            assert abs(a - b) <= (1e-4 if ref is g_32 else 1e-5) * scale, f"{name}: channel {ch} {a!r} vs {b!r}"
        if on_edge:
            assert float(g_32[6, y, x]) != 0.0
    # the tie pixels split the gradient: angle 0.5, gt 0 or 1 -> sign terms cancel, nothing flows into channel 6
    for k in (3, 4, 5):
        y, x = divmod((7 * k + 3) % (W * H), W)
        assert float(g_ref[6, y, x]) == 0.0 and float(g[6, y, x]) == 0.0


EDGE = {
    "gt_mask1_zero": dict(),
    "negative_confidence": dict(),
    "lambda_l1_zero": dict(lambdas=(0.0, 0.2, 0.1, 0.3)),
    "lambda_ssim_zero": dict(lambdas=(0.8, 0.0, 0.1, 0.3)),
    "lambda_mask_zero": dict(lambdas=(0.8, 0.2, 0.0, 0.3)),
    "lambda_orient_zero": dict(lambdas=(0.8, 0.2, 0.1, 0.0)),
}


@pytest.mark.parametrize("case", list(EDGE))
def test_loss_edge_inputs_against_float64(cuda_device, case):
    """An all-zero gt_mask[1] (SSIM of two zero images), a negative rendered confidence (Lorient is NaN, replaced by
    0: channels 5, 6 and 8 carry no gradient), and each lambda set to zero in turn."""
    W, H = 37, 35
    ins = make_case(W, H, seed=11)
    if case == "gt_mask1_zero":
        ins[2][1] = 0.0
    if case == "negative_confidence":
        ins[0][8, 4, 6] = -0.25
    g, g_ref, _, got = check_against_float64(cuda_device, ins, **EDGE[case])
    if case == "negative_confidence":
        assert got["Lorient"] == 0.0
        for ch in (5, 6, 8):
            assert float(g[ch].abs().max()) == 0.0, f"channel {ch} carries gradient though Lorient was replaced"
    if case == "gt_mask1_zero":
        assert abs(got["Lssim"]) <= 1e-6
        for ch in range(3):
            assert float(g[ch].abs().max()) == 0.0
    if case.startswith("lambda"):
        zero = EDGE[case]["lambdas"].index(0.0)
        chans = {0: (), 1: (), 2: (3, 4), 3: (5, 6, 8)}[zero]
        for ch in chans:
            assert float(g[ch].abs().max()) == 0.0, f"channel {ch} carries gradient of a term weighted 0"

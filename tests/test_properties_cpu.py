"""Property tests (hypothesis) of the host logic + oracle, CPU only: arbitrary (H, W, cut size, counts, power, gray portion)
-- the RNG record reproduces the reference's draw order and invariants, and (build container) the reference executed in
place agrees bit for bit with the oracle for every drawn configuration."""
import pytest
import torch
from hypothesis import given, settings
from hypothesis import strategies as st

from clip_diffusion_b200.rng_record import CUT_GRAY_PRE, CUT_OVERVIEW, draw_cutout_record
from oracle import cutouts as OC
from oracle import ref_stubs

configs = st.tuples(
    st.sampled_from([32, 48, 64]),          # cut size
    st.integers(0, 3), st.integers(0, 3),   # extra height / width in units of 32 (Config floors to multiples of 64)
    st.integers(0, 7), st.integers(0, 6),   # overview / inner cuts
    st.sampled_from([0.5, 1, 2, 5]), st.sampled_from([0.0, 0.3, 0.45, 0.7, 1.0]),
    st.integers(0, 2 ** 16),
)


@settings(max_examples=40, deadline=None)
@given(configs)
def test_record_invariants(cfg):
    cs, eh, ew, no, ni, power, gray, seed = cfg
    H, W = cs + 32 * eh, cs + 32 * ew
    g = torch.Generator().manual_seed(seed)
    rec = draw_cutout_record(H, W, cs, no, ni, power, gray, generator=g, noise="device")
    assert rec.num_cuts == no + ni
    longer, shorter = max(H, W), min(H, W)
    for n in range(no):  # overview: the zero-padded square of the longer side (cutouts.py:54-64)
        assert rec.flags[n] & CUT_OVERVIEW and rec.size[n] == longer
        assert (rec.y0[n], rec.x0[n]) == (-(longer - H) // 2, -(longer - W) // 2)
    if no > 4:
        assert len({rec.flags[n] for n in range(no)}) == 1  # identical copies (cutouts.py:77-79)
    for i in range(ni):
        n = no + i
        assert min(H, W, cs) <= rec.size[n] <= shorter
        assert 0 <= rec.x0[n] <= W - rec.size[n] and 0 <= rec.y0[n] <= H - rec.size[n]
        assert bool(rec.flags[n] & CUT_GRAY_PRE) == (i <= int(gray * ni))  # the reference's `<=` (cut 0 is always gray)
    assert -10.0 <= rec.angle <= 10.0 and abs(rec.tx) <= round(0.05 * cs) and abs(rec.ty) <= round(0.05 * cs)
    assert sorted(rec.perm) == [0, 1, 2, 3]
    assert 0.9 <= rec.brightness <= 1.1 and 0.9 <= rec.contrast <= 1.1 and 0.9 <= rec.saturation <= 1.1 and -0.1 <= rec.hue <= 0.1
    # same seed => same record (world-size-invariant crops); slices partition it
    rec2 = draw_cutout_record(H, W, cs, no, ni, power, gray, generator=torch.Generator().manual_seed(seed), noise="device")
    assert (rec.size, rec.x0, rec.y0, rec.flags, rec.angle, rec.perm) == (rec2.size, rec2.x0, rec2.y0, rec2.flags, rec2.angle, rec2.perm)


@pytest.mark.skipif(not ref_stubs.available(), reason="needs the original clip-diffusion source tree (set CLIPGUIDE_REFERENCE_ROOT)")
@settings(max_examples=15, deadline=None)
@given(configs)
def test_reference_in_place_equals_oracle_for_any_configuration(cfg):
    cs, eh, ew, no, ni, power, gray, seed = cfg
    if no + ni == 0:
        ni = 1
    H, W = cs + 32 * eh, cs + 32 * ew
    cut, _, _, _ = ref_stubs.install()
    x = torch.tanh(torch.randn(1, 3, H, W, generator=torch.Generator().manual_seed(seed))) * 1.1
    torch.manual_seed(seed)
    ref = cut.make_cutouts(x, cs, no, ni, power, gray)
    torch.manual_seed(seed)
    rec = draw_cutout_record(H, W, cs, no, ni, power, gray, noise="cpu")
    assert torch.equal(OC.make_cutouts(x, rec), ref)


@pytest.mark.parametrize("shape,groups", [((2, 16, 5, 7), 4), ((1, 32, 6, 6), 32), ((3, 24, 4, 9), 2)])
@pytest.mark.parametrize("silu", [False, True])
@pytest.mark.parametrize("with_ss", [False, True])
@pytest.mark.parametrize("with_bias", [False, True])
def test_unet_norm_folded_algebra_matches_autograd_of_the_definition(shape, groups, silu, with_ss, with_bias):
    """The formulas csrc/unet_norm.cu implements (oracle/unet_norm.folded_*: statistics of x + conv_bias from the per-channel sums
    of x, one per-channel affine, closed-form input gradient with the skip-path gradient added) against float64 autograd of the
    block arithmetic as guided-diffusion spells it (oracle/unet_norm.resblock_norm_reference)."""
    import numpy as np

    from oracle import unet_norm as U

    n, c, h, w = shape
    g = torch.Generator().manual_seed(n * 100 + c + (7 if silu else 0))
    x = (torch.randn(shape, generator=g, dtype=torch.float64) * 1.3 + torch.randn(1, c, 1, 1, generator=g, dtype=torch.float64)).requires_grad_()
    gamma = 1 + 0.3 * torch.randn(c, generator=g, dtype=torch.float64)
    beta = 0.2 * torch.randn(c, generator=g, dtype=torch.float64)
    ss = 0.4 * torch.randn(n, 2 * c, generator=g, dtype=torch.float64) if with_ss else None
    cb = 1.5 * torch.randn(c, generator=g, dtype=torch.float64) if with_bias else None
    dy = torch.randn(shape, generator=g, dtype=torch.float64)
    dres = torch.randn(shape, generator=g, dtype=torch.float64)
    y = U.resblock_norm_reference(x, gamma, beta, groups, 1e-5, ss, cb, silu)
    (dx,) = torch.autograd.grad((y * dy).sum() + (x * dres).sum(), x)  # x also feeds the block's skip path
    np_ = lambda t: None if t is None else t.detach().numpy()
    y2 = U.folded_forward(np_(x), np_(gamma), np_(beta), groups, 1e-5, np_(ss), np_(cb), silu)
    dx2 = U.folded_backward(np_(dy), np_(x), np_(gamma), np_(beta), groups, 1e-5, np_(ss), np_(cb), silu, np_(dres))
    assert np.abs(y2 - np_(y)).max() <= 1e-10 * max(1.0, np.abs(np_(y)).max())
    assert np.abs(dx2 - np_(dx)).max() <= 1e-9 * max(1.0, np.abs(np_(dx)).max())

"""GPU parity tests of csrc/ssim.cu through the fused_ssim-shaped host mirror (litegs_b200/ssim.py) against the CPU
oracle (fp64 restatement of fused_ssim/ssim.cu) and the committed golden vectors of the UNMODIFIED reference kernels.
Tolerance: 1e-4 of max(1, |ref|) per tensor (BASELINE.json north_star: fp32 within 1e-4) on well-conditioned inputs.  On
smooth images sigma = E[x^2] - mu^2 cancels and ANY fp32 evaluation (the reference's included: see the golden test in
test_oracle_ssim.py) is off by up to 1e-2 in dm_dmu1; there the bar is "no worse than 4x the error of the oracle's own
fp32 instantiation against its fp64 one", evaluated per tensor on the same input."""
import os

import numpy as np
import pytest
import torch

import oracle
from litegs_b200 import ssim

pytestmark = pytest.mark.gpu
C1, C2 = 0.01 ** 2, 0.03 ** 2
TOL = 1e-4


def serr(a, ref):
    ref = np.asarray(ref, np.float64)
    return float(np.abs(a.detach().cpu().numpy().astype(np.float64) - ref).max() / max(1.0, np.abs(ref).max()))


def images(shape, seed, smooth=False):
    rng = np.random.default_rng(seed)
    a = rng.random(shape, dtype=np.float32)
    b = rng.random(shape, dtype=np.float32)
    if smooth and shape[2] > 8 and shape[3] > 8:
        t = torch.nn.functional.avg_pool2d(torch.from_numpy(a), 7, 1, 3)
        a = t.numpy().copy()
        b = (a + 0.03 * (b - 0.5)).astype(np.float32)
        b[0, 0, 1:3, 2:6] = a[0, 0, 1:3, 2:6]
    return a, b


SHAPES = [(2, 3, 37, 53), (1, 1, 1, 1), (1, 2, 5, 7), (1, 3, 32, 64), (1, 3, 33, 65), (1, 1, 100, 200), (3, 1, 64, 129)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("l1", [0, 1])
@pytest.mark.parametrize("smooth", [False, True])
def test_forward_backward_match_oracle(cuda, shape, l1, smooth):
    a, b = images(shape, seed=sum(shape) + l1, smooth=smooth)
    up = np.random.default_rng(1).standard_normal(shape).astype(np.float32)
    w = 0.2
    ta, tb, tu = (torch.from_numpy(z).to(cuda) for z in (a, b, up))
    a64, b64, u64 = a.astype(np.float64), b.astype(np.float64), up.astype(np.float64)
    if l1:
        m, d0, d1, d2 = ssim.fusedl1ssim_loss(w, C1, C2, ta, tb, True)
        g = ssim.fusedl1ssim_loss_backward(w, C1, C2, ta, tb, tu, d0, d1, d2)
        om, o0, o1, o2 = oracle.fusedl1ssim_loss(w, C1, C2, a64, b64, True)
        og = oracle.fusedl1ssim_loss_backward(w, C1, C2, a64, b64, u64, o0, o1, o2)
    else:
        m, d0, d1, d2 = ssim.fusedssim(C1, C2, ta, tb, True)
        g = ssim.fusedssim_backward(C1, C2, ta, tb, tu, d0, d1, d2)
        om, o0, o1, o2 = oracle.fusedssim(C1, C2, a64, b64, True)
        og = oracle.fusedssim_backward(C1, C2, a64, b64, u64, o0, o1, o2)
    # conditioning of this input: what plain fp32 arithmetic (the oracle instantiated in float) loses against fp64
    if l1:
        fm, f0, f1, f2 = oracle.fusedl1ssim_loss(w, C1, C2, a, b, True)
        fg = oracle.fusedl1ssim_loss_backward(w, C1, C2, a, b, up, f0, f1, f2)
    else:
        fm, f0, f1, f2 = oracle.fusedssim(C1, C2, a, b, True)
        fg = oracle.fusedssim_backward(C1, C2, a, b, up, f0, f1, f2)
    for name, x, ref, f32 in (("map", m, om, fm), ("dm_dmu1", d0, o0, f0), ("dm_dsigma1_sq", d1, o1, f1), ("dm_dsigma12", d2, o2, f2),
                              ("grad", g, og, fg)):
        cond = float(np.abs(f32.astype(np.float64) - ref).max() / max(1.0, np.abs(ref).max()))
        bound = max(TOL, 4.0 * cond)
        if not smooth:
            assert bound == TOL, (name, cond)           # random images are well conditioned: the 1e-4 bar applies as is
        assert serr(x, ref) < bound, (name, serr(x, ref), cond)


def test_train_false_and_map_only(cuda):
    a, b = images((1, 3, 40, 70), 3)
    ta, tb = torch.from_numpy(a).to(cuda), torch.from_numpy(b).to(cuda)
    m, d0, d1, d2 = ssim.fusedssim(C1, C2, ta, tb, False)
    assert d0.numel() == 0 and d1.numel() == 0 and d2.numel() == 0
    assert serr(m, oracle.fusedssim(C1, C2, a.astype(np.float64), b.astype(np.float64), False)[0]) < TOL


@pytest.mark.parametrize("padding", ["same", "valid"])
def test_autograd_surface_matches_oracle(cuda, padding):
    """fused_ssim / fused_l1_ssim_loss (fused_ssim/__init__.py:44-90): scalar value and image gradient."""
    shape = (1, 3, 45, 83)
    a, b = images(shape, 9)
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    for l1 in (0, 1):
        ta = torch.from_numpy(a).to(cuda).requires_grad_(True)
        tb = torch.from_numpy(b).to(cuda)
        val = ssim.fused_l1_ssim_loss(ta, tb, 0.2, padding) if l1 else ssim.fused_ssim(ta, tb, padding)
        val.backward()
        if l1:
            om, o0, o1, o2 = oracle.fusedl1ssim_loss(0.2, C1, C2, a64, b64, True)
        else:
            om, o0, o1, o2 = oracle.fusedssim(C1, C2, a64, b64, True)
        up = np.zeros(shape)
        if padding == "valid":
            up[:, :, 5:-5, 5:-5] = 1.0 / om[:, :, 5:-5, 5:-5].size
            want = om[:, :, 5:-5, 5:-5].mean()
        else:
            up[:] = 1.0 / om.size
            want = om.mean()
        og = oracle.fusedl1ssim_loss_backward(0.2, C1, C2, a64, b64, up, o0, o1, o2) if l1 else \
            oracle.fusedssim_backward(C1, C2, a64, b64, up, o0, o1, o2)
        assert abs(float(val) - want) < 1e-5
        assert np.abs(ta.grad.cpu().numpy() - og).max() < TOL * max(np.abs(og).max(), 1e-12) + 1e-9


def test_fused_loss_and_grad_equals_the_autograd_path(cuda):
    """l1_ssim_loss_and_grad (no loss map, per-CTA partial sums, uniform upstream) == fused_l1_ssim_loss(...).backward()."""
    shape = (1, 3, 270, 480)
    a, b = images(shape, 11, smooth=True)
    ta = torch.from_numpy(a).to(cuda).requires_grad_(True)
    tb = torch.from_numpy(b).to(cuda)
    ref = ssim.fused_l1_ssim_loss(ta, tb, 0.2)
    ref.backward()
    loss, grad = ssim.l1_ssim_loss_and_grad(ta.detach(), tb, 0.2)
    assert abs(float(loss) - float(ref)) < 1e-6
    assert torch.allclose(grad, ta.grad, rtol=1e-5, atol=1e-10)
    loss2, grad2 = ssim.l1_ssim_loss_and_grad(ta.detach(), tb, 0.2, upstream=2.5)
    assert torch.allclose(grad2, 2.5 * grad, rtol=1e-4, atol=1e-9) and float(loss2) == float(loss)
    l3, g3 = ssim.l1_ssim_loss_and_grad(ta.detach(), tb, 0.2)
    assert float(l3) == float(loss) and torch.equal(g3, grad)            # deterministic


def test_full_hd_properties(cuda):
    """1080p x 3 channels (the size trainer.py:145 runs at): SSIM(x, x) = 1 and zero gradient of the SSIM term; the L1+SSIM
    loss of identical images is 0; symmetric in its arguments; matches the oracle on a seeded crop."""
    g = torch.Generator(device="cpu").manual_seed(5)
    x = torch.rand((1, 3, 1080, 1920), generator=g).to(cuda)
    y = torch.rand((1, 3, 1080, 1920), generator=g).to(cuda)
    m = ssim.fusedssim(C1, C2, x, x, False)[0]
    assert float((m - 1).abs().max()) < 1e-5
    loss, grad = ssim.l1_ssim_loss_and_grad(x, x, 0.2)
    assert abs(float(loss)) < 1e-6 and float(grad.abs().max()) < 1e-9
    mxy = ssim.fusedssim(C1, C2, x, y, False)[0]
    myx = ssim.fusedssim(C1, C2, y, x, False)[0]
    assert float((mxy - myx).abs().max()) < 1e-6
    # interior of a crop sees the same neighbourhood as in the full image
    cx, cy = x[:, :, 500:580, 900:1010].contiguous(), y[:, :, 500:580, 900:1010].contiguous()
    om = oracle.fusedssim(C1, C2, cx.cpu().numpy().astype(np.float64), cy.cpu().numpy().astype(np.float64), False)[0]
    assert np.abs(mxy[:, :, 505:575, 905:1005].cpu().numpy() - om[:, :, 5:-5, 5:-5]).max() < TOL


def test_errors(cuda):
    a = torch.zeros((1, 3, 8, 8), device=cuda)
    with pytest.raises(RuntimeError):
        ssim.fusedssim(C1, C2, a.cpu(), a.cpu(), True)
    with pytest.raises(RuntimeError):
        ssim.fusedssim(C1, C2, a, a[:, :2], True)
    with pytest.raises(RuntimeError):
        ssim.fusedssim(C1, C2, a.double(), a.double(), True)


GOLD = os.path.join(os.path.dirname(__file__), "golden", "ssim_small.npz")


@pytest.mark.skipif(not os.path.exists(GOLD), reason="tests/golden/ssim_small.npz not generated yet")
@pytest.mark.parametrize("name", ["rand", "smooth"])
def test_matches_reference_cuda_golden(cuda, name):
    """rand: 1e-4.  smooth: both sides are fp32 evaluations of a cancelling expression (the reference with --use_fast_math);
    they agree to the conditioning of the input, which test_oracle_ssim.py quantifies against fp64."""
    z = np.load(GOLD)
    ta, tb, tu = (torch.from_numpy(z[k]).to(cuda) for k in (f"{name}_img1", f"{name}_img2", "upstream"))
    c1, c2, w = float(z["C1"]), float(z["C2"]), float(z["ssim_weight"])
    m, d0, d1, d2 = ssim.fusedssim(c1, c2, ta, tb, True)
    g = ssim.fusedssim_backward(c1, c2, ta, tb, tu, d0, d1, d2)
    tol = {"rand": {}, "smooth": {"map": 1e-3, "dm_dmu1": 5e-2, "dm_dsigma1_sq": 1e-3, "dm_dsigma12": 1e-3, "grad": 3e-3}}[name]
    for k, v in zip(("map", "dm_dmu1", "dm_dsigma1_sq", "dm_dsigma12", "grad"), (m, d0, d1, d2, g)):
        assert serr(v, z[f"{name}_ssim_{k}"]) < tol.get(k, TOL), (k, serr(v, z[f"{name}_ssim_{k}"]))
    m, d0, d1, d2 = ssim.fusedl1ssim_loss(w, c1, c2, ta, tb, True)
    g = ssim.fusedl1ssim_loss_backward(w, c1, c2, ta, tb, tu, d0, d1, d2)
    for k, v in zip(("map", "dm_dmu1", "dm_dsigma1_sq", "dm_dsigma12", "grad"), (m, d0, d1, d2, g)):
        assert serr(v, z[f"{name}_l1_{k}"]) < tol.get(k, TOL), (k, serr(v, z[f"{name}_l1_{k}"]))


def test_against_reference_kernels_live(cuda):
    """The unmodified reference extension on the same 1080p inputs: its outputs at a fixed seeded sample of elements, and each
    tensor's largest magnitude (tests/golden/ssim_1080p_sample.npz, written by tests/golden/make_golden_ssim.py)."""
    from tests.golden.make_golden_ssim import inputs_1080p
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "ssim_1080p_sample.npz"))
    x, y, up = inputs_1080p(cuda)
    assert np.allclose([float(t.double().sum()) for t in (x, y, up)], z["input_sums"], rtol=1e-12, atol=1e-6)
    idx = torch.from_numpy(z["index"]).to(cuda)
    m, d0, d1, d2 = ssim.fusedl1ssim_loss(0.2, C1, C2, x, y, True)
    gg = ssim.fusedl1ssim_loss_backward(0.2, C1, C2, x, y, up, d0, d1, d2)
    for name, u in (("map", m), ("dm_dmu1", d0), ("dm_dsigma1_sq", d1), ("dm_dsigma12", d2), ("grad", gg)):
        v = z[name].astype(np.float64)
        err = float(np.abs(u.reshape(-1)[idx].cpu().numpy().astype(np.float64) - v).max() / max(1.0, float(z[f"{name}_absmax"])))
        assert err < TOL, (name, err)
        assert abs(float(u.abs().max()) - float(z[f"{name}_absmax"])) < TOL * max(1.0, float(z[f"{name}_absmax"])), name


def test_reference_own_consistency_check(cuda):
    """The reference's own test (fused_ssim/tests/test_fused_l1_ssim_loss.py:10-45) on our implementation: the fused
    L1+SSIM loss equals (1 - w) * L1 + w * (1 - fused_ssim) assembled from the separate SSIM op, value and gradient
    (torch.isclose defaults, as there), on a 1080p random pair."""
    w = 0.2
    g = torch.Generator(device="cpu").manual_seed(0)
    gt = torch.rand((3, 1080, 1920), generator=g).to(cuda)
    im = torch.rand((3, 1080, 1920), generator=g).to(cuda)
    a = im.clone().requires_grad_(True)
    before = (1.0 - w) * torch.abs(a - gt).mean() + w * (1.0 - ssim.fused_ssim(a.unsqueeze(0), gt.unsqueeze(0)))
    before.backward()
    b = im.clone().requires_grad_(True)
    after = ssim.fused_l1_ssim_loss(b.unsqueeze(0), gt.unsqueeze(0), w)
    after.backward()
    assert torch.isclose(before, after)
    assert torch.isclose(a.grad, b.grad).all()

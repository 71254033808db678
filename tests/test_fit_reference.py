"""The fit path's arithmetic against an independent reference (oracle/fit_ref.py: complex-step
Jacobian, math.fsum blocks), on the CPU: the reference checked against mpmath, then the C oracle's
Jacobian and blocks checked against the reference at the rotation angles where a closed-form
Rodrigues derivative loses accuracy.  tests/test_gpu_fit_reference.py holds the kernels to the
same reference."""
import math

import numpy as np
import pytest

from oracle import fit_ref as fr
from oracle import oracle_c as oc

U = fr.U


def _shared(intr):
    return intr[1], intr[2], intr[3], intr[4]


def _colerr(J, ref):
    """normwise error of every Jacobian column over the rows given, relative to the column's largest entry"""
    J, ref = J.reshape(-1, fr.NPAR), ref.reshape(-1, fr.NPAR)
    return np.abs(J - ref).max(0) / np.abs(ref).max(0)


def test_complex_step_jacobian_matches_mpmath():
    """The reference's Jacobian is itself checked: central differences in mpmath at 60 digits on a
    non-planar board, with distortion, aspect and checker size, at rotation angles from 0 to pi."""
    mpmath = pytest.importorskip("mpmath")
    thetas = (0.0, 1e-12, 1e-8, 1e-4, 1.0, math.pi - 1e-6)
    intr, views, obj, img = fr.case(4, len(thetas), k=-0.3, aspect=1.1, checker_size=0.025, planar=False,
                                    thetas=thetas, seed=11)
    J = fr.jacobian(views, _shared(intr), 0.025, 1.1, obj)
    with mpmath.workdps(60):
        for v in range(len(thetas)):
            p = list(views[v]) + list(_shared(intr))
            Jm = np.stack([fr.mp_jacobian(mpmath.mp, p, 0.025, 1.1, obj[c]) for c in range(len(obj))])
            err = _colerr(J[v], Jm)
            assert err.max() <= 32 * U, (thetas[v], err)
            assert np.all(np.abs(Jm).max((0, 1)) > 0)       # every column is exercised


@pytest.mark.parametrize("theta", fr.THETAS)
def test_oracle_jacobian_vs_reference(theta):
    """The oracle's Jacobian (the formula the kernel shares) within 32 u of every column's largest
    entry.  Forming (I - R) e_i as e_i - R e_i loses the (1 - cos theta) terms and the division by
    theta^2 magnifies the loss: about 2.3e-8 at theta = 1e-8."""
    intr, views, obj, img = fr.case(280, 3, k=-0.12, aspect=1.1, checker_size=0.025, thetas=(theta,), seed=3)
    _, _, Jo = oc.reproj_jtj(intr, 1.1, [(v[:3], v[3:]) for v in views], obj, img, want_jac=True)
    J = fr.jacobian(views, _shared(intr), 0.025, 1.1, obj)
    for v in range(len(views)):
        err = _colerr(Jo[v], J[v])
        assert err.max() <= 32 * U, (theta, err)


@pytest.mark.parametrize("nc,nv,k,aspect,cs,planar", [
    (280, 48, -0.12, 1.0, 1.0, True),
    (33, 17, 0.4, 1.1, 0.025, True),
    (64, 16, -0.3, 1.1, 1.0, False),
])
def test_oracle_blocks_vs_reference(nc, nv, k, aspect, cs, planar):
    """The oracle's per-view and shared blocks within the entry-wise bound of fit_ref.tolerance;
    the same data less one corner must fail that bound, so it is tight enough to see one term."""
    intr, views, obj, img = fr.case(nc, nv, k=k, aspect=aspect, checker_size=cs, planar=planar, seed=nc + nv)
    ref = fr.blocks(views, _shared(intr), cs, aspect, obj, img)
    pv, sh, _ = oc.reproj_jtj(intr, aspect, [(v[:3], v[3:]) for v in views], obj, img)
    assert np.all(np.abs(pv - ref["per_view"]) <= fr.tolerance(ref, "per_view"))
    assert np.all(np.abs(sh - ref["shared"]) <= fr.tolerance(ref, "shared"))
    # negative control: a corner short
    pv1, sh1, _ = oc.reproj_jtj(intr, aspect, [(v[:3], v[3:]) for v in views], obj[1:], img[:, 1:])
    assert np.all(np.any(np.abs(pv1 - ref["per_view"]) > fr.tolerance(ref, "per_view"), axis=1))
    assert np.any(np.abs(sh1 - ref["shared"]) > fr.tolerance(ref, "shared"))


def test_reference_residual_is_the_oracle_model():
    """fit_ref's residual is the oracle's world -> pixel chain (the same camera model)."""
    intr, views, obj, img = fr.case(31, 5, k=-0.12, aspect=1.25, checker_size=0.025, planar=False, seed=2)
    r = fr.residual(views, _shared(intr), 0.025, 1.25, obj, img)
    for v in range(len(views)):
        row, col = oc.world2img(oc.chain(intr, views[v, :3], views[v, 3:]), obj)
        assert np.allclose(r[v, :, 0], row - img[v, :, 0], rtol=0, atol=1e-10)
        assert np.allclose(r[v, :, 1], col - img[v, :, 1], rtol=0, atol=1e-10)

"""CPU checks of the remaining callers of SURVEY.md 8f (pyramids, resize family, lens model): the oracle's restatement
against the vectors recorded from the reference (tests/golden/wider.npz), the product wrappers' host logic with the
core functions swapped for the oracle, the signatures and the error behaviour."""
import inspect
from importlib import import_module

import pytest
import torch

import kornia_b200 as K
from conftest import golden
from helpers import family_grads, reference_package, rel_l2, run_family_case
from oracle import kornia_restated as R

WID = golden("wider")
FWD = [n for n in WID.names() if not WID.meta[n]["op"].endswith("_grad")]
GRAD = [n for n in WID.names() if WID.meta[n]["op"].endswith("_grad")]


def product_module(op):
    base = op[:-5] if op.endswith("_grad") else op
    return K.geometry.calibration if hasattr(K.geometry.calibration, base) else K.geometry.transform


def assert_outputs(got, outs, **tol):
    if isinstance(got, (list, tuple)):
        assert len(got) == len(outs), (len(got), len(outs))
        for i, g in enumerate(got):
            torch.testing.assert_close(g, outs[f"out{i}"], **tol)
    else:
        torch.testing.assert_close(got, outs["out"], **tol)


@pytest.mark.parametrize("name", FWD)
def test_oracle_forward_matches_reference(name):
    op, kw, ins, outs = WID.case(name)
    assert_outputs(run_family_case(R, op, kw, ins), outs, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", GRAD)
def test_oracle_grads_match_reference(name):
    op, kw, ins, outs = WID.case(name)
    got = family_grads(R, op, kw, ins, outs)
    for key, want in outs.items():
        if key != "cot":
            assert rel_l2(got[key], want) < 2e-6, (key, rel_l2(got[key], want))


@pytest.fixture
def core_on_cpu(monkeypatch):
    """Route the wrappers' calls into the core functions to the oracle (CPU); nothing else is touched."""
    pyramid, affwarp = (import_module("kornia_b200.geometry.transform." + m) for m in ("pyramid", "affwarp"))
    undistort = import_module("kornia_b200.geometry.calibration.undistort")
    monkeypatch.setattr(pyramid, "filter2d", R.filter2d)
    monkeypatch.setattr(affwarp, "gaussian_blur2d", R.gaussian_blur2d)
    monkeypatch.setattr(undistort, "remap", R.remap)


@pytest.mark.parametrize("name", FWD)
def test_wrapper_forward_on_cpu(core_on_cpu, name):
    op, kw, ins, outs = WID.case(name)
    assert_outputs(run_family_case(product_module(op), op, kw, ins), outs, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", GRAD)
def test_wrapper_grads_on_cpu(core_on_cpu, name):
    op, kw, ins, outs = WID.case(name)
    got = family_grads(product_module(op), op, kw, ins, outs)
    for key, want in outs.items():
        if key != "cot":
            assert rel_l2(got[key], want) < 2e-6, (key, rel_l2(got[key], want))


def test_reference_literals():
    # pyramid.py:435-438 (docstring example, pinned by the reference's doctest run)
    x = torch.arange(16, dtype=torch.float32).reshape(1, 1, 4, 4)
    torch.testing.assert_close(R.pyrdown(x, align_corners=True), torch.tensor([[[[3.75, 5.25], [9.75, 11.25]]]]))
    # tests/geometry/transform/test_pyramid.py: shapes of pyrdown / pyrup / build_pyramid
    assert R.pyrdown(torch.rand(1, 2, 5, 5)).shape == (1, 2, 2, 2)
    assert R.pyrup(torch.rand(1, 2, 3, 3)).shape == (1, 2, 6, 6)
    assert [tuple(t.shape[-2:]) for t in R.build_pyramid(torch.rand(1, 1, 20, 12), 3)] == [(20, 12), (10, 6), (5, 3)]
    # affwarp.py docstrings: resize / rescale shapes
    assert R.resize(torch.rand(1, 3, 4, 4), (6, 8)).shape == (1, 3, 6, 8)
    assert R.rescale(torch.rand(1, 3, 4, 4), (2, 3)).shape == (1, 3, 8, 12)
    # zero coefficients: the lens model is the identity on pixel coordinates
    pts = torch.rand(1, 5, 2) * 10
    cam = torch.tensor([[[8.0, 0, 5.0], [0, 9.0, 4.0], [0, 0, 1.0]]])
    torch.testing.assert_close(R.distort_points(pts, cam, torch.zeros(1, 4)), pts)


def test_signatures_match_reference():
    # pyramid.py:409-411,460,505-507,572-574; affwarp.py:588-595,679-686,718-724; undistort.py:138; distort.py:25,78-80
    KT, KC = K.geometry.transform, K.geometry.calibration
    want = {
        KT.pyrdown: "(input, border_type='reflect', align_corners=False, factor=2.0)",
        KT.pyrup: "(input, border_type='reflect', align_corners=False)",
        KT.build_pyramid: "(input, max_level, border_type='reflect', align_corners=False)",
        KT.build_laplacian_pyramid: "(input, max_level, border_type='reflect', align_corners=False)",
        KT.resize: "(input, size, interpolation='bilinear', align_corners=None, side='short', antialias=False)",
        KT.resize_to_be_divisible: "(input, divisible_factor, interpolation='bilinear', align_corners=None, side='short', antialias=False)",
        KT.rescale: "(input, factor, interpolation='bilinear', align_corners=None, antialias=False)",
        KC.undistort_image: "(image, K, dist)",
        KC.distort_points: "(points, K, dist, new_K=None)",
        KC.tilt_projection: "(taux, tauy, return_inverse=False)",
    }
    for fn, sig in want.items():
        params = inspect.signature(fn).parameters.values()
        got = "(" + ", ".join(p.name if p.default is inspect._empty else f"{p.name}={p.default!r}" for p in params) + ")"
        assert got == sig, fn.__name__


def test_validation_runs_before_device_work():
    KT, KC = K.geometry.transform, K.geometry.calibration
    img = torch.rand(1, 2, 6, 7)
    with pytest.raises(Exception, match="[Ss]hape"):
        KT.pyrdown(torch.rand(2, 6, 7))
    with pytest.raises(Exception, match="[Ss]hape"):
        KT.pyrup(torch.rand(6, 7))
    with pytest.raises(Exception, match="Invalid max_level"):
        KT.build_pyramid(img, 2.5)
    with pytest.raises(TypeError, match="not a torch.Tensor"):
        KT.resize([[1.0]], (2, 2))
    with pytest.raises(ValueError, match="at least two dimensions"):
        KT.resize(torch.rand(5), (2, 2))
    with pytest.raises(ValueError, match="side can be one of"):
        KT.resize(img, 4, side="diagonal")
    cam, d = torch.eye(3)[None], torch.zeros(1, 4)
    with pytest.raises(ValueError, match="Image shape is invalid"):
        KC.undistort_image(torch.rand(6, 7), cam, d)
    with pytest.raises(ValueError, match="K matrix shape is invalid"):
        KC.undistort_image(img, torch.eye(4)[None], d)
    with pytest.raises(ValueError, match="Invalid number of distortion coefficients"):
        KC.undistort_image(img, cam, torch.zeros(1, 6))
    with pytest.raises(ValueError, match="Input should be float"):
        KC.undistort_image((img * 255).to(torch.uint8), cam, d)
    with pytest.raises(ValueError, match="batch dimensions should match"):
        KC.undistort_image(torch.rand(2, 2, 6, 7), cam, d)
    with pytest.raises(ValueError, match="do not match"):
        KC.tilt_projection(torch.zeros(2), torch.zeros(3))
    # the product has no CPU path: a CPU image that passes validation is refused by the core function, not computed
    with pytest.raises(RuntimeError, match="CUDA-only"):
        KT.pyrdown(img)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        KC.undistort_image(img, cam, d)


def test_tilt_projection_matches_oracle():
    KC = K.geometry.calibration
    tx, ty = torch.tensor([0.02, -0.3]), torch.tensor([-0.015, 0.2])
    torch.testing.assert_close(KC.tilt_projection(tx, ty), R.tilt_matrix(tx, ty), rtol=0, atol=0)
    assert KC.tilt_projection(torch.tensor(0.1), torch.tensor(0.2)).shape == (3, 3)


def test_install_reaches_the_new_callers(monkeypatch):
    """install() rebinds filter2d / gaussian_blur2d / remap inside the reference's pyramid, affwarp and undistort modules,
    so the reference's own pyrdown / resize(antialias) / undistort_image run on the CUDA kernels unmodified (on the
    reference's import graph recorded in tests/golden/install.json)."""
    kornia, _ = reference_package(monkeypatch)
    pyr = import_module("kornia.geometry.transform.pyramid")
    aff = import_module("kornia.geometry.transform.affwarp")
    und = import_module("kornia.geometry.calibration.undistort")
    K.install(kornia)
    try:
        assert pyr.filter2d is K.filter2d and aff.gaussian_blur2d is K.gaussian_blur2d and und.remap is K.remap
    finally:
        K.uninstall()
    assert pyr.filter2d is not K.filter2d


def test_lens_packing_and_kernel_op_order():
    """The fused undistort kernel (csrc/remap_tiled.cuh:lens_distort) evaluates distort_points from 16 packed numbers.
    This mirrors its operation tree -- same indices into the packed row, same association, one torch op per device
    intrinsic -- and must reproduce the oracle's distort_points bit for bit on the exact pixel grid (CPU fp32): it
    pins the packing order of pack_lens and documents the op order the kernel transcribes."""
    from kornia_b200.geometry.calibration.undistort import pack_lens

    def lens_distort(L, px, py):
        fx, fy, cx, cy = L[0], L[1], L[2], L[3]
        x, y = (px - cx) / fx, (py - cy) / fy
        r2 = x * x + y * y
        r4 = r2 * r2
        r6 = r4 * r2
        num = ((1.0 + L[4] * r2) + L[5] * r4) + L[8] * r6
        den = ((1.0 + L[9] * r2) + L[10] * r4) + L[11] * r6
        rad = num / den
        xy1 = ((2.0 * L[6]) * x) * y
        xy2 = ((2.0 * L[7]) * x) * y
        rx = r2 + (2.0 * x) * x
        ry = r2 + (2.0 * y) * y
        xd = (((x * rad + xy1) + L[7] * rx) + L[12] * r2) + L[13] * r4
        yd = (((y * rad + L[6] * ry) + xy2) + L[14] * r2) + L[15] * r4
        return fx * xd + cx, fy * yd + cy

    H, W = 45, 64
    ys, xs = torch.meshgrid(torch.linspace(0, H - 1, H), torch.linspace(0, W - 1, W), indexing="ij")
    pts = torch.stack([xs, ys], -1).reshape(-1, 2)
    cam = torch.tensor([[[50.0, 0.0, 31.0], [0.0, 47.0, 22.5], [0.0, 0.0, 1.0]], [[61.0, 0.0, 30.0], [0.0, 60.0, 20.0], [0.0, 0.0, 1.0]]])
    g = torch.Generator().manual_seed(5)
    for n in (4, 5, 8, 12, 14):
        scale = torch.tensor([0.25, 0.08, 0.003, 0.003, 0.02, 0.05, 0.02, 0.004, 0.003, 0.001, 0.002, 0.0015, 0.0, 0.0])[:n]
        dist = (torch.rand(2, n, generator=g) - 0.5) * 2 * scale
        lens = pack_lens(cam, dist, pts)
        assert lens.shape == (2, 16)
        want = R.distort_points(pts, cam, dist)
        for b in range(2):
            mx, my = lens_distort(lens[b], pts[:, 0], pts[:, 1])
            assert torch.equal(mx, want[b, :, 0]) and torch.equal(my, want[b, :, 1]), n
    assert pack_lens(cam, torch.tensor([[0.0] * 12 + [0.01, 0.0]] * 2), pts) is None          # tilt: not covered
    assert pack_lens(cam[0], torch.zeros(4), pts).shape == (1, 16)                             # unbatched K and dist
    assert pack_lens(cam[:1], torch.zeros(3, 5), pts).shape == (3, 16)                         # broadcast intrinsics

"""CPU checks of the callers either side of the hot path (SURVEY.md 8f rows 1-3): the oracle's
restatement against the vectors recorded from the reference (tests/golden/family.npz), the host
logic of the product wrappers (signatures, tap generators, matrix builders: pure torch, runs on
CPU) and ``install()``."""
import inspect
import sys

import pytest
import torch

import kornia_b200 as K
from conftest import golden
from helpers import family_grads, reference_package, rel_l2, run_family_case
from oracle import kornia_restated as R

FAM = golden("family")
FWD = [n for n in FAM.names() if not FAM.meta[n]["op"].endswith("_grad")]
GRAD = [n for n in FAM.names() if FAM.meta[n]["op"].endswith("_grad")]


@pytest.mark.parametrize("name", FWD)
def test_oracle_forward_matches_reference(name):
    op, kw, ins, outs = FAM.case(name)
    got = run_family_case(R, op, kw, ins)
    torch.testing.assert_close(got, outs["out"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", GRAD)
def test_oracle_grads_match_reference(name):
    op, kw, ins, outs = FAM.case(name)
    got = family_grads(R, op, kw, ins, outs)
    for key, want in outs.items():
        if key != "cot":
            assert rel_l2(got[key], want) < 2e-6, (key, rel_l2(got[key], want))


# ---------------------------------------------------------------------------------- host logic of the product
MATRIX_OPS = [n for n in FAM.names() if FAM.meta[n]["op"].startswith(("get_rotation_matrix2d", "get_perspective_transform"))]


@pytest.mark.parametrize("name", MATRIX_OPS)
def test_matrix_builders_match_reference_on_cpu(name):
    """The (B,2,3)/(B,3,3) builders are torch ops: they run (and must agree with the reference) on CPU."""
    op, kw, ins, outs = FAM.case(name)
    if op.endswith("_grad"):
        got = family_grads(K.geometry.transform, op, kw, ins, outs)
        for key, want in outs.items():
            if key != "cot":
                assert rel_l2(got[key], want) < 2e-6, key
    else:
        torch.testing.assert_close(run_family_case(K.geometry.transform, op, kw, ins), outs["out"], rtol=1e-6, atol=1e-6)


def test_tap_generators_match_reference_literals():
    KF = K.filters
    # tests/filters/test_laplacian.py:45-57
    assert KF.get_laplacian_kernel1d(5).tolist() == [1.0, 1.0, -4.0, 1.0, 1.0]
    assert KF.get_laplacian_kernel2d(3).tolist() == [[1.0, 1.0, 1.0], [1.0, -8.0, 1.0], [1.0, 1.0, 1.0]]
    assert KF.get_laplacian_kernel2d((3, 5)).shape == (3, 5) and float(KF.get_laplacian_kernel2d((3, 5)).sum()) == 0.0
    assert KF.get_box_kernel1d(4).tolist() == [[0.25] * 4] and KF.get_box_kernel2d((2, 4)).shape == (1, 2, 4)
    sob = KF.get_sobel_kernel2d()
    assert sob[0].tolist() == [[-1.0, 0.0, 1.0], [-2.0, 0.0, 2.0], [-1.0, 0.0, 1.0]] and torch.equal(sob[1], sob[0].t())
    assert KF.get_spatial_gradient_kernel2d("sobel", 2).shape == (3, 5, 5)
    assert KF.get_spatial_gradient_kernel2d("diff", 2).shape == (3, 3, 3)
    for mode in ("sobel", "diff"):
        for order in (1, 2):
            torch.testing.assert_close(KF.get_spatial_gradient_kernel2d(mode, order), R.derivative_taps(mode, order, None, torch.float32),
                                       rtol=0, atol=0)
    with pytest.raises(Exception, match="Mode should be"):
        KF.get_spatial_gradient_kernel2d("prewitt", 1)
    with pytest.raises(Exception, match="Order should be"):
        KF.get_spatial_gradient_kernel2d("sobel", 3)
    with pytest.raises(Exception, match="Kernel size must be an odd"):
        KF.get_laplacian_kernel2d(4)


def test_family_signatures_match_reference():
    # filters/blur.py:29-31, laplacian.py:27-29, unsharp.py:27-32, sobel.py:32,134; geometry/transform/affwarp.py:136-142,
    # 257-264,401-407,455-462,522-528; crop2d.py:41-48,125-131,209-217,299-306; imgwarp.py:465,529
    KF, KT = K.filters, K.geometry.transform
    want = {
        KF.box_blur: "(input, kernel_size, border_type='reflect', separable=False)",
        KF.laplacian: "(input, kernel_size, border_type='reflect', normalized=True)",
        KF.unsharp_mask: "(input, kernel_size, sigma, border_type='reflect')",
        KF.spatial_gradient: "(input, mode='sobel', order=1, normalized=True)",
        KF.sobel: "(input, normalized=True, eps=1e-06)",
        KT.affine: "(tensor, matrix, mode='bilinear', padding_mode='zeros', align_corners=True)",
        KT.rotate: "(tensor, angle, center=None, mode='bilinear', padding_mode='zeros', align_corners=True)",
        KT.translate: "(tensor, translation, mode='bilinear', padding_mode='zeros', align_corners=True)",
        KT.scale: "(tensor, scale_factor, center=None, mode='bilinear', padding_mode='zeros', align_corners=True)",
        KT.shear: "(tensor, shear, mode='bilinear', padding_mode='zeros', align_corners=False)",
        KT.crop_and_resize: "(input_tensor, boxes, size, mode='bilinear', padding_mode='zeros', align_corners=True)",
        KT.center_crop: "(input_tensor, size, mode='bilinear', padding_mode='zeros', align_corners=True)",
        KT.crop_by_boxes: "(input_tensor, src_box, dst_box, mode='bilinear', padding_mode='zeros', align_corners=True, validate_boxes=True)",
        KT.crop_by_transform_mat: "(input_tensor, transform, out_size, mode='bilinear', padding_mode='zeros', align_corners=True)",
        KT.get_perspective_transform: "(points_src, points_dst)",
        KT.get_rotation_matrix2d: "(center, angle, scale)",
    }
    for fn, sig in want.items():
        params = inspect.signature(fn).parameters.values()
        got = "(" + ", ".join(p.name if p.default is inspect._empty else f"{p.name}={p.default!r}" for p in params) + ")"
        assert got == sig, fn.__name__


def test_family_validation_runs_before_device_work():
    KF, KT = K.filters, K.geometry.transform
    img = torch.rand(1, 2, 5, 6)
    with pytest.raises(TypeError):
        KT.rotate(img, 30.0)
    with pytest.raises(TypeError):
        KT.rotate(0.0, torch.tensor([30.0]))
    with pytest.raises(ValueError, match="Invalid tensor shape"):
        KT.rotate(torch.rand(5, 6), torch.tensor([30.0]))
    with pytest.raises(TypeError):
        KT.translate(img, (1.0, 2.0))
    with pytest.raises(TypeError):
        KT.crop_and_resize(img, [[0, 0]], (2, 2))
    with pytest.raises(ValueError, match="length 2"):
        KT.crop_and_resize(img, torch.zeros(1, 4, 2), (2,))
    with pytest.raises(AssertionError, match="shape \\(B, C, H, W\\)"):
        KT.center_crop(img[0], (2, 2))
    with pytest.raises(ValueError, match="Bx2"):
        KT.get_rotation_matrix2d(torch.zeros(2), torch.zeros(1), torch.ones(1, 2))
    with pytest.raises(K.core.TypeCheckError):
        KF.spatial_gradient([1.0])
    with pytest.raises(K.core.ShapeError):
        KF.sobel(torch.rand(2, 5, 6))
    with pytest.raises(K.core.TypeCheckError):
        KF.box_blur(None, 3)
    # no CPU path: a valid CPU call fails loudly instead of computing somewhere else
    for call in (lambda: KF.sobel(img), lambda: KF.spatial_gradient(img), lambda: KF.box_blur(img, 3), lambda: KF.laplacian(img, 3),
                 lambda: KF.unsharp_mask(img, (3, 3), (1.0, 1.0)), lambda: KT.rotate(img, torch.tensor([10.0])),
                 lambda: KT.center_crop(img, (2, 2))):
        with pytest.raises(RuntimeError, match="CUDA-only"):
            call()


def test_module_forms():
    KF = K.filters
    assert repr(KF.BoxBlur((3, 3))) == "BoxBlur(kernel_size=(3, 3), border_type=reflect, separable=False)"
    assert repr(KF.Laplacian(5)) == "Laplacian(kernel_size=5, normalized=True, border_type=reflect)"
    assert repr(KF.SpatialGradient("diff", 2)) == "SpatialGradient(order=2, normalized=True, mode=diff)"
    assert repr(KF.Sobel()) == "Sobel(normalized=True)"
    assert KF.UnsharpMask((3, 3), (1.0, 1.0)).border_type == "reflect"


def test_install_rebinds_every_importer_of_the_reference(monkeypatch):
    """On the reference's import graph (recorded in tests/golden/install.json): every module that holds one of the
    rebound functions gets the product's, and ``uninstall()`` puts the reference's back."""
    kornia, bindings = reference_package(monkeypatch)
    aug_persp = sys.modules["kornia.augmentation._2d.geometric.perspective"]
    aug_blur = sys.modules["kornia.augmentation._2d.intensity.gaussian_blur"]
    affwarp = sys.modules["kornia.geometry.transform.affwarp"]
    crop2d = sys.modules["kornia.geometry.transform.crop2d"]
    unsharp = sys.modules["kornia.filters.unsharp"]
    ours = {"warp_perspective": K.warp_perspective, "warp_affine": K.warp_affine, "remap": K.remap, "filter2d": K.filter2d,
            "filter2d_separable": K.filter2d_separable, "gaussian_blur2d": K.gaussian_blur2d,
            "get_perspective_transform": K.geometry.transform.get_perspective_transform, "spatial_gradient": K.filters.spatial_gradient,
            "sobel": K.filters.sobel, "ssim": K.metrics.ssim}
    before = {(m, name): getattr(sys.modules[m], name) for m, name in bindings}

    orig = kornia.geometry.transform.imgwarp.warp_perspective
    K.install(kornia)
    try:
        assert kornia.geometry.transform.warp_perspective is K.warp_perspective
        assert kornia.geometry.warp_affine is K.warp_affine
        assert kornia.filters.gaussian_blur2d is K.gaussian_blur2d
        assert aug_persp.warp_perspective is K.warp_perspective      # RandomPerspective.apply_transform
        assert affwarp.warp_affine is K.warp_affine                  # affine / rotate / translate / scale / shear
        assert crop2d.warp_perspective is K.warp_perspective and crop2d.warp_affine is K.warp_affine
        assert unsharp.gaussian_blur2d is K.gaussian_blur2d
        assert aug_blur.gaussian_blur2d is K.gaussian_blur2d                 # captured by RandomGaussianBlur.__init__
        assert aug_persp.get_perspective_transform is K.geometry.transform.get_perspective_transform
        assert kornia.filters.sobel is K.filters.sobel and kornia.filters.spatial_gradient is K.filters.spatial_gradient
        assert kornia.metrics.ssim is K.metrics.ssim and kornia.losses.ssim.metrics.ssim is K.metrics.ssim
        missed = [(m, name) for m, name in bindings if getattr(sys.modules[m], name) is not ours[name]]
        assert not missed, missed
        K.install(kornia)  # idempotent: the originals are remembered once
    finally:
        K.uninstall()
    assert kornia.geometry.transform.warp_perspective is orig and aug_persp.warp_perspective is orig
    assert kornia.metrics.ssim is not K.metrics.ssim and callable(kornia.filters.sobel)
    assert all(getattr(sys.modules[m], name) is before[m, name] for m, name in bindings)


def test_fused_unsharp_request_host_logic():
    """The envelope test + tap preparation in front of kb200_sepfilter_lerp_forward is pure host logic."""
    from kornia_b200.filters.unsharp import _fused_request

    x = torch.rand(2, 3, 20, 24)
    kx, ky, code = _fused_request(x, (5, 5), (1.5, 1.5), "reflect")
    assert kx.shape == (1, 5) and ky.shape == (1, 5) and code == K._lib.REFLECT
    composed = torch.lerp(R.filter2d_separable(x, kx, ky, "reflect"), x, 2.0)
    torch.testing.assert_close(composed, R.unsharp_mask(x, (5, 5), (1.5, 1.5)), rtol=0, atol=0)
    kx, ky, code = _fused_request(x, 5, torch.tensor([[1.0, 2.0], [0.5, 0.7]]), "replicate")
    assert kx.shape == (2, 5) and code == K._lib.REPLICATE
    torch.testing.assert_close(kx, R.gaussian_taps(5, torch.tensor([[2.0], [0.7]])), rtol=0, atol=0)   # x taps from sigma[:, 1]
    for bad in ((x, (3, 5), (1.0, 1.0), "reflect"), (x, (5, 5), (1.0, 1.0), "circular"), (x, (5, 5), (-1.0, 1.0), "reflect"),
                (x.double(), (5, 5), (1.0, 1.0), "reflect"), (x, 13, (1.0, 1.0), "reflect"), (x, 4, (1.0, 1.0), "reflect"),
                (x[0], 5, (1.0, 1.0), "reflect"), (x, 5, torch.ones(3, 2), "reflect"), (torch.rand(1, 1, 2, 9), 5, (1.0, 1.0), "reflect")):
        assert _fused_request(*bad) is None

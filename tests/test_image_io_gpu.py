"""GPU input path (mfr_b200.image_io: nvJPEG decode + cv2.resize restated as CUDA kernels) against OpenCV, the library
the reference's loaders call (SuperGlue/models/utils.py:263-285, lib/datasets/utils.py:58-75): uint8 fixed-point
resize bit-exact, float resize within fp32 round-off, JPEG luma within the +-2 levels two IDCT implementations differ by,
and the two offline matcher plugins end to end on image files."""
import cv2
import numpy as np
import pytest
import torch

from helpers import GOLDEN, synth

pytestmark = pytest.mark.gpu


def _img(seed, h, w, c=1):
    rng = np.random.default_rng(seed)
    im = synth.make_texture(rng, h, w)                       # band-limited RGB uint8
    im = (im.astype(np.int32) + rng.integers(-20, 20, im.shape)).clip(0, 255).astype(np.uint8)
    return im[:, :, 0].copy() if c == 1 else im


@pytest.mark.parametrize("src,dst", [((480, 640), (540, 720)), ((1920, 1440), (540, 720)), ((300, 401), (640, 480)), ((720, 540), (540, 720))])
def test_resize_u8_fixed_point(src, dst):
    from mfr_b200 import image_io
    for c in (1, 3):
        im = _img(sum(src) + c, src[1], src[0], c)
        ref = cv2.resize(im, dst)                            # uint8, INTER_LINEAR
        got = image_io.resize_linear(torch.from_numpy(im).cuda(), dst, image_io.MODE_U8_FIXED).cpu().numpy()
        assert np.array_equal(got, np.round(got)) and got.min() >= 0 and got.max() <= 255        # integer-valued uint8 range
        d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
        # the kernel restates OpenCV's generic fixed-point path; the wheel's dispatched (IPP / SIMD) code rounds a few
        # pixels per thousand the other way (measured here on the CPU: 0.05 - 0.08 % of the pixels off by one level)
        assert d.max() <= 1 and (d > 0).mean() < 3e-3


@pytest.mark.parametrize("src,dst", [((480, 640), (540, 720)), ((1296, 968), (640, 480)), ((333, 250), (540, 720))])
def test_resize_float_matches_cv2(src, dst):
    from mfr_b200 import image_io
    im = _img(sum(src), src[1], src[0])
    ref = cv2.resize(im.astype("float32"), dst) / 255.0       # read_image, resize_float=True
    got = image_io.resize_linear(torch.from_numpy(im).cuda(), dst, image_io.MODE_U8_AS_F32, 1.0 / 255.0)
    # OpenCV's generic float path is reproduced to fp32 round-off (scripts note in DESIGN.md: exact with cv2.setUseOptimized(False));
    # the IPP code the opencv-python wheel dispatches to differs from that generic path by up to 3e-3 gray levels itself
    np.testing.assert_allclose(got.cpu().numpy(), ref.astype(np.float32), rtol=0, atol=5e-3 / 255)
    cv2.setUseOptimized(False)
    try:
        ref_generic = cv2.resize(im.astype("float32"), dst) / 255.0
    finally:
        cv2.setUseOptimized(True)
    np.testing.assert_allclose(got.cpu().numpy(), ref_generic.astype(np.float32), rtol=0, atol=2e-5 / 255 + 1e-7)
    got2 = image_io.resize_linear(torch.from_numpy(im.astype(np.float32)).cuda(), dst, image_io.MODE_F32, 1.0 / 255.0)
    assert torch.equal(got, got2)


def test_jpeg_decode_and_plugins(tmp_path):
    from mfr_b200 import image_io, loftr, spsg
    rgb = _img(5, 720, 540, 3)
    p = str(tmp_path / "a.jpg")
    cv2.imwrite(p, rgb[:, :, ::-1], [cv2.IMWRITE_JPEG_QUALITY, 92])
    gray = image_io.decode_jpeg(p).cpu().numpy().astype(np.int32)
    ref = cv2.imread(p, cv2.IMREAD_GRAYSCALE).astype(np.int32)
    assert gray.shape == ref.shape and np.abs(gray - ref).max() <= 3 and np.abs(gray - ref).mean() < 0.5
    col = image_io.decode_jpeg(p, rgb=True).cpu().numpy().astype(np.int32)
    refc = cv2.imread(p, cv2.IMREAD_COLOR)[:, :, ::-1].astype(np.int32)
    # 4:2:0 chroma: nvJPEG replicates the subsampled chroma planes, libjpeg-turbo interpolates them ("fancy upsampling"); on this
    # synthetic image (independent noise per colour channel = maximal chroma detail) that is ~5 levels per channel on average.
    # The luma the matchers use is decoded at full resolution and unaffected: BT.601 gray of both decodes agrees within 2 levels.
    dc = np.abs(col - refc)
    assert dc.mean() < 8.0
    yg = (col * np.array([0.299, 0.587, 0.114])).sum(-1); yr = (refc * np.array([0.299, 0.587, 0.114])).sum(-1)
    assert np.abs(yg - yr).mean() < 1.0 and np.percentile(np.abs(yg - yr), 99) <= 3.0
    im = image_io.read_image(p, (270, 360), True)
    refr = cv2.resize(cv2.imread(p, cv2.IMREAD_GRAYSCALE).astype("float32"), (270, 360)) / 255.0
    assert im.shape == (360, 270) and np.abs(im.cpu().numpy() - refr).max() < 3.5 / 255
    ci = image_io.read_color_image(p, (270, 360))
    assert ci.shape == (3, 360, 270) and 0.0 <= float(ci.min()) and float(ci.max()) <= 1.0
    assert image_io.read_image(str(tmp_path / "missing.jpg"), (270, 360)) is None
    # offline plugins on files: match((path0, path1)) -> [N, 4]  (matchers.py:24-59, 93-120)
    q = str(tmp_path / "b.png")
    cv2.imwrite(q, np.roll(rgb, (6, 10), (0, 1))[:, :, ::-1])                      # PNG: host decode, GPU resize
    m = loftr.LoFTR_matcher((272, 360), weights=loftr.functional_state_dict(), cfg={"thr": 0.2})
    pts = m.match((p, q))
    assert pts.shape[1] == 4 and len(pts) > 50
    d = pts[:, 2:] - pts[:, :2]                              # image b is image a shifted by (10, 6) * 0.5 (resize 540 -> 272)
    assert np.abs(np.median(d, 0) - np.array([5.0, 3.0])).max() < 0.6
    sp, sg = spsg.synthetic_state_dicts(0)
    s = spsg.SuperGlue_matcher((272, 360), state_dicts=(sp, sg))
    out = s.match((p, q))
    assert out.shape[1] == 4


def test_readme_pair_through_the_gpu_loader():
    """Camera JPEGs (the SuperGlue README's 1296x968 ScanNet sample pair, stored re-encoded at quality 75) read by the GPU
    loader at the 640x480 of the README's known-answer test = OpenCV's decode and float resize up to the JPEG decoders'
    +-2 gray levels."""
    from mfr_b200 import image_io
    for n in ("scene0711_00_frame-001680.jpg", "scene0711_00_frame-001995.jpg"):
        path = GOLDEN + "/" + n
        got = image_io.read_image(path, (640, 480), True).cpu().numpy()
        ref = cv2.resize(cv2.imread(path, cv2.IMREAD_GRAYSCALE).astype("float32"), (640, 480)) / 255.0
        assert np.abs(got - ref).max() < 3.5 / 255 and np.abs(got - ref).mean() < 0.5 / 255

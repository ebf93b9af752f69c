"""CPU tier: the host side of the denoiser guide buffers — io.aov_images arithmetic and the PFM writer."""
import numpy as np
import pytest

from ray_tracer_archive_b200 import io


def _sums():
    # 2 x 3 image, 4 samples.  Pixel (0,0): every sample hit; (0,1): one of four; (1,2): none (background albedo only)
    s = np.zeros((2, 3, 8), dtype=np.float32)
    s[0, 0] = [2.0, 1.0, 4.0, 4.0, 0.0, 4.0, 0.0, 40.0]
    s[0, 1] = [3.0, 3.0, 3.0, 1.0, 1.0, 0.0, 0.0, 7.5]
    s[1, 2] = [0.4, 0.8, 1.2, 0.0, 0.0, 0.0, 0.0, 0.0]
    return s


def test_aov_images_divides_by_spp_and_coverage():
    img = io.aov_images(_sums(), 4)
    assert set(img) == {"albedo", "normal", "depth", "coverage"}
    assert img["albedo"].shape == (2, 3, 3) and img["normal"].shape == (2, 3, 3)
    assert img["depth"].shape == (2, 3) and img["coverage"].shape == (2, 3)
    assert all(v.dtype == np.float32 for v in img.values())
    np.testing.assert_allclose(img["albedo"][0, 0], [0.5, 0.25, 1.0])
    np.testing.assert_allclose(img["albedo"][1, 2], [0.1, 0.2, 0.3], rtol=1e-6)
    np.testing.assert_allclose(img["coverage"], [[1.0, 0.25, 0.0], [0.0, 0.0, 0.0]])
    np.testing.assert_allclose(img["normal"][0, 0], [0.0, 1.0, 0.0])
    np.testing.assert_allclose(img["normal"][0, 1], [0.25, 0.0, 0.0])
    # depth: mean over the samples that hit; 0 (not NaN) where nothing was hit
    np.testing.assert_allclose(img["depth"], [[10.0, 7.5, 0.0], [0.0, 0.0, 0.0]])
    assert np.isfinite(img["depth"]).all()


def test_aov_images_rejects_bad_input():
    with pytest.raises(ValueError):
        io.aov_images(np.zeros((2, 3, 4), np.float32), 1)
    with pytest.raises(ValueError):
        io.aov_images(_sums(), 0)


def _read_pfm(path):
    with open(path, "rb") as f:
        kind = f.readline().strip()
        w, h = map(int, f.readline().split())
        scale = float(f.readline())
        data = f.read()
    ch = 3 if kind == b"PF" else 1
    a = np.frombuffer(data, dtype="<f4" if scale < 0 else ">f4").reshape((h, w, ch) if ch == 3 else (h, w))
    return kind, w, h, scale, data, a[::-1]


@pytest.mark.parametrize("channels", [1, 3])
def test_save_pfm_header_row_order_and_round_trip(tmp_path, channels):
    rng = np.random.default_rng(channels)
    shape = (5, 7, 3) if channels == 3 else (5, 7)
    img = rng.standard_normal(shape).astype(np.float32)
    path = str(tmp_path / "x.pfm")
    io.save_pfm(path, img)
    kind, w, h, scale, data, back = _read_pfm(path)
    assert kind == (b"PF" if channels == 3 else b"Pf")
    assert (w, h) == (7, 5)
    assert scale == -1.0  # little-endian
    assert len(data) == img.nbytes
    # the file's first row is the image's BOTTOM row
    assert data[: 7 * channels * 4] == np.ascontiguousarray(img[-1], dtype="<f4").tobytes()
    assert back.tobytes() == img.tobytes()  # byte-exact round trip


def test_save_pfm_accepts_single_channel_last_axis_and_rejects_others(tmp_path):
    img = np.arange(12, dtype=np.float32).reshape(3, 4, 1)
    io.save_pfm(str(tmp_path / "a.pfm"), img)
    kind, w, h, _, _, back = _read_pfm(str(tmp_path / "a.pfm"))
    assert kind == b"Pf" and (w, h) == (4, 3) and np.array_equal(back, img[..., 0])
    with pytest.raises(ValueError):
        io.save_pfm(str(tmp_path / "b.pfm"), np.zeros((3, 4, 2), np.float32))

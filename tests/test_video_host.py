"""Host-side checks of the JPEG and Motion-JPEG output of a rendered camera path: the numpy reference encoder
(tests/jpeg_reference.py) against PIL, the header and capacity of the C library against the reference, the AVI
container parsed as RIFF (and read by OpenCV where it is installed), the assembly of per-rank part files, the path's
``seconds`` and the input errors."""
import io
import json
import struct

import numpy as np
import pytest
import torch

from soccernerfs_b200.cameras.camera_paths import get_path_from_json, get_seconds_from_json
from soccernerfs_b200.engine import path_renderer as pr
from tests import jpeg_reference as jr

QUALITIES = (1, 10, 50, 75, 95, 100)


def _image(kind, h, w, seed=0):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "constant":
        return np.full((h, w, 3), (200, 17, 90), dtype=np.uint8)
    if kind == "gradient":
        return np.stack([x * 255 // max(w - 1, 1), y * 255 // max(h - 1, 1), (x + y) * 255 // max(h + w - 2, 1)],
                        -1).astype(np.uint8)
    if kind == "saturated":
        return (np.stack([(x // 3) % 2, (y // 5) % 2, ((x + y) // 7) % 2], -1) * 255).astype(np.uint8)
    if kind == "checker":
        return np.repeat((((x + y) % 2) * 255).astype(np.uint8)[..., None], 3, -1)
    raise ValueError(kind)


def _pil(data):
    from PIL import Image

    im = Image.open(io.BytesIO(data))
    im.load()
    return im


@pytest.mark.parametrize("kind", ["noise", "constant", "gradient", "saturated", "checker"])
def test_reference_files_decode_and_round_trip(kind):
    for h, w in ((1, 1), (7, 9), (16, 16), (17, 33), (40, 72)):
        img = _image(kind, h, w)
        for q in (1, 50, 95, 100):
            data = jr.encode_image(img, q)
            im = _pil(data)
            assert im.size == (w, h) and im.mode == "RGB"
            dec = jr.decode(data)
            coefs, _ = jr.forward(img, q)
            assert np.array_equal(dec["coefs"], coefs), (kind, h, w, q)
            assert jr.encode(dec["coefs"], h, w, q) == data
            assert dec["restart"] == jr.RESTART_MCUS


def test_reference_stuffs_and_restarts():
    data = jr.encode_image(_image("noise", 48, 80), 100)  # 15 MCUs: 4 segments, RST0..RST2
    scan = data[len(jr.header(48, 80, 100)):-2]
    markers = [scan[i + 1] for i in range(len(scan) - 1) if scan[i] == 0xFF and scan[i + 1] != 0x00]
    assert markers == [0xD0, 0xD1, 0xD2]
    assert scan.count(b"\xff\x00") > 0


def test_quantisation_tables_match_pil():
    from PIL import Image

    img = _image("gradient", 32, 48)
    for q in QUALITIES:
        ours = _pil(jr.encode_image(img, q)).quantization
        buf = io.BytesIO()
        Image.fromarray(img).save(buf, "JPEG", quality=q, subsampling=2)
        theirs = _pil(buf.getvalue()).quantization
        for t in range(2):
            assert list(ours[t]) == list(jr.quant_tables(q)[t]) == list(theirs[t]), (q, t)


def test_huffman_tables_match_pil_defaults():
    from PIL import Image

    buf = io.BytesIO()
    Image.fromarray(_image("gradient", 16, 16)).save(buf, "JPEG", quality=75, subsampling=2)
    data = buf.getvalue()
    theirs, pos, tables = data[data.index(b"\xff\xc4"):], 0, {}
    while theirs[pos:pos + 2] == b"\xff\xc4":  # PIL (libjpeg) writes one DHT segment per table
        n = struct.unpack(">H", theirs[pos + 2:pos + 4])[0]
        body = theirs[pos + 4:pos + 2 + n]
        tables[body[0]] = body[1:]
        pos += 2 + n
    assert sorted(tables) == [0x00, 0x01, 0x10, 0x11]
    for (cls, tid), (bits, vals) in jr.HUFF.items():
        assert tables[cls << 4 | tid] == bytes(bits) + bytes(vals)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge

    ge.build()
    from soccernerfs_b200 import _lib

    return _lib.load()


def test_library_header_and_capacity(lib):
    from ctypes import c_void_p

    from soccernerfs_b200 import ops

    for h, w, q in ((1, 1, 1), (1080, 5760, 95), (65535, 8, 100), (17, 33, 50)):
        buf = torch.zeros(ops.JPEG_HEADER_BYTES, dtype=torch.uint8)
        assert lib.kp_jpeg_header(h, w, q, c_void_p(buf.data_ptr())) == 0
        assert bytes(buf.numpy()) == jr.header(h, w, q)
        segments = -(-(-(-h // 16) * -(-w // 16)) // jr.RESTART_MCUS)
        bound = 2 * -(-jr.RESTART_MCUS * 6 * (22 + 63 * 26) // 8) + 2
        assert ops.jpeg_capacity(h, w) == ops.JPEG_HEADER_BYTES + segments * bound + 2
    buf = torch.zeros(ops.JPEG_HEADER_BYTES, dtype=torch.uint8)
    for h, w, q in ((0, 5, 50), (5, 65536, 50), (5, 5, 0), (5, 5, 101)):
        assert lib.kp_jpeg_header(h, w, q, c_void_p(buf.data_ptr())) != 0
        assert b"jpeg_header" in lib.kp_last_error()


def test_capacity_holds_the_worst_reference_file():
    """Noise at quality 100 is about the largest file there is; it stays far inside the capacity."""
    from soccernerfs_b200 import ops

    for h, w in ((16, 16), (40, 72)):
        data = jr.encode_image(_image("noise", h, w), 100)
        assert len(data) < ops.jpeg_capacity(h, w) / 2


def test_encode_jpeg_input_errors():
    from soccernerfs_b200 import ops

    img = torch.zeros((4, 4, 3), dtype=torch.uint8)
    for q in (0, 101, 95.0, True):
        with pytest.raises(ValueError, match="quality"):
            ops.encode_jpeg(img, q)
    for shape in ((4, 4), (4, 4, 4), (1, 4, 4, 3)):
        with pytest.raises(ValueError, match="expected"):
            ops.encode_jpeg(torch.zeros(shape, dtype=torch.uint8))
    for shape in ((0, 4, 3), (1, 65536, 3)):
        with pytest.raises(ValueError, match="65535"):
            ops.encode_jpeg(torch.zeros(shape, dtype=torch.uint8))
    with pytest.raises(TypeError, match="uint8"):
        ops.encode_jpeg(img.float())
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.encode_jpeg(img)


# ---- AVI ----
def _chunks(data, start, end):
    """[(fourcc, offset of the payload, size)] of the RIFF chunks in data[start:end]; checks the even padding."""
    out, pos = [], start
    while pos < end:
        fourcc, size = data[pos:pos + 4], struct.unpack("<I", data[pos + 4:pos + 8])[0]
        out.append((fourcc, pos + 8, size))
        pos += 8 + size + (size & 1)
    assert pos == end
    return out


def _parse_avi(path):
    data = open(path, "rb").read()
    assert data[:4] == b"RIFF" and data[8:12] == b"AVI "
    assert struct.unpack("<I", data[4:8])[0] == len(data) - 8
    top = _chunks(data, 12, len(data))
    assert [c[0] for c in top] == [b"LIST", b"LIST", b"idx1"]
    (_, hdrl, hdrl_n), (_, movi, movi_n), (_, idx, idx_n) = top
    assert data[hdrl:hdrl + 4] == b"hdrl" and data[movi:movi + 4] == b"movi"
    hdr = _chunks(data, hdrl + 4, hdrl + hdrl_n)
    assert [c[0] for c in hdr] == [b"avih", b"LIST"] and hdr[0][2] == 56
    avih = struct.unpack("<14I", data[hdr[0][1]:hdr[0][1] + 56])
    strl = _chunks(data, hdr[1][1] + 4, hdr[1][1] + hdr[1][2])
    assert data[hdr[1][1]:hdr[1][1] + 4] == b"strl" and [c[0] for c in strl] == [b"strh", b"strf"]
    strh = data[strl[0][1]:strl[0][1] + strl[0][2]]
    assert strh[:8] == b"vidsMJPG" and len(strh) == 56
    scale, rate, _, length = struct.unpack("<IIII", strh[20:36])
    strf = data[strl[1][1]:strl[1][1] + strl[1][2]]
    assert len(strf) == 40 and strf[16:20] == b"MJPG"
    frames = _chunks(data, movi + 4, movi + movi_n)
    assert all(c[0] == b"00dc" for c in frames)
    assert avih[4] == length == len(frames) and idx_n == 16 * len(frames)
    for k, (_, off, size) in enumerate(frames):
        fourcc, flags, rel, n = struct.unpack("<4sIII", data[idx + 16 * k:idx + 16 * (k + 1)])
        assert fourcc == b"00dc" and flags == 0x10 and n == size
        assert data[movi + rel:movi + rel + 4] == b"00dc" and movi + rel + 8 == off  # the index lands on the chunk
    return {"fps": rate / scale, "width": avih[8], "height": avih[9], "frames": [data[o:o + n] for _, o, n in frames]}


def _write_parts(output_path, frames, world):
    for r in range(world):
        with open(pr.part_path(output_path, r), "wb") as f:
            for data in frames[r::world]:
                f.write(struct.pack("<I", len(data)) + data)


def _frames(n, h=24, w=40):
    out = [jr.encode_image(_image("gradient" if i % 2 else "noise", h, w, seed=i), 50 + i) for i in range(n)]
    assert any(len(d) % 2 for d in out) and any(len(d) % 2 == 0 for d in out)  # odd sizes get a pad byte
    return out


def test_avi_container(tmp_path):
    frames = _frames(7)
    path = tmp_path / "video.avi"
    _write_parts(path, frames, 1)
    pr.assemble_video(path, 1, 7 / 2.5)
    avi = _parse_avi(path)
    assert avi["frames"] == frames and avi["fps"] == pytest.approx(2.8, abs=1e-9)
    assert (avi["width"], avi["height"]) == (40, 24)
    assert not (tmp_path / "video.avi.part0").exists()
    try:
        import cv2
    except ImportError:
        return
    cap = cv2.VideoCapture(str(path), cv2.CAP_OPENCV_MJPEG)
    try:
        assert cap.isOpened()
        assert int(cap.get(cv2.CAP_PROP_FRAME_COUNT)) == 7
        assert cap.get(cv2.CAP_PROP_FPS) == pytest.approx(2.8, rel=1e-6)
        ok, first = cap.read()
        assert ok and first.shape == (24, 40, 3)
    finally:
        cap.release()


def test_assembled_parts_equal_one_part(tmp_path):
    frames = _frames(5)
    one, two, three = tmp_path / "one.avi", tmp_path / "two.avi", tmp_path / "three.avi"
    _write_parts(one, frames, 1)
    _write_parts(two, frames, 2)
    _write_parts(three, frames, 3)
    pr.assemble_video(one, 1, 24.0)
    pr.assemble_video(two, 2, 24.0)
    pr.assemble_video(three, 3, 24.0)
    assert one.read_bytes() == two.read_bytes() == three.read_bytes()
    assert sorted(p.name for p in tmp_path.iterdir()) == ["one.avi", "three.avi", "two.avi"]  # the parts are gone


def test_assemble_errors(tmp_path, monkeypatch):
    frames = _frames(4)
    path = tmp_path / "v.avi"
    _write_parts(path, frames, 1)
    step = [8 + len(d) + (len(d) & 1) for d in frames]
    monkeypatch.setattr(pr, "AVI_MAX_MOVI_BYTES", 4 + sum(step[:2]) + 1)
    with pytest.raises(ValueError, match="2 frames fit"):
        pr.assemble_video(path, 1, 30.0)
    assert not path.exists() and (tmp_path / "v.avi.part0").exists()  # nothing written, the part kept
    monkeypatch.setattr(pr, "AVI_MAX_MOVI_BYTES", 4 + sum(step))
    pr.assemble_video(path, 1, 30.0)  # exactly at the limit
    assert len(_parse_avi(path)["frames"]) == 4
    _write_parts(path, frames, 2)
    with open(pr.part_path(path, 1), "ab") as f:  # one frame too many in part 1
        f.write(struct.pack("<I", len(frames[0])) + frames[0])
    with pytest.raises(ValueError, match="interleave"):
        pr.assemble_video(path, 2, 30.0)
    for fps in (0.0, -1.0, float("inf")):
        with pytest.raises(ValueError, match="fps"):
            pr.assemble_video(path, 2, fps)


def test_frame_rates_are_exact_fractions(tmp_path):
    frames = _frames(3)
    for fps in (24.0, 30000 / 1001, 3 / 7.0, 120.0):
        path = tmp_path / "r.avi"
        _write_parts(path, frames, 1)
        pr.assemble_video(path, 1, fps)
        assert _parse_avi(path)["fps"] == pytest.approx(fps, rel=1e-9)


# ---- the path's length and the render errors ----
def _path(n=2, h=24, w=40, **extra):
    cams = [{"camera_to_world": [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 2, 0, 0, 0, 1], "fov": 50.0, "render_time": k / 2}
            for k in range(n)]
    return {"render_height": h, "render_width": w, "camera_path": cams, **extra}


def test_seconds_from_json():
    assert get_seconds_from_json(_path(seconds=4)) == 4.0
    assert get_seconds_from_json(json.loads(json.dumps(_path(seconds=2.5)))) == 2.5
    with pytest.raises(ValueError, match="seconds"):
        get_seconds_from_json(_path())
    for bad in (0, -1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="seconds"):
            get_seconds_from_json(_path(seconds=bad))
    cams, crop = pr.load_camera_path(_path(seconds=3))  # load_camera_path keeps its return value
    assert len(cams) == 2 and crop is None


def _stub_model():
    import types

    return types.SimpleNamespace(config=types.SimpleNamespace(num_proposal_iterations=2),
                                 field=types.SimpleNamespace(has_time_planes=True))


def test_render_output_errors(tmp_path):
    cams = get_path_from_json(_path())
    out = tmp_path / "frames"
    for fmt in ("PNG", "jpg", "video", None):
        with pytest.raises(ValueError, match="image_format"):
            pr.render_camera_path(_stub_model(), cams, out, image_format=fmt)
    for q in (0, 101, 9.5, True):
        with pytest.raises(ValueError, match="jpeg_quality"):
            pr.render_camera_path(_stub_model(), cams, out, image_format="jpeg", jpeg_quality=q)
        with pytest.raises(ValueError, match="jpeg_quality"):
            pr.render_camera_path_video(_stub_model(), cams, tmp_path / "v.avi", 2.0, jpeg_quality=q)
    for s in (0.0, -2.0, float("nan")):
        with pytest.raises(ValueError, match="seconds"):
            pr.render_camera_path_video(_stub_model(), cams, tmp_path / "v.avi", s)
    # the existing input checks apply to every output
    with pytest.raises(ValueError, match="available outputs"):
        pr.render_camera_path(_stub_model(), cams, out, rendered_output_names=("normals",), image_format="jpeg")
    with pytest.raises(ValueError, match="available outputs"):
        pr.render_camera_path_video(_stub_model(), cams, tmp_path / "v.avi", 2.0, rendered_output_names=("normals",))
    assert list(tmp_path.iterdir()) == []  # nothing was written

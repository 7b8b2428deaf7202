"""CPU: dynslam_b200/csrc/hostio.c — the on-disk formats either side of the path (SURVEY 8(f) rank 4) — against
(1) the reference's own ReadFilePFM (src/pfmLib), ReadMask (PrecomputedSegmentationProvider.cpp) and ITMMesh::WriteOBJ, compiled
    from the reference tree into oracle/_ref/libioref.so (oracle/build_ref.sh, oracle/ref_io_driver.cpp): byte for byte, against
    their outputs stored in tests/golden/reference_pins.json (tests/refpins.py); and
(2) known answers for the OpenCV XML depth dump and the max-depth clamp (OpenCV itself is not available to produce a pin)."""
import ctypes as C
import os

import numpy as np
import pytest

from dynslam_b200 import abi, formats
from tests import hostlib as H
from tests.refpins import pin

IOREF_SO = os.path.join(H.ROOT, "oracle", "_ref", "libioref.so")


def ioref():
    L = C.CDLL(IOREF_SO)
    P, vp = C.POINTER, C.c_void_p
    L.ref_read_pfm.argtypes = [C.c_char_p, P(C.c_int), P(C.c_int), P(C.c_int), vp, C.c_size_t]
    L.ref_read_mask.argtypes = [C.c_char_p, C.c_int, C.c_int, vp]
    L.ref_write_obj.argtypes = [C.c_char_p, vp, C.c_uint, C.c_long]
    return L


def write_pfm(path, a, little=True, crlf=False):
    h, w = a.shape[:2]
    with open(path, "wb") as f:
        f.write(b"Pf" if a.ndim == 2 else b"PF")
        f.write(b"\n%d %d\n%s" % (w, h, b"-1.0" if little else b"1.0"))
        f.write(b"\r\n" if crlf else b"\n")
        f.write(np.ascontiguousarray(a[::-1]).astype("<f4" if little else ">f4").tobytes())


@pytest.mark.parametrize("shape,little,crlf", [((37, 53), True, False), ((16, 9), False, False), ((12, 20, 3), True, True), ((5, 7, 3), False, False)])
def test_pfm_equals_reference_reader(tmp_path, shape, little, crlf):
    rng = np.random.default_rng(3)
    a = rng.normal(0, 30, shape).astype(np.float32)
    p = str(tmp_path / "d.pfm")
    write_pfm(p, a, little, crlf)
    got = formats.read_pfm(p)
    assert got.shape == a.shape and np.array_equal(got, a)                 # row 0 at the top, byte order undone

    def ref_read():
        w, h, b = C.c_int(), C.c_int(), C.c_int()
        ref = np.zeros(a.size, np.float32)
        rc = ioref().ref_read_pfm(p.encode(), C.byref(w), C.byref(h), C.byref(b), ref.ctypes.data, ref.size)
        return [rc, [h.value, w.value], ref]
    pin(f"hostio/read_pfm/{'x'.join(map(str, shape))}-{'le' if little else 'be'}{'-crlf' if crlf else ''}", [0, list(a.shape[:2]), got], ref_read)


def test_pfm_errors(tmp_path):
    with pytest.raises(RuntimeError):
        formats.read_pfm(str(tmp_path / "missing.pfm"))
    p = tmp_path / "bad.pfm"
    p.write_bytes(b"P6\n2 2\n-1.0\n" + b"\0" * 16)
    with pytest.raises(RuntimeError):
        formats.read_pfm(str(p))


def test_mask_txt_equals_reference_reader(tmp_path):
    rng = np.random.default_rng(5)
    m = (rng.uniform(size=(23, 31)) < 0.4).astype(np.float64)
    p = str(tmp_path / "m.mask.txt")
    np.savetxt(p, m)                                                        # numpy's default "%.18e" text dump, as the segmentation tool writes it
    got = formats.read_mask_txt(p, 31, 23)
    assert np.array_equal(got, m.astype(np.uint8))

    def ref_read(w, h):
        ref = np.zeros((23, 31), np.uint8)
        return [ioref().ref_read_mask(p.encode(), w, h, ref.ctypes.data), ref]
    pin("hostio/read_mask/float_dump", [0, got], lambda: ref_read(31, 23))
    # integer dumps and values other than 0 / 1 are truncated to a byte the same way
    np.savetxt(p, (m * 2.7), fmt="%.3f")
    got = formats.read_mask_txt(p, 31, 23)
    assert got.max() == 2
    pin("hostio/read_mask/fixed_dump", [0, got], lambda: ref_read(31, 23))
    # wrong size: both refuse
    with pytest.raises(RuntimeError):
        formats.read_mask_txt(p, 30, 23)
    pin("hostio/read_mask/too_narrow", -3, lambda: ref_read(30, 23)[0])
    with pytest.raises(RuntimeError):
        formats.read_mask_txt(p, 31, 22)
    pin("hostio/read_mask/too_short", -3, lambda: ref_read(31, 22)[0])


def test_obj_equals_reference_writer(tmp_path):
    rng = np.random.default_rng(9)
    n = 257
    t = np.zeros(n, abi.TRIANGLE_DTYPE)
    for k in ("p0", "p1", "p2"):
        t[k] = rng.uniform(-40, 40, (n, 3)).astype(np.float32)
    for k in ("c0", "c1", "c2"):
        t[k] = rng.uniform(0, 1, (n, 3)).astype(np.float32)
    ours, ref = str(tmp_path / "ours.obj"), str(tmp_path / "ref.obj")
    formats.write_obj(ours, t, n, 512)

    def ref_write():
        rc = ioref().ref_write_obj(ref.encode(), t.ctypes.data, n, 16)        # 16 blocks -> noMaxTriangles 512
        return [rc, open(ref, "rb").read()]
    pin("hostio/write_obj", [0, open(ours, "rb").read()], ref_write)
    # more triangles than the mesh can hold: the reference throws, we raise with its text
    with pytest.raises(RuntimeError, match="Too many triangles"):
        formats.write_obj(ours, t, n, 100)
    pin("hostio/write_obj/too_many_triangles", -3, lambda: ioref().ref_write_obj(ref.encode(), t.ctypes.data, 600, 16))


def test_depth_xml_and_clamp_known_answers(tmp_path):
    d = np.array([[0, 1500, 30000], [-3, 12, 20001]], np.int16)
    p = tmp_path / "000001.xml"
    p.write_text('<?xml version="1.0"?>\n<opencv_storage>\n<depth-frame type_id="opencv-matrix">\n  <rows>2</rows>\n  <cols>3</cols>\n  <dt>s</dt>\n'
                 '  <data>\n    0 1500 30000 -3\n    12 20001</data></depth-frame>\n</opencv_storage>\n')
    got = formats.read_depth_xml(str(p))
    assert got.dtype == np.int16 and np.array_equal(got, d)
    formats.clamp_max_depth(got, 20.0)                                       # max depth 20 m: 20001 mm and 30000 mm are dropped
    assert np.array_equal(got, np.array([[0, 1500, 0], [-3, 12, 0]], np.int16))
    f = np.array([100.0, 20000.0, 20000.5, 1e9], np.float32)
    formats.clamp_max_depth(f, 20.0)
    assert np.array_equal(f, np.array([100.0, 20000.0, 0.0, 0.0], np.float32))
    bad = tmp_path / "bad.xml"
    bad.write_text('<opencv_storage><depth-frame type_id="opencv-matrix"><rows>1</rows><cols>1</cols><dt>f</dt><data>1.</data></depth-frame></opencv_storage>')
    with pytest.raises(RuntimeError):
        formats.read_depth_xml(str(bad))                                     # "Precomputed depth map had the wrong format."

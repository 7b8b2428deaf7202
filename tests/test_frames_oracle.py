"""CPU: oracle/frames_oracle.c (instance splitting + compositing, SURVEY 8(f) ranks 2-3) against
(1) the reference's own ProcessSilhouette_CPU / RemoveSilhouette_CPU / CompositeDepth / CompositeColor, cut out of
    DS/InstRecLib/InstanceReconstructor.cpp at build time and compiled with the reference's Mask / BoundingBox / ORUtils headers
    (oracle/_ref/libinstrecref.so) — byte for byte on random inputs; and
(2) hand-computed known answers, which also cover the two pieces that cannot be cut out (the per-track dispatch loop and the
    background dimming of CompositeInstances)."""
import ctypes as C

import numpy as np

from dynslam_b200 import abi
from tests import frameslib as F
from tests import hostlib as H


def test_process_and_remove_silhouette_known_answers():
    L = H.oracle()
    w, h = 8, 6
    rgb = np.arange(w * h * 4, dtype=np.uint8).reshape(h, w, 4)
    depth = (np.arange(w * h, dtype=np.float32).reshape(h, w) + 1.0)
    rgb0, depth0 = rgb.copy(), depth.copy()
    copy = ((2, 1, 4, 3), np.array([[1, 1, 0], [1, 1, 1], [0, 1, 2]], np.uint8))          # 2 is not "inside" (== 1 test)
    dele = ((1, 0, 5, 4), np.zeros((5, 5), np.uint8))
    dele[1][1:4, 1:4] = 1                                                                  # frame x 2..4, y 1..3
    ops, dests = F.host_ops([dict(copy=copy, delete=dele)], [2], w, h)
    L.oracle_process_silhouettes(H.vptr(rgb), H.vptr(depth), w, h, ops, 1)
    drgb, ddep = dests[0]
    inside = np.zeros((h, w), bool)
    inside[1, 2] = inside[1, 3] = inside[2, 2] = inside[2, 3] = inside[2, 4] = inside[3, 3] = True
    assert np.array_equal(drgb[inside], rgb0[inside]) and np.array_equal(ddep[inside], depth0[inside])
    assert (drgb[~inside] == 255).all() and (ddep[~inside] == 0).all()                    # memset 255 / 0 everywhere else
    cut = np.zeros((h, w), bool); cut[1:4, 2:5] = True
    assert (rgb[cut] == 0).all() and (depth[cut] == 0).all()
    assert np.array_equal(rgb[~cut], rgb0[~cut]) and np.array_equal(depth[~cut], depth0[~cut])
    # a second detection copying from the already blanked area gets zeros (sequential semantics)
    rgb, depth = rgb0.copy(), depth0.copy()
    ops, dests = F.host_ops([dict(copy=copy, delete=dele), dict(copy=copy, delete=dele)], [1, 2], w, h)
    L.oracle_process_silhouettes(H.vptr(rgb), H.vptr(depth), w, h, ops, 2)
    assert (dests[1][1][inside] == 0).all() and (dests[1][0][inside] == 0).all()
    # action 0 touches nothing
    rgb, depth = rgb0.copy(), depth0.copy()
    ops, _ = F.host_ops([dict(copy=copy, delete=dele)], [0], w, h)
    L.oracle_process_silhouettes(H.vptr(rgb), H.vptr(depth), w, h, ops, 1)
    assert np.array_equal(rgb, rgb0) and np.array_equal(depth, depth0)


def test_composite_known_answers():
    L = H.oracle()
    t = np.array([0.0, 2.0, 3.0, 0.0, 5.0], np.float32)
    s = np.array([1.0, 0.0, 2.5, 0.0, 6.0], np.float32)
    L.oracle_composite_depth(H.vptr(t), H.vptr(s), 5)
    assert t.tolist() == [1.0, 2.0, 2.5, 0.0, 5.0]
    tc = np.array([[10, 20, 30, 40]] * 4, np.uint8)
    td = np.array([0.0, 4.0, 4.0, 4.0], np.float32)
    sc = np.array([[100, 200, 250, 9]] * 4, np.uint8)
    sd = np.array([3.0, 3.0, 5.0, 0.0], np.float32)
    tint = (C.c_int32 * 4)(0x1f, 0x77, 0xb4, 255)
    L.oracle_composite_color(H.vptr(tc), H.vptr(td), H.vptr(sc), H.vptr(sd), 4, tint, 1.0)
    # tint_strength 1: col_strength = 0.5 -> (100*.5+31, 200*.5+119, min(255, 250*.5+180)) ; alpha untouched
    assert tc[0].tolist() == [81, 219, 255, 40] and tc[1].tolist() == [81, 219, 255, 40]
    assert tc[2].tolist() == [10, 20, 30, 40] and tc[3].tolist() == [10, 20, 30, 40]
    assert td.tolist() == [3.0, 3.0, 4.0, 4.0]
    # dimming: uchar(c * (1.0 - 0.10f)) in double: 10*0.9 = 8.99999997 -> 8 ; 200 -> 179 (0.10f > 0.1)
    oc = np.array([[10, 200, 255, 77]], np.uint8)
    od = np.array([1.0], np.float32)
    layers = (abi.InstanceLayer * 1)()
    L.oracle_composite_instances(H.vptr(oc), H.vptr(od), 1, layers, 0, 0.10, 1.0)
    assert oc[0].tolist() == [8, 179, 229, 77]


# ---- pinned to the reference's own functions (oracle/_ref/libinstrecref.so, built by oracle/build_ref.sh from
# ---- DS/InstRecLib/InstanceReconstructor.cpp with the reference's Mask / BoundingBox / ORUtils headers); their outputs
# ---- on these inputs are stored in tests/golden/reference_pins.json (tests/refpins.py) -----------------------------------
import os

from tests.refpins import pin

INSTREC_SO = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libinstrecref.so")


def _instrec_ref():
    R = C.CDLL(INSTREC_SO)
    vp = C.c_void_p
    R.ref_process_silhouette.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.POINTER(abi.Mask)]
    R.ref_remove_silhouette.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(abi.Mask)]
    R.ref_composite_depth.argtypes = [vp, vp, C.c_int, C.c_int]
    R.ref_composite_color.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_float]
    for f in (R.ref_process_silhouette, R.ref_remove_silhouette, R.ref_composite_depth, R.ref_composite_color):
        f.restype = None
    return R


def _random_detection(rng, w, h):
    """A box that may stick out of the frame on any side, with a random 0/1/2 mask (2 is not 'inside')."""
    bw, bh = int(rng.integers(1, w)), int(rng.integers(1, h))
    x0, y0 = int(rng.integers(-bw // 2, w - 1)), int(rng.integers(-bh // 2, h - 1))
    data = rng.choice(np.array([0, 1, 1, 1, 2], np.uint8), size=(bh, bw)).astype(np.uint8)
    return (x0, y0, x0 + bw - 1, y0 + bh - 1), np.ascontiguousarray(data)


def test_silhouette_functions_equal_reference_code():
    """oracle_process_silhouettes (one op at a time) against ProcessSilhouette_CPU<float> / RemoveSilhouette_CPU<float> compiled
    from the reference file, on random frames, boxes (inside, clipped, mostly outside) and masks: every output byte equal."""
    L = H.oracle()
    rng = np.random.default_rng(5)
    for it in range(60):
        w, h = int(rng.integers(4, 70)), int(rng.integers(4, 40))
        rgb = rng.integers(0, 256, size=(h, w, 4), dtype=np.uint8)
        depth = rng.choice(np.array([0.0, -1.0, 1.5, 7.25, 19.0], np.float32), size=(h, w)).astype(np.float32)
        copy, dele = _random_detection(rng, w, h), _random_detection(rng, w, h)
        for action in (1, 2):
            o_rgb, o_dep = rgb.copy(), depth.copy()
            ops, dests = F.host_ops([dict(copy=copy, delete=dele)], [action], w, h)
            L.oracle_process_silhouettes(H.vptr(o_rgb), H.vptr(o_dep), w, h, ops, 1)

            def ref_silhouettes():
                R = _instrec_ref()
                r_rgb, r_dep = rgb.copy(), depth.copy()
                r_drgb, r_ddep = np.full((h, w, 4), 7, np.uint8), np.full((h, w), 7.0, np.float32)
                if action == 2:
                    cm = F.host_mask(*copy)
                    R.ref_process_silhouette(H.vptr(r_rgb), H.vptr(r_dep), H.vptr(r_drgb), H.vptr(r_ddep), w, h, C.byref(cm))
                dm = F.host_mask(*dele)
                R.ref_remove_silhouette(H.vptr(r_rgb), H.vptr(r_dep), w, h, C.byref(dm))
                return [r_rgb, r_dep, r_drgb, r_ddep]
            pin(f"frames/silhouettes/case{it}/action{action}", [o_rgb, o_dep, dests[0][0], dests[0][1]], ref_silhouettes)


def test_composite_functions_equal_reference_code():
    """oracle_composite_depth / oracle_composite_color against CompositeDepth / CompositeColor compiled from the reference file."""
    L = H.oracle()
    rng = np.random.default_rng(9)
    palette = [(0x1f, 0x77, 0xb4, 255), (0xff, 0x7f, 0x0e, 255), (0x17, 0xbe, 0xcf, 255), (0, 0, 0, 255), (255, 255, 255, 255)]
    for it in range(40):
        w, h = int(rng.integers(1, 50)), int(rng.integers(1, 30))
        vals = np.array([0.0, 0.5, 1.0, 2.5, 2.5000002, 30.0], np.float32)
        t, s = rng.choice(vals, size=(h, w)).astype(np.float32), rng.choice(vals, size=(h, w)).astype(np.float32)
        a = t.copy()
        L.oracle_composite_depth(H.vptr(a), H.vptr(s), w * h)

        def ref_depth():
            b = t.copy()
            _instrec_ref().ref_composite_depth(H.vptr(b), H.vptr(s), w, h)
            return b
        pin(f"frames/composite_depth/case{it}", a, ref_depth)
        tc, sc = rng.integers(0, 256, size=(h, w, 4), dtype=np.uint8), rng.integers(0, 256, size=(h, w, 4), dtype=np.uint8)
        tint = (C.c_int32 * 4)(*palette[it % len(palette)])
        for strength in (1.0, 0.35, 0.0, 1.5):
            oc, od = tc.copy(), t.copy()
            L.oracle_composite_color(H.vptr(oc), H.vptr(od), H.vptr(sc), H.vptr(s), w * h, tint, strength)

            def ref_color():
                rc, rd = tc.copy(), t.copy()
                _instrec_ref().ref_composite_color(H.vptr(rc), H.vptr(rd), H.vptr(sc), H.vptr(s), w, h, tint, strength)
                return [rc, rd]
            pin(f"frames/composite_color/case{it}/strength{strength}", [oc, od], ref_color)

"""CPU: oracle/eval_oracle.c (the evaluation consumer of the float raycast, SURVEY 8(f) rank 3) against
(1) the reference's own Evaluation::ProjectLidar / EvaluateDepth and EvaluationCallback::ProcessLidarPoint / ComputeAccuracy, cut
    out of DS/Evaluation/Evaluation.cpp and EvaluationCallback.cpp at build time (oracle/_ref/libevalref.so) — count for count on
    random clouds, with and without the static / dynamic association image, against their results stored in
    tests/golden/reference_pins.json (tests/refpins.py); and
(2) hand-computed known answers of the classification rules."""
import numpy as np
import pytest

from dynslam_b200 import abi, engine as E
from tests import evallib as V
from tests.refpins import pin

CBS = [(0.5, True, False)] + [(float(d), True, False) for d in range(1, 13)] + [(3.0, True, True)]     # Evaluation.cpp:176-195


def test_known_answers_of_the_classification():
    w, h = 64, 48
    p, rigt = V.params(w, h, 0.5, 30.0)
    v, pl, pr, b = rigt
    # one return straight ahead at 10 m: left pixel, disparity = fx * baseline / z
    cam = np.array([0.0, 0.0, 10.0, 1.0])
    velo = np.linalg.inv(v) @ cam
    pts = np.array([[velo[0], velo[1], velo[2], 0.3]], np.float32)
    left = pl @ cam; left /= left[2]
    row, col = int(round(left[1])), int(round(left[0]))
    lidar_disp = np.float32(left[0] - (pr @ cam / (pr @ cam)[2])[0])
    rendered = np.zeros((h, w), np.float32); inp = np.zeros((h, w), np.int16)
    fxb = np.float32(b) * np.float32(pl[0, 0])
    # rendered 2 px off, input 0.4 px off the ground-truth disparity
    rendered[row, col] = fxb / (lidar_disp + np.float32(2.0))
    inp[row, col] = int(round(1000.0 * float(fxb / (lidar_disp + np.float32(0.4)))))
    cbs = [(0.5, True, False), (1.0, True, False), (3.0, True, False), (3.0, True, True)]
    rc, st, _, summ = V.run_oracle(p, pts, rendered, inp, cbs)
    assert rc == 0 and summ.valid_lidar_points == 1
    assert [r["rendered"]["error"] for r in st] == [1, 1, 0, 0] and [r["rendered"]["correct"] for r in st] == [0, 0, 1, 1]
    assert [r["input"]["error"] for r in st] == [0, 0, 0, 0] and [r["input"]["correct"] for r in st] == [1, 1, 1, 1]
    # missing rendered depth: with compare_on_intersection both sides count the point as missing, without only the rendered side
    rendered[row, col] = 0.0
    rc, st, _, _ = V.run_oracle(p, pts, rendered, inp, [(1.0, True, False), (1.0, False, False)])
    assert st[0]["rendered"]["missing"] == 1 and st[0]["input"]["missing"] == 1 and st[0]["input"]["missing_separate"] == 0
    assert st[1]["rendered"]["missing"] == 1 and st[1]["input"]["missing"] == 0 and st[1]["input"]["correct"] == 1
    assert st[0]["rendered"]["missing_separate"] == 1
    # outside the depth range or the frame: not a measurement
    far = np.linalg.inv(v) @ np.array([0.0, 0.0, 31.0, 1.0])
    side = np.linalg.inv(v) @ np.array([50.0, 0.0, 10.0, 1.0])
    rc, st, _, summ = V.run_oracle(p, np.array([list(far[:3]) + [0], list(side[:3]) + [0]], np.float32), rendered, inp, cbs)
    assert summ.valid_lidar_points == 0 and all(r["measurement_count"] == 0 for r in st)


def test_negative_disparity_is_the_references_exception():
    w, h = 64, 48
    p, rigt = V.params(w, h)
    v, pl, pr, b = rigt
    p.proj_right[9] = p.proj_left[9] + 50.0          # right camera shifted the wrong way: negative disparities
    pts = V.lidar_cloud(50, 3, rigt, w, h)
    rendered, inp = V.depth_images(w, h, 4)
    rc, _, _, summ = V.run_oracle(p, pts, rendered, inp, CBS)
    assert rc == -1 and summ.negative_disparities == 1
    pin("eval/negative_disparity", rc, lambda: V.run_reference(p, pts, rendered, inp, CBS)[0])


@pytest.mark.parametrize("seed,w,h,with_assoc", [(1, 1242, 375, False), (2, 620, 188, True), (5, 1242, 375, True)])
def test_oracle_equals_reference_functions(seed, w, h, with_assoc):
    p, rigt = V.params(w, h)
    pts = V.lidar_cloud(60000, seed, rigt, w, h)
    rendered, inp = V.depth_images(w, h, seed + 100)
    assoc = None
    if with_assoc:
        assoc = (np.random.default_rng(seed).uniform(size=(h, w)) * 3).astype(np.uint8)       # static / dynamic / neither
        assoc[:, : w // 2] = abi.EVAL_STATIC
    rc_o, st_o, dy_o, summ = V.run_oracle(p, pts, rendered, inp, CBS, assoc, with_dynamic=with_assoc)
    assert rc_o == 0
    pin(f"eval/evaluate_depth/seed{seed}-{w}x{h}{'-assoc' if with_assoc else ''}", [rc_o, st_o, dy_o, summ.skipped_lidar_points],
        lambda: list(V.run_reference(p, pts, rendered, inp, CBS, assoc, with_dynamic=with_assoc)))
    assert st_o[0]["measurement_count"] > 10000
    for r in st_o:      # DepthResult's own invariants (Records.h:31-34)
        for side in ("rendered", "input"):
            assert r["measurement_count"] == r[side]["error"] + r[side]["missing"] + r[side]["correct"]
            assert r[side]["missing"] >= r[side]["missing_separate"]
    # accuracy grows with delta_max
    acc = [r["rendered"]["correct"] for r in st_o[:13]]
    assert acc == sorted(acc)


def test_default_callbacks_are_the_references_list():
    assert E.Evaluation.default_callbacks() == CBS

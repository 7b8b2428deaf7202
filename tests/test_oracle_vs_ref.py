"""Pins the oracle (oracle/tsdf_oracle.c) against the reference's own DeviceAgnostic functions
(compiled by oracle/build_ref.sh into oracle/_ref/libitmref.so): every stage bit-exact on a short
KITTI-shaped synthetic sequence. CPU only. The reference's outputs on these inputs are stored in
tests/golden/reference_pins.json (tests/refpins.py)."""
import ctypes as C

import numpy as np
import pytest

from dynslam_b200 import abi, synth
from tests import hostlib as H
from tests.refpins import pin

NB, NE = 0x100000, 0x80000  # compile-time sizes of the reference (Utils/ITMLibDefines.h:42-53)
SCALE = 0.25


def _hooks():
    L = H.oracle()
    L.oracle_mark_only.argtypes = [C.c_void_p, C.POINTER(abi.Scene), C.c_void_p, C.POINTER(abi.View)]
    L.oracle_mark_only.restype = None
    L.oracle_alloc_type.argtypes = [C.c_void_p]
    L.oracle_alloc_type.restype = C.POINTER(C.c_uint8)
    L.oracle_block_coords.argtypes = [C.c_void_p]
    L.oracle_block_coords.restype = C.POINTER(C.c_int16)
    L.oracle_block_visible.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_float, C.c_int, C.c_int]
    L.oracle_project_single_block.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int, C.c_int,
                                              C.c_float, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_float)]
    L.oracle_combine_block.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.oracle_combine_block.restype = None
    return L


@pytest.fixture(scope="module")
def seq():
    """Runs 6 frames through the oracle, keeping per-frame views and pre-integration voxel copies."""
    L = _hooks()

    def ref_sizes():
        nb, ne = C.c_int(), C.c_int()
        return [H.ref().ref_table_sizes(C.byref(nb), C.byref(ne)), nb.value, ne.value]
    pin("oracle_vs_ref/table_sizes", [20, NB, NE], ref_sizes)
    scene = synth.StreetScene(seed=6, length_m=80.0)
    w, h = int(round(synth.KITTI_W * SCALE)), int(round(synth.KITTI_H * SCALE))
    vol = H.HostVolume(20000, NB, NE, w, h, H.SceneParams(voxelSize=0.05, mu=0.75, maxW=50))
    frames = []
    for f in range(6):
        depth, rgb, M, proj = synth.kitti_frame(scene, f * 3, scale=SCALE)
        view = H.make_view(depth, rgb, M, proj, depthWeighting=(f % 2))
        # stage pin 1: marking, on the table state before this frame's allocation
        vis_o = vol.visType.copy()
        L.oracle_mark_only(vol.engine, C.byref(vol.scene), H.vptr(vis_o), C.byref(view))
        n = NB + NE
        at_o = np.ctypeslib.as_array(L.oracle_alloc_type(vol.engine), shape=(n,)).copy()
        bc_o = np.ctypeslib.as_array(L.oracle_block_coords(vol.engine), shape=(n * 4,)).copy()

        def ref_mark():
            vis_r = vol.visType.copy()
            at_r = np.zeros(n, dtype=np.uint8)
            bc_r = np.zeros(n * 4, dtype=np.int16)
            H.ref().ref_mark_image(H.vptr(at_r), H.vptr(vis_r), H.vptr(bc_r), C.byref(vol.scene), C.byref(view))
            return [at_r, vis_r, bc_r.reshape(-1, 4)[np.nonzero(at_r)[0]]]
        req = np.nonzero(at_o)[0]
        pin(f"oracle_vs_ref/mark/frame{f}", [at_o, vis_o, bc_o.reshape(-1, 4)[req]], ref_mark)
        if f == 0:
            assert len(req) > 500
        rc = L.oracle_allocate_from_depth(vol.engine, C.byref(vol.scene), C.byref(vol.rs), C.byref(view), 0, 0)
        assert rc == 0
        pre = vol.voxels.copy()
        L.oracle_integrate(vol.engine, C.byref(vol.scene), C.byref(vol.rs), C.byref(view), 0)
        frames.append((view, pre, vol.voxels.copy(), vol.visiblePos[:vol.rs.noVisibleBlocks].copy()))
    return vol, frames


def test_mat4_inv_and_mul():
    L = H.oracle()
    rng = np.random.RandomState(0)
    mats, ours = [], []
    for i in range(50):
        M = synth.kitti_pose(i * 7).astype(np.float32)
        M[:3, 3] += rng.randn(3).astype(np.float32)
        c = abi.mat_to_c(M)
        a, m1 = abi.f16(), abi.f16()
        rc = L.oracle_mat4_inv(c, a)
        L.oracle_mat4_mul(c, a, m1)
        mats.append(c)
        ours.append([rc, bytes(a), bytes(m1)])

    def ref_inv_mul():
        R, out = H.ref(), []
        for c in mats:
            b, m2 = abi.f16(), abi.f16()
            rc = R.ref_mat4_inv(c, b)
            R.ref_mat4_mul(c, b, m2)
            out.append([rc, bytes(b), bytes(m2)])
        return out
    assert all(o[0] == 1 for o in ours)
    pin("oracle_vs_ref/mat4_inv_mul", ours, ref_inv_mul)


def test_integrate_blocks_bit_exact(seq):
    vol, frames = seq
    L = H.oracle()
    rng = np.random.RandomState(1)
    checked = changed = 0
    for f, (view, pre, post, vis) in enumerate(frames):
        pick = rng.choice(len(vis), size=min(400, len(vis)), replace=False)
        coords = [tuple(int(t) for t in vis[i]) for i in pick]
        idxs = np.array([L.oracle_find_block(H.vptr(vol.hash), NB, x, y, z) for x, y, z in coords], dtype=np.int32)
        # the final table may have moved the block (no decay here, so ptr is stable)
        ptrs = [int(vol.hash[idx]["ptr"]) for idx in idxs if idx >= 0]
        ours = b"".join(post[p * 512:(p + 1) * 512].tobytes() for p in ptrs)

        def ref_integrate():
            R, out = H.ref(), []
            ridx = np.array([R.ref_find_block(H.vptr(vol.hash), x, y, z) for x, y, z in coords], dtype=np.int32)
            for (x, y, z), idx in zip(coords, ridx):
                if idx < 0:
                    continue
                ptr = int(vol.hash[idx]["ptr"])
                blk = pre[ptr * 512:(ptr + 1) * 512].copy()
                R.ref_integrate_block(H.vptr(blk), H.vptr(np.array([x, y, z], dtype=np.int16)), C.byref(vol.scene), C.byref(view))
                out.append(blk.tobytes())
            return [ridx, b"".join(out)]
        pin(f"oracle_vs_ref/integrate_blocks/frame{f}", [idxs, ours], ref_integrate)
        checked += len(ptrs)
        changed += sum(int(post[p * 512:(p + 1) * 512].tobytes() != pre[p * 512:(p + 1) * 512].tobytes()) for p in ptrs)
    assert checked > 1000 and changed > 300


def test_block_visibility_and_projection(seq):
    vol, frames = seq
    L = _hooks()
    used = np.nonzero(vol.hash["ptr"] >= 0)[0]
    rng = np.random.RandomState(2)
    w, h = vol.w, vol.h
    n_vis = n_proj = 0

    def visible_and_projected(lib, prefix, pos, view):
        """[visible, projected, ul, lr] and the z range of one block (corners and z range only where it projects)"""
        a = getattr(lib, prefix + "block_visible")(H.vptr(pos), view.M_d, view.proj_d, vol.scene.voxelSize, w, h)
        ul, lr, zr = (C.c_int * 2)(), (C.c_int * 2)(), (C.c_float * 2)()
        o = getattr(lib, prefix + "project_single_block")(H.vptr(pos), view.M_d, view.proj_d, w, h, vol.scene.voxelSize, ul, lr, zr)
        return [a, o] + (list(ul) + list(lr) if o else [0] * 4), (bytes(zr) if o else b"")

    for f, (view, _, _, _) in enumerate(frames[::2]):
        blocks = [vol.hash[i]["pos"].astype(np.int16).copy() for i in rng.choice(used, size=600, replace=False)]

        def table(lib, prefix):
            rows = [visible_and_projected(lib, prefix, pos, view) for pos in blocks]
            return [np.array([r[0] for r in rows], dtype=np.int32), b"".join(r[1] for r in rows)]
        ours = table(L, "oracle_")
        pin(f"oracle_vs_ref/visibility_projection/frame{2 * f}", ours, lambda: table(H.ref(), "ref_"))
        n_vis += int(ours[0][:, 0].sum())
        n_proj += int((ours[0][:, 1] != 0).sum())
    assert n_vis > 100 and n_proj > 100


def test_raycast_shading_icp_bit_exact(seq):
    vol, frames = seq
    L = H.oracle()
    view = frames[-1][0]
    cam = abi.Camera()
    cam.M, cam.invM, cam.proj = view.M_d, view.invM_d, view.proj_d
    L.oracle_expected_depths(C.byref(vol.scene), C.byref(vol.rs), C.byref(cam))
    mm = vol.minmax.copy()
    assert (mm[..., 0] < mm[..., 1]).sum() > 200  # some 1/8-res cells are covered
    # raycast
    L.oracle_raycast(C.byref(vol.scene), C.byref(vol.rs), view.invM_d, view.proj_d, 0)
    ray_o = vol.raycastResult.copy()

    def ref_raycast():
        vol.raycastResult[:] = 0
        H.ref().ref_raycast(C.byref(vol.scene), C.byref(vol.rs), view.invM_d, view.proj_d)
        return vol.raycastResult.copy()
    pin("oracle_vs_ref/raycast", ray_o, ref_raycast)
    assert (ray_o[..., 3] > 0).mean() > 0.3
    # all five render types
    for t in range(5):
        oc = np.zeros((vol.h, vol.w, 4), dtype=np.uint8)
        of = np.zeros((vol.h, vol.w), dtype=np.float32)
        L.oracle_render_image(C.byref(vol.scene), C.byref(vol.rs), C.byref(cam), H.vptr(oc), H.vptr(of), t, 0)
        # drawPixelNormal leaves alpha untouched (DA/ITMVisualisationEngine.h:283-288)
        channels = 3 if t == abi.RENDER_COLOUR_FROM_NORMAL else 4

        def ref_shade():
            rc_, rf = np.zeros_like(oc), np.zeros_like(of)
            H.ref().ref_shade(C.byref(vol.scene), C.byref(vol.rs), C.byref(cam), H.vptr(rc_), H.vptr(rf), t)
            return [rc_[..., :channels], rf]
        pin(f"oracle_vs_ref/render_type{t}", [oc[..., :channels], of], ref_shade)
        if t == abi.RENDER_DEPTH_MAP:
            assert (of > 0).mean() > 0.3
        else:
            assert oc[..., :3].any()
    # ICP maps
    L.oracle_icp_maps(C.byref(vol.scene), C.byref(vol.rs), C.byref(view), H.vptr(vol.points), H.vptr(vol.normals), 0)
    img_o, p_o, n_o = vol.raycastImage.copy(), vol.points.copy(), vol.normals.copy()

    def ref_icp():
        vol.raycastImage[:] = 0
        p_r, n_r = np.zeros_like(p_o), np.zeros_like(n_o)
        H.ref().ref_icp(C.byref(vol.scene), C.byref(vol.rs), view.invM_d, H.vptr(p_r), H.vptr(n_r))
        return [vol.raycastImage.copy(), p_r, n_r]
    pin("oracle_vs_ref/icp_maps", [img_o, p_o, n_o], ref_icp)
    assert (p_o[..., 3] > 0).mean() > 0.2


def test_combine_voxels(seq):
    vol, frames = seq
    L = _hooks()
    used = np.nonzero(vol.hash["ptr"] >= 0)[0][:64]
    pairs = [(vol.voxels[int(vol.hash[i]["ptr"]) * 512:][:512].copy(), vol.voxels[int(vol.hash[used[k + 1]]["ptr"]) * 512:][:512].copy())
             for k, i in enumerate(used[:-1])]

    def combined(fn):
        out = []
        for a, b in pairs:
            d = b.copy()
            fn(H.vptr(a), H.vptr(d), 50)
            out.append(d.tobytes())
        return b"".join(out)
    pin("oracle_vs_ref/combine_voxels", combined(L.oracle_combine_block), lambda: combined(H.ref().ref_combine_block))


# ---- view builder (oracle/view_oracle.c vs DeviceAgnostic/ITMViewBuilder.h) ---------------------------
def _vb_inputs():
    from tests import viewlib
    raw, _ = viewlib.raw_kitti_frame(scale=0.25)
    return [raw, viewlib.raw_noise_frame()]


def test_view_convert_bit_exact():
    L = H.oracle()
    for k, raw in enumerate(_vb_inputs()):
        h, w = raw.shape
        a = np.zeros((h, w), np.float32)
        L.oracle_convert_depth_affine_to_float(H.vptr(a), H.vptr(raw), w, h, 1.0 / 1000.0, 0.0)

        def ref_affine():
            b = np.zeros((h, w), np.float32)
            H.ref().ref_view_convert_affine(H.vptr(b), H.vptr(raw), w, h, 1.0 / 1000.0, 0.0)
            return b
        pin(f"oracle_vs_ref/view_convert_affine/input{k}", a, ref_affine)
        assert (a == -1.0).any() and (a > 0).any()
        # Kinect disparity trafo (Objects/ITMDisparityCalib.h:25-26) with the calib-file style parameters
        disp = (raw // 4).astype(np.int16)
        disp[0, :5] = 1135                                   # disparity_tmp == 0 -> depth 0 -> -1
        L.oracle_convert_disparity_to_depth(H.vptr(a), H.vptr(disp), w, h, 1135.09, 0.0819141, 573.71)

        def ref_disparity():
            b = np.zeros((h, w), np.float32)
            H.ref().ref_view_convert_disparity(H.vptr(b), H.vptr(disp), w, h, 1135.09, 0.0819141, 573.71)
            return b
        pin(f"oracle_vs_ref/view_convert_disparity/input{k}", a, ref_disparity)


def test_view_filter_and_update_view_bit_exact():
    L = H.oracle()
    for k, raw in enumerate(_vb_inputs()):
        h, w = raw.shape
        d0 = np.zeros((h, w), np.float32)
        L.oracle_convert_depth_affine_to_float(H.vptr(d0), H.vptr(raw), w, h, 1.0 / 1000.0, 0.0)   # pinned in test_view_convert_bit_exact
        # one pass: the target's 2-pixel border must stay what it was
        a = np.full((h, w), 7.0, np.float32)
        L.oracle_depth_filtering(H.vptr(a), H.vptr(d0), w, h)

        def ref_filter_pass():
            b = np.full((h, w), 7.0, np.float32)
            H.ref().ref_view_filter_pass(H.vptr(b), H.vptr(d0), w, h)
            return b
        pin(f"oracle_vs_ref/view_filter_pass/input{k}", a, ref_filter_pass)
        assert (a[:2] == 7.0).all() and (a[:, -2:] == 7.0).all()
        calib = abi.ViewCalib()
        calib.trafoType, calib.useBilateralFilter, calib.modelSensorNoise = 1, 1, 1
        calib.params = (C.c_float * 2)(1.0 / 1000.0, 0.0)
        calib.intrinsics_d = (C.c_float * 4)(707.0912, 707.0912, w / 2.0, h / 2.0)
        depth_o, float_o = np.zeros((h, w), np.float32), np.zeros((h, w), np.float32)
        nrm_o, sig_o = np.zeros((h, w, 4), np.float32), np.zeros((h, w), np.float32)
        L.oracle_update_view(H.vptr(raw), w, h, C.byref(calib), H.vptr(depth_o), H.vptr(float_o), H.vptr(nrm_o), H.vptr(sig_o))

        def ref_update_view():
            """UpdateView: the reference's own sequence (ITMViewBuilder_CUDA.cu:64-79) composed from its functions"""
            R = H.ref()
            depth_r, float_r = d0.copy(), np.zeros((h, w), np.float32)
            for _ in range(2):
                R.ref_view_filter_pass(H.vptr(float_r), H.vptr(depth_r), w, h)
                R.ref_view_filter_pass(H.vptr(depth_r), H.vptr(float_r), w, h)
            R.ref_view_filter_pass(H.vptr(float_r), H.vptr(depth_r), w, h)
            nrm_r, sig_r = np.zeros((h, w, 4), np.float32), np.zeros((h, w), np.float32)
            R.ref_view_normal_weight(H.vptr(float_r), H.vptr(nrm_r), H.vptr(sig_r), w, h, calib.intrinsics_d)
            return [float_r, nrm_r, sig_r]
        pin(f"oracle_vs_ref/update_view/input{k}", [depth_o, nrm_o, sig_o], ref_update_view)
        assert (depth_o[:2] == 0).all() and (depth_o[-2:] == 0).all() and (depth_o[:, :2] == 0).all()   # floatImage's border
        assert (nrm_o[..., 3] == 1.0).sum() > 0.3 * w * h


def test_mesh_oracle_equals_reference_cpu_engine():
    """Meshing (SURVEY 8(f) rank 4): oracle/mesh_oracle.c against the reference's OWN serial engine,
    ITMMeshingEngine_CPU<ITMVoxel, ITMVoxelBlockHash>::MeshScene (Engine/DeviceSpecific/CPU/ITMMeshingEngine_CPU.cpp:19-80, live
    code, compiled from its source into oracle/_ref/libitmref.so), on a map fused by the oracle: same triangle count, every
    vertex and colour bit for bit, same order."""
    from dynslam_b200 import abi, synth
    from tests import parity as P
    L = H.oracle()
    cfg = P.Cfg(scale=0.25, frames=4, numBlocks=16384, numBuckets=0x100000, excessSize=0x80000)    # the reference's compile-time table size
    w, h = int(round(synth.KITTI_W * cfg.scale)), int(round(synth.KITTI_H * cfg.scale))
    vol = H.HostVolume(cfg.numBlocks, cfg.numBuckets, cfg.excessSize, w, h)
    for depth, rgb, M, proj in P.frames_of(cfg):
        hv = H.make_view(depth, rgb, M, proj)
        assert L.oracle_allocate_from_depth(vol.engine, C.byref(vol.scene), C.byref(vol.rs), C.byref(hv), 0, 0) == 0
        L.oracle_integrate(vol.engine, C.byref(vol.scene), C.byref(vol.rs), C.byref(hv), 0)
    nmax = cfg.numBlocks * 512 // 16
    a = np.zeros(nmax, dtype=abi.TRIANGLE_DTYPE)
    na = L.oracle_mesh_scene(C.byref(vol.scene), H.vptr(a), nmax)

    def ref_mesh():
        b = np.zeros(nmax, dtype=abi.TRIANGLE_DTYPE)
        nb = H.ref().ref_mesh_scene(H.vptr(vol.hash), H.vptr(vol.voxels), cfg.numBlocks, C.c_float(cfg.voxelSize), H.vptr(b), nmax)
        return [nb, b[:nb]]
    pin("oracle_vs_ref/mesh_scene", [na, a[:na]], ref_mesh)
    assert na > 20000
    # colours are really interpolated from the volume, vertices lie inside the fused region
    assert a["c0"][:na].max() > 0.2 and np.isfinite(a["p0"][:na]).all()

"""GPU parity at the places where the VIO kernels have their special cases, against the CPU oracle:
  * tap footprints at the image border (parity_util.border_frame): one stride inside, on the last row / column, one stride
    past, half outside, the corners and points left / right of the image, at every tap stride 1 .. 32; the linear-index
    reads wrap to the neighbouring row left and right and read 0 above / below the buffer (DESIGN §4);
  * reference-image selection (ref_img_index over three images) in warpAffine and the inverse-compositional precompute;
  * the TMA tap path (ESIKF_TUNE_VIO_TMA) at its eligibility boundary and on images whose pitch rules it out;
  * patch and point counts on both sides of the persistent kernels' work-split boundaries (cached / uncached VIO slices,
    resident / tiled LIO slices, and launches that mix both);
  * search levels outside [0, 8] rejected on input."""
import dataclasses
import functools

import numpy as np
import pytest

import oracle_bind as O
from conftest import get_frame
from fast_livo2_b200 import api
from fast_livo2_b200 import synthetic as S
from parity_util import border_frame, last_origin, tap_origin
from test_gpu_loop_modes import LIO_KEYS, VIO_KEYS, _bits_equal
from test_gpu_vio import _compare_vio, _setup, _vio_prior

pytestmark = pytest.mark.gpu

FISHEYE = S.CamCfg(model=1, width=720, height=540, fx=351.31400364193297, fy=351.4911744656785, cx=367.8522793375995, cy=253.8402144980996,
                   d=(-0.03696737352869157, -0.008917880497032812, 0.008912969593422046, -0.0037685977496087313, 0.0))
CAMERAS = {
    "640x512": dict(seed=2),  # BASELINE config-2 camera: row pitch a multiple of 16, the TMA variant is eligible
    "612x512": dict(seed=13, cam=S.CamCfg(width=612, height=512, fx=612.0 * 0.72, fy=612.0 * 0.72, cx=306.0, cy=256.0),
                    vio=S.VioCfg(levels=5, img_point_cov=1000.0)),  # config-5 camera: pitch not a multiple of 16
    "720x540_fisheye": dict(seed=9, cam=FISHEYE, vio=S.VioCfg(img_point_cov=1000.0), ext=S.hilti_extrinsics()),
    "641x481": dict(seed=5, cam=S.CamCfg(width=641, height=481, fx=470.0, fy=470.0, cx=320.3, cy=240.7)),
}


@functools.lru_cache(maxsize=None)
def _border(name):
    kw = dict(CAMERAS[name])
    seed = kw.pop("seed")
    fr = get_frame(seed=seed, n_pts=1000, n_map=100_000, n_patches=100, scene_scale=0.5, **kw)
    prior = _vio_prior(fr, seed)
    return border_frame(fr, prior, seed=seed), prior


def _args(b, prior, idx=slice(None)):
    return (b["img"], b["vis_pos"][idx], b["warp_patch"][idx], b["search_levels"][idx], b["inv_ref_expo"][idx], prior, prior)


def _oracle(b, *args):
    return O.OracleVIO(b["cam_cfg"], b["ext"], b["vio_cfg"]).update(*args)


def _third_image(img):
    """A third reference image with content unlike the other two (mirrored, inverted)."""
    return np.ascontiguousarray(255 - img[::-1, ::-1])


def _run_modes(ctx, args, modes, tuning=0):
    out = []
    try:
        ctx.set_tuning(tuning)
        for m in modes:
            ctx.set_loop_mode(m)
            out.append(ctx.vio_update(*args))
    finally:
        ctx.set_loop_mode(api.DEFAULT_LOOP_MODE)
        ctx.set_tuning(0)
    return out


# ---------------------------------------------------------------------------------------------------------------- coverage
def _footprints(b, state):
    """Per border patch at its target stride: (x0, y0, s) for the pose in `state`."""
    m = b["bp_level"] >= 0
    s = 1 << np.maximum(b["bp_level"], 0)
    x0, y0 = tap_origin(b["cam_cfg"], b["ext"], state, b["vis_pos"], s)
    return m, x0, y0, s


def _assert_edges_are_hit(b, prior, posterior):
    """The frame really exercises the border: per target stride, footprints past each edge, on the TMA boundary (last tap on
    the first / last column / row) and one stride past it, and border patches whose integer tap base moves during the update."""
    w, h = b["cam_cfg"].width, b["cam_cfg"].height
    m, x0, y0, s = _footprints(b, prior)
    for p in sorted(set(b["bp_level"][m])):
        k = m & (b["bp_level"] == p)
        sp = 1 << p
        assert np.any(k & (x0 < 0)) and np.any(k & (x0 + 10 * s >= w)) and np.any(k & (y0 < 0)) and np.any(k & (y0 + 10 * s >= h)), p
        assert np.any(k & (x0 == 0)) and np.any(k & (x0 == -sp)) and np.any(k & (y0 == 0)) and np.any(k & (y0 == -sp)), p
        lx, ly = last_origin(w, sp), last_origin(h, sp)
        assert np.any(k & (x0 == lx)) and np.any(k & (x0 == lx + sp)) and np.any(k & (y0 == ly)) and np.any(k & (y0 == ly + sp)), p
        if p == 0:
            assert np.any(k & (x0 + 10 == w - 1)) and np.any(k & (y0 + 10 == h - 1))
    assert np.any(b["bp_label"] == "outside")
    _, x1, y1, _ = _footprints(b, posterior)
    crossing = m & ((np.minimum(x0, x1) < 0) | (np.maximum(x0, x1) + 10 * s >= w) | (np.minimum(y0, y1) < 0) | (np.maximum(y0, y1) + 10 * s >= h))
    moved = (x0 != x1) | (y0 != y1)
    assert np.count_nonzero(crossing & moved) >= 4, "no border patch changes its tap base during the update"


# ---------------------------------------------------------------------------------------------------------------- getImagePatch
@pytest.mark.parametrize("name", list(CAMERAS))
def test_image_patch_at_the_border(gpu_ctx, name):
    b, _ = _border(name)
    _setup(gpu_ctx, b)
    vio = O.OracleVIO(b["cam_cfg"], b["ext"], b["vio_cfg"])
    pc = np.concatenate([b["bp_px"], -b["bp_px"][:12], [[0.0, 0.0], [b["cam_cfg"].width - 1.0, b["cam_cfg"].height - 1.0]]])
    assert np.any(pc < 0)
    for level in range(b["vio_cfg"].levels):
        g = gpu_ctx.vio_get_image_patch(pc, level)
        for i in range(len(pc)):
            assert np.array_equal(g[i], vio.get_image_patch(b["img"], pc[i], level)), (level, pc[i])


# ---------------------------------------------------------------------------------------------------------------- warpAffine
def _warp_refs(b):
    return [b["img_ref"], b["img"], _third_image(b["img_ref"])]


def _check_warp(g, o_rows, n):
    """atol 2e-3 and >= 98 % of the patches bit-exact; every sample the oracle zeroes stays exactly 0 on the GPU."""
    o = np.stack(o_rows)
    np.testing.assert_allclose(g, o, atol=2e-3)
    assert np.sum([np.array_equal(g[i], o[i]) for i in range(n)]) >= 0.98 * n
    assert np.all(g[o == 0] == 0)
    return o


def test_warp_affine_at_the_border_with_three_reference_images(gpu_ctx):
    b, prior = _border("640x512")
    refs = _warp_refs(b)
    cols, rows = b["cam_cfg"].width, b["cam_cfg"].height
    L = b["vio_cfg"].levels
    _setup(gpu_ctx, b)
    gpu_ctx.vio_set_ref_images(refs)
    vio = O.OracleVIO(b["cam_cfg"], b["ext"], b["vio_cfg"])
    try:
        # (1) vio_warp_patches on the border frame, reference image by patch
        n = len(b["vis_pos"])
        ridx = (np.arange(n) % 3).astype(np.int32)
        st = S.unpack_state(prior)
        T_cur = api.pack_T(*S.camera_pose(b["ext"], st["R"], st["p"]))
        w = gpu_ctx.vio_warp_patches(ridx, b["px_ref"], b["vis_pos"], b["vis_normal"], np.tile(api.pack_T(*b["T_ref"]), (n, 1)), T_cur)
        o = _check_warp(w["warp_patch"], [vio.warp_affine(refs[ridx[i]], w["A_cur_ref"][i], b["px_ref"][i], w["search_levels"][i]) for i in range(n)], n)
        assert np.count_nonzero(o == 0) > 1000
        # (2) vio_warp_affine with caller matrices: integer reference pixels put samples exactly on 0 and on cols-1 / rows-1
        #     (identity A: sample x = px_ref + (x - 4) 2^(search_level + level)), fractional ones on both sides of them
        rng = np.random.default_rng(7)
        px, A, sl = [], [], []
        for s_l in range(3):
            for u, v in ((4.0, rows / 2), (cols - 4.0, rows / 2), (cols / 2, 4.0), (cols / 2, rows - 4.0), (4.0, 4.0), (cols - 4.0, rows - 4.0),
                         (1.37, 3.62), (cols - 2.41, rows - 1.73), (cols - 5.5, 0.25), (-2.75, rows / 3), (cols + 1.5, rows / 3)):
                for shear in (0.0, 0.07):
                    px.append((u, v)), sl.append(s_l)
                    A.append(np.eye(2) if shear == 0 else np.eye(2) + rng.uniform(-shear, shear, (2, 2)))
        px, A, sl = np.array(px), np.array(A), np.array(sl, np.int32)
        m = len(px)
        ridx = (np.arange(m) % 3).astype(np.int32)
        g = gpu_ctx.vio_warp_affine(ridx, px, A, sl)
        _check_warp(g, [vio.warp_affine(refs[ridx[i]], A[i], px[i], sl[i]) for i in range(m)], m)
        # samples at exactly cols-1 / rows-1 exist (identity A, integer px_ref) and are outside (0); those at exactly 0 are inside
        y, x = np.divmod(np.arange(64), 8)
        hit_last = hit_zero = 0
        for i in range(m):
            if not np.array_equal(A[i], np.eye(2)):
                continue
            for lvl in range(L):
                sc = (1 << int(sl[i])) * (1 << lvl)
                sx, sy = px[i, 0] + (x - 4) * sc, px[i, 1] + (y - 4) * sc
                on_last = (sx == cols - 1) | (sy == rows - 1)
                hit_last += np.count_nonzero(on_last)
                assert np.all(g[i, 64 * lvl:64 * lvl + 64][on_last] == 0)
                hit_zero += np.count_nonzero((sx == 0) & (sy >= 0) & (sy < rows - 1))
        assert hit_last > 0 and hit_zero > 0
        # the image actually depends on ref_img_index: the same request against another image differs
        assert not np.array_equal(g, gpu_ctx.vio_warp_affine(np.zeros(m, np.int32), px, A, sl))
    finally:
        gpu_ctx.vio_set_ref_images([b["img_ref"]])


# ---------------------------------------------------------------------------------------------------------------- forward update
@pytest.mark.parametrize("name", list(CAMERAS))
def test_forward_update_with_border_patches_matches_oracle(gpu_ctx, name):
    b, prior = _border(name)
    _setup(gpu_ctx, b)
    args = _args(b, prior)
    o = _oracle(b, *args)
    L = b["vio_cfg"].levels
    assert o["total_iters"] >= 4
    assert np.any(o["accepted_per_level"][:L] < o["iters_per_level"][:L]), "no rollback"
    _assert_edges_are_hit(b, prior, o["state"])
    g2, g0 = _run_modes(gpu_ctx, args, (2, 0))
    _compare_vio(g2, o, L)
    _compare_vio(g0, o, L)
    assert g0["total_iters"] == g2["total_iters"]
    _bits_equal(g0, g2, VIO_KEYS)


@pytest.mark.parametrize("name", list(CAMERAS))
def test_tma_taps_at_the_eligibility_boundary_are_bit_identical(gpu_ctx, name):
    """On 640 px the footprints exactly at x0 == 0, on the last column / row and one stride past each exist at strides 1 .. 8
    (asserted by _assert_edges_are_hit); on 612 / 641 px and the fisheye camera (pitch not a multiple of 16 / 720 = 45 x 16
    with its own boundary) the flag changes nothing and raises nothing."""
    b, prior = _border(name)
    _setup(gpu_ctx, b)
    args = _args(b, prior)
    a = _run_modes(gpu_ctx, args, (2,))[0]
    t1, t2 = _run_modes(gpu_ctx, args, (2, 2), tuning=api.TUNE_VIO_TMA)
    assert a["total_iters"] == t1["total_iters"] == t2["total_iters"] and a["total_iters"] >= 4
    _bits_equal(a, t1, VIO_KEYS)
    _bits_equal(a, t2, VIO_KEYS)


# ---------------------------------------------------------------------------------------------------------------- inverse variant
def _inverse_refs_at_the_border(b, prior, imgs):
    """Reference features seen from the prior camera pose itself: ref_px are the border pixels (footprints across every edge
    of the reference images), images by patch from `imgs`."""
    st = S.unpack_state(prior)
    R, t = S.camera_pose(b["ext"], st["R"], st["p"])
    n = len(b["vis_pos"])
    pc = b["vis_pos"] @ R.T + t
    return dict(ref_imgs=imgs, ref_img_index=(np.arange(n) % len(imgs)).astype(np.int32), ref_px=np.ascontiguousarray(S.cam_project(b["cam_cfg"], pc)),
                ref_f=np.ascontiguousarray(pc / np.linalg.norm(pc, axis=1, keepdims=True)), ref_R=np.tile(R.reshape(1, 9), (n, 1)), ref_pos=np.tile(-R.T @ t, (n, 1)))


def test_inverse_compositional_at_the_border_with_three_reference_images(gpu_ctx):
    b, prior = _border("640x512")
    imgs = [b["img"], b["img_ref"], _third_image(b["img"])]
    refs = _inverse_refs_at_the_border(b, prior, imgs)
    assert np.any(refs["ref_px"] < 0) and np.any(refs["ref_px"][:, 0] > b["cam_cfg"].width - 1)
    inv_cfg = dataclasses.replace(b["vio_cfg"], inverse_composition_en=True)
    n = len(b["vis_pos"])
    args = (b["img"], b["vis_pos"], b["warp_patch"], b["search_levels"], np.ones(n), prior, prior)
    vio = O.OracleVIO(b["cam_cfg"], b["ext"], b["vio_cfg"])
    vio.set_inverse_refs(**refs)
    vio.set_inverse(True)
    o = vio.update(*args)
    assert o["total_iters"] >= 3
    try:
        _setup(gpu_ctx, b)
        gpu_ctx.vio_set_ref_images(imgs)
        gpu_ctx.vio_set_camera(b["cam_cfg"], inv_cfg)
        gpu_ctx.vio_set_inverse_refs(refs["ref_img_index"], refs["ref_px"], refs["ref_f"], refs["ref_R"], refs["ref_pos"])
        g2, g0 = _run_modes(gpu_ctx, args, (2, 0))
        # new reference images invalidate the reference features (their indices pointed into the released images)
        swapped = [imgs[1], imgs[2], imgs[0]]
        gpu_ctx.vio_set_ref_images(swapped)
        for mode in (2, 0):
            with pytest.raises(api.EsikfError):
                _run_modes(gpu_ctx, args, (mode,))
        gpu_ctx.vio_set_inverse_refs(refs["ref_img_index"], refs["ref_px"], refs["ref_f"], refs["ref_R"], refs["ref_pos"])
        gs = _run_modes(gpu_ctx, args, (2,))[0]
    finally:
        gpu_ctx.set_loop_mode(api.DEFAULT_LOOP_MODE)
        gpu_ctx.vio_set_camera(b["cam_cfg"], b["vio_cfg"])
        gpu_ctx.vio_set_ref_images([b["img_ref"]])
    L = b["vio_cfg"].levels
    _compare_vio(g2, o, L)
    _compare_vio(g0, o, L)
    _bits_equal(g0, g2, VIO_KEYS)
    vio.set_inverse_refs(**dict(refs, ref_imgs=swapped))
    _compare_vio(gs, vio.update(*args), L)


# ---------------------------------------------------------------------------------------------------------------- work split
def _sm_count():
    import torch

    return min(torch.cuda.get_device_properties(0).multi_processor_count, 160)  # partial_blocks caps the grid at 160


@pytest.mark.parametrize("per_cta", ["16S", "16S+1", "32S", "32S+1"])
def test_vio_patch_counts_at_the_work_split_edges_match_oracle(gpu_ctx, per_cta):
    """A CTA of the persistent kernel keeps its patches cached across iterations while its slice holds at most
    16 warps x VIO_KMAX = 32 patches: 16 S -> one per warp, 16 S + 1 -> the second slot comes into use, 32 S -> full,
    32 S + 1 -> uncached (slot 0 refilled per patch). The border frame's patches repeated to the count."""
    S_ = _sm_count()
    k, plus = per_cta.split("S")
    n = int(k) * S_ + (1 if plus else 0)
    b, prior = _border("640x512")
    _setup(gpu_ctx, b)
    rep = np.arange(n) % len(b["vis_pos"])
    args = (b["img"], b["vis_pos"][rep], b["warp_patch"][rep], b["search_levels"][rep], b["inv_ref_expo"][rep], prior, prior)
    g2, g0 = _run_modes(gpu_ctx, args, (2, 0))
    o = _oracle(b, *args)
    L = b["vio_cfg"].levels
    _compare_vio(g2, o, L)
    _bits_equal(g0, g2, VIO_KEYS)


LIO_COUNTS = ["32S-1", "32S", "32S+1", "704S-31", "704S", "704S+1", "704S+33"]


def _lio_n(label, S_):
    k, rest = label.split("S")
    return int(k) * S_ + int(rest or 0)


def _lio_slices(n, S_):
    """Points per CTA of lio_block_range: 32-point chunks dealt over min(S, chunks) CTAs."""
    chunks = (n + 31) // 32
    g = min(S_, chunks)
    q, r = divmod(chunks, g)
    return [min(32 * (q + (c < r)), n - 32 * (c * q + min(c, r))) for c in range(g)]


@functools.lru_cache(maxsize=None)
def _lio_frame():
    # points for the largest count at the 160-CTA cap; every count is a prefix of the same scan
    return get_frame(seed=0, n_pts=704 * 160 + 64, n_map=1_000_000)


def test_lio_counts_cover_a_launch_with_resident_and_tiled_ctas():
    for S_ in (148, 160):
        kinds = [{s <= 704 for s in _lio_slices(_lio_n(lab, S_), S_)} for lab in LIO_COUNTS]
        assert {True, False} in kinds  # some CTAs keep their slice resident while others walk tiles
        assert {True} in kinds and {False} not in kinds


@pytest.mark.parametrize("label", LIO_COUNTS)
def test_lio_point_counts_at_the_work_split_edges_match_oracle(gpu_ctx, label):
    """lio_block_range deals 32-point chunks over min(S, chunks) CTAs; a CTA whose slice fits its 704 lanes keeps points,
    slots and outputs resident and writes the per-point outputs once at the end, a larger slice walks tiles and writes them
    every iteration. 704 S + 1 / + 33: one / two tiled CTAs next to resident ones in the same launch."""
    from test_gpu_lio import _compare

    S_ = _sm_count()
    n = _lio_n(label, S_)
    fr = _lio_frame()
    assert len(fr["pts"]) >= n
    pts = np.ascontiguousarray(fr["pts"][:n])
    cfg = fr["lio_cfg"]
    gpu_ctx.set_extrinsics(fr["ext"])
    gpu_ctx.map_upload(fr["map"], cfg.voxel_size)
    out = []
    try:
        for mode, tune in ((2, 0), (0, 0), (2, api.TUNE_STAGE_LDG)):
            gpu_ctx.set_loop_mode(mode)
            gpu_ctx.set_tuning(tune)
            out.append(gpu_ctx.lio_update(pts, fr["state_prior"], fr["state_prior"], cfg))
    finally:
        gpu_ctx.set_tuning(0)
        gpu_ctx.set_loop_mode(api.DEFAULT_LOOP_MODE)
    lio = O.OracleLIO(cfg, fr["ext"])
    lio.set_map(fr["map"])
    o = lio.state_estimation(pts, fr["state_prior"], fr["state_prior"])
    g2, g0, gl = out
    _compare(g2, o)  # association / distances bit-exact for every point, those of the tiled CTAs included
    assert g0["iters"] == g2["iters"] == gl["iters"]
    _bits_equal(g0, g2, LIO_KEYS)
    _bits_equal(gl, g2, LIO_KEYS)
    slices = _lio_slices(n, S_)
    tiled = np.repeat([s > 704 for s in slices], slices)
    if tiled.any():  # the tiled CTAs' points are matched too (not just left at their initial values)
        assert np.count_nonzero(o["match_plane"][tiled] >= 0) > 0.5 * np.count_nonzero(tiled)


# ---------------------------------------------------------------------------------------------------------------- input checks
def test_search_levels_outside_0_to_8_are_rejected(gpu_ctx, small_vio_frame):
    """Checked on the host before anything is launched (TMA off: even without the check only the bounds-checked per-lane
    loads would run); a valid update afterwards is unaffected."""
    fr = small_vio_frame
    _setup(gpu_ctx, fr)
    prior = _vio_prior(fr)
    w = O.oracle_warp_patches(fr, prior)
    args = lambda sl: (fr["img"], fr["vis_pos"], w["warp_patch"], sl, fr["inv_ref_expo"], prior, prior)
    gpu_ctx.set_tuning(0)
    for bad in (-1, 9, 1 << 30):
        sl = w["search_levels"].copy()
        sl[len(sl) // 2] = bad
        with pytest.raises(api.EsikfError, match="search level"):
            gpu_ctx.vio_update(*args(sl))
        with pytest.raises(api.EsikfError, match="search level"):
            gpu_ctx.vio_set_patches(fr["vis_pos"], w["warp_patch"], sl, fr["inv_ref_expo"])
    g = gpu_ctx.vio_update(*args(w["search_levels"]))
    _compare_vio(g, _oracle(fr, *args(w["search_levels"])), fr["vio_cfg"].levels)


# ---------------------------------------------------------------------------------------------------------------- reference source
def test_vio_wrapping_footprints_match_reference_source_outputs(gpu_ctx):
    """The CUDA path against the REFERENCE SOURCE's stored outputs (tests/golden/ref_vio_pins.npz, `edge_wrap`): footprints
    crossing the left / right edges wrap to the neighbouring row in both (DESIGN §4), in the update and in getImagePatch."""
    from parity_util import assert_state_close, digest, load_golden
    from test_oracle_ref_pin_vio import PINS, edge_wrap_inputs

    b, prior, _, centres = edge_wrap_inputs()
    ref = load_golden(PINS, "edge_wrap")
    assert digest(b["warp_patch"]) == ref["warp_patch"]
    _setup(gpu_ctx, b)
    for g in _run_modes(gpu_ctx, _args(b, prior), (2, 0)):
        assert_state_close(g["state"], ref["state"], rot_tol=1e-8, pos_tol=1e-8, cov_tol=1e-6, rest_tol=1e-8)
        np.testing.assert_allclose(g["errors"], ref["errors"], rtol=2e-6, atol=1e-3)
    got = np.array([[digest(p) for p in gpu_ctx.vio_get_image_patch(centres, lvl)] for lvl in range(b["vio_cfg"].levels)]).T
    assert (got == ref["image_patch"]).all()

"""GPU: a context torn down with every buffer populated, and contexts that keep working after an entry point failed.

One sequence touches every kind of context-owned device memory: both arenas of the device-resident map (init, build,
update, slide, download), the LIO scan buffers, two sets of reference images (the first released by the second), the
warped patches kept on the device, the inverse-compositional references, the warpAffine / getImagePatch scratch, and the
timing events of a per-iteration update. Run on fresh contexts and on a context that has just returned an error, it
must give the same bits every time."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

import map_bind as MB
import oracle_bind as O
from fast_livo2_b200 import api
from fast_livo2_b200 import synthetic as S
from test_gpu_vio import _vio_prior
from test_map_host import _tick_points

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _need_gpu():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _sequence(ctx, fr):
    """The whole sequence on `ctx`; returns every array it produced (maps as flat downloads)."""
    cfg, vio_cfg = fr["lio_cfg"], fr["vio_cfg"]
    out = {}
    ctx.set_loop_mode(2)
    ctx.set_kernel_timing(False)
    ctx.set_extrinsics(fr["ext"])
    # device-resident map: build from the scan, absorb more points, slide to the inner part of the scan's footprint
    ctx.map_device_init(cfg, root_capacity=1 << 16)
    ctx.lio_set_scan(fr["pts"])
    ctx.map_device_build(fr["state_prior"])
    out["map_built"] = ctx.map_device_download()
    keys = out["map_built"]["keys"]
    lo, hi = np.percentile(keys, 10, axis=0).astype(np.int64), np.percentile(keys, 90, axis=0).astype(np.int64)
    pw, var = _tick_points(np.random.default_rng(4), S.make_scene("room", 0.5), 3000, np.array([-12.0, -9.0, -3.0]), np.array([12.0, 9.0, 5.0]))
    ctx.map_device_update_points(pw, var)
    roots_before = ctx.map_device_stats()["roots"]
    ctx.map_device_slide(lo, hi)
    assert 0 < ctx.map_device_stats()["roots"] < roots_before
    out["map_slid"] = ctx.map_device_download()
    # LIO on the device map
    g = ctx.lio_update(fr["pts"], fr["state_prior"], fr["state_prior"], cfg)
    assert g["M"][0] > 0
    out["lio_state"], out["lio_M"], out["lio_dis"] = g["state"], g["M"], g["dis_to_plane"]
    # record ids depend on the order the map kernels allocated them in: compare the association by what it points at
    out["lio_matched"], out["lio_has_normal"] = g["match_plane"] >= 0, g["normal_plane"] >= 0
    out["lio_normals"] = ctx.lio_fetch_normals()
    out["body_cov"], out["cross_mat"] = ctx.lio_fetch_point_cov()
    # VIO: the second set of reference images replaces (and releases) the first
    ctx.vio_set_camera(fr["cam_cfg"], vio_cfg)
    ctx.vio_set_image(fr["img"])
    ctx.vio_set_ref_images([fr["img"], fr["img_ref"], fr["img"]])
    ctx.vio_set_ref_images([fr["img_ref"]])
    prior = _vio_prior(fr)
    st = S.unpack_state(prior)
    n = len(fr["vis_pos"])
    T_cur = api.pack_T(*S.camera_pose(fr["ext"], st["R"], st["p"]))
    T_ref = np.tile(api.pack_T(*fr["T_ref"]), (n, 1))
    w = ctx.vio_warp_patches(np.zeros(n, np.int32), fr["px_ref"], fr["vis_pos"], fr["vis_normal"], T_ref, T_cur, keep_on_device=True)
    out.update(warp_A=w["A_cur_ref"], warp_levels=w["search_levels"], warp_patch=w["warp_patch"])
    refs = O.inverse_refs_from_frame(fr)
    ctx.vio_set_camera(fr["cam_cfg"], dataclasses.replace(vio_cfg, inverse_composition_en=True))
    ctx.vio_set_inverse_refs(refs["ref_img_index"], refs["ref_px"], refs["ref_f"], refs["ref_R"], refs["ref_pos"])
    ctx.vio_run(prior, prior)
    v = ctx.vio_fetch()
    assert v["total_iters"] > 0
    out["inv_state"], out["inv_errors"] = v["state"], v["errors"]
    ctx.vio_set_camera(fr["cam_cfg"], vio_cfg)
    out["affine"] = ctx.vio_warp_affine(np.zeros(n, np.int32), fr["px_ref"], w["A_cur_ref"], w["search_levels"])
    out["image_patch"] = ctx.vio_get_image_patch(fr["px_ref"][:64], 1)
    # one per-iteration update with kernel timing (the timing events are created on demand and owned by the context)
    ctx.set_loop_mode(0)
    ctx.set_kernel_timing(True)
    ctx.vio_run(prior, prior)
    v = ctx.vio_fetch()
    out["fwd_state"], out["fwd_errors"] = v["state"], v["errors"]
    assert ctx.get_kernel_timing()["vio_patch_ms"][0] > 0
    return out


def _fresh(fr):
    ctx = api.Context(0)
    try:
        return _sequence(ctx, fr)
    finally:
        ctx.close()


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if k.startswith("map_"):
            MB.compare_flat_maps(a[k], b[k], exact=True, what=(k, k))
        else:
            assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k


def test_three_fresh_contexts_give_the_same_bits(small_vio_frame):
    rounds = [_fresh(small_vio_frame) for _ in range(3)]
    for r in rounds[1:]:
        _assert_same(rounds[0], r)


def test_error_paths_leave_the_context_usable(small_vio_frame):
    fr = small_vio_frame
    ref = _fresh(fr)
    ctx = api.Context(0)
    try:
        with pytest.raises(api.EsikfError, match="no resident LIO frame"):
            ctx.profile_kernel(0, reps=2, flush_l2=False)
        with pytest.raises(api.EsikfError, match="no resident VIO frame"):
            ctx.profile_kernel(2, reps=2, flush_l2=False)
        with pytest.raises(api.EsikfError, match="which=7"):
            ctx.profile_kernel(7, reps=2, flush_l2=False)
        _assert_same(ref, _sequence(ctx, fr))
        # the map has far more than one root: a one-root buffer is rejected after the device-side count
        keys, first, count = np.zeros((1, 3), np.int64), np.zeros(1, np.int32), np.zeros(1, np.int32)
        planes = np.zeros(1 << 16, S.PLANE_DTYPE)
        nr, npl = C.c_int32(0), C.c_int32(0)
        rc = ctx.lib.esikf_map_device_download(ctx.h, keys.ctypes.data, first.ctypes.data, count.ctypes.data, 1, planes.ctypes.data, len(planes), C.byref(nr),
                                               C.byref(npl))
        assert rc != 0 and "do not fit" in ctx.lib.esikf_last_error(ctx.h).decode() and nr.value > 1
        _assert_same(ref, _sequence(ctx, fr))
    finally:
        ctx.close()

"""Pins the VIO oracle (oracle/orc_vio.cpp, a restatement) against the REFERENCE'S OWN SOURCE: FAST-LIVO2's src/vio.cpp (+
frame.cpp, visual_point.cpp) compiled against stand-in headers (oracle/ref_shim/: matrix library, cv::Mat, Sophus::SE3,
boost::noncopyable, PCL / ROS shells; oracle/ref_vio.cpp -> oracle/_ref/libfl2_ref_vio.so).

What this pins: everything VIOManager::computeJacobianAndUpdateEKF -> updateState (projection, bilinear weights, taps, the
Jacobian chain, H^T H, the gain, boxplus, the error-gated accept / rollback, P -= G P), the inverse-compositional variant
(precomputeReferencePatches, updateStateInverse), getImagePatch, warpAffine, getWarpMatrixAffineHomography / getBestSearchLevel
compute — the reference's own arithmetic. What it cannot pin: vikit (un-vendored, no version pin): the pinhole model and
vk::interpolateMat_8u inside the stand-in are restatements of the published algorithm, shared by both sides.

The reference's outputs are stored in tests/golden/ref_vio_pins.npz (and tests/golden/ref_vio_golden.npz), so the pin holds on
machines without the FAST-LIVO2 sources; tests/golden/make_ref_golden.py regenerates them from oracle/_ref/. Patches that must
agree bit for bit are stored as SHA-256 digests (parity_util.digest)."""
import dataclasses
import os

import numpy as np
import pytest

import oracle_bind as O
from conftest import get_frame
from fast_livo2_b200 import synthetic as S
from parity_util import assert_state_close, digest, load_golden

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vio_golden.npz")
PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vio_pins.npz")

CASES = {
    "small": dict(seed=2, n_pts=2000, n_map=120_000, n_patches=150, scene_scale=0.5),
    "exposure": dict(seed=6, n_pts=1000, n_map=120_000, n_patches=200, scene_scale=0.5, vio=S.VioCfg(exposure_estimate_en=True)),
    "three_levels": dict(seed=8, n_pts=1000, n_map=120_000, n_patches=300, scene_scale=0.5, vio=S.VioCfg(levels=3, img_point_cov=400.0)),
    "distorted_pinhole": dict(seed=9, n_pts=1000, n_map=120_000, n_patches=200, scene_scale=0.5,
                              cam=S.CamCfg(d=(-0.05, 0.02, 0.001, -0.0005, 0.0))),
    # config 3's camera (HILTI22 fisheye, vk::EquidistantCamera) behind the same abstract interface
    "fisheye": dict(seed=10, n_pts=1000, n_map=120_000, n_patches=200, scene_scale=0.5, vio=S.VioCfg(img_point_cov=1000.0),
                    cam=S.CamCfg(model=1, width=720, height=540, fx=351.31400364193297, fy=351.4911744656785, cx=367.8522793375995, cy=253.8402144980996,
                                 d=(-0.03696737352869157, -0.008917880497032812, 0.008912969593422046, -0.0037685977496087313, 0.0))),
}


def _prior(fr, seed=3):
    rng = np.random.default_rng(seed)
    t = S.unpack_state(fr["state_true"])
    return S.pack_state(t["R"] @ S.so3_exp(rng.normal(0, np.deg2rad(0.15), 3)), t["p"] + rng.normal(0, 0.01, 3), 1.0 + rng.normal(0, 0.01), t["v"], g=t["g"],
                        cov=S.random_prior_cov(rng, scale=0.2))


def _inputs(name):
    fr = get_frame(**CASES[name])
    prior = _prior(fr)
    w = O.oracle_warp_patches(fr, prior)
    return fr, prior, w


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_vio_update_reproduces_the_reference_source(name):
    fr, prior, w = _inputs(name)
    args = (fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], fr["inv_ref_expo"], prior, prior)
    ref = load_golden(PINS, f"update.{name}")
    assert digest(w["warp_patch"]) == ref["warp_patch"]  # same inputs as when the reference's outputs were stored
    orc = O.OracleVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"]).update(*args)
    assert orc["total_iters"] >= 4
    # same decisions (accept / rollback / stop) or the states would differ grossly; the sums differ only in association order
    assert_state_close(orc["state"], ref["state"], rot_tol=1e-11, pos_tol=1e-11, cov_tol=1e-9, rest_tol=1e-11)
    # per-patch photometric error: float accumulation in both, same order (one thread)
    np.testing.assert_allclose(orc["errors"], ref["errors"], rtol=1e-6, atol=1e-4)
    # the H_T_H member (vio.h:121) holds the normal matrix of the last ACCEPTED iteration: one of the oracle's per-iteration blocks
    blocks = orc["HTH"].reshape(-1, 7, 7)
    blocks = blocks[np.abs(blocks).max(axis=(1, 2)) > 0]
    want = ref["H_T_H"][:7, :7]
    rel = [np.abs(b - want).max() / np.abs(want).max() for b in blocks]
    assert min(rel) < 1e-10, min(rel)


def test_oracle_inverse_compositional_variant_reproduces_the_reference_source():
    fr, prior, w = _inputs("small")
    refs = O.inverse_refs_from_frame(fr)
    n = len(fr["vis_pos"])
    args = (fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], np.ones(n))
    ref = load_golden(PINS, "inverse")
    assert digest(w["warp_patch"]) == ref["warp_patch"]
    vio = O.OracleVIO(fr["cam_cfg"], fr["ext"], dataclasses.replace(fr["vio_cfg"], inverse_composition_en=True))
    vio.set_inverse_refs(**refs)
    vio.set_inverse(True)
    orc = vio.update(*args, prior, prior)
    assert_state_close(orc["state"], ref["state"], rot_tol=1e-11, pos_tol=1e-11, cov_tol=1e-9, rest_tol=1e-11)
    np.testing.assert_allclose(orc["errors"], ref["errors"], rtol=1e-6, atol=1e-4)


def patch_producer_calls(vio, ref=None):
    """getWarpMatrixAffineHomography + getBestSearchLevel, warpAffine and getImagePatch of `vio` (the oracle or the reference)
    on every 7th patch of the distorted-pinhole case: per patch the warp matrix, its search level, the digest of the reference
    patch warped with the REFERENCE's matrix and level (`ref`'s stored ones, else vio's own) and the digests of a current
    image patch at every pyramid level."""
    fr, prior, w = _inputs("distorted_pinhole")
    st = S.unpack_state(prior)
    T_cur = S.camera_pose(fr["ext"], st["R"], st["p"])
    rng = np.random.default_rng(1)
    for k, i in enumerate(range(0, len(fr["vis_pos"]), 7)):
        A, sl = vio.warp_matrix(fr["px_ref"][i], fr["vis_pos"][i], fr["vis_normal"][i], fr["T_ref"], T_cur)
        Ar, sr = (A, sl) if ref is None else (ref["A"][k], int(ref["search_level"][k]))
        warp = digest(vio.warp_affine(fr["img_ref"], Ar, fr["px_ref"][i], sr))
        pc = np.array([rng.uniform(40, fr["cam_cfg"].width - 40), rng.uniform(40, fr["cam_cfg"].height - 40)])
        yield A, sl, warp, [digest(vio.get_image_patch(fr["img"], pc, lvl)) for lvl in range(fr["vio_cfg"].levels)]


def test_oracle_patch_producers_reproduce_the_reference_source():
    """getImagePatch, getWarpMatrixAffineHomography + getBestSearchLevel, warpAffine (vio.cpp:203-331)."""
    fr = _inputs("distorted_pinhole")[0]
    ref = load_golden(PINS, "patch")
    orc = O.OracleVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"])
    k = -1
    for k, (Ao, so, warp, patches) in enumerate(patch_producer_calls(orc, ref)):
        assert int(ref["search_level"][k]) == so
        np.testing.assert_allclose(Ao, ref["A"][k], rtol=1e-11, atol=1e-13)
        assert warp == ref["warp_affine"][k], f"warpAffine of patch {7 * k} differs"
        assert patches == ref["image_patch"][k].tolist(), f"getImagePatch of sample {k} differs"
    assert k + 1 == len(ref["A"])


def test_oracle_matches_reference_vio_golden():
    """The reference library's own outputs, committed: the pin survives where the library cannot be built."""
    if not os.path.exists(GOLDEN):
        pytest.skip("tests/golden/ref_vio_golden.npz not generated")
    g = np.load(GOLDEN, allow_pickle=False)
    for name in ("small", "exposure"):
        fr, prior, w = _inputs(name)
        np.testing.assert_array_equal(w["warp_patch"], g[f"{name}_warp_patch"])  # same inputs as when the vectors were made
        orc = O.OracleVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"]).update(fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], fr["inv_ref_expo"], prior, prior)
        assert_state_close(orc["state"], g[f"{name}_state"], rot_tol=1e-11, pos_tol=1e-11, cov_tol=1e-9, rest_tol=1e-11)
        np.testing.assert_allclose(orc["errors"], g[f"{name}_errors"], rtol=1e-6, atol=1e-4)


def edge_wrap_inputs():
    """The "small" frame with visual points whose tap footprints cross the LEFT and RIGHT image edges at every tap stride
    1 .. 32 (parity_util.border_frame: one stride inside, on the edge column, one stride past, half outside), rows kept to
    h/2 +- 50. There the reference's raw linear-index reads (img.data + v * width + u) wrap to the neighbouring row, which is
    defined behaviour as long as every index stays inside [0, width * height): asserted here for every patch at every
    pyramid level at the prior and at the oracle's posterior, with 8 rows to spare for the iterates in between. Returns
    (frame, prior, oracle update, getImagePatch centres)."""
    from parity_util import border_frame, tap_origin

    fr = get_frame(**CASES["small"])
    prior = _prior(fr)
    cam, L = fr["cam_cfg"], fr["vio_cfg"].levels
    b = border_frame(fr, prior, seed=21, n_interior=0, edges=("left", "right"), corners=False, outside=False, rows=(cam.height / 2 - 50, cam.height / 2 + 50))
    o = O.OracleVIO(cam, fr["ext"], fr["vio_cfg"]).update(b["img"], b["vis_pos"], b["warp_patch"], b["search_levels"], b["inv_ref_expo"], prior, prior)
    w, h = cam.width, cam.height
    crosses = np.zeros(len(b["vis_pos"]), bool)
    for state in (prior, o["state"]):
        for level in range(L):
            s = 1 << (level + b["search_levels"].astype(np.int64))
            x0, y0 = tap_origin(cam, fr["ext"], state, b["vis_pos"], s)
            assert np.all(y0 * w + x0 >= 8 * w) and np.all((y0 + 10 * s) * w + x0 + 10 * s < (h - 8) * w), "a footprint leaves the buffer"
            crosses |= (x0 < 0) | (x0 + 10 * s >= w)
    assert crosses.mean() > 0.5
    return b, prior, o, b["bp_px"]


def edge_wrap_image_patches(vio, img, centres, levels):
    """Digests of getImagePatch at every pyramid level for centres on the left / right edges (wrapping footprints)."""
    return np.array([[digest(vio.get_image_patch(img, c, lvl)) for lvl in range(levels)] for c in centres])


def test_oracle_reproduces_the_reference_source_where_footprints_wrap_rows():
    """Left / right border footprints at tap strides up to 32: the oracle's linear-index reads (pix()) against the reference
    source's raw img.data reads, through the whole update and through getImagePatch."""
    b, prior, orc, centres = edge_wrap_inputs()
    ref = load_golden(PINS, "edge_wrap")
    assert digest(b["warp_patch"]) == ref["warp_patch"] and np.array_equal(b["search_levels"], ref["search_levels"])
    assert orc["total_iters"] >= 4
    assert_state_close(orc["state"], ref["state"], rot_tol=1e-11, pos_tol=1e-11, cov_tol=1e-9, rest_tol=1e-11)
    np.testing.assert_allclose(orc["errors"], ref["errors"], rtol=1e-6, atol=1e-4)
    vio = O.OracleVIO(b["cam_cfg"], b["ext"], b["vio_cfg"])
    assert (edge_wrap_image_patches(vio, b["img"], centres, b["vio_cfg"].levels) == ref["image_patch"]).all()


BASELINE_COUNTS = {  # per-iteration matched points / VIO iterations the CUDA bench lines report for these frames (profiles/bench_r02_*)
    "cfg2": ([99663, 99869, 99883, 99892, 99896], 18),
    "cfg3": (None, -1),  # HILTI fisheye + corridor scene: no CUDA bench line this round, the pin itself is what is checked
    "cfg4": ([259473, 259653, 259654, 259637, 259637], None),
    "cfg5": ([299848, 299903, 299906, 299902, 299902], 13),
}


@pytest.mark.parametrize("name", ["cfg2", "cfg3", "cfg4", "cfg5"])
def test_oracle_reproduces_the_reference_source_on_the_baseline_configs(name):
    """The frames bench.py times (BASELINE config 2: 100 k points against a 1 M-point map + 2 000 patches; config 4: 260 k
    points; config 5: 300 k points + 4 000 patches, 5 levels, voxel 2.0): VoxelMapManager::StateEstimation and
    VIOManager::computeJacobianAndUpdateEKF of the REFERENCE SOURCE against the oracle — the per-iteration matched counts the
    CUDA path reports in its bench lines, posteriors and per-patch errors. The VIO update of both starts from the oracle's LIO
    posterior as it was when the reference's outputs were stored (`vio_prior`)."""
    from fast_livo2_b200 import workloads as W

    fr = W.frame(name)
    want_M, want_vio = BASELINE_COUNTS[name]
    r = load_golden(PINS, f"baseline.{name}")
    lio = O.OracleLIO(fr["lio_cfg"], fr["ext"])
    lio.set_map(fr["map"])
    o = lio.state_estimation(fr["pts"], fr["state_prior"], fr["state_prior"])
    assert o["iters"] == r["iters"] and np.array_equal(o["M"], r["M"]) and (want_M is None or o["M"].tolist() == want_M)
    assert_state_close(o["state"], r["state"], rot_tol=1e-12, pos_tol=1e-12, cov_tol=1e-10, rest_tol=1e-12)
    if want_vio is None:
        return
    w = O.oracle_warp_patches(fr, r["vio_prior"])
    assert digest(w["warp_patch"]) == r["vio_warp_patch"]  # same inputs as when the reference's outputs were stored
    args = (fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], fr["inv_ref_expo"], r["vio_prior"], r["vio_prior"])
    rv = dict(state=r["vio_state"], errors=r["vio_errors"])
    ov = O.OracleVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"]).update(*args)
    assert want_vio < 0 or ov["total_iters"] == want_vio
    assert_state_close(ov["state"], rv["state"], rot_tol=1e-11, pos_tol=1e-11, cov_tol=1e-9, rest_tol=1e-11)
    np.testing.assert_allclose(ov["errors"], rv["errors"], rtol=1e-6, atol=1e-4)

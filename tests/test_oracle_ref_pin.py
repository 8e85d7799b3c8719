"""Pins the LIO oracle (oracle/orc_lio.cpp, a restatement) against the REFERENCE'S OWN SOURCE: FAST-LIVO2's src/voxel_map.cpp
compiled against stand-in headers for Eigen / PCL / ROS (oracle/ref_shim/, oracle/ref_voxel_map.cpp ->
oracle/_ref/libfl2_ref_lio.so). The reference ships no tests or golden vectors of its own; its compiled update loop
(VoxelMapManager::StateEstimation with BuildResidualListOMP / build_single_residual, OpenMP on) is the next best thing.

The oracle must reproduce the reference source on every case below: iteration count, effective feature number per iteration
(parsed from the reference's own console line), the final ptpl_list_ (matched plane centres and signed distances, in order),
pv.normal of every point — all bit-exact — and the posterior state / covariance to 1e-12 (the two differ only in the
summation order of small fixed-size products). The reference's outputs are stored in tests/golden/ref_lio_pins.npz (and, in
full for two cases, tests/golden/ref_lio_golden.npz), so the pin holds on machines without the FAST-LIVO2 sources;
tests/golden/make_ref_golden.py regenerates them from oracle/_ref/ (make -C oracle REF=<FAST-LIVO2 source tree>). Per-point
arrays and map structures are stored as SHA-256 digests (parity_util.digest) and the map tests keep every root's structure
and a seeded sample of roots' plane records (map_bind.map_record)."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_bind as O
from conftest import get_frame
from fast_livo2_b200 import synthetic as S
from parity_util import digest, load_golden

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_lio_golden.npz")
PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_lio_pins.npz")

CASES = {
    "small": dict(frame=dict(seed=1, n_pts=4000, n_map=150_000, scene_scale=0.5)),
    "seed3": dict(frame=dict(seed=3, n_pts=5000, n_map=150_000, scene_scale=0.5)),
    "20k": dict(frame=dict(seed=4, n_pts=20000, n_map=150_000, scene_scale=0.5)),
    "three_iterations": dict(frame=dict(seed=0, n_pts=5000, n_map=150_000, scene_scale=0.5), cfg=dict(max_iterations=3)),
    "hilti_voxel_04_non_identity_extrinsics": dict(frame=dict(seed=5, n_pts=6000, n_map=400_000, lio=S.LioCfg(voxel_size=0.4, min_eigen_value=1e-4, max_points_num=100),
                                                            ext=S.hilti_extrinsics(), scene="corridor", scene_scale=0.25)),
    "voxel_2m": dict(frame=dict(seed=7, n_pts=6000, n_map=300_000, lio=S.LioCfg(voxel_size=2.0, min_eigen_value=0.005), scene_scale=2.0)),
}


EDGE_FRAMES = {
    "voxel_0.5": dict(seed=1, n_pts=4000, n_map=150_000, scene_scale=0.5),
    "voxel_0.4": dict(seed=5, n_pts=6000, n_map=400_000, lio=S.LioCfg(voxel_size=0.4, min_eigen_value=1e-4, max_points_num=100), ext=S.hilti_extrinsics(), scene="corridor",
                      scene_scale=0.25),
    "voxel_2.0": dict(seed=7, n_pts=6000, n_map=300_000, lio=S.LioCfg(voxel_size=2.0, min_eigen_value=0.005), scene_scale=2.0),
}


def _case(name):
    c = CASES[name]
    fr = get_frame(**c["frame"])
    cfg = fr["lio_cfg"]
    if "cfg" in c:
        cfg = S.LioCfg(**{**cfg.__dict__, **c["cfg"]})
    return fr, cfg


def _oracle(fr, cfg, state_in=None):
    lio = O.OracleLIO(cfg, fr["ext"])
    lio.set_map(fr["map"])
    s = fr["state_prior"] if state_in is None else state_in
    return lio.state_estimation(fr["pts"], s, fr["state_prior"])


def lio_record(r):
    """A StateEstimation result of the reference source as stored in tests/golden/ref_lio_pins.npz: iteration count, matched
    counts and state in full, the per-point arrays as digests."""
    return dict(iters=np.int32(r["iters"]), M=np.asarray(r["M"], np.int32), state=np.asarray(r["state"]), n_ptpl=np.int32(len(r["ptpl_dis"])),
                ptpl_center=np.str_(digest(r["ptpl_center"])), ptpl_dis=np.str_(digest(r["ptpl_dis"])), normals=np.str_(digest(r["normals"])))


def _check(o, r, planes):
    assert o["iters"] == r["iters"]
    assert np.array_equal(o["M"], r["M"])  # effective feature number of every iteration
    mk = o["match_plane"] >= 0
    assert mk.sum() == r["n_ptpl"]
    # ptpl_list_ keeps the scan order of the matched points: plane by plane and distance by distance
    assert digest(planes["center"][o["match_plane"][mk]]) == r["ptpl_center"], "matched plane centres (ptpl_list_) differ"
    assert digest(o["dis_to_plane"][mk]) == r["ptpl_dis"], "point-to-plane distances (ptpl_list_) differ"
    want = np.where(o["normal_plane"][:, None] >= 0, planes["normal"][np.maximum(o["normal_plane"], 0)], 0.0)
    assert digest(want) == r["normals"], "pv.normal differs"  # zero when the point never matched
    d = np.abs(o["state"] - r["state"])
    assert d[:25].max() <= 1e-12 * max(1.0, np.abs(r["state"][:25]).max())
    assert d[25:].max() <= 1e-12 * np.abs(r["state"][25:]).max()


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_reproduces_the_reference_source(name):
    fr, cfg = _case(name)
    o = _oracle(fr, cfg)
    r = load_golden(PINS, name)
    assert r["iters"] >= 2
    _check(o, r, fr["map"]["planes"])


def early_stop_frame():
    """A tight prior converges twice in a row: the rematch / stop rule (voxel_map.cpp:477-499) ends the loop after 2 iterations."""
    fr, cfg = _case("small")
    st = _oracle(fr, cfg)["state"].copy()
    st[25:] = (np.eye(19) * 1e-12).reshape(-1)
    return dict(fr, state_prior=st), cfg


def test_oracle_reproduces_the_reference_source_on_early_stop():
    fr2, cfg = early_stop_frame()
    o = _oracle(fr2, cfg)
    r = load_golden(PINS, "early_stop")
    assert r["iters"] == 2
    _check(o, r, fr2["map"]["planes"])


def edge_frame(kind):
    from parity_util import edge_scan

    fr = get_frame(**EDGE_FRAMES[kind])
    pts, ext, state = edge_scan(fr)
    return dict(fr, ext=ext, pts=pts, state_prior=state)


@pytest.mark.parametrize("kind", list(EDGE_FRAMES))
def test_edge_scan_oracle_reproduces_the_reference_source(kind):
    """Voxel corners / faces with both signs, float neighbours of them, z == 0 and off-plane points that exercise the
    neighbour rule (parity_util.edge_scan), for voxel sizes 0.5 / 0.4 / 2.0: oracle against the reference source."""
    fr2 = edge_frame(kind)
    lio = O.OracleLIO(fr2["lio_cfg"], fr2["ext"])
    lio.set_map(fr2["map"])
    o = lio.state_estimation(fr2["pts"], fr2["state_prior"], fr2["state_prior"])
    r = load_golden(PINS, f"edge_{kind}")
    assert o["M"][0] > 20
    # the neighbour rule is exercised: some points match a plane that is not in their own voxel's candidate list
    _check(o, r, fr2["map"]["planes"])


def body_cov_points():
    rng = np.random.default_rng(0)
    p = np.concatenate([rng.normal(0, 5, (50, 3)), [[1.0, 2.0, 0.001], [0.3, -0.2, 7.0]]])
    return np.ascontiguousarray(p.astype(np.float32).astype(np.float64))


def test_calc_body_cov_matches_the_reference_source():
    olib = O.load()
    want = load_golden(PINS, "body_cov")["cov"]
    for p, a in zip(body_cov_points(), want):
        b, cm = np.zeros(9), np.zeros(9)
        olib.orc_calc_body_cov(O.dptr(p.copy()), C.c_float(0.02), C.c_float(0.05), O.dptr(b), O.dptr(cm))
        np.testing.assert_allclose(b, a, rtol=1e-13, atol=1e-300)


@pytest.mark.parametrize("name", ["small", "hilti_voxel_04_non_identity_extrinsics"])
def test_oracle_matches_reference_golden(name):
    """Same check against the committed full outputs of the reference source (generated by tests/golden/make_ref_golden.py)."""
    g = np.load(GOLDEN)
    fr, cfg = _case(name)
    o = _oracle(fr, cfg)
    r = dict(iters=int(g[f"{name}_iters"]), M=g[f"{name}_M"], ptpl_center=g[f"{name}_ptpl_center"], ptpl_dis=g[f"{name}_ptpl_dis"], normals=g[f"{name}_normals"],
             state=g[f"{name}_state"])
    _check(o, lio_record(r), fr["map"]["planes"])


MAP_CFGS = {"avia_defaults": S.LioCfg(), "voxel0.4_layer3_max20": S.LioCfg(voxel_size=0.4, max_layer=3, max_points_num=20)}


def update_voxel_map_run(cfg, update, clear_out_of_map, flatten):
    """The tick sequence of test_oracle_update_voxel_map_reproduces_the_reference_source on one map (the oracle's or the
    reference's, through its three callables): yields (label, flattened map) after every tick and after the clearMemOutOfMap."""
    from test_map_host import _tick_points

    rng = np.random.default_rng(5)
    rects = S.make_scene("room", 0.5)
    for tick in range(8):
        lo = np.array([-10.0 + 1.5 * tick, -8.0, -2.0])
        pw, var = _tick_points(rng, rects, 6000, lo, lo + np.array([8.0, 16.0, 6.0]))
        update(pw, var)
        yield f"tick{tick}", flatten()
        if tick == 5:
            # mapSliding's clearMemOutOfMap (:950-971) in between, then more ticks on the pruned maps
            c, half = np.array([4, -2, 1]), 14
            assert clear_out_of_map([int(c[0] + half), int(c[0] - half), int(c[1] + half), int(c[1] - half), int(c[2] + half), int(c[2] - half)]) > 0
            yield "cleared", flatten()


@pytest.mark.parametrize("cfg_id", list(MAP_CFGS))
def test_oracle_update_voxel_map_reproduces_the_reference_source(cfg_id):
    """The map construction (f1's oracle): VoxelMapManager::UpdateVoxelMap / UpdateOctoTree / init_octo_tree / cut_octo_tree /
    init_plane of the REFERENCE SOURCE against the oracle's restatement, tick by tick on the same (point_w, var) lists: the same
    root voxels, the same octree shape (candidate planes per root in DFS order, layer / path), the plane's centre, normal,
    plane_var, d and radius of every plane of the sampled roots. Tolerance, not bits: the reference calls Eigen::EigenSolver,
    which in the stored outputs is the stand-in's Jacobi and in the oracle another Jacobi — a genuine Eigen would differ in the
    last bits just the same."""
    import map_bind as MB
    from test_map_host import _oracle_update

    cfg = MAP_CFGS[cfg_id]
    orc = O.OracleLIO(cfg, S.avia_extrinsics())
    n = 0
    for label, f in update_voxel_map_run(cfg, lambda pw, var: _oracle_update(orc, pw, var), lambda b: orc.lib.orc_lio_clear_out_of_map(orc.h, *b), orc.flatten):
        n = MB.compare_map_record(f, load_golden(PINS, f"map_update.{cfg_id}.{label}"), rtol=1e-9, what=(f"oracle ({label})", "reference source"))
        if label == "tick5":
            assert f["count"].max() > 1 and (f["planes"]["layer"] > 0).any()  # octrees were cut: several candidates per root
    assert n > 1500


def build_voxel_map_inputs():
    cfg, ext = S.LioCfg(), S.hilti_extrinsics()
    rng = np.random.default_rng(21)
    rects = S.make_scene("room", 0.5)
    R0, p0 = S.so3_exp(np.array([0.01, -0.02, 0.3])), np.array([-2.0, 0.5, 0.3])
    st0 = S.pack_state(R0, p0, cov=S.random_prior_cov(np.random.default_rng(3), scale=0.05), g=np.array([0, 0, -9.81]))
    scan = S.scan_at(rects, ext, R0, p0, 60000, cfg, rng)
    return cfg, ext, scan, st0


def test_oracle_build_voxel_map_reproduces_the_reference_source():
    """First LiDAR frame (LIVMapper.cpp:356-366): TransformLidar + BuildVoxelMap (per-point covariance with the raw body point's
    cross matrix and calcBodyCov's own z fix, all points pushed, then init_octo_tree with the recursive cut) of the REFERENCE
    SOURCE against the oracle's tick_build_map on a 60 k-point scan with non-identity extrinsics — the form the device map's
    esikf_map_device_build is held to."""
    import map_bind as MB

    cfg, ext, scan, st0 = build_voxel_map_inputs()
    orc = O.OracleLIO(cfg, ext)
    orc.tick_build_map(scan, st0)
    n = MB.compare_map_record(orc.flatten(), load_golden(PINS, "map_build"), rtol=1e-9, what=("oracle BuildVoxelMap", "reference source"))
    assert n > 1500

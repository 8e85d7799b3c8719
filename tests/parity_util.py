"""Shared comparison helpers for the GPU-vs-oracle parity tests."""
import numpy as np

import oracle_bind as O
from fast_livo2_b200 import synthetic as S

# north_star tolerance: "bit-identical for voxel indexing, within 1e-5 relative on the pose/covariance".
# The tests hold the CUDA path to much tighter bounds (fp64 reduction-order noise only).
POSE_RTOL = 1e-9
COV_RTOL = 1e-6
INFO_RTOL = 1e-10


def cov_rel_per_element(cov, ref):
    """Covariance error PER ELEMENT: |dP_ij| / sqrt(P_ii P_jj) — every entry, small cross-covariances included, against the
    scale of its own two variances (the north star's "1e-5 relative on the covariance" read element-wise, with the absolute
    floor a correlation-like normalisation gives: an exactly-zero reference entry is held to 1e-5 of sqrt(P_ii P_jj))."""
    d = np.sqrt(np.abs(np.diag(ref)))
    return float((np.abs(cov - ref) / np.maximum(np.outer(d, d), 1e-300)).max())


def pose_diff(a, b):
    ua, ub = S.unpack_state(a), S.unpack_state(b)
    rot = O.rot_err(ua["R"], ub["R"])
    pos = float(np.linalg.norm(ua["p"] - ub["p"]) / max(np.linalg.norm(ub["p"]), 1e-3))
    rest = float(np.abs(a[12:25] - b[12:25]).max())
    cov = cov_rel_per_element(ua["cov"], ub["cov"])
    return rot, pos, rest, cov


def assert_state_close(gpu, ref, rot_tol=POSE_RTOL, pos_tol=POSE_RTOL, cov_tol=COV_RTOL, rest_tol=1e-9):
    rot, pos, rest, cov = pose_diff(gpu, ref)
    assert rot < rot_tol, f"rotation differs by {rot} rad"
    assert pos < pos_tol, f"position differs by {pos} (relative)"
    assert rest < rest_tol, f"expo/v/bias/gravity differ by {rest}"
    assert cov < cov_tol, f"covariance differs by {cov} (per element, relative to sqrt(P_ii P_jj))"


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def digest(a):
    """SHA-256 of an array's shape and values, for bit-exact comparisons with stored outputs too large to commit in full.
    Floats are widened to float64 (exact) with -0.0 folded into 0.0, integers to int64: for arrays without NaN, equal digests <=> np.array_equal."""
    import hashlib

    a = np.asarray(a)
    a = np.ascontiguousarray(a.astype(np.float64) + 0.0 if a.dtype.kind == "f" else a.astype(np.int64))
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()


def load_golden(path, prefix):
    """The record stored under `prefix.` in a golden .npz (keys `prefix.field`), as {field: array}."""
    with np.load(path, allow_pickle=False) as g:
        return {k[len(prefix) + 1:]: g[k] for k in g.files if k.startswith(prefix + ".")}


def edge_scan(fr, seed=4):
    """World-frame points where the voxel indexing and the neighbour rule of BuildResidualListOMP (src/voxel_map.cpp:665-691)
    are fragile, for a frame's map (identity pose and extrinsics, so p_w is the float point itself):
      * exactly on voxel corners and faces of occupied voxels, both signs (trunc(q - 1) vs floor at negative integers),
      * one float ulp to either side of those,
      * uniformly inside occupied voxels, and the same with z == 0 (the 0.001 substitution of :352),
      * displaced off the local plane by 3-30 cm inside occupied voxels, towards every face: the home voxel fails and the
        unit-mixing neighbour rule (:683-688, voxel units against metres) picks the one neighbour that is probed.
    Returns (pts float32 [n,3], extrinsics with identity lidar->imu, packed state with identity pose and the frame's covariance)."""
    ext = S.Extrinsics(np.eye(3), np.zeros(3), fr["ext"].Rcl, fr["ext"].Pcl)
    st = S.unpack_state(fr["state_prior"])
    state = S.pack_state(np.eye(3), np.zeros(3), 1.0, st["v"], g=st["g"], cov=st["cov"])
    vs = fr["lio_cfg"].voxel_size
    keys = fr["map"]["keys"]
    rng = np.random.default_rng(seed)
    pick = keys[rng.choice(len(keys), 80, replace=False)].astype(np.float64)
    on_corner = (pick * vs).astype(np.float32)
    on_face = on_corner.copy()
    on_face[:, 1] += np.float32(0.37 * vs)
    inside = ((pick + rng.uniform(0.05, 0.95, pick.shape)) * vs).astype(np.float32)
    zero_z = inside.copy()
    zero_z[:, 2] = 0.0
    # off-plane points: first plane of the voxel, point = centre + in-plane jitter + offset along the normal, pushed towards a face
    first = fr["map"]["first"][rng.choice(len(keys), 400, replace=False)]
    pl = fr["map"]["planes"][first]
    off = rng.choice([-1.0, 1.0], (len(pl), 1)) * rng.uniform(0.03, 0.3, (len(pl), 1))
    jitter = rng.normal(0, 0.2 * vs, (len(pl), 3))
    jitter -= (jitter * pl["normal"]).sum(1, keepdims=True) * pl["normal"]
    off_plane = (pl["center"] + jitter + off * pl["normal"]).astype(np.float32)
    pts = np.ascontiguousarray(np.concatenate([on_corner, on_face, np.nextafter(on_corner, np.float32(-np.inf)), np.nextafter(on_corner, np.float32(np.inf)),
                                               inside, zero_z, off_plane]))
    return pts, ext, state

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


# ---------------------------------------------------------------------------------------------------------------------
# Border frames. A visual patch at tap stride s = 2^(level + search_level) reads an 11 x 11 footprint of the level-0 image:
# tile (0, 0) at x0 = u_i - 5 s, y0 = v_i - 5 s, the last tap at x0 + 10 s, with u_i = floorf(u / s) s (src/vio.cpp:1580-1597).
# The helpers below place visual points so that these footprints sit at prescribed places against the image edges.
EDGE_KINDS = ("margin", "touch", "past", "half")  # one stride inside / last tap on the edge row or column / one stride past / half out


def tap_origin(cam, ext, state, pos, stride):
    """(x0, y0) of the tap footprints of world points `pos` at tap strides `stride` for the pose in `state`, by the kernels'
    float rule (u_i = (int)(floorf((float)(u / s)) * s))."""
    st = S.unpack_state(state)
    Rcw, Pcw = S.camera_pose(ext, st["R"], st["p"])
    px = S.cam_project(cam, np.asarray(pos, np.float64) @ Rcw.T + Pcw)
    s = np.asarray(stride, np.int64)
    ui = np.floor((px[:, 0] / s).astype(np.float32)).astype(np.int64) * s
    vi = np.floor((px[:, 1] / s).astype(np.float32)).astype(np.int64) * s
    return ui - 5 * s, vi - 5 * s


def last_origin(size, s):
    """Largest footprint origin (a multiple of s) whose last tap x0 + 10 s is still inside [0, size)."""
    return (size - 1 - 10 * s) // s * s


def border_pixels(cam, levels, seed=0, edges=("left", "right", "top", "bottom"), corners=True, outside=True, rows=None):
    """Pixels whose footprint, at the target tap stride s = 2^p (p = 0 .. 5, search level p % 3 at level p - p % 3), sits
    at each EDGE_KINDS place against each edge, plus the four corners (touching and one stride past) and a few points up to
    200 px left / right of the image. Sub-pixel offsets of 0.2 .. 0.8 s keep every bilinear weight non-zero and the integer
    tap base away from rounding ties. rows: (lo, hi) range of v for the left / right edges (default the middle half).
    Returns px (n, 2), search_level (n,), target p (n,) (-1: outside the image) and a label per pixel."""
    rng = np.random.default_rng(seed)
    w, h = cam.width, cam.height
    rows = rows or (0.25 * h, 0.75 * h)
    px, sl, tp, lab = [], [], [], []

    def put(x0, y0, s, p, label, fu=None, fv=None):
        # x0 / y0 are multiples of s, so u_i = x0 + 5 s exactly
        px.append((x0 + 5 * s + (rng.uniform(0.2, 0.8) if fu is None else fu) * s, y0 + 5 * s + (rng.uniform(0.2, 0.8) if fv is None else fv) * s))
        sl.append(p % 3), tp.append(p), lab.append(label)

    for p in range(6):
        s = 1 << p
        if p - p % 3 > levels - 1:
            continue
        lx, ly = last_origin(w, s), last_origin(h, s)
        at = {"left": (s, 0, -s, -5 * s), "right": (lx - s, lx, lx + s, lx + 5 * s), "top": (s, 0, -s, -5 * s), "bottom": (ly - s, ly, ly + s, ly + 5 * s)}
        for e in edges:
            for kind, o in zip(EDGE_KINDS, at[e]):
                if e in ("left", "right"):
                    v = rng.uniform(*rows)
                    put(o, int(np.floor(v / s)) * s - 5 * s, s, p, f"{e}_{kind}")
                else:
                    u = rng.uniform(0.25 * w, 0.75 * w)
                    put(int(np.floor(u / s)) * s - 5 * s, o, s, p, f"{e}_{kind}")
        if corners:
            for kind, d in (("touch", 0), ("past", s)):
                for cx, cy in ((-d, -d), (lx + d, -d), (-d, ly + d), (lx + d, ly + d)):
                    put(cx, cy, s, p, f"corner_{kind}")
    if outside:
        for k, u in enumerate((-37.3, -120.6, -199.2, w + 15.4, w + 88.8, w + 190.1)):
            px.append((u, rng.uniform(*rows))), sl.append(k % 3), tp.append(-1), lab.append("outside")
    return np.array(px), np.array(sl, np.int32), np.array(tp), np.array(lab)


def border_frame(fr, state, seed=0, n_interior=64, extra_refs=(), **kw):
    """A copy of frame `fr` whose visual points are border_pixels(...) back-projected from the camera pose of `state` onto
    the scene (3 m deep where the ray misses it), followed by the first `n_interior` patches of `fr`. Warp patches and
    search levels come from the oracle (getWarpMatrixAffineHomography / warpAffine at the pose of `state`); the border
    patches then get their prescribed search levels. Adds bp_level (target p, -1 for interior and outside points) and
    bp_label per patch."""
    cam, ext = fr["cam_cfg"], fr["ext"]
    px, sl, tp, lab = border_pixels(cam, fr["vio_cfg"].levels, seed, **kw)
    st = S.unpack_state(state)
    Rcw, Pcw = S.camera_pose(ext, st["R"], st["p"])
    vio = O.OracleVIO(cam, ext, fr["vio_cfg"])
    f = np.stack([vio.cam2world(q) for q in px])  # unit bearings in the camera frame
    o = -Rcw.T @ Pcw
    d = f @ Rcw
    t, idx, hit = S.raycast(fr["rects"], o, d)
    miss = idx < 0
    hit = np.where(miss[:, None], o + 3.0 * d, hit)
    normals = np.where(miss[:, None], -d, np.stack([r.n for r in fr["rects"]])[np.maximum(idx, 0)])
    # keep the pixels the camera model maps back onto themselves (a fisheye's far-off-image pixels do not round-trip)
    keep = np.abs(S.cam_project(cam, hit @ Rcw.T + Pcw) - px).max(axis=1) < 1e-3
    assert keep.mean() > 0.9, keep.mean()
    px, sl, tp, lab, hit, normals = px[keep], sl[keep], tp[keep], lab[keep], hit[keep], normals[keep]
    R_ref, t_ref = fr["T_ref"]
    k = min(n_interior, len(fr["vis_pos"]))
    out = dict(fr)
    out.update(vis_pos=np.ascontiguousarray(np.concatenate([hit, fr["vis_pos"][:k]])), vis_normal=np.ascontiguousarray(np.concatenate([normals, fr["vis_normal"][:k]])),
               px_ref=np.ascontiguousarray(np.concatenate([S.cam_project(cam, hit @ R_ref.T + t_ref), fr["px_ref"][:k]])),
               inv_ref_expo=np.ones(len(px) + k), bp_level=np.concatenate([tp, np.full(k, -1)]), bp_label=np.concatenate([lab, np.full(k, "interior")]),
               bp_px=px)
    w = O.oracle_warp_patches(out, state)
    w["search_levels"][: len(px)] = sl
    out.update(warp_patch=w["warp_patch"], search_levels=w["search_levels"])
    return out

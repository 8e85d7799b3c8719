"""ctypes binding of tests/map_host_harness.cu (the device voxel-map state machine compiled for the host) + the comparison of
two flattened maps (keys / candidate lists / plane records) used by the CPU and GPU map tests."""
import ctypes as C
import os
import subprocess

import numpy as np

from fast_livo2_b200.synthetic import PLANE_DTYPE

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libmap_host.so")
SRC = os.path.join(HERE, "map_host_harness.cu")
HDR = os.path.join(HERE, "..", "fast_livo2_b200", "csrc", "esikf_map.cuh")


def build():
    if os.path.exists(SO) and os.path.getmtime(SO) >= max(os.path.getmtime(SRC), os.path.getmtime(HDR)):
        return
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC", "-o", SO, SRC], check=True)


class HostMap:
    def __init__(self, cfg, hash_cap=1 << 16, node_cap=1 << 16, pool_cap=1 << 19, rec_cap=1 << 16):
        build()
        self.lib = C.CDLL(SO)
        self.lib.maph_create.restype = C.c_void_p
        self.lib.maph_create.argtypes = [C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_int]
        self.lib.maph_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        self.lib.maph_flatten.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        self.lib.maph_usage.argtypes = [C.c_void_p, C.c_void_p]
        self.lib.maph_destroy.argtypes = [C.c_void_p]
        self.lib.maph_slide.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lin = np.zeros(8, np.int32)
        lin[:len(cfg.layer_init_num)] = cfg.layer_init_num
        lin[len(cfg.layer_init_num):] = cfg.layer_init_num[-1]
        self.h = self.lib.maph_create(cfg.voxel_size, cfg.min_eigen_value, cfg.max_layer, cfg.max_points_num, lin.ctypes.data, hash_cap, node_cap, pool_cap, rec_cap)

    def __del__(self):
        try:
            self.lib.maph_destroy(self.h)
        except Exception:
            pass

    def apply(self, pw, var, build=False):
        pt = np.ascontiguousarray(np.concatenate([np.asarray(pw, np.float64).reshape(-1, 3), np.asarray(var, np.float64).reshape(-1, 9)], axis=1))
        return self.lib.maph_apply(self.h, pt.ctypes.data, len(pt), 1 if build else 0)

    def flatten(self):
        nr, npl = C.c_int(0), C.c_int(0)
        self.lib.maph_flatten(self.h, C.byref(nr), C.byref(npl), None, None, None, None)
        keys, first, count = np.zeros((nr.value, 3), np.int64), np.zeros(nr.value, np.int32), np.zeros(nr.value, np.int32)
        planes = np.zeros(npl.value, PLANE_DTYPE)
        self.lib.maph_flatten(self.h, C.byref(nr), C.byref(npl), keys.ctypes.data, first.ctypes.data, count.ctypes.data, planes.ctypes.data)
        return dict(keys=keys, first=first, count=count, planes=planes)

    def slide(self, lo, hi):
        """mapSliding: keep the roots whose key lies in [lo, hi] (component-wise); everything is rebuilt into a fresh arena."""
        lo, hi = np.ascontiguousarray(lo, np.int64), np.ascontiguousarray(hi, np.int64)
        return self.lib.maph_slide(self.h, lo.ctypes.data, hi.ctypes.data)

    def usage(self):
        u = np.zeros(4, np.int64)
        self.lib.maph_usage(self.h, u.ctypes.data)
        return dict(nodes=int(u[0]), recs=int(u[1]), pool_points=int(u[2]), roots=int(u[3]))


def _by_key(flat):
    """Roots sorted by key, their candidate counts and candidate records in that order."""
    keys = np.asarray(flat["keys"]).reshape(-1, 3)
    order = np.lexsort(keys.T[::-1])
    count = np.asarray(flat["count"])[order]
    sel = np.concatenate([np.arange(f, f + c) for f, c in zip(np.asarray(flat["first"])[order], count)] or [np.zeros(0, np.int64)]).astype(np.int64)
    return keys[order], count, flat["planes"][sel]


def _structure_digest(keys, count, planes):
    from parity_util import digest

    return "/".join(digest(a) for a in (keys, count, planes["layer"], planes["path"]))


def map_record(flat, n_roots, seed):
    """A flattened map reduced to what a golden file can hold: a digest of its whole structure (root keys, candidates per root,
    layer / path of every candidate) and the complete records of a seeded sample of `n_roots` roots that hold planes
    (compare_map_record)."""
    keys, count, planes = _by_key(flat)
    held = np.nonzero(count > 0)[0]
    pick = np.sort(np.random.default_rng(seed).choice(held, min(n_roots, len(held)), replace=False))
    start = np.concatenate([[0], np.cumsum(count)[:-1]]).astype(np.int64)
    sel = np.concatenate([np.arange(start[i], start[i] + count[i]) for i in pick]).astype(np.int64)
    return dict(structure=np.str_(_structure_digest(keys, count, planes)), keys=keys[pick], count=count[pick].astype(np.int32),
                first=np.concatenate([[0], np.cumsum(count[pick])[:-1]]).astype(np.int32), planes=planes[sel])


def compare_map_record(flat, rec, rtol=1e-9, what=("a", "b")):
    """compare_flat_maps against a map_record: the structure of the whole map bit for bit, the sampled roots' plane records
    within the tolerances of compare_flat_maps. Returns the number of planes in the map."""
    keys, count, planes = _by_key(flat)
    assert _structure_digest(keys, count, planes) == str(rec["structure"]), f"root voxels, candidate counts or candidate order differ between {what[0]} and {what[1]}"
    compare_flat_maps(flat, dict(keys=rec["keys"], first=rec["first"], count=rec["count"], planes=rec["planes"]), rtol=rtol, what=what, subset=True)
    return len(planes)


def compare_flat_maps(a, b, rtol=1e-9, what=("a", "b"), exact=False, subset=False):
    """Same root keys, same candidate count per root, candidate j of a root = the same plane (centre, +-normal, plane_var, d,
    radius, layer, path) within rtol. Returns the number of planes compared. The eigenvector sign of a fit is free: a flipped
    normal flips d and the normal-position cross block of plane_var. subset: b holds some of a's roots, only those are compared."""
    ka = {tuple(k): i for i, k in enumerate(a["keys"].tolist())}
    kb = {tuple(k): i for i, k in enumerate(b["keys"].tolist())}
    if subset:
        assert set(kb) <= set(ka), f"{len(set(kb) - set(ka))} root voxels of {what[1]} missing in {what[0]}"
    else:
        assert set(ka) == set(kb), f"root voxels differ: {len(set(ka) - set(kb))} only in {what[0]}, {len(set(kb) - set(ka))} only in {what[1]}"
    common = list(kb) if subset else list(ka)
    ia = np.array([ka[k] for k in common], np.int64)
    ib = np.array([kb[k] for k in common], np.int64)
    assert np.array_equal(a["count"][ia], b["count"][ib]), "candidate counts per root differ"
    sel_a = np.concatenate([np.arange(f, f + c) for f, c in zip(a["first"][ia], a["count"][ia])] or [np.zeros(0, np.int64)]).astype(np.int64)
    sel_b = np.concatenate([np.arange(f, f + c) for f, c in zip(b["first"][ib], b["count"][ib])] or [np.zeros(0, np.int64)]).astype(np.int64)
    pa, pb = a["planes"][sel_a], b["planes"][sel_b]
    if exact:  # every byte of every candidate record (centre, normal incl. its sign, plane_var, d, radius, layer, path)
        bad = np.nonzero(pa.view(np.uint8).reshape(len(pa), -1) != pb.view(np.uint8).reshape(len(pb), -1))[0]
        assert len(bad) == 0, f"{len(np.unique(bad))} of {len(pa)} plane records differ between {what[0]} and {what[1]}"
        return len(pa)
    assert np.array_equal(pa["layer"], pb["layer"]) and np.array_equal(pa["path"], pb["path"]), "candidate order (layer / path) differs"
    np.testing.assert_allclose(pa["center"], pb["center"], rtol=rtol, atol=1e-12)
    sign = np.sign((pa["normal"] * pb["normal"]).sum(1))
    assert np.all(sign != 0)
    np.testing.assert_allclose(pa["normal"], pb["normal"] * sign[:, None], rtol=0, atol=1e-8)
    np.testing.assert_allclose(pa["d"], pb["d"] * sign, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(pa["radius"], pb["radius"], rtol=1e-6)
    # plane_var upper triangle: the normal block is rows / cols 0..2, the centre block 3..5; the cross block changes sign with the normal
    tri = [(i, j) for i in range(6) for j in range(i, 6)]
    flip = np.array([-1.0 if (i < 3) != (j < 3) else 1.0 for i, j in tri])
    va, vb = pa["plane_var"], pb["plane_var"] * np.where(sign[:, None] < 0, flip[None, :], 1.0)
    scale = np.abs(vb).max(axis=1, keepdims=True) + 1e-300
    # the refit sums are ill-conditioned where two eigenvalues nearly coincide (1 / (l_min - l_m)): relative to the plane's largest entry
    assert np.max(np.abs(va - vb) / scale) < max(rtol, 1e-7), f"plane_var differs by {np.max(np.abs(va - vb) / scale):.3e} (relative to the largest entry)"
    return len(pa)

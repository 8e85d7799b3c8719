"""Regenerates the stored outputs of the REFERENCE SOURCE that the pin tests compare the oracle with:
  ref_lio_golden.npz / ref_vio_golden.npz : full outputs on a few seeded synthetic frames (also read by the GPU tests),
  ref_lio_pins.npz / ref_vio_pins.npz     : every case of tests/test_oracle_ref_pin.py and tests/test_oracle_ref_pin_vio.py.
The reference source is FAST-LIVO2's src/voxel_map.cpp and src/vio.cpp compiled against oracle/ref_shim/ into oracle/_ref/,
which needs the FAST-LIVO2 source tree:   make -C oracle REF=<FAST-LIVO2 source tree> && python tests/golden/make_ref_golden.py"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import map_bind as MB  # noqa: E402
import oracle_bind as O  # noqa: E402
import test_oracle_ref_pin as L  # noqa: E402
from parity_util import digest  # noqa: E402
from test_oracle_ref_pin import _case  # noqa: E402

MAP_SAMPLE_ROOTS = 12  # roots per stored map whose plane records are kept in full (the structure of all roots is digested)

assert O.ref_lio_available() and O.ref_vio_available(), "build oracle/_ref first (make -C oracle REF=<FAST-LIVO2 source tree>)"
out = {}
for name in ("small", "hilti_voxel_04_non_identity_extrinsics"):
    fr, cfg = _case(name)
    r = O.ref_lio_state_estimation(fr, cfg=cfg)
    out[f"{name}_iters"] = np.int32(r["iters"])
    for k in ("M", "ptpl_center", "ptpl_dis", "normals", "state"):
        out[f"{name}_{k}"] = r[k]
np.savez_compressed(os.path.join(HERE, "ref_lio_golden.npz"), **out)
print("wrote", os.path.join(HERE, "ref_lio_golden.npz"), {k: np.asarray(v).shape for k, v in out.items()})

# ---- VIO half: oracle/_ref/libfl2_ref_vio.so = src/vio.cpp (+ frame.cpp, visual_point.cpp, voxel_map.cpp)
import test_oracle_ref_pin_vio as V  # noqa: E402
from test_oracle_ref_pin_vio import _inputs  # noqa: E402

vout = {}
for name in ("small", "exposure"):
    fr, prior, w = _inputs(name)
    r = O.RefVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"]).update(fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], fr["inv_ref_expo"], prior, prior)
    vout[f"{name}_state"], vout[f"{name}_errors"], vout[f"{name}_warp_patch"] = r["state"], r["errors"], w["warp_patch"]
    vout[f"{name}_search_levels"], vout[f"{name}_prior"] = w["search_levels"], prior
np.savez_compressed(os.path.join(HERE, "ref_vio_golden.npz"), **vout)
print("wrote", os.path.join(HERE, "ref_vio_golden.npz"), {k: np.asarray(v).shape for k, v in vout.items()})


# ---- the pin tests' cases, stored as `case.field`
def put(store, prefix, rec):
    for k, v in rec.items():
        store[f"{prefix}.{k}"] = v


lio = {}
for name in L.CASES:
    fr, cfg = _case(name)
    put(lio, name, L.lio_record(O.ref_lio_state_estimation(fr, cfg=cfg)))
fr, cfg = L.early_stop_frame()
put(lio, "early_stop", L.lio_record(O.ref_lio_state_estimation(fr, cfg=cfg)))
for kind in L.EDGE_FRAMES:
    put(lio, f"edge_{kind}", L.lio_record(O.ref_lio_state_estimation(L.edge_frame(kind))))
ref_lib = C.CDLL(O.REF_LIO_SO)
pts = L.body_cov_points()
cov = np.zeros((len(pts), 9))
for p, c in zip(pts, cov):
    ref_lib.ref_calc_body_cov(p.ctypes.data_as(C.c_void_p), C.c_float(0.02), C.c_float(0.05), c.ctypes.data_as(C.c_void_p))
put(lio, "body_cov", dict(cov=cov))
for cfg_id, cfg in L.MAP_CFGS.items():
    ref = O.RefMap(cfg)

    def clear(b, ref=ref):
        n0 = len(ref.flatten()["keys"])
        ref.lib.ref_map_clear_out_of_map(C.c_void_p(ref.h), *b)
        return n0 - len(ref.flatten()["keys"])

    for j, (label, f) in enumerate(L.update_voxel_map_run(cfg, ref.update, clear, ref.flatten)):
        put(lio, f"map_update.{cfg_id}.{label}", MB.map_record(f, MAP_SAMPLE_ROOTS, seed=j))
cfg, ext, scan, st0 = L.build_voxel_map_inputs()
ref = O.RefMap(cfg)
ref.build(scan, st0, ext, cfg)
put(lio, "map_build", MB.map_record(ref.flatten(), 4 * MAP_SAMPLE_ROOTS, seed=0))
np.savez_compressed(os.path.join(HERE, "ref_lio_pins.npz"), **lio)
print("wrote", os.path.join(HERE, "ref_lio_pins.npz"), len(lio), "arrays")

vio = {}
for name in V.CASES:
    fr, prior, w = _inputs(name)
    r = O.RefVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"]).update(fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], fr["inv_ref_expo"], prior, prior)
    put(vio, f"update.{name}", dict(state=r["state"], errors=r["errors"], H_T_H=r["H_T_H"][:7, :7], warp_patch=np.str_(digest(w["warp_patch"]))))
fr, prior, w = _inputs("small")
n = len(fr["vis_pos"])
r = O.RefVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"]).update_inverse(fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], np.ones(n),
                                                                      O.inverse_refs_from_frame(fr), prior, prior)
put(vio, "inverse", dict(state=r["state"], errors=r["errors"], warp_patch=np.str_(digest(w["warp_patch"]))))
fr = _inputs("distorted_pinhole")[0]
rows = list(V.patch_producer_calls(O.RefVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"])))
put(vio, "patch", dict(A=np.stack([a for a, _, _, _ in rows]), search_level=np.array([s for _, s, _, _ in rows], np.int32),
                       warp_affine=np.array([wd for _, _, wd, _ in rows]), image_patch=np.array([p for _, _, _, p in rows])))
b, prior, _, centres = V.edge_wrap_inputs()
rv = O.RefVIO(b["cam_cfg"], b["ext"], b["vio_cfg"])
r = rv.update(b["img"], b["vis_pos"], b["warp_patch"], b["search_levels"], b["inv_ref_expo"], prior, prior)
put(vio, "edge_wrap", dict(state=r["state"], errors=r["errors"], warp_patch=np.str_(digest(b["warp_patch"])), search_levels=b["search_levels"],
                           image_patch=V.edge_wrap_image_patches(rv, b["img"], centres, b["vio_cfg"].levels)))
from fast_livo2_b200 import workloads as W  # noqa: E402

for name, (_, want_vio) in V.BASELINE_COUNTS.items():
    fr = W.frame(name)
    r = O.ref_lio_state_estimation(fr)
    rec = dict(iters=np.int32(r["iters"]), M=np.asarray(r["M"], np.int32), state=r["state"])
    if want_vio is not None:
        lio_o = O.OracleLIO(fr["lio_cfg"], fr["ext"])
        lio_o.set_map(fr["map"])
        st = lio_o.state_estimation(fr["pts"], fr["state_prior"], fr["state_prior"])["state"]
        w = O.oracle_warp_patches(fr, st)
        rv = O.RefVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"]).update(fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], fr["inv_ref_expo"], st, st)
        rec.update(vio_prior=st, vio_warp_patch=np.str_(digest(w["warp_patch"])), vio_state=rv["state"], vio_errors=rv["errors"])
    put(vio, f"baseline.{name}", rec)
np.savez_compressed(os.path.join(HERE, "ref_vio_pins.npz"), **vio)
print("wrote", os.path.join(HERE, "ref_vio_pins.npz"), len(vio), "arrays")

#!/usr/bin/env python
"""bench.py — ESIKF update iterations/sec on synthetic frames (BASELINE.json metric).

A "step" is one LIVMapper tick pair on one synthetic frame: the LIO update (StateEstimation, <= 5 iterations over the
LiDAR points) followed by the VIO update (computeJacobianAndUpdateEKF, levels x <= 5 iterations over the visual patches).
One ESIKF iteration = residual/Jacobian build over all points or patches -> information reduction -> 19x19 gain solve ->
boxplus. --config selects the BASELINE.json workload (default cfg2 = configs[1], the one the metric is quoted on).

  value    : iterations/s with the frame resident in HBM (scan, image, patches, map on the device; only the 3 KB packed
             state crosses PCIe per update), device-timed with CUDA events on the library's stream, L2 flushed between steps.
  e2e      : same metric through the C ABI's host-buffer path: per step the scan / image / patches are copied from pinned
             host memory and the posterior state + per-point association + patch errors are read back.
  e2e_shim : same through the drop-in C++ classes (fl2b200::VoxelMapManager::StateEstimation + VIOManager::
             computeJacobianAndUpdateEKF, pageable std::vector buffers, pv_list_ / ptpl_list_ filled) via libfl2_shim.so.
  parity   : every run compares the first update's result (per-iteration matched counts, iteration counts per level, posterior
             states and covariances) with the CPU oracle and the last timed update with the first; any figure over the
             tolerance fails the run (exit code 1) — at every N.
  --impl reference : the CPU oracle restatement of the reference (the reference itself cannot be built in this image,
             see DESIGN.md) compiled ON THIS HOST with the reference's flags, OpenMP as in the reference.

Multi-GPU (torchrun, one rank per GPU): the residual point / patch set is sharded across ranks; the compact information
vector is exchanged inside the persistent kernel over NVLink peer memory (or with ncclAllReduce per iteration, --comm nccl);
every rank solves redundantly ("scaling": "strong" — the frame is fixed).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ next to the imported modules
# seeded frames take tens of seconds to generate: cached per user in the temporary directory, never in the tree
FRAME_CACHE = os.path.join(tempfile.gettempdir(), f"fast_livo2_b200_frames_{os.getuid()}")

METRIC = "ESIKF update iters/sec @100k LiDAR pts+2k patches"
UNIT = "iters/s"
LIO_BYTES_PER_POINT = 268.0   # SURVEY.md §8d: 12 (xyz f32) + 32 (hash slot) + 224 (plane record), h = c = 1
VIO_BYTES_PER_PATCH = 413.0   # SURVEY.md §8d
TOL = 1e-5                    # north star: pose / covariance within 1e-5 relative of the reference


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"], help="BASELINE.json workload (cfg2 = configs[1], the metric's own)")
    ap.add_argument("--cpu-baseline-frames", type=int, default=30)  # bounded by 30 s of wall time
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-shim", action="store_true", help="skip the e2e_shim leg")
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"], help="N>1: in-kernel NVLink peer-memory exchange (default) or NCCL per iteration")
    ap.add_argument("--tuning", type=int, default=0, help="esikf_set_tuning flags (1: stage plane records with __ldg copies instead of cp.async.bulk)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (posterior states, iteration statistics, per-point association and per-patch "
                         "errors) to DIR/<name>.npy, float64 / float32, for comparing two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


# ----------------------------------------------------------------------------------------------------------------------
def make_workload(args):
    from fast_livo2_b200 import workloads as W

    t0 = time.time()
    fr = W.frame(args.config, cache_dir=FRAME_CACHE)
    fr["gen_seconds"] = time.time() - t0
    return fr


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            time.sleep(0.3)  # the first sample is in before the timed region starts
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the persistent LIO kernel from the committed ncu capture (profiles/), else None."""
    p = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("lio_update_kernel_r02", {}).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ---------------------------------------------------------------------------------------------------------------------- CPU oracle legs
def native_baseline_build():
    """Build liborc_baseline.so ON THIS HOST (-march=native must mean the machine the number is taken on). Returns the path or None."""
    out_dir = os.path.join(tempfile.gettempdir(), f"orc_native_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "liborc_baseline.so")
    src = [os.path.join(ROOT, "oracle", f) for f in ("orc_lio.cpp", "orc_vio.cpp", "orc_capi.cpp")]
    try:
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
            subprocess.run(["/usr/bin/g++", "-std=c++17", "-fPIC", "-shared", "-fopenmp", "-O3", "-march=native", "-mtune=native", "-funroll-loops", "-o", so, *src],
                           check=True, capture_output=True, timeout=300)
        return so
    except Exception:
        return None


def run_cpu_reference(fr, threads, frames, warm=1, kind="baseline", budget_s=None):
    """Time the oracle restatement (compiled like the reference) on up to `frames` repetitions of the frame (bounded by budget_s)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_bind as O

    has_vio = len(fr.get("vis_pos", [])) > 0
    lio = O.OracleLIO(fr["lio_cfg"], fr["ext"], threads=threads, kind=kind)
    lio.set_map(fr["map"])
    vio = O.OracleVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"], threads=threads, kind=kind) if has_vio else None
    r = lio.state_estimation(fr["pts"], fr["state_prior"], fr["state_prior"])
    w = O.oracle_warp_patches(fr, r["state"]) if has_vio else None
    t_l = t_v = 0.0
    it_l = it_v = 0
    done = 0
    v = None
    t_start = time.time()
    for k in range(warm + frames):
        r = lio.state_estimation(fr["pts"], fr["state_prior"], fr["state_prior"])
        if k >= warm:
            t_l += r["secs"]
            it_l += r["iters"]
        if has_vio:
            v = vio.update(fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], fr["inv_ref_expo"], r["state"], r["state"])
            if k >= warm:
                t_v += v["secs"]
                it_v += v["total_iters"]
        if k >= warm:
            done += 1
            if budget_s is not None and time.time() - t_start > budget_s:
                break
    return dict(value=(it_l + it_v) / (t_l + t_v), lio_iters_per_s=it_l / t_l if t_l else None, vio_iters_per_s=it_v / t_v if t_v else None,
                ms_per_frame=1e3 * (t_l + t_v) / done, iters_per_frame=(it_l + it_v) / done, seconds=t_l + t_v, frames=done,
                lio=r, vio=v, warp=w)


def state_error(s, ref):
    """Pose / covariance error of a packed state against the oracle's: rotation angle of R_ref^T R [rad], |p - p_ref| / |p_ref|,
    the other state blocks relative to their norm, and the covariance PER ELEMENT: |dP_ij| / sqrt(P_ii P_jj) (each entry against
    the scale of its own two variances — small cross-covariances are held to the same relative bound as the diagonal)."""
    from fast_livo2_b200 import synthetic as S

    a, b = S.unpack_state(np.asarray(s, dtype=np.float64)), S.unpack_state(np.asarray(ref, dtype=np.float64))
    dR = b["R"].T @ a["R"]
    rot = float(np.linalg.norm(dR - dR.T) / (2.0 * np.sqrt(2.0)))  # = sin(angle), exact to first order where acos() loses digits
    pos = float(np.linalg.norm(a["p"] - b["p"]) / max(np.linalg.norm(b["p"]), 1e-3))
    rest = float(np.abs(np.asarray(s)[12:25] - np.asarray(ref)[12:25]).max() / max(np.abs(np.asarray(ref)[12:25]).max(), 1e-3))
    d = np.sqrt(np.abs(np.diag(b["cov"])))
    cov = float((np.abs(a["cov"] - b["cov"]) / np.maximum(np.outer(d, d), 1e-300)).max())
    return {"rot_rad": rot, "pos_rel": pos, "rest_rel": rest, "cov_rel_per_element": cov}


def dump_outputs(out_dir, rl, vl, per_point):
    """What a caller of the timed path (esikf_lio_run + esikf_lio_fetch, esikf_vio_run + esikf_vio_fetch) receives for the last
    timed step, one DIR/<name>.npy per array; integer outputs are stored as float64 (exact). The largest workload (cfg5:
    300 k points, 4 k patches) writes about 6 MB."""
    arrays = {"lio_state": rl["state"], "lio_iters": [rl["iters"]], "lio_matched_points": rl["M"], "lio_total_residual": rl["total_residual"],
              "lio_converged": rl["converged"]}
    if per_point:
        arrays.update(lio_match_plane=rl["match_plane"], lio_normal_plane=rl["normal_plane"], lio_dis_to_plane=rl["dis_to_plane"])
    if vl is not None:
        arrays.update(vio_state=vl["state"], vio_total_iters=[vl["total_iters"]], vio_iters_per_level=vl["iters_per_level"],
                      vio_accepted_per_level=vl["accepted_per_level"])
        if per_point:
            arrays["vio_errors"] = vl["errors"]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, f"{name}.npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def parity_block(fr, r0, v0, world):
    """First update of this run against the CPU oracle (the -ffp-contract=off checker build, 4 threads)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_bind as O

    has_vio = v0 is not None
    lio = O.OracleLIO(fr["lio_cfg"], fr["ext"], threads=4)
    lio.set_map(fr["map"])
    o = lio.state_estimation(fr["pts"], fr["state_prior"], fr["state_prior"])
    out = {"tolerance": TOL, "lio": state_error(r0["state"], o["state"]), "lio_iters": [int(r0["iters"]), int(o["iters"])],
           "matched_points_per_iteration_equal": [int(m) for m in r0["M"]] == [int(m) for m in o["M"]],
           "matched_points": [int(m) for m in r0["M"]]}
    if world == 1:  # per-point outputs are complete on a single rank
        out["association_identical"] = bool(np.array_equal(r0["match_plane"], o["match_plane"]) and np.array_equal(r0["dis_to_plane"], o["dis_to_plane"]))
    ok = out["matched_points_per_iteration_equal"] and out["lio_iters"][0] == out["lio_iters"][1] and out.get("association_identical", True)
    ok = ok and all(v <= TOL for v in out["lio"].values())
    if has_vio:
        vio = O.OracleVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"], threads=4)
        ov = vio.update(fr["img"], fr["vis_pos"], fr["_warp"]["warp_patch"], fr["_warp"]["search_levels"], fr["inv_ref_expo"], r0["state"], r0["state"])
        L = fr["vio_cfg"].levels
        out["vio"] = state_error(v0["state"], ov["state"])
        out["vio_iters_per_level"] = [v0["iters_per_level"][:L].tolist(), ov["iters_per_level"][:L].tolist()]
        ok = ok and out["vio_iters_per_level"][0] == out["vio_iters_per_level"][1] and all(v <= TOL for v in out["vio"].values())
    out["ok"] = bool(ok)
    return out


def reference_source_timing(fr, restatement, budget_s=20.0):
    """The reference's OWN translation units (oracle/_ref/*_timing.so: src/voxel_map.cpp and src/vio.cpp compiled against the
    stand-in headers with -O3 -funroll-loops -fopenmp, MP_PROC_NUM=4; built where /root/reference exists, shipped with the
    snapshot) timed on the same frame, next to the restatement that the arm's `value` comes from. Their linear algebra is the
    stand-in matrix library (plain loops), not Eigen: a cross-check of the restatement's figure, not a replacement for it."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_bind as O

        lio_so = os.path.join(ROOT, "oracle", "_ref", "libfl2_ref_lio_timing.so")
        vio_so = os.path.join(ROOT, "oracle", "_ref", "libfl2_ref_vio_timing.so")
        if not os.path.exists(lio_so):
            return {"unavailable": "oracle/_ref/*_timing.so not in this checkout (built only where /root/reference exists)"}
        has_vio = len(fr.get("vis_pos", [])) > 0 and os.path.exists(vio_so) and fr["cam_cfg"].model == 0
        t_l = t_v = 0.0
        it_l = it_v = frames = 0
        t0 = time.time()
        rv = O.RefVIO(fr["cam_cfg"], fr["ext"], fr["vio_cfg"], so=vio_so) if has_vio else None
        w = restatement.get("warp")
        while frames < 8 and time.time() - t0 < budget_s:
            r = O.ref_lio_state_estimation(fr, so=lio_so)
            if frames > 0 or budget_s < 1:
                t_l += r["secs"]
                it_l += r["iters"]
            if has_vio:
                v = rv.update(fr["img"], fr["vis_pos"], w["warp_patch"], w["search_levels"], fr["inv_ref_expo"], r["state"], r["state"])
                if frames > 0:
                    t_v += v["secs"]
                    it_v += int(restatement["vio"]["total_iters"])  # the reference does not export its count; the restatement's is the same (pinned)
            frames += 1
        if it_l == 0:
            return {"unavailable": "no timed frame inside the budget"}
        return {"value": (it_l + it_v) / (t_l + t_v), "unit": UNIT, "lio_iters_per_s": it_l / t_l, "vio_iters_per_s": (it_v / t_v) if t_v else None,
                "frames": frames - 1, "threads": 4,
                "note": "reference source (voxel_map.cpp / vio.cpp) against stand-in headers, -O3 -funroll-loops -fopenmp, no -march=native (built on another host)"}
    except Exception as e:  # a cross-check: never lose the arm's line over it
        return {"error": repr(e)}


def reference_arm(args, rank, world):
    if rank != 0:
        return
    fr = make_workload(args)
    ncpu = os.cpu_count() or 1
    so = native_baseline_build()
    if so:
        os.environ["ORC_BASELINE_SO"] = so
    has_vio = len(fr.get("vis_pos", [])) > 0
    # the reference hard-caps OpenMP at 4 threads (CMakeLists.txt:46-58): that is the reference's own configuration. All host
    # cores are tried on a short sample as well (the per-point mutex makes it slower); the faster of the two is reported.
    probe = run_cpu_reference(fr, ncpu, 2, warm=1, budget_s=20) if ncpu > 4 else None
    res4 = run_cpu_reference(fr, 4, args.steps, warm=args.warmup, budget_s=150)
    best, cores = (res4, 4)
    if probe is not None and probe["value"] > res4["value"]:
        best, cores = run_cpu_reference(fr, ncpu, args.steps, warm=args.warmup, budget_s=150), ncpu
    ref_src = reference_source_timing(fr, best)
    out = {
        "impl": "reference", "metric": METRIC, "value": best["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": best["frames"], "warmup": args.warmup,
        "ms_per_step": best["ms_per_frame"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": fr["workload"], "n_pts": len(fr["pts"]), "n_patches": len(fr["vis_pos"]) if has_vio else 0,
                   "image": f"{fr['cam_cfg'].width}x{fr['cam_cfg'].height}" if has_vio else None, "levels": fr["vio_cfg"].levels if has_vio else 0},
        "cpu_baseline": {"value": best["value"], "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{best['frames']} frames of the workload after {args.warmup} warm-up frames ({best['seconds']:.1f} s of CPU work, capped at 150 s); oracle "
                                   f"restatement built {'on this host' if so else 'in the build container (native build failed)'} with the reference's flags "
                                   f"(-O3 -march=native -funroll-loops -fopenmp); 4 threads (reference cap): {res4['value']:.2f} it/s"
                                   + (f", {ncpu} threads (short sample): {probe['value']:.2f} it/s" if probe else "") + f"; host: {ncpu} logical cores"},
        "e2e": {"value": best["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_source": ref_src,
    }
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------------------------------- drop-in shim leg
def shim_session(fr, warp):
    """A persistent fl2b200::VoxelMapManager (+ VIOManager) holding the frame's map: returns step() -> (iterations, lio_state, vio_state)."""
    import ctypes as C

    from fast_livo2_b200 import api

    shim = C.CDLL(os.path.join(ROOT, "fast_livo2_b200", "libfl2_shim.so"))
    shim.fl2_shim_session_create.restype = C.c_void_p
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    m = fr["map"]
    k, f, c, p = (np.ascontiguousarray(m["keys"]), np.ascontiguousarray(m["first"]), np.ascontiguousarray(m["count"]), np.ascontiguousarray(m["planes"]))
    lcfg = api.lio_cfg_c(fr["lio_cfg"])
    ext = api.ExtrinsicsC()
    ext.extR[:] = fr["ext"].extR.reshape(9)
    ext.extT[:] = fr["ext"].extT
    ext.Rcl[:] = fr["ext"].Rcl.reshape(9)
    ext.Pcl[:] = fr["ext"].Pcl
    has_vio = warp is not None
    cam = vcfg = None
    if has_vio:
        cc, vc = fr["cam_cfg"], fr["vio_cfg"]
        cam = api.CameraC(cc.model, cc.width, cc.height, 0, cc.fx, cc.fy, cc.cx, cc.cy)
        cam.d[:] = list(cc.d)
        vcfg = api.VioCfgC(vc.img_point_cov, vc.levels, vc.max_iterations, int(vc.exposure_estimate_en), 0)
    h = C.c_void_p(shim.fl2_shim_session_create(vp(k), vp(f), vp(c), len(f), vp(p), len(p), C.byref(lcfg), C.byref(ext), C.byref(cam) if has_vio else None,
                                                C.byref(vcfg) if has_vio else None, 0))
    if not h:
        raise RuntimeError("fl2_shim_session_create failed")
    pts = np.ascontiguousarray(fr["pts"])
    sp = np.ascontiguousarray(fr["state_prior"])
    lio_out, vio_out = np.zeros(386), np.zeros(386)
    iters = (C.c_int32 * 2)()
    n = len(pts)
    if has_vio:
        img = np.ascontiguousarray(fr["img"])
        pos, wp, sl, ie = (np.ascontiguousarray(fr["vis_pos"]), np.ascontiguousarray(warp["warp_patch"]), np.ascontiguousarray(warp["search_levels"]),
                           np.ascontiguousarray(fr["inv_ref_expo"]))
        npatch = len(pos)

    def step():
        if has_vio:
            rc = shim.fl2_shim_session_step(h, vp(pts), n, vp(sp), vp(sp), vp(img), npatch, vp(pos), vp(wp), vp(sl), vp(ie), vp(lio_out), vp(vio_out), iters)
        else:
            rc = shim.fl2_shim_session_step(h, vp(pts), n, vp(sp), vp(sp), None, 0, None, None, None, None, vp(lio_out), vp(vio_out), iters)
        if rc:
            raise RuntimeError(f"fl2_shim_session_step failed: {rc}")
        return int(iters[0] + iters[1])

    def close():
        shim.fl2_shim_session_destroy(h)

    def point_lists(mode):
        shim.fl2_shim_session_point_lists(h, mode)

    shim.fl2_shim_session_manager_ns.restype = C.c_longlong
    shim.fl2_shim_session_manager_ns.argtypes = [C.c_void_p]
    step.point_lists = point_lists
    step.manager_ns = lambda: int(shim.fl2_shim_session_manager_ns(h))
    return step, close, lio_out, vio_out


def map_update_leg(fr, torch, api, dev, ticks=6):
    """SURVEY §8 f1, the step right after the LIO update of every tick (LIVMapper.cpp:413-424 + UpdateVoxelMap, the
    "updateVoxelMap" row of the reference's timing table): device-resident map absorbing the scan, timed with CUDA events on
    the context's stream and by wall clock (the call returns after its status read-back), next to the oracle's UpdateVoxelMap
    on the host for the same sequence (BuildVoxelMap from the scan at the true pose, then `ticks` x {StateEstimation, update})."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_bind as O

    cfg, ext, pts = fr["lio_cfg"], fr["ext"], np.ascontiguousarray(fr["pts"])
    ctx = api.Context(dev.index)
    orc = O.OracleLIO(cfg, ext, threads=4, kind="baseline")
    try:
        ctx.set_extrinsics(ext)
        ctx.map_device_init(cfg, root_capacity=1 << 19)
        ctx.lio_set_scan(pts)
        t0 = time.perf_counter()
        ctx.map_device_build(fr["state_true"])
        build_ms = 1e3 * (time.perf_counter() - t0)
        t0 = time.perf_counter()
        orc.tick_build_map(pts, fr["state_true"])
        cpu_build_ms = 1e3 * (time.perf_counter() - t0)
        stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
        dev_ms, wall_ms, cpu_ms, touched, same = [], [], [], [], []
        for k in range(ticks):
            g = ctx.lio_update(pts, fr["state_prior"], fr["state_prior"], cfg)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            t0 = time.perf_counter()
            ctx.map_device_update()
            wall_ms.append(1e3 * (time.perf_counter() - t0))
            e1.record(stream)
            e1.synchronize()
            dev_ms.append(e0.elapsed_time(e1))
            touched.append(ctx.map_device_stats()["touched_roots"])
            o = orc.state_estimation(pts, fr["state_prior"], fr["state_prior"])
            t0 = time.perf_counter()
            orc.tick_update_map()
            cpu_ms.append(1e3 * (time.perf_counter() - t0))
            same.append(bool(g["iters"] == o["iters"] and np.array_equal(np.asarray(g["M"])[:g["iters"]], o["M"]) and
                             state_error(g["state"], o["state"])["rot_rad"] < 1e-9))
        st = ctx.map_device_stats()
        return {"device_ms_per_tick": dev_ms, "wall_ms_per_tick": wall_ms, "cpu_oracle_ms_per_tick": cpu_ms, "touched_roots_per_tick": touched,
                "device_build_ms_wall": build_ms, "cpu_oracle_build_ms": cpu_build_ms, "n_pts": int(len(pts)), "roots": st["roots"], "nodes": st["nodes"],
                "lio_update_on_device_map_tracks_oracle": all(same),
                "what": "esikf_map_device_update after esikf_lio_update of the same scan (world points + covariances with the posterior, voxel keys, "
                        "stable sort by root, one warp per touched root replaying UpdateOctoTree / init_plane, candidate records re-emitted); map built by "
                        "esikf_map_device_build from the scan at the true pose; the same scan is absorbed every tick, so later ticks meet saturated "
                        "(update_enable_ == false) voxels like a mature map does; CPU column: the oracle's UpdateVoxelMap (single thread, like the reference)"}
    finally:
        ctx.close()


# ---------------------------------------------------------------------------------------------------------------------- B200 arm
def b200_arm(args, rank, world, local_rank):
    import torch

    from fast_livo2_b200 import api
    from fast_livo2_b200 import synthetic as S

    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
        import torch.distributed as dist_mod

        dist = dist_mod
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    # one rank builds (or finds) the seeded frame, the others read the same pickle: every rank works on bit-identical inputs
    if dist is not None and rank != 0:
        dist.barrier()
    fr = make_workload(args)
    if dist is not None and rank == 0:
        dist.barrier()
    has_vio = len(fr.get("vis_pos", [])) > 0
    ctx = api.Context(local_rank)
    if world > 1:
        if args.comm == "p2p":
            handles = [None] * world
            dist.all_gather_object(handles, ctx.peer_export())
            ctx.peer_attach(rank, world, handles)
        else:
            uid = [api.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            ctx.comm_init(rank, world, uid[0])
    if args.tuning:
        ctx.set_tuning(args.tuning)
    ctx.set_extrinsics(fr["ext"])
    ctx.map_upload(fr["map"], fr["lio_cfg"].voxel_size)
    if has_vio:
        ctx.vio_set_camera(fr["cam_cfg"], fr["vio_cfg"])

    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    pts_h = pin(fr["pts"])
    prior_h = pin(fr["state_prior"])
    n, npatch, L = len(fr["pts"]), (len(fr["vis_pos"]) if has_vio else 0), (fr["vio_cfg"].levels if has_vio else 0)

    # ---------------- first update: LIO posterior (what the VIO tick starts from), warp patches by the product's own kernels, VIO
    ctx.lio_set_scan(pts_h)
    ctx.lio_run(prior_h, prior_h, fr["lio_cfg"])
    r0 = ctx.lio_fetch()
    r0 = dict(r0, state=r0["state"].copy())
    v0 = w = None
    post_h = pin(r0["state"])
    if has_vio:
        img_h = pin(fr["img"])
        post = S.unpack_state(r0["state"])
        ctx.vio_set_image(img_h)
        ctx.vio_set_ref_images([fr["img_ref"]])
        T_cur = api.pack_T(*S.camera_pose(fr["ext"], post["R"], post["p"]))
        T_ref = np.tile(api.pack_T(*fr["T_ref"]), (npatch, 1))
        w = ctx.vio_warp_patches(np.zeros(npatch, np.int32), fr["px_ref"], fr["vis_pos"], fr["vis_normal"], T_ref, T_cur)
        fr["_warp"] = w
        pos_h, wp_h, sl_h, ie_h = pin(fr["vis_pos"]), pin(w["warp_patch"]), pin(w["search_levels"]), pin(fr["inv_ref_expo"])
        ctx.vio_set_patches(pos_h, wp_h, sl_h, ie_h)
        ctx.vio_run(post_h, post_h)
        v0 = ctx.vio_fetch()
        v0 = dict(v0, state=v0["state"].copy())
    iters_per_step = int(r0["iters"] + (v0["total_iters"] if has_vio else 0))

    # ---------------- parity of THIS run against the CPU oracle — at every N, and it fails the run
    parity = parity_block(fr, r0, v0, world) if rank == 0 else None
    if dist is not None:
        torch.cuda.synchronize()
        dist.barrier()  # the oracle runs for seconds on rank 0: nobody launches an update that would wait for it inside a kernel

    ext_stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        # Drain the update stream BEFORE the collective: a persistent update kernel occupies every SM (co-resident cooperative
        # grid) and spins on its peers, and an NCCL kernel of the barrier that slips in between two queued updates on one rank
        # keeps that rank's next cooperative launch from becoming resident while the peers wait for it inside their kernels.
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        ctx.lio_run(prior_h, prior_h, fr["lio_cfg"])
        if has_vio:
            ctx.vio_run(post_h, post_h)

    # ---------------- value: frame resident in HBM, device-timed per step, L2 flushed (untimed) between steps
    W, K = args.warmup, args.steps
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    sampler = ClockSampler(local_rank)
    for k in range(W):
        with torch.cuda.stream(ext_stream):
            flush.zero_()
        one_step()
    if rank == 0:
        sampler.start()  # before the barrier: nobody spins on a peer while rank 0 forks nvidia-smi
    barrier()
    l0 = ctx.launch_count()
    for k in range(K):
        with torch.cuda.stream(ext_stream):
            flush.zero_()
            evs[k][0].record(ext_stream)
        ctx.lio_run(prior_h, prior_h, fr["lio_cfg"])
        with torch.cuda.stream(ext_stream):
            evs[k][2].record(ext_stream)  # LIO update done (persistent kernel: ONE launch = all its iterations)
        if has_vio:
            ctx.vio_run(post_h, post_h)
        with torch.cuda.stream(ext_stream):
            evs[k][1].record(ext_stream)
    barrier()
    launches = ctx.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    step_ms = np.array([a.elapsed_time(b) for a, b, _ in evs])
    lio_ms = float(np.mean([a.elapsed_time(c) for a, _, c in evs]))   # LIO update (launch + its state copy), in the timed region
    vio_ms = float(np.mean([c.elapsed_time(b) for _, b, c in evs]))
    stat = torch.tensor([float(step_ms.sum()), float(np.median(step_ms)), float(step_ms.max())], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(stat, op=dist.ReduceOp.MAX)
    total_ms, med_ms, max_ms = (float(x) for x in stat.tolist())
    # the last timed update must reproduce the first bit for bit (same inputs, deterministic reduction order)
    per_point = args.dump_outputs is not None and world == 1  # a rank of a sharded run holds only its slice of the per-point outputs
    vl = ctx.vio_fetch(errors=per_point) if has_vio else None
    rl = ctx.lio_fetch(per_point=per_point)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, rl, vl, per_point)
    same = rl["iters"] == r0["iters"] and rl["M"].tolist() == r0["M"].tolist()
    if has_vio:
        same = same and vl["total_iters"] == v0["total_iters"] and np.array_equal(vl["state"], v0["state"])
    else:
        same = same and np.array_equal(rl["state"], r0["state"])
    value = iters_per_step * K / (total_ms * 1e-3)

    # ---------------- e2e: host buffers through the C ABI, H2D + D2H inside the timed region (wall clock, blocking calls)
    st_out, st_out2 = torch.empty(386, dtype=torch.float64).pin_memory(), torch.empty(386, dtype=torch.float64).pin_memory()
    m_h, nm_h = torch.empty(n, dtype=torch.int32).pin_memory(), torch.empty(n, dtype=torch.int32).pin_memory()
    d_h, err_h = torch.empty(n, dtype=torch.float32).pin_memory(), torch.empty(max(npatch, 1), dtype=torch.float32).pin_memory()
    lio_cfg_c = api.lio_cfg_c(fr["lio_cfg"])

    def e2e_step():
        a = ctx.lio_update_into(pts_h, prior_h, prior_h, lio_cfg_c, st_out, m_h, nm_h, d_h)
        b = ctx.vio_update_into(img_h, pos_h, wp_h, sl_h, ie_h, st_out, st_out, st_out2, err_h) if has_vio else 0
        return a + b

    for _ in range(W):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e2e_iters = 0
    for _ in range(K):
        e2e_iters += e2e_step()
    torch.cuda.synchronize()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = e2e_iters / float(t_e2e.item())
    h2d = n * 12 + 2 * 386 * 8 + (fr["cam_cfg"].width * fr["cam_cfg"].height + npatch * (24 + 256 * L + 4 + 8) + 2 * 386 * 8 if has_vio else 0)
    d2h = 386 * 8 + n * 12 + 1288 + 64 + ((386 * 8 + npatch * 4 + 33096 + 64) if has_vio else 0)  # states + match/normal/dis + errors + stats + loop control

    # ---------------- e2e through the drop-in C++ classes (single GPU): pageable buffers, pv_list_ / ptpl_list_ filled
    e2e_shim = None
    if world == 1 and not args.no_shim:
        try:
            step, close, s_lio, s_vio = shim_session(fr, w)

            def timed():
                for _ in range(W):
                    step()
                t0 = time.perf_counter()
                its, inside = 0, 0
                for _ in range(K):
                    its += step()
                    inside += step.manager_ns()
                return its, time.perf_counter() - t0, inside * 1e-9

            step.point_lists(1)  # lazy: the lists are there on request (MaterializePointLists), not built inside the tick
            its, dt_h, dt = timed()
            step.point_lists(0)  # eager: the reference's member contract, pv_list_ / ptpl_list_ / covariance lists rebuilt every tick
            its_e, dt_eh, dt_e = timed()
            e2e_shim = {"value": its / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / K, "iters_per_step": its / K,
                        "value_with_point_lists": its_e / dt_e, "ms_per_step_with_point_lists": 1e3 * dt_e / K,
                        "ms_per_step_including_harness": 1e3 * dt_h / K,
                        "timed": "wall clock inside the two manager calls LIVMapper makes per tick pair (StateEstimation, computeJacobianAndUpdateEKF), host<->device "
                                 "copies included; `ms_per_step_including_harness` adds this bench's own copies of its flat numpy buffers into the managers' "
                                 "reference-shaped members (feats_down_body_, SubSparseMap vectors), which LIVMapper already holds in that shape",
                        "path": "fl2b200::VoxelMapManager::StateEstimation + VIOManager::computeJacobianAndUpdateEKF (libfl2_shim.so): caller-owned pageable "
                                "std::vector buffers in, reference-shaped members out; `value`: pv_list_ / ptpl_list_ / body_cov_list_ / cross_mat_list_ "
                                "materialised on request only (lazy_point_lists_), `value_with_point_lists`: rebuilt on the host inside every tick (14 MB of "
                                "per-point covariances D2H + a host loop over the scan — what a LIVMapper that still runs UpdateVoxelMap on the host reads)",
                        "state_equal_to_c_abi": bool(np.array_equal(s_lio, r0["state"]) and (not has_vio or np.array_equal(s_vio, v0["state"]))),
                        "max_abs_state_diff_to_c_abi": [float(np.abs(s_lio - r0["state"]).max()), float(np.abs(s_vio - v0["state"]).max()) if has_vio else 0.0]}
            close()
        except Exception as e:  # measurement extra: never lose the bench line over it
            e2e_shim = {"error": repr(e)}

    # ---------------- f1: the map absorbing the scan on the device (single GPU; every rank of a sharded run would repeat it identically)
    map_update = None
    if world == 1 and not args.no_shim:
        try:
            map_update = map_update_leg(fr, torch, api, dev)
        except Exception as e:  # measurement extra: never lose the bench line over it
            map_update = {"error": repr(e)}

    # ---------------- per-kernel device times inside the loop (separate instrumented pass) -> roofline of the LIO residual kernel
    per_iter_ok = (world == 1) or args.comm == "nccl"  # per-launch event timing uses the per-iteration launch path
    ctx.set_kernel_timing(per_iter_ok)
    res_ms, patch_ms, solve_ms = [], [], []
    for k in range(max(5, min(K, 10)) if per_iter_ok else 0):
        with torch.cuda.stream(ext_stream):
            flush.zero_()
        one_step()
        ctx.synchronize()
        tm = ctx.get_kernel_timing()
        res_ms += list(tm["lio_residual_ms"][: rl["iters"]])
        solve_ms += list(tm["lio_solve_ms"][: rl["iters"]])
        for lvl in range(L):
            base = (L - 1 - lvl) * fr["vio_cfg"].max_iterations
            patch_ms += list(tm["vio_patch_ms"][base: base + v0["iters_per_level"][lvl]])
    ctx.set_kernel_timing(False)
    # in-kernel phase stamps (%globaltimer, CTA 0) of the persistent kernels, separate untimed pass
    phase = None
    try:
        ctx.set_phase_stamps(True)
        for _ in range(3):
            with torch.cuda.stream(ext_stream):
                flush.zero_()
            one_step()
        ctx.synchronize()
        st_ns = ctx.get_phase_stamps().astype(np.int64)
        lio_rows = [k for k in range(8) if st_ns[k, 0] > 0 and st_ns[k, 3] > st_ns[k, 1]]
        vio_rows = [k for k in range(8, 72) if st_ns[k, 0] > 0 and st_ns[k, 3] > st_ns[k, 1]]
        us = lambda rows, a, b: float(np.mean([(st_ns[k, b] - st_ns[k, a]) / 1e3 for k in rows])) if rows else None
        if lio_rows:
            phase = {"lio_build_us_per_iteration": us(lio_rows, 1, 3), "lio_iteration_us": us(lio_rows, 0, 5),
                     "lio_tail_us_all_arrived_to_solved": us(lio_rows, 3, 5),
                     "vio_build_us_per_iteration": us(vio_rows, 1, 3), "vio_iteration_us": us(vio_rows, 0, 5), "vio_tail_us_all_arrived_to_solved": us(vio_rows, 3, 5),
                     "note": "CTA 0's %globaltimer stamps, measured in a separate pass with stamping on; build = constants in place until the grid "
                             "barrier is passed, i.e. until the slowest CTA has finished its slice; tail = all CTAs arrived until the state is updated"}
    except Exception as e:  # measurement extra: never lose the bench line over it
        phase = {"error": repr(e)}
    finally:
        try:
            ctx.set_phase_stamps(False)
        except Exception:
            pass
    k1_iso_ms = ctx.profile_kernel(0, reps=20, flush_l2=True)
    k1_iso_warm_ms = ctx.profile_kernel(0, reps=20, flush_l2=False)
    k1_ms = float(np.mean(res_ms)) if res_ms else k1_iso_ms
    k2_iso_ms = ctx.profile_kernel(2, arg=0, reps=20, flush_l2=False) if has_vio else None
    k3_iso_ms = ctx.profile_kernel(1, reps=20, flush_l2=False)
    peak, peak_src = measured_peak_hbm()
    shard_pts = n // world + (1 if rank < n % world else 0)
    alg_bytes_iter = LIO_BYTES_PER_POINT * shard_pts
    # dominant residual kernel = the persistent LIO update kernel: one launch runs all LIO iterations of the step, so its
    # algorithmic bytes are iterations x 268 B x points, and its duration is measured by CUDA events INSIDE the timed region
    alg_bytes = alg_bytes_iter * int(rl["iters"])
    achieved = alg_bytes / (lio_ms * 1e-3) / 1e9
    achieved_iter_kernel = alg_bytes_iter / (k1_ms * 1e-3) / 1e9

    failed = False
    if rank == 0:
        cam = fr["cam_cfg"]
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms / K,
            "ms_per_step_median": med_ms, "ms_per_step_max": max_ms, "ms_per_step_all_rank0": [round(float(x), 4) for x in step_ms],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": fr["workload"], "name": args.config, "n_pts": n, "n_patches": npatch, "image": f"{cam.width}x{cam.height}" if has_vio else None,
                       "levels": L, "iters_per_step": iters_per_step,
                       "lio_iters": int(rl["iters"]), "vio_iters": int(v0["total_iters"]) if has_vio else 0, "l2": "flushed between steps (256 MiB write, untimed)",
                       "parallelism": (f"points/patches sharded over {world} ranks, compact information vector (29 / 37 doubles) exchanged per iteration " +
                                       ("inside the persistent kernel over NVLink peer memory" if args.comm == "p2p" else "with ncclAllReduce")) if world > 1 else "single GPU",
                       "map_planes": int(len(fr["map"]["planes"])), "matched_points": int(rl["M"][-1]), "tuning_flags": int(args.tuning),
                       "loop": ("residual + all-reduce + solve launches per iteration (loop_mode 0)" if (world > 1 and args.comm == "nccl") else
                                "one persistent cooperative kernel per update, gain solve replicated in every CTA")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": 1e3 * float(t_e2e.item()) / K, "path": "esikf_lio_update + esikf_vio_update (C ABI), pinned host buffers"},
            "e2e_shim": e2e_shim,
            "map_update": map_update,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"kernel": "lio_update_kernel (persistent: all LIO iterations of a step in one launch)",
                         "bound": "hbm", "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_point": LIO_BYTES_PER_POINT, "points_per_launch": shard_pts,
                         "iterations_per_launch": int(rl["iters"]), "avg_launch_ms_in_timed_region": lio_ms, "vio_update_ms_in_timed_region": vio_ms,
                         "residual_build_phase": (dict(phase, achieved=LIO_BYTES_PER_POINT * shard_pts / (phase["lio_build_us_per_iteration"] * 1e-6) / 1e9,
                                                       frac=LIO_BYTES_PER_POINT * shard_pts / (phase["lio_build_us_per_iteration"] * 1e-6) / 1e9 / peak)
                                                  if phase and phase.get("lio_build_us_per_iteration") else phase),
                         "per_iteration_kernel": {"kernel": "lio_residual_kernel (cold: nothing resident)", "achieved": achieved_iter_kernel, "frac": achieved_iter_kernel / peak,
                                                  "algorithmic_bytes_per_launch": alg_bytes_iter},
                         "avg_launch_ms_in_loop": k1_ms,
                         "avg_launch_ms_isolated_l2_flushed": k1_iso_ms, "avg_launch_ms_isolated_l2_warm": k1_iso_warm_ms,
                         "vio_patch_kernel_ms_in_loop": float(np.mean(patch_ms)) if patch_ms else None, "vio_patch_kernel_ms_isolated": k2_iso_ms,
                         "lio_solve_kernel_ms_in_loop": float(np.mean(solve_ms)) if solve_ms else None, "lio_solve_kernel_ms_isolated": k3_iso_ms,
                         "vio_achieved_gbs": (VIO_BYTES_PER_PATCH * npatch / world) / (float(np.mean(patch_ms)) * 1e-3) / 1e9 if patch_ms else None},
            "parity_vs_oracle": dict(parity, last_update_bit_identical_to_first=bool(same)),
        }
        if world == 1 and not args.no_cpu_baseline:
            so = native_baseline_build()
            if so:
                os.environ["ORC_BASELINE_SO"] = so
            frames = max(1, args.cpu_baseline_frames)
            cb = run_cpu_reference(fr, 4, frames, warm=1, budget_s=30)
            out["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": 4, "kind": "port",
                                   "sample": f"{cb['frames']} frames of the same workload ({cb['seconds']:.1f} s of CPU work); oracle restatement compiled "
                                             f"{'on this host' if so else 'in the build container'} with the "
                                             f"reference's flags, OpenMP capped at 4 threads like the reference (CMakeLists.txt:46-58); host has {os.cpu_count()} logical cores",
                                   "lio_iters_per_s": cb["lio_iters_per_s"], "vio_iters_per_s": cb["vio_iters_per_s"], "ms_per_frame": cb["ms_per_frame"]}
        print(json.dumps(out), flush=True)
        failed = not (parity["ok"] and same)
        if failed:
            print(f"PARITY FAILURE: {json.dumps(out['parity_vs_oracle'])}", file=sys.stderr, flush=True)
    elif not same:
        failed = True
        print(f"[rank {rank}] last timed update differs from the first", file=sys.stderr, flush=True)
    ctx.close()
    if dist is not None:
        f = torch.tensor([1 if failed else 0], device=dev)
        dist.all_reduce(f, op=dist.ReduceOp.MAX)
        failed = bool(f.item())
        dist.barrier()
        dist.destroy_process_group()
    if failed:
        sys.exit(1)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    b200_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()

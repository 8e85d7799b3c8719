"""Named synthetic workloads = the BASELINE.json configs (SURVEY.md Appendix C gives the YAML behind each).

Data generation only (fast_livo2_b200.synthetic); no ESIKF arithmetic, nothing from oracle/.
"""
from __future__ import annotations

from . import synthetic as S

# name -> (description, named GPU count in BASELINE.json, kwargs of synthetic.make_frame)
_HILTI_CAM = dict(model=1, width=720, height=540, fx=351.31400364193297, fy=351.4911744656785, cx=367.8522793375995, cy=253.8402144980996,
                  d=(-0.03696737352869157, -0.008917880497032812, 0.008912969593422046, -0.0037685977496087313, 0.0))


def _spec(name):
    if name == "small":  # quick functional case, not a BASELINE config
        return ("small test frame: 20 k LiDAR pts + 150 patches", 1,
                dict(seed=4, n_pts=20_000, n_map=150_000, n_patches=150, scene_scale=0.5))
    if name == "cfg1":
        return ("configs[0]: single synthetic frame, 5 k LiDAR pts, LIO-only, 3 iterations", 1,
                dict(seed=1, n_pts=5000, n_map=150_000, scene_scale=0.5, lio=S.LioCfg(max_iterations=3)))
    if name == "cfg2":
        return ("configs[1]: avia.yaml synthetic frame, 100k LiDAR pts + 640x512 image + 2k visual patches, LIO(<=5 it)+VIO(4 levels x <=5 it)", 1,
                dict(seed=0, n_pts=100_000, n_map=1_000_000, n_patches=2000))
    if name == "cfg3":
        return ("configs[2]: HILTI22 fisheye, 50k LiDAR pts + 720x540 image + 1k patches, voxel 0.4, non-identity extrinsic_R, corridor (degenerate) scene", 1,
                dict(seed=5, n_pts=50_000, n_map=600_000, n_patches=1000, lio=S.LioCfg(voxel_size=0.4, min_eigen_value=1e-4, max_points_num=100),
                     vio=S.VioCfg(img_point_cov=1000.0), cam=S.CamCfg(**_HILTI_CAM), ext=S.hilti_extrinsics(), scene="corridor", scene_scale=0.5))
    if name == "cfg4":
        return ("configs[3]: NTU_VIRAL Ouster, 260k LiDAR pts, LIO-only, beam_err 0.01", 4,
                dict(seed=12, n_pts=260_000, n_map=1_000_000, lio=S.LioCfg(beam_err=0.01)))
    if name == "cfg5":
        return ("configs[4]: MARS_LVIG, 300k LiDAR pts + 612x512 image + 4k patches, voxel 2.0, 5 pyramid levels", 8,
                dict(seed=13, n_pts=300_000, n_map=1_200_000, n_patches=4000, scene_scale=2.0, lio=S.LioCfg(voxel_size=2.0, min_eigen_value=0.005),
                     vio=S.VioCfg(levels=5, img_point_cov=1000.0), cam=S.CamCfg(width=612, height=512, fx=612.0 * 0.72, fy=612.0 * 0.72, cx=306.0, cy=256.0)))
    raise KeyError(name)


NAMES = ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5")


def describe(name):
    d, gpus, kw = _spec(name)
    return dict(workload=d, named_gpus=gpus)


def frame(name, cache_dir=None, **override):
    """The seeded frame of a named config (pickle-cached under cache_dir, default .frame_cache/); keyword overrides replace
    generator arguments."""
    d, gpus, kw = _spec(name)
    kw = dict(kw, **override)
    fr = S.cached_frame(cache_dir=cache_dir, **kw)
    fr.setdefault("vis_pos", [])
    fr["workload"] = d
    fr["named_gpus"] = gpus
    return fr

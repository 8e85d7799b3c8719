"""Second, independent restatement (plain numpy, written against the reference text, not against oracle/) of ONE LIO
iteration: TransformLidar + per-point covariance (voxel_map.cpp:376-390), voxel key / neighbour rule (:665-691), plane gate
and max-probability choice (:721-754), Jacobian / R^-1 (:414-458) and the information sums (:464-466). The C++ oracle must
agree with it point by point — this is what stands in for the golden vectors the reference does not ship."""
import numpy as np

import oracle_bind as O
from fast_livo2_b200 import synthetic as S

f32 = np.float32


def _body_cov(p, dept, beam):
    p = p.copy()
    if p[2] == 0:
        p[2] = 0.0001
    rng = f32(np.sqrt(p @ p))
    rv = f32(dept) * f32(dept)
    dv = np.sin(float(f32(beam)) * 0.017453293) ** 2
    d = p / np.linalg.norm(p)
    b1 = np.array([1.0, 1.0, -(d[0] + d[1]) / d[2]])
    b1 /= np.linalg.norm(b1)
    b2 = np.cross(b1, d)
    b2 /= np.linalg.norm(b2)
    A = float(rng) * S.skew(d) @ np.stack([b1, b2], 1)
    return np.outer(d, d) * float(rv) + A @ (np.eye(2) * dv) @ A.T


def _key(pw, vs):
    loc = np.zeros(3, f32)
    for j in range(3):
        loc[j] = f32(pw[j] / vs)
        if loc[j] < 0:
            loc[j] = f32(float(loc[j]) - 1.0)
    return loc, tuple(int(np.trunc(float(x))) for x in loc)


def _eval(pl, pw, var, sigma_num):
    n, c = pl["normal"], pl["center"]
    pv = np.zeros((6, 6))
    iu = np.triu_indices(6)
    pv[iu] = pl["plane_var"]
    pv = pv + pv.T - np.diag(np.diag(pv))
    sd = n @ pw + float(pl["d"])
    dtp = f32(abs(sd))
    dtc = f32(((c - pw) ** 2).sum())
    with np.errstate(invalid="ignore"):
        rd = np.sqrt(f32(dtc - f32(dtp * dtp)))
    if not (float(rd) <= 3.0 * float(pl["radius"])):
        return None
    J = np.concatenate([pw - c, -n])
    sig = J @ pv @ J + n @ var @ n
    if not (float(dtp) < sigma_num * np.sqrt(sig)):
        return None
    return 1.0 / np.sqrt(sig) * np.exp(-0.5 * float(dtp) * float(dtp) / sig), f32(sd)


def _check_one_lio_iteration(fr, pts, state):
    """One LIO pass of the C++ oracle against the numpy restatement, point by point; returns (matched, via neighbour, multi-plane)."""
    cfg, ext, vm = fr["lio_cfg"], fr["ext"], fr["map"]
    st = S.unpack_state(state)
    R, t, P = st["R"], st["p"], st["cov"]
    roots = {tuple(k): (f, c) for k, f, c in zip(vm["keys"].tolist(), vm["first"], vm["count"])}
    vsf = float(f32(cfg.voxel_size))
    ql = float(f32(f32(cfg.voxel_size) / f32(4)))
    lio = O.OracleLIO(cfg, ext)
    lio.set_map(vm)
    sp = lio.single_pass(pts, state, state)
    HTH, HTz, n_match, n_neigh, n_multi = np.zeros((6, 6)), np.zeros(6), 0, 0, 0
    for i, pb in enumerate(pts.astype(np.float64)):
        pz = pb.copy()
        if pz[2] == 0:
            pz[2] = 0.001
        bc = _body_cov(pz, cfg.dept_err, cfg.beam_err)
        cm = S.skew(ext.extR @ pz + ext.extT)
        pi = ext.extR @ pb + ext.extT
        pw = (R @ pi + t).astype(f32).astype(np.float64)
        var = R @ bc @ R.T + (-cm) @ P[0:3, 0:3] @ (-cm).T + P[3:6, 3:6]
        np.testing.assert_allclose(sp["point_w"][i], pw, rtol=0, atol=0)
        np.testing.assert_allclose(sp["var"][i], var, rtol=1e-11, atol=1e-18)
        loc, key = _key(pw, cfg.voxel_size)
        best = None
        if key in roots:
            f, c = roots[key]
            n_multi += c > 1
            for j in range(f, f + c):
                e = _eval(vm["planes"][j], pw, var, cfg.sigma_num)
                if e is not None and (best is None or e[0] > best[0]):
                    best = (e[0], j, e[1])
            if best is None:
                nk = list(key)
                for a in range(3):
                    center = (0.5 + key[a]) * vsf
                    if float(loc[a]) > center + ql:
                        nk[a] += 1
                    elif float(loc[a]) < center - ql:
                        nk[a] -= 1
                if tuple(nk) in roots:
                    f, c = roots[tuple(nk)]
                    for j in range(f, f + c):
                        e = _eval(vm["planes"][j], pw, var, cfg.sigma_num)
                        if e is not None and (best is None or e[0] > best[0]):
                            best = (e[0], j, e[1])
                    n_neigh += best is not None
        if best is None:
            assert sp["plane"][i] == -1
            continue
        n_match += 1
        assert sp["plane"][i] == best[1] and sp["dis"][i] == best[2]
        pl = vm["planes"][best[1]]
        n, c = pl["normal"], pl["center"]
        pv = np.zeros((6, 6))
        iu = np.triu_indices(6)
        pv[iu] = pl["plane_var"]
        pv = pv + pv.T - np.diag(np.diag(pv))
        J = np.concatenate([R @ pi + t - c, -n])  # prior pose == current pose in this single pass
        RE = R @ ext.extR
        rinv = 1.0 / (0.001 + J @ pv @ J + n @ (RE @ bc @ RE.T) @ n)
        A = S.skew(pi) @ R.T @ n
        H = np.concatenate([A, n])
        np.testing.assert_allclose(sp["H"][i], H, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(sp["R_inv"][i], rinv, rtol=1e-11)
        HTH += rinv * np.outer(H, H)
        HTz += rinv * H * (-float(best[2]))
    # the full oracle's first-iteration information matrix over the same points
    r = lio.state_estimation(pts, state, state)
    assert r["M"][0] == n_match
    if n_match:
        np.testing.assert_allclose(r["HTH"][0], HTH, rtol=1e-11)
        np.testing.assert_allclose(r["HTz"][0], HTz, rtol=1e-9, atol=1e-9)
    return n_match, n_neigh, n_multi


def test_numpy_restatement_agrees_with_cpp_oracle(small_frame):
    fr = small_frame
    n_match, _, n_multi = _check_one_lio_iteration(fr, fr["pts"][:700], fr["state_prior"])
    assert n_match > 500 and n_multi > 0


def test_numpy_restatement_agrees_on_voxel_boundaries_and_negative_keys(small_frame):
    """The float voxel key (voxel_map.cpp:665-671: double quotient narrowed to float, "-1 if negative", truncation) and the
    unit-mixing neighbour rule (:680-691) where they are fragile: world points EXACTLY on voxel boundaries (identity pose and
    extrinsics, coordinates that are exact multiples of the voxel size, both signs — trunc(q - 1) differs from floor there),
    z == 0 (the 0.001 substitution of :352) and points half a float ulp away from a boundary."""
    fr = dict(small_frame)
    fr["ext"] = S.Extrinsics(np.eye(3), np.zeros(3), small_frame["ext"].Rcl, small_frame["ext"].Pcl)
    st = S.unpack_state(small_frame["state_prior"])
    state = S.pack_state(np.eye(3), np.zeros(3), 1.0, st["v"], g=st["g"], cov=st["cov"])
    vs = fr["lio_cfg"].voxel_size
    keys = fr["map"]["keys"]
    rng = np.random.default_rng(4)
    pick = keys[rng.choice(len(keys), 60, replace=False)].astype(np.float64)
    on_corner = (pick * vs).astype(np.float32)                      # the low corner of existing voxels: exact multiples
    on_face = on_corner.copy()
    on_face[:, 1] += np.float32(0.37 * vs)                          # exact in x and z only
    just_below = np.nextafter(on_corner, np.float32(-np.inf))
    just_above = np.nextafter(on_corner, np.float32(np.inf))
    inside = ((pick + rng.uniform(0.05, 0.95, pick.shape)) * vs).astype(np.float32)
    zero_z = inside.copy()
    zero_z[:, 2] = 0.0
    pts = np.ascontiguousarray(np.concatenate([on_corner, on_face, just_below, just_above, inside, zero_z]))
    assert (pts < 0).any() and (pts > 0).any()
    n_match, n_neigh, _ = _check_one_lio_iteration(fr, pts, state)
    assert n_match > 20


def test_numpy_restatement_of_one_vio_iteration(small_vio_frame):
    """First iteration of updateState at the coarsest level (vio.cpp:1540-1634, 1660-1662) restated in numpy with the
    reference's float / double narrowing points; the oracle's H^T H, H^T z and mean squared error must agree."""
    fr = small_vio_frame
    ext, cam, vcfg = fr["ext"], fr["cam_cfg"], fr["vio_cfg"]
    w = O.oracle_warp_patches(fr, fr["state_prior"])
    n = 40
    pos, wp, sl = fr["vis_pos"][:n], w["warp_patch"][:n], w["search_levels"][:n]
    st = S.unpack_state(fr["state_prior"])
    Rli, Pli = ext.extR.T, -ext.extR.T @ ext.extT
    Rci = ext.Rcl @ Rli
    Pci = ext.Rcl @ Pli + ext.Pcl
    Pic = -Rci.T @ Pci
    Jdp_dR = -Rci @ S.skew(Pic)
    Rcw = Rci @ st["R"].T
    Pcw = -Rci @ st["R"].T @ st["p"] + Pci
    level = vcfg.levels - 1
    img = fr["img"].astype(np.int64)
    width = cam.width
    flat = img.reshape(-1)
    HTH, HTz, err, nm = np.zeros((7, 7)), np.zeros(7), f32(0), 0
    for i in range(n):
        scale = 1 << (level + int(sl[i]))
        inv_scale = f32(1.0) / f32(scale)
        pf = Rcw @ pos[i] + Pcw
        pc = np.array([cam.fx * pf[0] / pf[2] + cam.cx, cam.fy * pf[1] / pf[2] + cam.cy])
        zi = 1.0 / pf[2]
        Jdpi = np.array([[cam.fx * zi, 0, -cam.fx * pf[0] * zi * zi], [0, cam.fy * zi, -cam.fy * pf[1] * zi * zi]])
        u_ref, v_ref = f32(pc[0]), f32(pc[1])
        u_i = int(np.floor(f32(pc[0] / scale)) * scale)
        v_i = int(np.floor(f32(pc[1] / scale)) * scale)
        su, sv = f32((u_ref - f32(u_i)) / f32(scale)), f32((v_ref - f32(v_i)) / f32(scale))
        wtl, wtr = f32((1.0 - float(su)) * (1.0 - float(sv))), f32(float(su) * (1.0 - float(sv)))
        wbl, wbr = f32((1.0 - float(su)) * float(sv)), f32(su * sv)
        bil = lambda a, b, c, d: f32(f32(f32(wtl * f32(a)) + f32(wtr * f32(b))) + f32(wbl * f32(c))) + f32(wbr * f32(d))
        perr = f32(0)
        for x in range(8):
            for y in range(8):
                b = (v_i + x * scale - 4 * scale) * width + u_i - 4 * scale + y * scale
                sw = scale * width
                T = lambda o: flat[b + o]
                du = f32(0.5) * f32(bil(T(scale), T(2 * scale), T(sw + scale), T(sw + 2 * scale)) - bil(T(-scale), T(0), T(sw - scale), T(sw)))
                dv = f32(0.5) * f32(bil(T(sw), T(scale + sw), T(2 * sw), T(2 * sw + scale)) - bil(T(-sw), T(-sw + scale), T(0), T(scale)))
                Jimg = np.array([float(du), float(dv)]) * st["inv_expo"] * float(inv_scale)
                Jdphi = Jimg @ Jdpi @ S.skew(pf)
                Jdp = -Jimg @ Jdpi
                JdR = Jdphi @ Rci + Jdp @ Jdp_dR
                Jdt = Jdp @ Rcw
                cur = float(bil(T(0), T(scale), T(sw), T(sw + scale)))
                res = st["inv_expo"] * cur - 1.0 * float(wp[i][64 * level + x * 8 + y])
                h = np.concatenate([JdR, Jdt, [cur]])
                HTH += np.outer(h, h)
                HTz += h * res
                perr = f32(float(perr) + res * res)
                nm += 1
        err = f32(err + perr)
    err = f32(err / f32(nm))
    vio = O.OracleVIO(cam, ext, vcfg)
    o = vio.update(fr["img"], pos, wp, sl, np.ones(n), fr["state_prior"], fr["state_prior"])
    np.testing.assert_allclose(o["HTH"][level][0], HTH, rtol=1e-11)
    np.testing.assert_allclose(o["HTz"][level][0], HTz, rtol=1e-10, atol=1e-8)
    assert o["error_trace"][level][0] == err


def _numpy_gain_solution(HTH_m, HTz_m, P, sign):
    """K_1 = (H^T H + P^-1)^-1 with the information block zero-padded to 19 x 19; first-iteration solution (vec = 0):
    sign * K_1[:, :m] H^T z   (voxel_map.cpp:462-472 with sign +1, vio.cpp:1660-1667 with sign -1)."""
    m = len(HTz_m)
    H = np.zeros((19, 19))
    H[:m, :m] = HTH_m
    K1 = np.linalg.inv(H + np.linalg.inv(P))
    return sign * K1[:, :m] @ HTz_m


def test_first_iteration_solutions_match_numpy_gain_formula(small_frame, small_vio_frame):
    """The gain algebra (a7 / a9) restated with numpy's LAPACK inverses instead of the oracle's own 19 x 19 elimination."""
    fr = small_frame
    lio = O.OracleLIO(fr["lio_cfg"], fr["ext"])
    lio.set_map(fr["map"])
    r = lio.state_estimation(fr["pts"], fr["state_prior"], fr["state_prior"])
    P = S.unpack_state(fr["state_prior"])["cov"]
    want = _numpy_gain_solution(r["HTH"][0], r["HTz"][0], P, +1.0)
    np.testing.assert_allclose(r["solution"][0], want, rtol=1e-7, atol=1e-10 * np.abs(want).max())

    fv = small_vio_frame
    w = O.oracle_warp_patches(fv, fv["state_prior"])
    vio = O.OracleVIO(fv["cam_cfg"], fv["ext"], fv["vio_cfg"])
    o = vio.update(fv["img"], fv["vis_pos"], w["warp_patch"], w["search_levels"], fv["inv_ref_expo"], fv["state_prior"], fv["state_prior"])
    top = fv["vio_cfg"].levels - 1
    assert o["accepted_per_level"][top] >= 1
    Pv = S.unpack_state(fv["state_prior"])["cov"] / fv["vio_cfg"].img_point_cov
    want = _numpy_gain_solution(o["HTH"][top][0], o["HTz"][top][0], Pv, -1.0)
    np.testing.assert_allclose(o["solution"][top][0], want, rtol=1e-7, atol=1e-10 * np.abs(want).max())


def test_numpy_restatement_of_the_inverse_compositional_variant(small_vio_frame):
    """precomputeReferencePatches (vio.cpp:1327-1396) and the first iteration of updateStateInverse (:1398-1518) restated in
    numpy: reference-image gradients -> world-frame Jacobian rows, float residual, 6 x 6 information block."""
    fr = small_vio_frame
    ext, cam, vcfg = fr["ext"], fr["cam_cfg"], fr["vio_cfg"]
    n = 24
    w = O.oracle_warp_patches(fr, fr["state_prior"])
    pos, wp = fr["vis_pos"][:n], w["warp_patch"][:n]
    refs = O.inverse_refs_from_frame(fr)
    refs = {k: (v if k == "ref_imgs" else v[:n]) for k, v in refs.items()}
    vio = O.OracleVIO(cam, ext, vcfg)
    vio.set_inverse_refs(**refs)
    level = vcfg.levels - 1
    scale = 1 << level
    H_inv = vio.precompute_reference_patches(pos, level)

    def taps(img_flat, width, pc):
        u_i = int(np.floor(f32(pc[0] / scale)) * scale)
        v_i = int(np.floor(f32(pc[1] / scale)) * scale)
        su = f32((f32(pc[0]) - f32(u_i)) / f32(scale))
        sv = f32((f32(pc[1]) - f32(v_i)) / f32(scale))
        wts = (f32((1.0 - float(su)) * (1.0 - float(sv))), f32(float(su) * (1.0 - float(sv))), f32((1.0 - float(su)) * float(sv)), f32(su * sv))
        bil = lambda a, b, c, d: f32(f32(f32(wts[0] * f32(a)) + f32(wts[1] * f32(b))) + f32(wts[2] * f32(c))) + f32(wts[3] * f32(d))
        return u_i, v_i, bil

    width = cam.width
    ref_flat = fr["img_ref"].astype(np.int64).reshape(-1)
    R_ref = fr["T_ref"][0]
    for i in range(n):
        depth = np.linalg.norm(pos[i] - refs["ref_pos"][i])
        pf = refs["ref_f"][i] * depth
        zi = 1.0 / pf[2]
        Jdpi = np.array([[cam.fx * zi, 0, -cam.fx * pf[0] * zi * zi], [0, cam.fy * zi, -cam.fy * pf[1] * zi * zi]])
        u_i, v_i, bil = taps(ref_flat, width, refs["ref_px"][i])
        sw = scale * width
        for x in (0, 3, 7):
            for y in (0, 4, 7):
                b = (v_i + x * scale - 4 * scale) * width + u_i - 4 * scale + y * scale
                T = lambda o: ref_flat[b + o]
                du = f32(0.5) * f32(bil(T(scale), T(2 * scale), T(sw + scale), T(sw + 2 * scale)) - bil(T(-scale), T(0), T(sw - scale), T(sw)))
                dv = f32(0.5) * f32(bil(T(sw), T(scale + sw), T(2 * sw), T(2 * sw + scale)) - bil(T(-sw), T(-sw + scale), T(0), T(scale)))
                Jimg = np.array([float(du), float(dv)]) * (1.0 / scale)
                JdR = Jimg @ Jdpi @ R_ref @ S.skew(pos[i])
                Jdt = -Jimg @ Jdpi @ R_ref
                np.testing.assert_allclose(H_inv[i, x * 8 + y], np.concatenate([JdR, Jdt]), rtol=1e-12, atol=1e-12)

    # first iteration at the coarsest level: H rows rotated into the current IMU frame, float residual, H^T H / H^T z / error
    st = S.unpack_state(fr["state_prior"])
    Rwi, Pwi = st["R"], st["p"]
    Rcw, Pcw = S.camera_pose(ext, Rwi, Pwi)
    cur_flat = fr["img"].astype(np.int64).reshape(-1)
    HTH, HTz, err, nm = np.zeros((6, 6)), np.zeros(6), f32(0), 0
    for i in range(n):
        pf = Rcw @ pos[i] + Pcw
        pc = np.array([cam.fx * pf[0] / pf[2] + cam.cx, cam.fy * pf[1] / pf[2] + cam.cy])
        u_i, v_i, bil = taps(cur_flat, width, pc)
        sw = scale * width
        perr = f32(0)
        for x in range(8):
            for y in range(8):
                b = (v_i + x * scale - 4 * scale) * width + u_i - 4 * scale + y * scale
                T = lambda o: cur_flat[b + o]
                res = float(f32(bil(T(0), T(scale), T(sw), T(sw + scale)) - f32(wp[i][64 * level + x * 8 + y])))
                J_dR, J_dt = H_inv[i, x * 8 + y, :3], H_inv[i, x * 8 + y, 3:]
                h = np.concatenate([J_dR @ Rwi + (J_dt @ S.skew(Pwi)) @ Rwi, J_dt @ Rwi])
                HTH += np.outer(h, h)
                HTz += h * res
                perr = f32(float(perr) + res * res)
                nm += 1
        err = f32(err + perr)
    err = f32(err / f32(nm))
    vio.set_inverse(True)
    o = vio.update(fr["img"], pos, wp, np.zeros(n, np.int32), np.ones(n), fr["state_prior"], fr["state_prior"])
    np.testing.assert_allclose(o["HTH"][level][0][:6, :6], HTH, rtol=1e-10, atol=1e-10 * np.abs(HTH).max())
    np.testing.assert_allclose(o["HTz"][level][0][:6], HTz, rtol=1e-9, atol=1e-9 * np.abs(HTz).max())
    assert not o["HTH"][level][0][6].any() and not o["HTH"][level][0][:, 6].any()
    assert o["error_trace"][level][0] == err
    P = S.unpack_state(fr["state_prior"])["cov"] / vcfg.img_point_cov
    want = _numpy_gain_solution(HTH, HTz, P, -1.0)
    np.testing.assert_allclose(o["solution"][level][0], want, rtol=1e-6, atol=1e-9 * np.abs(want).max())
    vio.set_inverse(False)
    fwd = vio.update(fr["img"], pos, wp, np.zeros(n, np.int32), np.ones(n), fr["state_prior"], fr["state_prior"])
    assert fwd["HTH"][level][0][6, 6] > 0  # the forward variant is untouched by the switch


def _numpy_image_patch(img, pc, level):
    """getImagePatch (vio.cpp:203-225) with the oracle's border rule written out: raw linear indices v * width + u (left /
    right overhangs wrap to the neighbouring row) and 0 where the index leaves [0, width * height) (DESIGN §4)."""
    h, w = img.shape
    flat = img.reshape(-1)
    s = 1 << level
    u_ref, v_ref = f32(pc[0]), f32(pc[1])
    ui = int(np.floor(f32(pc[0] / s)) * f32(s))
    vi = int(np.floor(f32(pc[1] / s)) * f32(s))
    su, sv = (u_ref - f32(ui)) / f32(s), (v_ref - f32(vi)) / f32(s)
    wtl, wtr = f32((1.0 - float(su)) * (1.0 - float(sv))), f32(float(su) * (1.0 - float(sv)))
    wbl, wbr = f32((1.0 - float(su)) * float(sv)), su * sv
    pix = lambda i: f32(flat[i]) if 0 <= i < w * h else f32(0)
    out = np.zeros(64, f32)
    for x in range(8):
        base = (vi - 4 * s + x * s) * w + (ui - 4 * s)
        for y in range(8):
            b = base + y * s
            out[x * 8 + y] = wtl * pix(b) + wtr * pix(b + s) + wbl * pix(b + s * w) + wbr * pix(b + s * w + s)
    return out


def test_numpy_restatement_of_image_patch_at_the_border(small_vio_frame):
    """Centres whose footprints wrap left / right and leave the buffer above / below, at every level: the oracle's pix()
    rule bit for bit. The reference source pins the in-buffer wrap (test_oracle_ref_pin_vio); this pins the 0 outside."""
    from parity_util import border_pixels

    fr = small_vio_frame
    cam = fr["cam_cfg"]
    vio = O.OracleVIO(cam, fr["ext"], fr["vio_cfg"])
    px = border_pixels(cam, fr["vio_cfg"].levels, seed=3)[0]
    px = np.concatenate([px, [[-3.5, -2.25], [cam.width + 2.75, cam.height + 1.5], [0.0, 0.0]]])
    n_outside = 0
    for level in range(fr["vio_cfg"].levels):
        s = 1 << level
        for c in px:
            want = _numpy_image_patch(fr["img"], c, level)
            assert np.array_equal(vio.get_image_patch(fr["img"], c, level), want), (level, c)
            n_outside += (np.floor(c[1] / s) * s - 4 * s) * cam.width + np.floor(c[0] / s) * s - 4 * s < 0
    assert n_outside > 20

"""CPU: pin the oracle (oracle/*.py) against the third-party arithmetic the reference calls, and against the
committed fixtures.  Pinned: torch grid_sample (= torch::grid_sampler, superpoint_tensorrt.cpp:209),
cv2.BFMatcher(NORM_L2, True) (= cv::BFMatcher, loop_cam.cpp:147), Jacobians vs central differences,
NMS2 vs a literal 2-D re-implementation of the C++ loops."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from omniswarm_b200 import synth
from oracle import frontend_ref as fr
from oracle import solver_ref as sr


def nms2_literal(prob, thres, max_num, dist=4):
    """NMS2 as the C++ is written (superpoint_tensorrt.cpp:237-310) with 2-D indexing and explicit flat-address
    emulation of cv::Mat::at for out-of-row columns; independent of oracle.nms2's vectorised form."""
    H, W = prob.shape
    pts = [(x, y) for y in range(H) for x in range(W) if prob[y, x] > np.float32(thres)]
    grid = np.zeros(H * W, np.int8); inds = np.zeros(H * W, np.uint16); conf = np.zeros(H * W, np.float32)
    for i, (x, y) in enumerate(pts):
        grid[y * W + x] = 1; inds[y * W + x] = i & 0xFFFF; conf[y * W + x] = prob[y, x]
    for (x, y) in pts:
        if grid[y * W + x] != 1:
            continue
        for k in range(-dist, dist + 1):
            for j in range(-dist, dist + 1):
                if j == 0 and k == 0:
                    continue
                L = (y + k) * W + (x + j)
                if 0 <= L < H * W and conf[L] < conf[y * W + x]:
                    grid[L] = 0
        grid[y * W + x] = 2
    out = []
    for v in range(H):
        for u in range(W):
            if grid[v * W + u] == 2:
                out.append((pts[int(inds[v * W + u])], float(conf[v * W + u]), v * W + u))
    out.sort(key=lambda t: (-t[1], t[2]))
    out = out[:max_num]
    return np.array([p for p, _, _ in out], np.float32).reshape(-1, 2), np.array([c for _, c, _ in out], np.float32)


@pytest.mark.parametrize("seed,density", [(1, 0.03), (2, 0.2), (3, 0.6)])
def test_nms2_matches_literal_loops(seed, density):
    rng = np.random.default_rng(seed)
    H, W = 24, 40
    p = rng.uniform(0, 0.014, (H, W)).astype(np.float32)
    m = rng.uniform(size=(H, W)) < density
    p[m] = rng.choice(np.linspace(0.02, 0.9, 12).astype(np.float32), m.sum())   # many exact ties
    k1, c1 = fr.get_keypoints(p, 0.015, 30)
    k2, c2 = nms2_literal(p, 0.015, 30)
    assert np.array_equal(k1, k2) and np.array_equal(c1, c2)


def test_nms2_is_order_dependent_not_local_max():
    """A suppressed point never suppresses others (SURVEY.md A.2 consequence i)."""
    p = np.zeros((16, 32), np.float32)
    p[5, 5], p[5, 8], p[5, 11] = 0.9, 0.5, 0.3     # 0.9 kills 0.5; 0.5 (dead) does NOT kill 0.3
    k, c = fr.get_keypoints(p, 0.015, 10)
    assert {tuple(x) for x in k.tolist()} == {(5.0, 5.0), (11.0, 5.0)}
    p[5, 5], p[5, 8], p[5, 11] = 0.3, 0.5, 0.9     # raster order reversed: 0.3 active first, later zeroed by 0.5,
    k, c = fr.get_keypoints(p, 0.015, 10)          # 0.5 zeroed by 0.9 -> only 0.9 survives
    assert {tuple(x) for x in k.tolist()} == {(11.0, 5.0)}


def test_grid_sample_pin():
    """Restated bilinear formula of SURVEY.md A.3 == torch.grid_sample(align_corners=False, zeros)."""
    rng = np.random.default_rng(0)
    H, W = 64, 96
    desc = rng.standard_normal((256, H // 8, W // 8)).astype(np.float32)
    kpts = np.stack([rng.integers(0, W, 40), rng.integers(0, H, 40)], 1).astype(np.float32)
    kpts[:4] = [[0, 0], [W - 1, H - 1], [0, H - 1], [W - 1, 0]]           # corners: taps fall outside -> zeros
    comp, mean = synth.pca_matrices(0)
    got = fr.compute_descriptors(desc, kpts, W, H, comp, mean)
    S = np.zeros((len(kpts), 256), np.float64)
    Hc, Wc = H // 8, W // 8
    for n, (x, y) in enumerate(kpts):
        fx, fy = x / 8 - 0.5, y / 8 - 0.5
        x0, y0 = int(np.floor(fx)), int(np.floor(fy))
        for dy in (0, 1):
            for dx in (0, 1):
                xx, yy = x0 + dx, y0 + dy
                if 0 <= xx < Wc and 0 <= yy < Hc:
                    S[n] += desc[:, yy, xx] * (1 - abs(fx - xx)) * (1 - abs(fy - yy))
    S /= np.sqrt((S ** 2).sum(0, keepdims=True))      # per-CHANNEL norm over keypoints
    ref = (S - mean) @ comp.T.astype(np.float64)
    assert np.abs(got - ref).max() < 2e-5


def test_bfmatcher_pin():
    cv2 = pytest.importorskip("cv2")
    for seed, (nq, nt) in enumerate([(57, 43), (200, 200), (1, 5), (5, 1)]):
        a = synth.local_descriptors(nq, 10 + seed)
        b = synth.local_descriptors(nt, 20 + seed, base=a) if nt <= nq else synth.local_descriptors(nt, 20 + seed)
        qi, ti, dist = fr.bf_crosscheck(a, b)
        ms = sorted(cv2.BFMatcher(cv2.NORM_L2, True).match(a, b), key=lambda m: m.queryIdx)
        assert [m.queryIdx for m in ms] == qi.tolist() and [m.trainIdx for m in ms] == ti.tolist()
        assert np.allclose([m.distance for m in ms], dist, rtol=1e-5, atol=1e-6)


def test_jacobians_vs_central_differences():
    g = synth.pose_graph(3, 12, n_uwb=20, n_loop=15, n_det=8, n_bearing=9, seed=3)
    worst = 0.0
    for f in range(len(g["ftype"])):
        a, b = g["ia"][f], g["ib"][f]
        pa, pb = g["init"][a], g["init"][b]
        _, Ja, Jb = sr.factor_residual_jacobian(int(g["ftype"][f]), pa, pb, g["payload"][f])
        for which, J in ((0, Ja), (1, Jb)):
            for j in range(4):
                h = 1e-6
                p1, p2 = [pa.copy(), pb.copy()], [pa.copy(), pb.copy()]
                p1[which][j] += h; p2[which][j] -= h
                r1 = sr.factor_residual_jacobian(int(g["ftype"][f]), p1[0], p1[1], g["payload"][f])[0]
                r2 = sr.factor_residual_jacobian(int(g["ftype"][f]), p2[0], p2[1], g["payload"][f])[0]
                worst = max(worst, np.max(np.abs((r1 - r2) / (2 * h) - J[:, j])) / (1 + np.max(np.abs(J[:, j]))))
    assert worst < 1e-6


def test_create_cov6d_sqrt_information():
    """RelativePoseFactor4d::CreateCov6d (factors.hpp:255-263): element-wise sqrt(|inv(cov4)|)."""
    cov6 = np.diag([1e-4, 2e-4, 3e-4, 1.0, 1.0, 5e-5])
    cov6[0, 1] = cov6[1, 0] = 5e-5
    S = sr.create_cov6d_sqrt_inf(cov6)
    cov4 = np.zeros((4, 4)); cov4[:3, :3] = cov6[:3, :3]; cov4[3, 3] = cov6[5, 5]
    assert np.allclose(S * S, np.abs(np.linalg.inv(cov4)))


def test_golden_fixtures_reproduce():
    """The committed fixtures are what the oracle produces today."""
    comp, mean = synth.pca_matrices(0)
    z = np.load(os.path.join(GOLDEN, "postproc.npz"))
    for n in "abc":
        k, c = fr.get_keypoints(z[f"{n}_semi"], 0.015, 50)
        assert np.array_equal(k, z[f"{n}_kpts"]) and np.array_equal(c, z[f"{n}_conf"])
        d = fr.compute_descriptors(z[f"{n}_desc"], k, 96, 64, comp, mean)
        assert np.allclose(d, z[f"{n}_out"], atol=1e-6, equal_nan=True)
    z = np.load(os.path.join(GOLDEN, "matcher.npz"))
    qi, ti, dist = fr.bf_crosscheck(z["q"], z["t"])
    assert np.array_equal(qi, z["qi"]) and np.array_equal(ti, z["ti"]) and np.array_equal(dist, z["dist"])
    z = np.load(os.path.join(GOLDEN, "superpoint_net.npz"))
    semi, desc = fr.superpoint_net(z["img"], synth.superpoint_weights(0))
    assert np.allclose(semi, z["semi"], atol=1e-6) and np.allclose(desc, z["desc"].astype(np.float32), atol=2e-3)
    z = np.load(os.path.join(GOLDEN, "netvlad.npz"))
    assert np.allclose(fr.netvlad_net(z["img"], synth.netvlad_weights(0)), z["out"], atol=1e-6)
    z = np.load(os.path.join(GOLDEN, "graph_small.npz"))
    g = synth.pose_graph(3, 12, n_uwb=20, n_loop=15, n_det=8, n_bearing=9, seed=3)
    res = sr.solve(g)
    assert np.allclose(res["poses"], z["poses"], atol=1e-9) and abs(res["final_cost"] - z["final_cost"]) < 1e-9


def test_query_rule_quirks():
    """SURVEY.md A.4: `<=` on the index test, stale `distance` from the remote search, fall-through id."""
    dim = 16
    rng = np.random.default_rng(0)
    rows = rng.standard_normal((12, dim)).astype(np.float32)
    rows /= np.linalg.norm(rows, axis=1, keepdims=True)
    det = fr.LoopDetectorDB(self_id=1, dim=dim, inner_product_thres=0.5, match_index_dist=5)
    for i, r in enumerate(rows[:8]):
        det.add_frame(i, 1, [r], [10])
    # query == newest row (7): score 1.0 but label 7 > ntotal - max_index = 3 -> rejected; falls through
    idq, dist = det.query(1, rows[7], False, False)
    assert dist == -1.0 and idq != -1              # last valid label returned, distance untouched
    # query == old row 2: accepted with its score
    idq, dist = det.query(1, rows[2], False, False)
    assert idq == 2 and abs(dist - 1.0) < 1e-6
    # remote hit leaves a stale distance that validates a failing local search
    det.add_frame(100, 2, [rows[9]], [10])
    idq, dist = det.query(1, rows[9], False, False)
    assert abs(dist - 1.0) < 1e-6 and idq < fr.REMOTE_MAGIN_NUMBER     # local id, remote score
    # remote keyframe queries the LOCAL db with max_index 1
    idq, dist = det.query(2, rows[7], False, False)
    assert idq == 7 and abs(dist - 1.0) < 1e-6


# ---------------------------------------------------------------------------------------------------------------
# geometric filter (SURVEY 8f-1): the deterministic homography RANSAC pinned against the real OpenCV
# ---------------------------------------------------------------------------------------------------------------
def _homography_case(seed, n=200, n_out=60, noise=0.3):
    rng = np.random.default_rng(seed)
    src = rng.uniform(0, 640, (n, 2)).astype(np.float32); src[:, 1] *= 0.75
    H = np.array([[1.0 + rng.normal(0, 0.03), rng.normal(0, 0.03), rng.normal(0, 15)],
                  [rng.normal(0, 0.03), 1.0 + rng.normal(0, 0.03), rng.normal(0, 15)],
                  [rng.normal(0, 2e-5), rng.normal(0, 2e-5), 1.0]])
    p = np.c_[src, np.ones(n)] @ H.T
    dst = (p[:, :2] / p[:, 2:]).astype(np.float32) + rng.normal(0, noise, (n, 2)).astype(np.float32)
    out = rng.choice(n, n_out, replace=False)
    dst[out] += (rng.uniform(25, 80, (n_out, 2)) * rng.choice([-1, 1], (n_out, 2))).astype(np.float32)
    truth = np.ones(n, np.uint8); truth[out] = 0
    return src, dst, truth


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_homography_mask_equals_opencv_on_separated_data(seed):
    """cv::findHomography(old_2d, new_2d, CV_RANSAC, 3, mask) (loop_detector.cpp:590) through the Python binding of the
    same OpenCV function: inliers with 0.3 px noise, outliers 25-80 px away -> the masks must be identical."""
    import cv2
    from oracle import geometry_ref as gr
    src, dst, truth = _homography_case(seed)
    m, c, h = gr.homography_ransac_mask(src, dst, 3.0, seed=seed)
    _, mc = cv2.findHomography(src, dst, cv2.RANSAC, 3.0)
    assert np.array_equal(m, mc.ravel()) and np.array_equal(m, truth) and c == int(truth.sum()) and h >= 0


def test_homography_edge_cases_and_pair_filter():
    from oracle import geometry_ref as gr
    src, dst, truth = _homography_case(5, n=40, n_out=10)
    assert gr.homography_ransac_mask(src[:3], dst[:3])[1] == 0              # fewer than 4 points: nothing passes
    m4 = gr.homography_ransac_mask(src[truth == 1][:4], dst[truth == 1][:4])
    assert m4[1] == 4                                                       # exactly 4: the model fits them
    same = np.repeat(src[:1], 10, 0)
    assert gr.homography_ransac_mask(same, same)[2] == -1                   # all points identical: every sample degenerate
    # the reference's filter: matches whose NEW landmark has no 3-D flag are dropped first (loop_detector.cpp:572-586)
    n = len(src)
    flags = np.ones(n, np.uint8); flags[::5] = 0
    qn, qo = gr.loop_pair_filter(list(range(n)), list(range(n)), flags, dst, src)
    assert set(qn.tolist()) == {i for i in range(n) if flags[i] and truth[i]} and np.array_equal(qn, qo)
    assert gr.loop_pair_filter([0, 1, 2], [0, 1, 2], flags, dst, src) is None


def test_c_restatement_of_nms2_agrees_with_numpy_oracle():
    """oracle/c/nms2_ref.c (plain C, compiled by __graft_entry__.build) and oracle/frontend_ref.py::nms2 (numpy) are two
    independent statements of superpoint_tensorrt.cpp:164-189,237-310: golden fixtures, exact ties, the flat-address column
    wrap at the image edge and the u16 index-plane wrap above 65535 candidates must all agree bit for bit."""
    from oracle import nms2_c
    z = np.load(os.path.join(GOLDEN, "postproc.npz"))
    for n in "abc":
        k, c = nms2_c.get_keypoints(z[f"{n}_semi"], 0.015, 50)
        assert np.array_equal(k, z[f"{n}_kpts"]) and np.array_equal(c, z[f"{n}_conf"])
    rng = np.random.default_rng(11)
    cases = [rng.choice(np.array([0.0, 0.02, 0.3, 0.3, 0.7], np.float32), (64, 96)),        # dense ties
             np.full((40, 56), 0.5, np.float32),                                             # all equal
             np.zeros((32, 32), np.float32),                                                 # empty
             rng.uniform(0.0, 1.0, (48, 80)).astype(np.float32),
             rng.uniform(0.02, 0.9, (256, 320)).astype(np.float32)]                          # > 65535 candidates
    cases[3][:, 0] = 0.95; cases[3][:, -1] = 0.9                                             # strong columns at both edges
    for prob in cases:
        for max_num in (7, 200):
            k, c = nms2_c.get_keypoints(prob, 0.015, max_num)
            rk, rc = fr.get_keypoints(prob, 0.015, max_num)
            assert np.array_equal(k, rk) and np.array_equal(c, rc)


def test_pcm_oracle_clique_heuristic_and_consistency():
    """oracle/pcm_ref.py: (a) the restated FMC::maxCliqueHeu returns a clique and, on small random graphs, one as large as
    the exact maximum clique in most cases (it is a heuristic: never larger, always a clique); (b) the pairwise consistency
    test separates inliers from gross outliers on the synthetic loop edges, is symmetric under storing a loop b -> a, and
    never links edges of different drone pairs."""
    from oracle import pcm_ref as pr
    rng = np.random.default_rng(0)
    hits = 0
    for trial in range(30):
        n = int(rng.integers(5, 13))
        a = (rng.uniform(size=(n, n)) < 0.55).astype(np.uint8)
        a = np.triu(a, 1); a = a + a.T
        clique, size = pr.max_clique_heu(a)
        assert size == len(clique) and len(set(clique)) == len(clique)
        assert all(a[u, v] for i, u in enumerate(clique) for v in clique[i + 1:]), "heuristic returned a non-clique"
        exact = pr.max_clique_exact(a)
        assert size <= exact
        hits += size == exact
    assert hits >= 20
    edges = synth.pcm_edges(40, 0.35, 3, other_pair=4)
    clique, adj, size = pr.pcm(edges, 15.0, 1e-4, 1e-5)
    inl = np.array([e["inlier"] for e in edges])
    assert size >= 0.5 * inl.sum() and all(edges[i]["inlier"] for i in clique)
    pair = np.array([{e["id_a"], e["id_b"]} == {1, 2} for e in edges])
    assert adj[np.ix_(pair, ~pair)].sum() == 0 and adj[np.ix_(~pair, pair)].sum() == 0    # across drone pairs: never consistent
    assert np.array_equal(adj, adj.T) and adj.diagonal().sum() == 0
    # a loop stored b -> a (same_robot_pair == 2, :214-224): with exact data the error pose is the identity in either statement
    e, other = dict(edges[0]), dict(edges[1])
    for x in (e, other):
        x["rel"] = pr.pose_mul(pr.pose_inv(x["odom_a"]), x["odom_b"])
    flipped = dict(id_a=e["id_b"], id_b=e["id_a"], rel=pr.pose_inv(e["rel"]), cov=e["cov"], odom_a=e["odom_b"],
                   odom_b=e["odom_a"], len_a=e["len_b"], len_b=e["len_a"])
    if pr.same_robot_pair(e, other):
        assert pr.pair_smd(e, other, 1e-4, 1e-5) < 1e-18 and pr.pair_smd(flipped, other, 1e-4, 1e-5) < 1e-18


def test_pnp_oracle_pinned_against_opencv():
    """oracle/pnp_ref.py (deterministic RANSAC + LM, the definition of cv::solvePnPRansac's result) against the real OpenCV
    on correspondences whose outliers are gross: same inlier set, same pose.  Also the reference's own setting (reprojection
    error 3 in NORMALISED coordinates, loop_detector.cpp:393): every correspondence is an inlier and the pose is the
    least-squares fit over all of them -- cv2 agrees on that too."""
    import cv2
    from oracle import pnp_ref as pn, pcm_ref as pr
    for seed, out in ((0, 0.25), (1, 0.4), (2, 0.0)):
        c = synth.pnp_case(160, out, seed)
        res = pn.pnp_ransac(c["X"], c["uv"], c["prior"], iterations=100, thresh=0.03, seed=seed)
        assert res["success"] and np.array_equal(res["mask"].astype(bool), c["inlier"])
        ok, rvec, tvec, inl = cv2.solvePnPRansac(c["X"].astype(np.float64), c["uv"].astype(np.float64), np.eye(3), None,
                                                 iterationsCount=100, reprojectionError=0.03, confidence=0.99)
        m = np.zeros(len(c["X"]), bool); m[inl.ravel()] = True
        assert ok and np.array_equal(m, res["mask"].astype(bool))
        R, _ = cv2.Rodrigues(rvec)
        Ro = np.stack([pr.q_rot(res["pose"][3:], e) for e in np.eye(3)], 1)
        assert np.abs(R - Ro).max() < 1e-6 and np.abs(tvec.ravel() - res["pose"][:3]).max() < 1e-6
        assert np.abs(res["pose"][:3] - c["pose_true"][:3]).max() < 0.02
    c = synth.pnp_case(120, 0.0, 5)
    res = pn.pnp_ransac(c["X"], c["uv"], c["prior"], iterations=100, thresh=3.0, seed=0)
    ok, rvec, tvec, inl = cv2.solvePnPRansac(c["X"].astype(np.float64), c["uv"].astype(np.float64), np.eye(3), None,
                                             iterationsCount=100, reprojectionError=3.0, confidence=0.99)
    assert res["n_inliers"] == 120 == len(inl) and np.abs(tvec.ravel() - res["pose"][:3]).max() < 1e-6
    # the acceptance chain on the true geometry: small roll/pitch error, the loop's 4-DoF pose = old drone -> new drone
    prm = dict(extrinsic=c["extrinsic"], drone_pose_now=c["drone_pose_now"], drone_pose_old=c["drone_pose_old"], is_4dof=1,
               min_loop_num=15, rperr_thres=0.1, accept_loop_yaw_rad=0.8, max_loop_dis=5.0)
    v = pn.loop_from_pnp(res, prm)
    assert v["verified"] and v["rperr"] < 0.01
    old_in_wn = pr.pose_mul(pr.pose_inv(res["pose"]), pr.pose_inv(c["extrinsic"]))      # old drone in the new drone's frame
    d = pn.delta_pose(old_in_wn, c["drone_pose_now"], True)
    assert np.abs(v["dp"][:3] - d[:3]).max() < 1e-9 and abs(v["dp"][3] - 0.3 * -1) < 0.02   # yaw(new) - yaw(old) = -0.3


def test_solver_oracle_minimum_agrees_with_an_independent_optimiser():
    """Pins the oracle's Levenberg-Marquardt (step control, Huber corrector, fixed nodes) against an optimiser that shares no
    code with it: scipy's trust-region-reflective least_squares on the SAME objective, written as plain residuals
    r' = r * sqrt(rho(s) / s) per factor (so that |r'|^2 = rho(|r|^2), Ceres' robustified cost).  Both must land on the same
    minimum of a small swarm graph with outliers (some Huber terms active) -- poses and cost."""
    import scipy.optimize as so
    from oracle import solver_ref as sr
    from omniswarm_b200 import synth
    g = synth.pose_graph(3, 10, n_uwb=18, n_loop=12, n_det=8, n_bearing=0, seed=11, outlier_frac=0.15)
    ref = sr.solve(g)
    free = np.nonzero(g["fixed"] == 0)[0]

    def residuals(xf):
        x = g["init"].astype(np.float64).copy()
        x[free] = xf.reshape(-1, 4)
        out = []
        for f in range(len(g["ftype"])):
            r, _, _ = sr.factor_residual_jacobian(int(g["ftype"][f]), x[int(g["ia"][f])], x[int(g["ib"][f])], g["payload"][f])
            s = float(r @ r)
            if g["huber"][f] and s > 1.0:
                r = r * np.sqrt((2.0 * np.sqrt(s) - 1.0) / s)
            out.append(np.pad(r, (0, 4 - len(r))))
        return np.concatenate(out)

    x0 = g["init"].astype(np.float64)[free].reshape(-1)
    sol = so.least_squares(residuals, x0, method="trf", xtol=1e-15, ftol=1e-15, gtol=1e-13, max_nfev=400)
    n_active = sum(1 for f in range(len(g["ftype"])) if g["huber"][f] and
                   float(np.sum(sr.factor_residual_jacobian(int(g["ftype"][f]), ref["poses"][int(g["ia"][f])],
                                                            ref["poses"][int(g["ib"][f])], g["payload"][f])[0] ** 2)) > 1.0)
    assert n_active >= 1, "the graph should keep some Huber terms active at the minimum"
    assert abs(sol.cost - ref["final_cost"]) <= 1e-9 * max(1.0, ref["final_cost"])
    assert np.abs(sol.x.reshape(-1, 4) - ref["poses"][free]).max() < 1e-6


def test_pose_algebra_agrees_with_homogeneous_matrices():
    """The 4-DoF relative pose of RelativePoseFactor4d (DeltaPose, factors.hpp:139-149) and the 7-vector Swarm::Pose algebra the
    PCM / PnP oracles define (swarm_msgs is not in the reference tree) are checked against the textbook statement of the same
    things: 4x4 homogeneous transforms composed and inverted with numpy, rotations from scipy."""
    from scipy.spatial.transform import Rotation as Rot
    from oracle import solver_ref as sr, pcm_ref as pr
    rng = np.random.default_rng(5)

    def T4(p):                                   # (x y z yaw) -> 4x4
        T = np.eye(4); T[:3, :3] = Rot.from_euler("z", p[3]).as_matrix(); T[:3, 3] = p[:3]; return T

    def T7(p):                                   # (x y z, qw qx qy qz) -> 4x4
        T = np.eye(4); T[:3, :3] = Rot.from_quat([p[4], p[5], p[6], p[3]]).as_matrix(); T[:3, 3] = p[:3]; return T

    for _ in range(50):
        pa = np.concatenate([rng.normal(0, 3, 3), rng.uniform(-3.1, 3.1, 1)])
        pb = np.concatenate([rng.normal(0, 3, 3), rng.uniform(-3.1, 3.1, 1)])
        pl = np.zeros(24); pl[4:20] = np.eye(4).reshape(-1)          # measurement 0, sqrt information I: r = -est
        r, _, _ = sr.factor_residual_jacobian(sr.FACTOR_RELPOSE, pa, pb, pl)
        D = np.linalg.inv(T4(pa)) @ T4(pb)
        est = np.array([D[0, 3], D[1, 3], D[2, 3], np.arctan2(D[1, 0], D[0, 0])])
        assert np.allclose(-r[:3], est[:3], atol=1e-12)
        assert abs(sr.normalize_angle(-r[3] - est[3])) < 1e-12
        # Swarm::Pose: composition, inverse, log map
        qa, qb = Rot.random(random_state=int(rng.integers(1 << 30))), Rot.random(random_state=int(rng.integers(1 << 30)))
        A = np.concatenate([rng.normal(0, 2, 3), np.roll(qa.as_quat(), 1)])
        B = np.concatenate([rng.normal(0, 2, 3), np.roll(qb.as_quat(), 1)])
        assert np.allclose(T7(pr.pose_mul(A, B)), T7(A) @ T7(B), atol=1e-12)
        assert np.allclose(T7(pr.pose_inv(A)), np.linalg.inv(T7(A)), atol=1e-12)
        lm = pr.log_map(A)
        assert np.allclose(lm[:3], A[:3]) and np.allclose(lm[3:], qa.as_rotvec(), atol=1e-10)


def test_network_oracle_matches_the_references_own_module():
    """The SuperPoint stage of the oracle against the REFERENCE ITSELF: tests/golden/ref_superpoint.npz holds the outputs of the
    `SuperPointNet` class of swarm_loop/superpoint.ipynb (the module the reference exports its TensorRT engine from),
    executed in place by tests/golden/make_ref_superpoint.py with the seeded weights.  oracle/frontend_ref.py must
    reproduce them (same torch kernels underneath: a few ulp).  `make_ref_superpoint.py --check` executes the notebook again
    and compares its outputs with the fixture."""
    import os
    from oracle import frontend_ref as fr
    from omniswarm_b200 import synth
    here = os.path.dirname(os.path.abspath(__file__))
    z = np.load(os.path.join(here, "golden", "ref_superpoint.npz"))
    w = synth.superpoint_weights(0)
    seeds = sorted(int(k.split("_")[1]) for k in z.files if k.startswith("img_"))
    assert len(seeds) == 3
    for s in seeds:
        img = z[f"img_{s}"]
        assert np.array_equal(img, synth.image(s, *img.shape))            # the fixture's inputs are reproducible
        semi, desc = fr.superpoint_net(img, w, num_threads=1)
        assert semi.shape == z[f"semi_{s}"].shape and desc.shape == z[f"desc_{s}"].shape
        assert np.abs(semi - z[f"semi_{s}"]).max() <= 2e-7 and np.abs(desc - z[f"desc_{s}"]).max() <= 2e-7
        # the decision the pipeline takes on it -- which pixels exceed the threshold -- is identical
        assert np.array_equal(semi > np.float32(0.015), z[f"semi_{s}"] > np.float32(0.015))
    # the notebook scales its input with `/255`, the C++ runtime with `* (float)(1/255.0)` (what runs on the drone, and what the
    # oracle restates): one ulp on some pixels, a few 1e-6 on the heat map
    semi0, _ = fr.superpoint_net(z["img_0"], w, num_threads=1)
    assert 0 < np.abs(semi0 - z["semi_div_0"]).max() < 1e-5


def test_euler_convention_matches_the_references_python_helpers():
    """`quat2eulers` and the angle wrap that the PnP / PCM oracles define (their C++ originals live in swarm_msgs, which is not in
    the tree) against the reference's own Python statement of them, swarm_localization/scripts/utils.py, executed in place by
    tests/golden/make_ref_utils.py (`--check` compares them with the fixture again)."""
    import os
    from oracle import pnp_ref as pr
    from oracle import solver_ref as sr
    here = os.path.dirname(os.path.abspath(__file__))
    z = np.load(os.path.join(here, "golden", "ref_utils.npz"))
    for q, ypr in zip(z["quat_wxyz"], z["ypr"]):
        rpy = pr.quat2eulers(q)
        assert np.allclose(rpy[::-1], ypr, atol=1e-12)                # the reference returns (yaw, pitch, roll)
    for a, w in zip(z["angle"], z["wrapped"]):
        assert abs(pr.wrap(a) - w) < 1e-12 and abs(sr.normalize_angle(a) - w) < 1e-12


def ref_fmc_graphs():
    """the graphs of tests/golden/ref_fmc.npz with the clique and size the reference's own maxCliqueHeu returned on each"""
    z = np.load(os.path.join(GOLDEN, "ref_fmc.npz"))
    adj_end, clq_end = np.cumsum(z["pin_adj_bytes"]), np.cumsum(z["pin_clique_len"])
    for g, n in enumerate(z["pin_n"]):
        iu = np.triu_indices(n, 1)
        a = np.zeros((n, n), np.uint8)
        a[iu] = np.unpackbits(z["pin_adj"][adj_end[g] - z["pin_adj_bytes"][g]:adj_end[g]])[:len(iu[0])]
        yield a | a.T, z["pin_clique"][clq_end[g] - z["pin_clique_len"][g]:clq_end[g]].tolist(), int(z["pin_size"][g])


def test_max_clique_restatement_equals_the_references_own_library():
    """FMC::maxCliqueHeu is plain C++ inside the reference tree (third_party/fast_max-clique_finder), so it is COMPILED from its
    sources in place (oracle/ref_build/Makefile -> oracle/_ref/libfmc_ref.so, nothing copied); tests/golden/ref_fmc.npz holds
    what it returns on 423 graphs of every density, PCM-shaped and degenerate ones (tests/golden/make_ref_fmc.py).  The
    restatement in oracle/pcm_ref.py -- what the CUDA clique kernel is compared with -- must return the same clique, vertex by
    vertex in the same order; where the library has been built, it is asked again, so the fixture cannot drift from it."""
    from oracle import fmc_ref, pcm_ref
    graphs = list(ref_fmc_graphs())
    assert len(graphs) == 423
    for a, ref_clique, ref_size in graphs:
        clique, size = pcm_ref.max_clique_heu(a)
        assert clique == ref_clique and size == ref_size
        assert all(a[u, v] for i, u in enumerate(clique) for v in clique[i + 1:])      # and it is a clique
        if fmc_ref.available():
            assert fmc_ref.max_clique_heu(a) == (ref_clique, ref_size)

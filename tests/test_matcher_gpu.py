"""GPU parity tests of the matcher half of the hot path (through the C-ABI): tcgen05 kNN vs exact brute force,
RANSAC vs its CPU restatement."""
import os

import numpy as np
import pytest

from bundletrack_b200 import synth
from oracle import matcher_oracle as mo

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def matcher(cuda_device):
    from bundletrack_b200.matcher import KnnMatcher
    m = KnnMatcher(max_pairs=64, max_feats=5120)
    yield m
    m.close()


def _check(matcher, dev, a, b, k=5):
    import torch
    ta, tb = torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)
    iAB, dAB, iBA, dBA = matcher.knn_match_pairs([(ta, tb)], k=k)
    i1, d1 = mo.knn(a, b, k)
    i2, d2 = mo.knn(b, a, k)
    assert np.array_equal(iAB[0].cpu().numpy(), i1)
    assert np.array_equal(iBA[0].cpu().numpy(), i2)
    f = np.isfinite(d1)
    assert np.array_equal(np.isfinite(dAB[0].cpu().numpy()), f)
    if f.any():
        assert np.abs(dAB[0].cpu().numpy()[f] - d1[f]).max() <= 1e-6
    f2 = np.isfinite(d2)
    if f2.any():
        assert np.abs(dBA[0].cpu().numpy()[f2] - d2[f2]).max() <= 1e-6


@pytest.mark.parametrize("na,nb", [(500, 500), (2000, 2000), (1000, 3000), (129, 257), (5, 3), (1, 700), (300, 2)])
def test_knn_equals_exact_brute_force(matcher, cuda_device, na, nb):
    a, b, _, _ = synth.make_descriptors(na * 7 + nb, na, nb)
    _check(matcher, cuda_device, a, b)


@pytest.mark.parametrize("every,na,nb", [(7, 900, 1300), (1, 40, 33), (1, 1500, 2100)])
def test_knn_exact_fallback_paths(matcher, cuda_device, every, na, nb):
    """The brute-force fallback in both of its shapes (few rows: train set split over 16 CTAs + ticketed merge; many rows: one
    CTA per row) returns exactly what the tensor-core path + proof returns."""
    a, b, _, _ = synth.make_descriptors(na + nb, na, nb)
    b[5] = b[6] = a[3]                      # ties across segment boundaries resolve to the lower index
    matcher.force_fallback(every)
    matcher.enable_timing(True)
    try:
        _check(matcher, cuda_device, a, b)
        assert matcher.timing()["fallback_rows"] >= (na + nb) // every - 1
    finally:
        matcher.force_fallback(0)
        matcher.enable_timing(False)


def test_knn_cfg5_5000x5000(matcher, cuda_device):
    a, b, _, _ = synth.make_descriptors(55, 5000, 5000)
    _check(matcher, cuda_device, a, b)


def test_knn_duplicates_and_unnormalised(matcher, cuda_device):
    """Exact ties (duplicate descriptors) must come out lowest-index-first; non-unit norms must not break the proof."""
    rng = np.random.default_rng(3)
    a = rng.normal(size=(300, 256)).astype(np.float32)
    b = rng.normal(size=(400, 256)).astype(np.float32) * 3.0
    b[10] = b[200]; b[11] = b[200]; b[350] = b[200]
    a[5] = b[200] * 0.999
    _check(matcher, cuda_device, a, b)


def test_knn_pitched_rows_and_batch(matcher, cuda_device):
    """GpuMat rows are pitched; a keyframe's descriptor set is shared by many pairs of one call."""
    import torch
    frames = []
    for f in range(4):
        d = synth.make_descriptors(200 + f, 600 + 50 * f, 8)[0]
        buf = torch.zeros((d.shape[0], 320), device=cuda_device)      # pitch 1280 B
        buf[:, :256] = torch.from_numpy(d).to(cuda_device)
        frames.append((d, buf[:, :256]))
    pairs = [(frames[j][1], frames[i][1]) for i in range(4) for j in range(i + 1, 4)]
    iAB, dAB, iBA, dBA = matcher.knn_match_pairs(pairs)
    p = 0
    for i in range(4):
        for j in range(i + 1, 4):
            i1, _ = mo.knn(frames[j][0], frames[i][0])
            i2, _ = mo.knn(frames[i][0], frames[j][0])
            assert np.array_equal(iAB[p].cpu().numpy(), i1)
            assert np.array_equal(iBA[p].cpu().numpy(), i2)
            p += 1


def test_knn_descriptor_pool_slots(matcher, cuda_device):
    """bt_desc_pool_store once per frame + bt_knn_match_slots == bt_knn_match_pairs on the raw views, bit for bit; a slot can be
    overwritten; an empty slot is an error; steady-state calls launch no descriptor conversion."""
    import torch
    from bundletrack_b200 import _lib
    descs = [synth.make_descriptors(300 + f, 500 + 130 * f, 8)[0] for f in range(4)]
    dev = [torch.from_numpy(d).to(cuda_device) for d in descs]
    matcher.pool_reserve(6)
    for f in range(4):
        matcher.pool_store(f, dev[f])
    idx = [(j, i) for i in range(4) for j in range(i + 1, 4)]
    want = matcher.knn_match_pairs([(dev[a], dev[b]) for a, b in idx])
    got = matcher.knn_match_slots(idx, [(len(descs[a]), len(descs[b])) for a, b in idx], device=cuda_device)
    for w4, g4 in zip(want, got):
        for w, g in zip(w4, g4):
            assert torch.equal(w, g)
    matcher.enable_timing(True)
    matcher.knn_match_slots(idx, [(len(descs[a]), len(descs[b])) for a, b in idx], device=cuda_device)
    assert matcher.timing()["prep_ms"] < 0.04             # only the table upload sits between the two events: no conversion kernel in steady state
    matcher.enable_timing(False)
    matcher.pool_store(1, dev[3])                          # overwrite: slot 1 now holds frame 3's descriptors
    iAB, _, iBA, _ = matcher.knn_match_slots([(1, 0)], [(len(descs[3]), len(descs[0]))], device=cuda_device)
    assert np.array_equal(iAB[0].cpu().numpy(), mo.knn(descs[3], descs[0])[0])
    assert np.array_equal(iBA[0].cpu().numpy(), mo.knn(descs[0], descs[3])[0])
    with pytest.raises(_lib.BtError):
        matcher.knn_match_slots([(5, 0)], [(10, 10)], device=cuda_device)


def test_knn_cta_pair_kernel_equals_exact_brute_force(cuda_device, monkeypatch):
    """The cta_group::2 form of the tensor pass (clusters of two CTAs, M = 256, double-buffered B half tiles; BT_KNN_CTA_PAIRS=1, not the
    default) gives the same exact result, incl. A sets that do not fill a 256-row unit and several pairs per call."""
    import torch
    from bundletrack_b200.matcher import KnnMatcher
    monkeypatch.setenv("BT_KNN_CTA_PAIRS", "1")
    m = KnnMatcher(max_pairs=4, max_feats=1024)
    shapes = [(700, 900), (129, 257), (1000, 300)]
    sets = [synth.make_descriptors(40 + i, na, nb)[:2] for i, (na, nb) in enumerate(shapes)]
    pairs = [(torch.from_numpy(a).to(cuda_device), torch.from_numpy(b).to(cuda_device)) for a, b in sets]
    iAB, dAB, iBA, dBA = m.knn_match_pairs(pairs, k=5)
    for p, (a, b) in enumerate(sets):
        i1, d1 = mo.knn(a, b, 5)
        i2, d2 = mo.knn(b, a, 5)
        assert np.array_equal(iAB[p].cpu().numpy(), i1) and np.array_equal(iBA[p].cpu().numpy(), i2)
        assert np.abs(dAB[p].cpu().numpy() - d1).max() <= 1e-6 and np.abs(dBA[p].cpu().numpy() - d2).max() <= 1e-6
    m.close()


def test_knn_matches_opencv(matcher, cuda_device):
    pytest.importorskip("cv2")
    import torch
    a, b, _, _ = synth.make_descriptors(9, 800, 700)
    iAB, dAB, _, _ = matcher.knn_match_pairs([(torch.from_numpy(a).to(cuda_device), torch.from_numpy(b).to(cuda_device))])
    ic, dc = mo.knn_cv2(a, b)
    assert np.array_equal(iAB[0].cpu().numpy(), ic)
    assert np.abs(dAB[0].cpu().numpy() - dc).max() < 1e-5


# ------------------------------------------------------------------------------------------------------------ RANSAC
def _ransac_case(seed, n, inlier_frac=0.7, noise=0.0005, big=False):
    return synth.make_ransac_case(seed, n, inlier_frac, noise)


def _ransac_vs_reference(A4, B4, got, ref, u3, best_trial, thresh):
    """How bt_ransac_pairs' inlier set relates to the one the reference's ransacMultiPairGPU returned for the same points.
    'identical': same ids.  'better': another trial won here with at least as many inliers - the reference's McAdams-SVD fit is
    approximate and its arg-max is racy (SURVEY.md Q8), so among near-tied trials either may win.  'borderline': same winner, the
    sets differ only in points whose distance under the winning model is within 5e-6 m of the threshold (the two fits of the same
    three points differ by ~1e-6).  Anything else is a failure."""
    if np.array_equal(got, ref):
        return "identical"
    A = A4[:, :3].astype(np.float64); B = B4[:, :3].astype(np.float64)
    n = len(A)
    ids = np.floor(u3[best_trial].astype(np.float32) * np.float32(n - 1) + np.float32(0.5)).astype(np.int64)
    s, d = A[ids], B[ids]
    sm, dm = s.mean(0), d.mean(0)
    U, _, Vt = np.linalg.svd((s - sm).T @ (d - dm))
    R = Vt.T @ U.T
    if np.linalg.det(R) < 0:
        Vt[2] *= -1; R = Vt.T @ U.T
    dist = np.linalg.norm(B - (A @ R.T + (dm - R @ sm)), axis=1)
    diff = np.setxor1d(got, ref)
    if np.all(np.abs(dist[diff] - thresh) <= 5e-6):
        return "borderline"
    if len(got) >= len(ref):
        return "better"
    return "worse"


def test_ransac_sampler_is_curand_xorwow(cuda_device):
    """The sampler's uniforms must be the reference's: curand_init(0, trial, 0) + 3 x curand_uniform (golden table made
    with that very call on a B200 by scripts/make_golden_curand.py)."""
    from bundletrack_b200.matcher import Ransac
    import torch
    r = Ransac(max_pairs=2, max_pts=256, max_trials=2000)
    A4, B4, _ = _ransac_case(0, 50)
    r.ransac_pairs([torch.from_numpy(A4).to(cuda_device)], [torch.from_numpy(B4).to(cuda_device)], 2000, 0.005)
    u3, _ = r.debug(2000, 1)
    gold = np.load(os.path.join(GOLD, "curand_xorwow_seed0.npy"))
    assert np.array_equal(u3, gold[:2000])
    r.close()


@pytest.mark.parametrize("n", [8, 60, 400, 3000])
def test_ransac_matches_oracle(cuda_device, n):
    from bundletrack_b200.matcher import Ransac
    import torch
    r = Ransac(max_pairs=4, max_pts=4096, max_trials=2000)
    cases = [_ransac_case(10 * n + k, n) for k in range(3)]
    ids = r.ransac_pairs([torch.from_numpy(c[0]).to(cuda_device) for c in cases], [torch.from_numpy(c[1]).to(cuda_device) for c in cases], 2000, 0.005)
    u3, best = r.debug(2000, 3)
    for k, (A4, B4, truth) in enumerate(cases):
        got = ids[k].cpu().numpy()
        want, wbest, counts = mo.ransac_pair(A4, B4, u3, 0.005)
        assert (np.diff(got) > 0).all()
        # the winning count can differ by a borderline point or two (fp32 pose vs float64 SVD); the SET must be the true inliers
        assert abs(len(got) - len(want)) <= max(2, len(want) // 200)
        inter = len(np.intersect1d(got, want))
        assert inter >= len(want) - max(2, len(want) // 200)
        assert counts[best[k]] >= counts.max() - max(2, len(want) // 200)      # our winner is (near-)optimal for the oracle too
        if n >= 60:
            assert np.array_equal(np.nonzero(truth)[0], got) or inter >= truth.sum() - 2
    r.close()


def test_ransac_edge_cases(cuda_device):
    from bundletrack_b200.matcher import Ransac
    import torch
    r = Ransac(max_pairs=4, max_pts=64, max_trials=500)
    A4, B4, _ = _ransac_case(1, 2)          # fewer than 3 points: no model, no inliers
    z = torch.zeros((0, 4), device=cuda_device)
    ids = r.ransac_pairs([torch.from_numpy(A4).to(cuda_device), z], [torch.from_numpy(B4).to(cuda_device), z], 500, 0.005)
    assert len(ids[0]) == 0 and len(ids[1]) == 0
    A4, B4, _ = _ransac_case(2, 30, inlier_frac=0.0)   # all outliers: at most the 3 sampled points agree
    ids = r.ransac_pairs([torch.from_numpy(A4).to(cuda_device)], [torch.from_numpy(B4).to(cuda_device)], 500, 0.0005)
    assert len(ids[0]) <= 6
    r.close()


def _ransac_reference_check(cuda_device, A, B, ref_ids, thresh, label):
    """bt_ransac_pairs (seed 0 = the reference's XORWOW sequence) against the reference's own ransacMultiPairGPU outputs."""
    from bundletrack_b200.matcher import Ransac
    import torch
    r = Ransac(max_pairs=max(len(A), 1), max_pts=4096, max_trials=2000)
    ids = r.ransac_pairs([torch.from_numpy(a).to(cuda_device) for a in A], [torch.from_numpy(b).to(cuda_device) for b in B], 2000, thresh)
    u3, best = r.debug(2000, len(A))
    r.close()
    verdicts = []
    for p in range(len(A)):
        got = ids[p].cpu().numpy()
        v = _ransac_vs_reference(A[p], B[p], got, ref_ids[p], u3, best[p], thresh)
        verdicts.append(v)
        assert v != "worse", (label, p, len(got), len(ref_ids[p]))
        # whichever trial won on either side, the two inlier sets describe the same rigid motion: they overlap almost entirely
        inter = len(np.intersect1d(got, ref_ids[p]))
        assert inter >= min(len(got), len(ref_ids[p])) - max(2, len(ref_ids[p]) // 100), (label, p, inter, len(got), len(ref_ids[p]))
    return verdicts


def test_ransac_matches_reference_golden(cuda_device):
    """tests/golden/ref_ransac.npz: inputs + the inlier ids the reference's ransacMultiPairGPU (cuda_ransac.cu:1228-1323, compiled
    verbatim into oracle/_ref) returned on a B200 (scripts/make_golden_ransac.py)."""
    path = os.path.join(GOLD, "ref_ransac.npz")
    if not os.path.exists(path):
        pytest.skip("tests/golden/ref_ransac.npz not generated yet")
    g = np.load(path)
    verdicts = []
    for k in range(int(g["n_cases"])):
        verdicts += _ransac_reference_check(cuda_device, [g[f"A{k}"]], [g[f"B{k}"]], [g[f"ref{k}"]], float(g["thresh"][k]), f"golden{k}")
    assert verdicts.count("identical") >= (len(verdicts) + 1) // 2, verdicts


def test_ransac_matches_reference_live(cuda_device):
    """The reference's own ransacMultiPairGPU (its inlier sets recorded on a B200 in tests/golden/ref_matcher_runs.npz, made by
    scripts/make_golden_reference_runs.py): n = 8 ... 3000 points, and the 45 pairs of a 10-keyframe window at cfg2 sizes in one
    call.  Identical inlier sets are the rule; a pair may differ only as _ransac_vs_reference allows."""
    g = np.load(os.path.join(GOLD, "ref_matcher_runs.npz"))
    def ref_ids(key, n):
        return np.flatnonzero(np.unpackbits(g[key], count=n)).astype(np.int32)
    verdicts = []
    for n, thresh in ((8, 0.005), (60, 0.005), (300, 0.01), (1000, 0.005), (3000, 0.005)):
        cases = [_ransac_case(7000 + 10 * n + k, n, inlier_frac=0.5 + 0.1 * k) for k in range(3)]
        ref = [ref_ids(f"ransac_n{n}_{k}", n) for k in range(3)]
        verdicts += _ransac_reference_check(cuda_device, [c[0] for c in cases], [c[1] for c in cases], ref, thresh, f"n{n}")
    rng = np.random.default_rng(5)
    cases = [_ransac_case(8000 + p, int(rng.integers(300, 1600)), inlier_frac=float(rng.uniform(0.3, 0.9))) for p in range(45)]
    assert np.array_equal([len(c[0]) for c in cases], g["ransac_cfg2_n"])      # the inputs the reference was run on
    ref = [ref_ids(f"ransac_cfg2_{p}", len(c[0])) for p, c in enumerate(cases)]
    verdicts += _ransac_reference_check(cuda_device, [c[0] for c in cases], [c[1] for c in cases], ref, 0.005, "cfg2")
    print("RANSAC vs reference:", {v: verdicts.count(v) for v in sorted(set(verdicts))})
    assert verdicts.count("identical") >= int(0.6 * len(verdicts)), verdicts


# ------------------------------------------------------------------------------------------------- prune / fused pipeline
def _feature_window(seed, N, n_feats, dev):
    import torch
    w = synth.make_window(seed, n_frames=N, n_corr=10)
    fr = synth.make_feature_frames(w, n_feats, seed=seed)
    host, devf = [], []
    for k in range(N):
        h = {"kpts": fr[k]["kpts"], "desc": fr[k]["desc"], "depth": w.depth[k], "normal": w.normal[k], "pose": w.poses_init[k], "id": k}
        host.append(h)
        devf.append({"kpts": torch.from_numpy(h["kpts"]).to(dev), "desc": torch.from_numpy(h["desc"]).to(dev), "depth": torch.from_numpy(w.depth[k]).to(dev),
                     "normal": torch.from_numpy(w.normal[k]).to(dev), "pose": h["pose"], "id": k, "window_index": k})
    return w, host, devf


def test_prune_mutual_equals_oracle(cuda_device):
    from bundletrack_b200.matcher import MatchPipeline
    import torch
    w, host, devf = _feature_window(3, 4, 400, cuda_device)
    mp = MatchPipeline(None, max_pairs=8, max_feats=512)
    pairs_idx = [(j, i) for i in range(4) for j in range(i + 1, 4)]           # (newer, older), incl. neighbours |j-i| == 1
    idxAB = [mo.knn(host[a]["desc"], host[b]["desc"])[0] for a, b in pairs_idx]
    idxBA = [mo.knn(host[b]["desc"], host[a]["desc"])[0] for a, b in pairs_idx]
    got = mp.prune_mutual([(devf[a], devf[b]) for a, b in pairs_idx], torch.from_numpy(np.concatenate(idxAB)).to(cuda_device),
                          torch.from_numpy(np.concatenate(idxBA)).to(cuda_device), w.H, w.W, w.K)
    prm = (mp.prune.max_dist_no_neighbor, mp.prune.cos_max_normal_no_neighbor, mp.prune.max_dist_neighbor, mp.prune.cos_max_normal_neighbor)
    total = 0
    for p, (a, b) in enumerate(pairs_idx):
        nb = abs(a - b) == 1
        md, cm = (prm[2], prm[3]) if nb else (prm[0], prm[1])
        want = mo.collect_mutual(host[a], host[b], mo.prune_matches(host[a], host[b], idxAB[p], w.K, md, cm), mo.prune_matches(host[b], host[a], idxBA[p], w.K, md, cm))
        g = got[p].cpu().numpy()
        assert g.shape == want.shape, (p, g.shape, want.shape)
        assert np.allclose(g, want, atol=2e-6)
        total += len(want)
    assert total > 50
    mp.close()


def test_fused_pipeline_matches_oracle_and_feeds_solver(cuda_device):
    """descriptors -> kNN -> prune -> mutual -> RANSAC -> EntryJ on the device, compared stage by stage with the oracle, then the
    resulting correspondences drive the solver to the same poses as the oracle solver fed with the oracle correspondences."""
    from bundletrack_b200.matcher import MatchPipeline
    from bundletrack_b200.optimizer import OptimizerGpu, SolveWindow
    import oracle
    yml = {"bundle": {"num_iter_outter": 7, "num_iter_inner": 5, "robust_delta": 0.005, "image_downscale": 4}, "p2p": {"max_dist": 0.02, "max_normal_angle": 45},
           "feature_corres": {"max_dist_no_neighbor": 0.02, "max_normal_no_neighbor": 45, "max_dist_neighbor": 10000, "max_normal_neighbor": 180},
           "ransac": {"max_iter": 2000, "inlier_dist": 0.01}}
    w, host, devf = _feature_window(5, 4, 500, cuda_device)
    mp = MatchPipeline(yml, max_pairs=8, max_feats=512)
    pairs_idx = [(j, i) for i in range(4) for j in range(i + 1, 4)]
    ent, n_ent, off = mp.match_pairs([(devf[a], devf[b]) for a, b in pairs_idx], w.H, w.W, w.K)
    u3 = np.load(os.path.join(GOLD, "curand_xorwow_seed0.npy"))[:2000]
    prm = (mp.prune.max_dist_no_neighbor, mp.prune.cos_max_normal_no_neighbor, mp.prune.max_dist_neighbor, mp.prune.cos_max_normal_neighbor)
    want_entries = []
    for p, (a, b) in enumerate(pairs_idx):
        rows, ids = mo.find_corres(host[a], host[b], w.K, prm, u3, 0.01)
        n_want = 0 if ids is None else len(ids)
        assert abs(int(n_ent[p]) - n_want) <= max(2, n_want // 50), (p, n_ent[p], n_want)
        e = ent[off[p]:off[p] + n_ent[p]]
        assert (e["imgIdx_i"] == b).all() and (e["imgIdx_j"] == a).all()
        if ids is not None:
            wp = rows[ids]
            # every emitted entry is one of the oracle's mutual rows (pos_i = ptB_cam, pos_j = ptA_cam)
            allrows = np.concatenate([rows[:, 7:10], rows[:, 4:7]], 1)
            for x in e:
                got = np.concatenate([x["pos_i"], x["pos_j"]])
                assert np.abs(allrows - got).max(axis=1).min() <= 2e-6
            for r in wp:
                want_entries.append((b, a, r[7:10], r[4:7]))
    assert n_ent.sum() >= 20
    # hand the device-produced correspondences to the solver; compare with the oracle solver on the oracle's correspondences
    corr_o = np.zeros(len(want_entries), synth.ENTRYJ_DTYPE)
    for k, (i, j, pi, pj) in enumerate(want_entries):
        corr_o[k] = (i, j, pi, pj)
    opt = OptimizerGpu(yml, max_windows=1, max_frames=8, max_corr=8192)
    depth = [f["depth"] for f in devf]; normal = [f["normal"] for f in devf]
    out = opt.optimizeWindows([SolveWindow(ent, w.H, w.W, depth, normal, w.poses_init, w.K)])[0]
    # same RANSAC winner on both sides (the device's own entries handed to the oracle solver): north_star's 1e-4 rad / 1e-4 m
    # the reference's own kernels on an EntryJ list of this chain (recorded on a B200 with its pair directions and a second run of the
    # same call, tests/golden/ref_matcher_runs.npz): the library solves that very list
    g = np.load(os.path.join(GOLD, "ref_matcher_runs.npz"))
    assert np.allclose(w.poses_init, g["fused_init"], rtol=0, atol=1e-6)
    ent_ref = g["fused_ent"].view(synth.ENTRYJ_DTYPE).reshape(-1)
    ref_same, pairs, ref_again = g["fused_poses"], g["fused_pairs"], g["fused_poses_again"]
    out_same = opt.optimizeWindows([SolveWindow(ent_ref, w.H, w.W, depth, normal, w.poses_init, w.K, dense_pairs=pairs)])[0]
    r, t = synth.pose_errors(out_same, ref_same)
    # yardsticks on this very window: the reference against itself (float atomics: its sums change from run to run) and the IEEE
    # restatement of the same arithmetic (oracle A, same pair directions) against the reference.  On a window whose hard dense gates
    # amplify rounding (tests/test_solver_gpu.py::test_gate_sensitive_window) no implementation can be closer to the reference than
    # those two are; on all others the plain 1e-4 applies.
    a_same = oracle.solve_window(w.depth, w.normal, w.K, ent_ref, w.poses_init, pairs=pairs)
    yard = max(max(synth.pose_errors(ref_again, ref_same)), max(synth.pose_errors(a_same, ref_same)))
    print(f"fused chain -> solver vs the reference's kernels on the same entries: rot {r:.2e} rad trans {t:.2e} m "
          f"(reference run-to-run {max(synth.pose_errors(ref_again, ref_same)):.2e}, oracle A vs reference {max(synth.pose_errors(a_same, ref_same)):.2e})")
    a64_same = oracle.solve_window(w.depth, w.normal, w.K, ent_ref, w.poses_init, pairs=pairs, precision="f64")
    print(f"   pair directions {np.asarray(pairs).tolist()}; oracle float vs double {max(synth.pose_errors(a_same, a64_same)):.2e}; library vs oracle float {max(synth.pose_errors(out_same, a_same)):.2e}, vs oracle double {max(synth.pose_errors(out_same, a64_same)):.2e}")
    if max(r, t) > max(1e-4, 1.25 * yard):
        # ONE source pixel of pair (3,0) of this window sits on the 2 cm distance gate: depending on rounding-level differences of the
        # poses of the earlier iterations (e.g. the order in which the pairs' sums are added - the reference's pair list changes with
        # its allocation addresses) it is gated in or out, the pair's count is 771 or 772, and the result moves by 1.5e-4
        # (scripts/dev_pair_order.py: same pair SET in five orders -> 3e-6 or 1.5e-4, in round 1's solver as well).  When the
        # tolerance is missed it must be exactly that: a gate count that differs from the oracle's, and poses still within a few 1e-4.
        opt.enable_debug(True)
        opt.optimizeWindows([SolveWindow(ent_ref, w.H, w.W, depth, normal, w.poses_init, w.K, dense_pairs=pairs)])
        cnt = opt.debug_counts(0, len(pairs)).astype(np.int64)
        opt.enable_debug(False)
        before_last = oracle.solve_window(w.depth, w.normal, w.K, ent_ref, w.poses_init, pairs=pairs, params=oracle.default_params(num_iter_outer=6))
        _, _, nf = oracle.dense_system(w.depth, w.normal, w.K, before_last, pairs=pairs)
        print(f"   gate counts of the last iteration: library {cnt.tolist()}, oracle {nf.tolist()}")
        assert (cnt != nf).any() and np.abs(cnt - nf).sum() <= 4 and max(r, t) <= 5e-4, (r, t, yard, cnt, nf)
    ref_same = oracle.solve_window(w.depth, w.normal, w.K, ent, w.poses_init)
    r, t = synth.pose_errors(out, ref_same)
    assert r <= 2e-4 and t <= 1e-4, (r, t)      # Oracle A on this window sits 1.5e-4 from the CUDA path (a gate-sensitive one, see tests/test_solver_gpu.py)
    # the oracle's own correspondences (its float64 RANSAC may keep or drop a borderline inlier): still the same poses to ~1e-3
    ref = oracle.solve_window(w.depth, w.normal, w.K, corr_o, w.poses_init)
    r, t = synth.pose_errors(out, ref)
    assert r <= 2e-3 and t <= 1e-3, (r, t)
    opt.close(); mp.close()


def test_device_resident_handoff_equals_host_path(cuda_device):
    """bt_match_pairs' EntryJ list consumed by the solver straight from device memory (bt_window::corr_dev + block arrays: only
    2 x n_pairs ints come back to the host) gives the poses of the host round trip, bit for bit - also next to a host-fed window."""
    from bundletrack_b200.matcher import MatchPipeline
    from bundletrack_b200.optimizer import OptimizerGpu, SolveWindow
    from bundletrack_b200 import _lib
    w, host, devf = _feature_window(8, 5, 600, cuda_device)
    mp = MatchPipeline(None, max_pairs=16, max_feats=640)
    pairs_idx = [(j, i) for i in range(5) for j in range(i + 1, 5)]
    prs = [(devf[a], devf[b]) for a, b in pairs_idx]
    ent_h, n_h, off_h = mp.match_pairs(prs, w.H, w.W, w.K)
    ent_d, n_d, off_d = mp.match_pairs(prs, w.H, w.W, w.K, keep_on_device=True)
    assert np.array_equal(n_h, n_d) and np.array_equal(off_h, off_d) and n_d.sum() >= 20
    depth = [f["depth"] for f in devf]; normal = [f["normal"] for f in devf]
    opt = OptimizerGpu(None, max_windows=2, max_frames=8, max_corr=8192)
    via_host = opt.optimizeWindows([SolveWindow(ent_h, w.H, w.W, depth, normal, w.poses_init, w.K)])[0]
    blocks = MatchPipeline.solver_blocks(prs, n_d, off_d)
    wd = SolveWindow(None, w.H, w.W, depth, normal, w.poses_init, w.K, corr_dev=ent_d, blocks=blocks)
    via_dev = opt.optimizeWindows([wd])[0]
    assert np.array_equal(via_host, via_dev)
    w2 = synth.make_window(9, n_frames=4, n_corr=300)
    d2 = [torch_from(x, cuda_device) for x in w2.depth]; n2 = [torch_from(x, cuda_device) for x in w2.normal]
    alone = opt.optimizeWindows([SolveWindow(w2.corr, w2.H, w2.W, d2, n2, w2.poses_init, w2.K)])[0]
    for order in ((0, 1), (1, 0)):      # host-fed and device-fed windows in one batch, either order
        ws = [SolveWindow(w2.corr, w2.H, w2.W, d2, n2, w2.poses_init, w2.K), wd]
        out = opt.optimizeWindows([ws[k] for k in order])
        assert np.array_equal(out[order.index(0)], alone) and np.array_equal(out[order.index(1)], via_dev)
    bad = (blocks[0].copy(), blocks[1], blocks[2], blocks[3]); bad[0][1] += 1       # not back to back
    if len(bad[0]) > 1:
        with pytest.raises(_lib.BtError):
            opt.optimizeWindows([SolveWindow(None, w.H, w.W, depth, normal, w.poses_init, w.K, corr_dev=ent_d, blocks=bad)])
    opt.close(); mp.close()


def torch_from(x, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def test_find_corres_sequence_with_propagation_cache_and_fail(cuda_device):
    """SiftManager::findCorres over a 5-frame sequence on the device chain (FindCorres): every new frame is matched against its
    neighbour first, then against the older frames WITH the map-point matches propagated through the frames in between
    (findCorresByMapPoints), pair by pair like the reference; compared with the oracle's find_corres + Tracks restatement.  Then the
    cache: a second request matches nothing, the window's EntryJ list comes straight from the cache and drives the solver to the
    poses of the host path; a frame with too few neighbour matches is reported Frame::FAIL."""
    import torch
    from bundletrack_b200.matcher import MatchPipeline, FindCorres
    from bundletrack_b200.optimizer import OptimizerGpu, SolveWindow
    from oracle import policy_oracle as po
    yml = {"bundle": {"num_iter_outter": 7, "num_iter_inner": 5, "robust_delta": 0.005, "image_downscale": 4}, "p2p": {"max_dist": 0.02, "max_normal_angle": 45},
           "feature_corres": {"max_dist_no_neighbor": 0.02, "max_normal_no_neighbor": 45, "max_dist_neighbor": 10000, "max_normal_neighbor": 180},
           "ransac": {"max_iter": 2000, "inlier_dist": 0.01}}
    N = 5
    w, host, devf = _feature_window(21, N, 500, cuda_device)
    mp = MatchPipeline(yml, max_pairs=8, max_feats=512)
    mp.pool_reserve(N)
    for f in range(N):
        mp.pool_store(f, devf[f]["desc"])
    fc = FindCorres(mp)
    u3 = np.load(os.path.join(GOLD, "curand_xorwow_seed0.npy"))[:2000]
    prm = (mp.prune.max_dist_no_neighbor, mp.prune.cos_max_normal_no_neighbor, mp.prune.max_dist_neighbor, mp.prune.cos_max_normal_neighbor)
    otracks = po.Tracks()
    n_prop_used = 0
    host_entries = {}
    for f in range(1, N):
        for a, b in [(f, f - 1)] + [(f, j) for j in range(f - 2, -1, -1)]:
            res = fc.find_corres([(devf[a], devf[b])], [(a, b)], w.H, w.W, w.K)
            n_dev, st_dev = res[(a, b)]
            neighbor = a - b == 1
            prop = None if neighbor else otracks.propagate(a, b, np.zeros((0, 4), np.float32))
            rows, ids = mo.find_corres(host[a], host[b], w.K, prm, u3, 0.01, propagated=prop)
            n_want = 0 if ids is None else len(ids)
            assert abs(n_dev - n_want) <= max(2, n_want // 50), (a, b, n_dev, n_want)
            if n_want >= 8 or n_want == 0 and n_dev == 0:
                assert st_dev == (0 if n_want else (2 if neighbor else 1)), (a, b, st_dev)
            # the device's entries are rows of the oracle's candidate list (mutual matches + appended propagated ones), bit for bit
            ent, blocks = fc.window_entries([{"id": b}, {"id": a}], cuda_device)
            e = ent[: int(blocks[1][0])].cpu().numpy().view(np.uint8).reshape(-1).view(synth.ENTRYJ_DTYPE)
            assert len(e) == n_dev and (e["imgIdx_i"] == 0).all() and (e["imgIdx_j"] == 1).all()
            host_entries[(a, b)] = e
            if n_dev:
                allrows = np.concatenate([rows[:, 7:10], rows[:, 4:7]], 1)
                n_nn = len(mo.find_corres(host[a], host[b], w.K, prm, u3, 0.01)[0])
                for x in e:
                    d = np.abs(allrows - np.concatenate([x["pos_i"], x["pos_j"]])).max(axis=1)
                    assert d.min() <= 2e-6
                    n_prop_used += int(d.argmin() >= n_nn)
            if ids is not None:      # updateFramePairMapPoints of the restatement
                otracks.update_pair(a, b, rows[ids][:, :4])
    assert n_prop_used >= 3, n_prop_used                      # propagated map-point matches made it through RANSAC into the EntryJ list
    assert fc.tracks.stats()[0] > 20
    # ---- the cache: nothing is matched twice; a window's list is assembled from it
    assert fc.find_corres([(devf[4], devf[2]), (devf[3], devf[0])], [(4, 2), (3, 0)], w.H, w.W, w.K) == {}
    frames = [{"id": k} for k in range(N)]
    ent, blocks = fc.window_entries(frames, cuda_device)
    total = int(blocks[1].sum())
    assert total == sum(len(v) for v in host_entries.values()) and total >= 40
    corr_h = ent[:total].cpu().numpy().view(np.uint8).reshape(-1).view(synth.ENTRYJ_DTYPE)
    opt = OptimizerGpu(yml, max_windows=1, max_frames=8, max_corr=8192)
    depth = [f["depth"] for f in devf]; normal = [f["normal"] for f in devf]
    via_dev = opt.optimizeWindows([SolveWindow(None, w.H, w.W, depth, normal, w.poses_init, w.K, corr_dev=ent, blocks=blocks)])[0]
    via_host = opt.optimizeWindows([SolveWindow(corr_h, w.H, w.W, depth, normal, w.poses_init, w.K)])[0]
    assert np.array_equal(via_dev, via_host)
    opt.close()
    # ---- forgetFrame drops the frame's pairs; a neighbour pair with (almost) no features is a Frame::FAIL
    fc.forget_frame(4)
    assert not fc.has(4, 3) and fc.has(3, 2)
    few = dict(devf[4], kpts=devf[4]["kpts"][:0].contiguous(), id=4)       # feature detection found nothing
    mp.pool_store(4, devf[4]["desc"][:0].contiguous())
    res = fc.find_corres([(few, devf[3])], [(4, 3)], w.H, w.W, w.K)
    assert res[(4, 3)] == (0, 2) and 4 in fc.failed
    mp.close()

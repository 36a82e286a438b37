"""Generates tests/golden/ref_{solver,matcher,frontend}_runs.npz on a B200: what the GPU parity tests compare against the
reference's own kernels (oracle/_ref/libbt_ref.so, `make -C oracle ref`), recorded once so that the tests need neither the
reference sources nor oracle/_ref.  The inputs are the tests' seeded synthetic ones (bundletrack_b200/synth.py); next to the
reference's outputs each file keeps a few input values the tests check first, so that a change of the generator shows as
such and not as a parity failure.

    python scripts/make_golden_reference_runs.py OUT_DIR      # then copy OUT_DIR/ref_*_runs.npz to tests/golden/
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import oracle
from bundletrack_b200 import synth

out_dir = sys.argv[1]
os.makedirs(out_dir, exist_ok=True)
dev = torch.device("cuda:0")


def ref_solve(w, corr=None):
    depth = [torch.from_numpy(np.ascontiguousarray(w.depth[k])).to(dev) for k in range(w.n_frames)]
    normal = [torch.from_numpy(np.ascontiguousarray(w.normal[k])).to(dev) for k in range(w.n_frames)]
    args = ([d.data_ptr() for d in depth], [n.data_ptr() for n in normal], w.H, w.W, w.K, w.corr if corr is None else corr, w.poses_init)
    poses, pairs, _, _ = oracle.ref_optimize_frames(*args)
    again = oracle.ref_optimize_frames(*args)[0]      # the reference's float atomics: a second run is its own run-to-run yardstick
    return poses, pairs, again


# ---- tests/test_solver_gpu.py
sv = {}
for seed, N, C in ((0, 10, 2000), (40, 6, 1200)):
    w = synth.make_window(seed, n_frames=N, n_corr=C)
    sv[f"w{seed}_poses"], sv[f"w{seed}_pairs"], _ = ref_solve(w)
    sv[f"w{seed}_init"] = w.poses_init
w = synth.make_window(63, n_frames=30, n_corr=3000, occlusion=True)
sv["n30_poses"], sv["n30_pairs"], _ = ref_solve(w)
sv["n30_init"] = w.poses_init
poses, pairs, n_pairs, jitter, init_sum = [], [], [], [], []
for seed in range(200):
    N = 3 + seed % 6
    w = synth.make_window(5000 + seed, n_frames=N, n_corr=200 * N)
    p, pr, again = ref_solve(w)
    poses.append(p); pairs.append(pr); n_pairs.append(len(pr))
    jitter.append(max(synth.pose_errors(again, p)))
    init_sum.append(w.poses_init.astype(np.float64).sum())
sv.update(sweep_poses=np.concatenate(poses), sweep_pairs=np.concatenate(pairs).astype(np.uint8), sweep_n_pairs=np.asarray(n_pairs, np.int32),
          sweep_jitter=np.asarray(jitter), sweep_init_sum=np.asarray(init_sum))
print(f"parity sweep: reference run-to-run median {np.median(jitter):.2e}, max {np.max(jitter):.2e}")
np.savez_compressed(os.path.join(out_dir, "ref_solver_runs.npz"), **sv)

# ---- tests/test_matcher_gpu.py: RANSAC inlier sets (bit masks) and the fused chain's EntryJ list solved by the reference
mt = {}
for n, thresh in ((8, 0.005), (60, 0.005), (300, 0.01), (1000, 0.005), (3000, 0.005)):
    cases = [synth.make_ransac_case(7000 + 10 * n + k, n, 0.5 + 0.1 * k) for k in range(3)]
    ids, _ = oracle.ref_ransac_pairs([c[0] for c in cases], [c[1] for c in cases], 2000, thresh)
    for k, i in enumerate(ids):
        m = np.zeros(n, bool); m[i] = True
        mt[f"ransac_n{n}_{k}"] = np.packbits(m)
rng = np.random.default_rng(5)
cases = [synth.make_ransac_case(8000 + p, int(rng.integers(300, 1600)), float(rng.uniform(0.3, 0.9))) for p in range(45)]
ids, _ = oracle.ref_ransac_pairs([c[0] for c in cases], [c[1] for c in cases], 2000, 0.005)
mt["ransac_cfg2_n"] = np.asarray([len(c[0]) for c in cases], np.int32)
for p, i in enumerate(ids):
    m = np.zeros(len(cases[p][0]), bool); m[i] = True
    mt[f"ransac_cfg2_{p}"] = np.packbits(m)
from bundletrack_b200.matcher import MatchPipeline
yml = {"bundle": {"num_iter_outter": 7, "num_iter_inner": 5, "robust_delta": 0.005, "image_downscale": 4}, "p2p": {"max_dist": 0.02, "max_normal_angle": 45},
       "feature_corres": {"max_dist_no_neighbor": 0.02, "max_normal_no_neighbor": 45, "max_dist_neighbor": 10000, "max_normal_neighbor": 180},
       "ransac": {"max_iter": 2000, "inlier_dist": 0.01}}
w = synth.make_window(5, n_frames=4, n_corr=10)
fr = synth.make_feature_frames(w, 500, seed=5)
devf = [{"kpts": torch.from_numpy(fr[k]["kpts"]).to(dev), "desc": torch.from_numpy(fr[k]["desc"]).to(dev), "depth": torch.from_numpy(w.depth[k]).to(dev),
         "normal": torch.from_numpy(w.normal[k]).to(dev), "pose": w.poses_init[k], "id": k, "window_index": k} for k in range(4)]
mp = MatchPipeline(yml, max_pairs=8, max_feats=512)
ent, _, _ = mp.match_pairs([(devf[a], devf[b]) for a, b in [(j, i) for i in range(4) for j in range(i + 1, 4)]], w.H, w.W, w.K)
mp.close()
mt["fused_ent"] = np.ascontiguousarray(ent).view(np.uint8).reshape(-1, 32)
mt["fused_poses"], mt["fused_pairs"], mt["fused_poses_again"] = ref_solve(w, corr=ent)
mt["fused_init"] = w.poses_init
np.savez_compressed(os.path.join(out_dir, "ref_matcher_runs.npz"), **mt)

# ---- tests/test_frontend_gpu.py: one 640x480 frame through the reference's front end, kept at a seeded sample of pixels
raw, K = synth.make_raw_depth(7, 480, 640)
d, xyz, nrm, _ = oracle.ref_frame_preprocess(raw, K)
idx = np.sort(np.random.default_rng(7).choice(raw.size, 16384, replace=False)).astype(np.uint32)
np.savez_compressed(os.path.join(out_dir, "ref_frontend_runs.npz"), idx=idx, raw_sum=raw.astype(np.float64).sum(), depth=d.reshape(-1)[idx],
                    xyz=xyz.reshape(-1, 4)[idx, :3], normal=nrm.reshape(-1, 4)[idx, :3])
for f in ("ref_solver_runs.npz", "ref_matcher_runs.npz", "ref_frontend_runs.npz"):
    print(f, os.path.getsize(os.path.join(out_dir, f)), "bytes")

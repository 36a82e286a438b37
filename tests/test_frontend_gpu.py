"""GPU parity tests of the fused frame front end (bt_frames_preprocess through the C-ABI) against the CPU restatement
(oracle/frame_oracle.py) and the committed golden vectors of the reference's kernels (a 640x480 frame among them, kept at a
seeded sample of its pixels).  Tolerances: filtered depth 2e-6 m (a few float ulps at ~1 m; the reference build uses
fast-math exp/division), normals 1e-3 (unit vectors from ~1e-3 m differences amplify depth ulps), both allowing a small
fraction of pixels where a hard threshold (1 cm filter gate, 2 cm normal gate, 0.1 m validity) flips."""
import glob
import os

import numpy as np
import pytest

from bundletrack_b200 import synth
from oracle import frame_oracle

pytestmark = pytest.mark.gpu
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "ref_frame_*.npz")))


@pytest.fixture(scope="module")
def fe(cuda_device):
    from bundletrack_b200.frontend import FrameFrontEnd
    f = FrameFrontEnd()
    yield f
    f.close()


def _run(fe, raws, K, dev, dp=None, want_xyz=True):
    import torch
    from bundletrack_b200 import _lib
    if dp:
        full = dict(frame_oracle.DEFAULTS, **dp)
        fe.params = _lib.DepthParams(int(full["erode_radius"]), full["erode_diff"], full["erode_ratio"], int(full["bf_radius"]), full["sigma_D"], full["sigma_R"])
    else:
        from bundletrack_b200.config import depth_params
        fe.params = depth_params(None)
    H, W = raws[0].shape
    tin = [torch.from_numpy(np.ascontiguousarray(r)).to(dev) for r in raws]
    dout = [torch.full((H, W), -7.0, device=dev) for _ in raws]
    nout = [torch.full((H, W, 4), -7.0, device=dev) for _ in raws]
    xout = [torch.full((H, W, 4), -7.0, device=dev) for _ in raws] if want_xyz else None
    fe.process(tin, H, W, K, dout, nout, xout)
    torch.cuda.synchronize()
    return [d.cpu().numpy() for d in dout], [n.cpu().numpy() for n in nout], ([x.cpu().numpy() for x in xout] if want_xyz else None)


def _check(d, n, x, rd, rn, rx, frac=2e-3):
    bad_d = np.abs(d - rd) > 2e-6
    assert bad_d.mean() <= frac, f"depth: {bad_d.mean():.2e} of the pixels differ by > 2e-6 (max {np.abs(d - rd).max():.2e})"
    ok = ~bad_d
    if x is not None:
        assert np.abs(x[..., :3] - rx[..., :3])[ok].max() <= 3e-6
        assert np.array_equal(x[..., 3][ok], (rd >= 0.1).astype(np.float32)[ok])
    bad_n = np.abs(n[..., :3] - rn[..., :3]).max(-1) > 1e-3
    assert bad_n.mean() <= 2 * frac, f"normals: {bad_n.mean():.2e} of the pixels differ by > 1e-3"
    assert np.all(n[..., 3] == 0)


@pytest.mark.parametrize("seed,H,W", [(0, 120, 160), (1, 97, 131), (2, 480, 640)])
def test_matches_oracle(fe, cuda_device, seed, H, W):
    raw, K = synth.make_raw_depth(seed, H, W)
    d, n, x = _run(fe, [raw], K, cuda_device)
    rd, rx, rn = frame_oracle.preprocess(raw, K)
    _check(d[0], n[0], x[0], rd, rn, rx)
    assert (d[0] > 0).sum() > 0.02 * H * W          # the filter fills small holes and keeps the object


def test_other_parameters_and_batch(fe, cuda_device):
    dp = {"erode_radius": 2, "erode_diff": 0.004, "erode_ratio": 0.5, "bf_radius": 1, "sigma_D": 1.5, "sigma_R": 0.05}
    raws, K = [], None
    for s in (3, 4, 5):
        r, K = synth.make_raw_depth(s, 100, 140)
        raws.append(r)
    d, n, x = _run(fe, raws, K, cuda_device, dp)
    for i, r in enumerate(raws):
        rd, rx, rn = frame_oracle.preprocess(r, K, dp)
        _check(d[i], n[i], x[i], rd, rn, rx)
    # a batch equals the same frames one at a time, bit for bit; xyz is optional
    d1, n1, _ = _run(fe, [raws[1]], K, cuda_device, dp, want_xyz=False)
    assert np.array_equal(d1[0], d[1]) and np.array_equal(n1[0], n[1])


def test_edge_cases(fe, cuda_device):
    import torch
    from bundletrack_b200 import _lib
    K = synth.NOCS_K
    zero = np.zeros((70, 90), np.float32)
    d, n, x = _run(fe, [zero], K, cuda_device)
    assert not d[0].any() and not n[0].any() and not x[0].any()
    # constant plane: interior depth unchanged to rounding, normals point at the camera; the image border has no normal
    plane = np.full((64, 80), 0.75, np.float32)
    d, n, x = _run(fe, [plane], K, cuda_device)
    assert np.abs(d[0] - 0.75).max() < 1e-6
    assert np.allclose(n[0][1:-1, 1:-1, :3], [0, 0, -1], atol=1e-3)     # (x - cx) / fx * d differences cancel to ~1e-4 relative
    assert not n[0][0].any() and not n[0][-1].any() and not n[0][:, 0].any() and not n[0][:, -1].any()
    # an isolated flying pixel is eroded away and refilled from its neighbours by the filter
    spike = plane.copy(); spike[30, 40] = 0.80
    d, _, _ = _run(fe, [spike], K, cuda_device)
    assert abs(d[0][30, 40] - 0.75) < 1e-6
    # errors are reported, not fatal
    t = torch.zeros((64, 80), device=cuda_device)
    nn = torch.zeros((64, 80, 4), device=cuda_device)
    with pytest.raises(_lib.BtError):
        fe.process([t], 64, 80, K, [t], [nn])                       # in place
    fe.params = _lib.DepthParams(5, 0.001, 0.8, 4, 2.0, 1e5)         # halo 14 > supported
    with pytest.raises(_lib.BtError):
        fe.process([t], 64, 80, K, [torch.zeros_like(t)], [nn])


@pytest.mark.skipif(not GOLDEN, reason="no golden vectors")
@pytest.mark.parametrize("path", GOLDEN)
def test_golden_reference_kernels(fe, cuda_device, path):
    g = np.load(path)
    dp = {k: float(g[k]) for k in frame_oracle.DEFAULTS}
    d, n, x = _run(fe, [g["raw"]], tuple(g["K"]), cuda_device, dp)
    rn = np.concatenate([g["normal"], np.zeros(g["normal"].shape[:2] + (1,), np.float32)], -1)
    rx = np.concatenate([g["xyz"], (g["depth"] >= 0.1).astype(np.float32)[..., None]], -1)
    _check(d[0], n[0], x[0], g["depth"], rn, rx)


def test_matches_reference_kernels_live(fe, cuda_device):
    """The reference's front end on a 640x480 frame, recorded on a B200 at 16384 seeded pixels (tests/golden/ref_frontend_runs.npz,
    scripts/make_golden_reference_runs.py); the library processes the whole frame and is compared at those pixels."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_frontend_runs.npz"))
    raw, K = synth.make_raw_depth(7, 480, 640)
    assert abs(raw.astype(np.float64).sum() - float(g["raw_sum"])) <= 1e-6 * abs(float(g["raw_sum"]))     # the frame the reference saw
    d, n, x = _run(fe, [raw], K, cuda_device)
    i = g["idx"]
    _check(d[0].reshape(-1)[i], n[0].reshape(-1, 4)[i], x[0].reshape(-1, 4)[i], g["depth"], g["normal"], g["xyz"])


def test_feeds_the_solver(fe, cuda_device):
    """Front-end outputs are exactly the maps bt_solve_windows consumes: solving on GPU-filtered maps equals the oracle solving
    on oracle-filtered maps (1e-4 rad / 1e-4 m, north_star's gate)."""
    import torch
    import oracle
    from bundletrack_b200.optimizer import OptimizerGpu, SolveWindow
    w = synth.make_window(11, n_frames=3, n_corr=400, H=240, W=320, K=tuple(v * 0.5 for v in synth.NOCS_K))
    rng = np.random.default_rng(5)
    raws = [(w.depth[k] + (w.depth[k] > 0) * rng.normal(0, 0.0003, w.depth[k].shape)).astype(np.float32) for k in range(3)]
    d, n, _ = _run(fe, raws, w.K, cuda_device, want_xyz=False)
    td = [torch.from_numpy(v).to(cuda_device) for v in d]
    tn = [torch.from_numpy(v).to(cuda_device) for v in n]
    opt = OptimizerGpu(None, max_windows=1, max_frames=3, max_corr=400, H=240, W=320)
    got = opt.optimizeWindows([SolveWindow(w.corr, 240, 320, td, tn, w.poses_init, w.K)])[0]
    opt.close()
    od = np.stack([frame_oracle.preprocess(r, w.K)[0] for r in raws])
    on = np.stack([frame_oracle.preprocess(r, w.K)[2] for r in raws])
    ref = oracle.solve_window(od, on, w.K, w.corr, w.poses_init)
    r, t = synth.pose_errors(got, ref)
    assert r <= 1e-4 and t <= 1e-4

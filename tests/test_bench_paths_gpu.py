"""GPU parity tests of exactly the entry points bench.py times (VERDICT r1 weak #2): orbx_extract_batch_device with several
handles on several CUDA streams at the bench batch size (level 0 read straight from the caller's tensor), the host slab
variant, the host and device batched last-frame matchers fed from those slabs, and the blurred planes -- all against the CPU
oracle, bit for bit."""
import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

W, H = 640, 480


@pytest.fixture(scope='module')
def orb():
    import orb_slam3_modified_b200 as m
    m.lib()
    return m


@pytest.fixture(scope='module')
def bench():
    import bench as b
    return b


@pytest.fixture(scope='module')
def oracle_sets(bench):
    """Oracle extraction of the bench's distinct source frames (both parities)."""
    oe = O.OracleExtractor(1000, 1.2, 8, 20, 7)
    out = []
    for k in range(2):
        fr = bench.make_frames(bench.DISTINCT, k)
        out.append((fr, [oe(f, (0, 1000)) for f in fr]))
    return out


def test_extract_batch_device_four_stream_groups_at_bench_batch(orb, bench, oracle_sets):
    import torch
    B, DG = 256, 4
    dev = torch.device('cuda')
    frames = bench.make_frames(B, 1)
    d_img = torch.from_numpy(frames).to(dev)
    gb = [(g * B // DG, (g + 1) * B // DG) for g in range(DG)]
    exs = [orb.ORBextractor(1000, 1.2, 8, 20, 7, W, H, b1 - b0) for b0, b1 in gb]
    cap = exs[0].max_keypoints
    d_kps = torch.zeros((B, cap, 7), dtype=torch.float32, device=dev)
    d_desc = torch.zeros((B, cap, 32), dtype=torch.uint8, device=dev)
    d_n = torch.zeros(B, dtype=torch.int32, device=dev)
    d_mono = torch.zeros(B, dtype=torch.int32, device=dev)
    streams = [torch.cuda.Stream() for _ in gb]
    torch.cuda.synchronize()
    for rep in range(2):     # the second pass runs over warm handles, like the timed loop
        for g, (b0, b1) in enumerate(gb):
            exs[g].extract_batch_device(d_img[b0:b1], d_kps[b0:b1], d_desc[b0:b1], d_n[b0:b1], d_mono[b0:b1], (0, 1000), streams[g].cuda_stream)
    torch.cuda.synchronize()
    n = d_n.cpu().numpy(); mono = d_mono.cpu().numpy()
    kps = d_kps.cpu().numpy().view(np.uint8).reshape(B, cap, 28); desc = d_desc.cpu().numpy()
    for b in range(B):
        omono, okps, odesc = oracle_sets[1][1][b % bench.DISTINCT]
        assert n[b] == len(okps) and mono[b] == omono, b
        assert kps[b, :n[b]].tobytes() == okps.tobytes(), b
        assert np.array_equal(desc[b, :n[b]], odesc), b


def test_extract_batch_slabs_and_host_batch_matcher(orb, bench, oracle_sets):
    """The e2e path of bench.py: host slabs out of orbx_extract_batch, then orbm_search_last_frame_batch on them."""
    from orb_slam3_modified_b200 import synth
    B = 48
    frames = bench.make_frames(B, 1)
    ex = orb.ORBextractor(1000, 1.2, 8, 20, 7, W, H, B)
    cap = ex.max_keypoints
    kps = np.zeros((B, cap), orb.KP_DTYPE); desc = np.zeros((B, cap, 32), np.uint8)
    nK = np.zeros(B, np.int32); mono = np.zeros(B, np.int32)
    ex.extract_batch_slabs(frames, kps, desc, nK, mono, (0, 1000))
    for b in range(B):
        omono, okps, odesc = oracle_sets[1][1][b % bench.DISTINCT]
        assert nK[b] == len(okps) and mono[b] == omono
        assert kps[b, :nK[b]].tobytes() == okps.tobytes() and np.array_equal(desc[b, :nK[b]], odesc)
    # last frame = parity 0 of every stream, as bench.last_frame_slabs builds it
    kl = [oracle_sets[0][1][b % bench.DISTINCT][1] for b in range(B)]
    dl = [oracle_sets[0][1][b % bench.DISTINCT][2] for b in range(B)]
    L = bench.last_frame_slabs(kl, dl, 0, cap)
    poses = np.stack([bench.stream_pose(s, 1) for s in range(B)])
    sf = ex.GetScaleFactors()
    cam = [float(c) for c in synth.camera(W, H)]
    matcher = orb.ORBmatcher(0.9, True, max_batch=B, max_keypoints=cap, max_mappoints=cap)
    d = dict(batch=B, kcap=cap, mcap=cap, nlevels=8, kps=kps, desc=desc, nK=nK, scaleFactors=sf, nM=L['nM'], valid=L['valid'], xyz=L['xyz'],
             octave=L['octave'], angle=L['angle'], hasObs=L['hasObs'], mpDesc=L['mpDesc'], Tcw7=poses, bounds=(0.0, 0.0, float(W), float(H)), cam=cam, reset=1)
    match = np.full((B, cap), 123, np.int32); claimed = np.full((B, cap), 1, np.uint8); nm = np.zeros(B, np.int32)   # garbage in: reset=1 must ignore it
    matcher.search_last_frame_batch(d, bench.TH_PROJ, match, claimed, nm)
    for b in range(B):
        k = int(nK[b]); m = int(L['nM'][b])
        last = dict(valid=L['valid'][b, :m], xyz=L['xyz'][b, :m], octave=L['octave'][b, :m], angle=L['angle'][b, :m], hasObs=L['hasObs'][b, :m],
                    descriptors=L['mpDesc'][b, :m])
        om = np.full(k, -1, np.int32); oc = np.zeros(k, np.uint8)
        on = O.search_last_frame(kps[b, :k], desc[b, :k], (0.0, 0.0, float(W), float(H)), sf, poses[b], cam, last, bench.TH_PROJ, True, om, oc)
        assert nm[b] == on and on > 300, (b, nm[b], on)
        assert np.array_equal(match[b, :k], om) and np.array_equal(claimed[b, :k], oc), b


def test_bench_dump_outputs_are_the_timed_loop_results(bench, oracle_sets, tmp_path):
    """bench.py --dump-outputs at a small size: the dumped keypoints, descriptors and matches of every stream are the oracle's on the
    frames bench.make_frames rebuilds from their seeds, a dumped bundle adjustment is the oracle's solution of its problem, and the
    kernel launches the timed loop counted grow in proportion to --steps."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.abspath(bench.__file__))
    out = str(tmp_path / 'dump')
    runs = {}
    for steps in (1, 3):
        cmd = [sys.executable, os.path.join(root, 'bench.py'), '--steps', str(steps), '--warmup', '1', '--batch', '10', '--rounds', '2', '--lba-rounds', '2',
               '--no-cpu-baseline', '--no-e2e', '--no-extra'] + (['--dump-outputs', out] if steps == 3 else [])
        runs[steps] = json.loads(subprocess.check_output(cmd, cwd=root, timeout=900).decode().strip().splitlines()[-1])
    assert runs[3]['gpu_launches'] == 3 * runs[1]['gpu_launches'] > 0 and runs[3]['config']['frames_per_gpu_per_step'] == 20
    d = {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}
    assert all(v.dtype in (np.float32, np.float64) for v in d.values()) and sum(v.nbytes for v in d.values()) <= 64 << 20
    assert np.array_equal(d['frame_streams'], np.arange(10)) and np.array_equal(d['lba_problems'], np.arange(2))
    from orb_slam3_modified_b200 import synth
    kl = [oracle_sets[0][1][b][1] for b in range(10)]
    L = bench.last_frame_slabs(kl, [oracle_sets[0][1][b][2] for b in range(10)], 0, max(len(k) for k in kl))
    sf = O.OracleExtractor(1000, 1.2, 8, 20, 7).tables()['scale']
    cam = [float(c) for c in synth.camera(W, H)]
    o = 0
    for b in range(10):       # 6 timed rounds: the last one extracted parity 1 and matched it against parity 0
        omono, okps, odesc = oracle_sets[1][1][b]
        k, m = len(okps), int(L['nM'][b])
        assert d['frame_n_keypoints'][b] == k and d['frame_mono'][b] == omono
        kp = d['frame_keypoints'][o:o + k]
        assert np.array_equal(kp[:, 0], okps['x']) and np.array_equal(kp[:, 5], okps['octave']) and np.array_equal(d['frame_descriptors'][o:o + k], odesc)
        last = {n: L[v][b, :m] for n, v in (('valid', 'valid'), ('xyz', 'xyz'), ('octave', 'octave'), ('angle', 'angle'), ('hasObs', 'hasObs'),
                                            ('descriptors', 'mpDesc'))}
        om = np.full(k, -1, np.int32); oc = np.zeros(k, np.uint8)
        on = O.search_last_frame(okps, odesc, (0.0, 0.0, float(W), float(H)), sf, bench.stream_pose(b, 1), cam, last, bench.TH_PROJ, True, om, oc)
        assert d['frame_n_matches'][b] == on and np.array_equal(d['frame_match'][o:o + k], om) and np.array_equal(d['frame_claimed'][o:o + k], oc)
        o += k
    assert o == len(d['frame_keypoints'])
    # problem 1 (bench's own parity gate checks problem 0): poses / points / statistics are the oracle's solution of that problem
    nP, nL = bench.LBA_CFG['n_kf'], bench.LBA_CFG['n_pts']
    prob = bench.lba_problems(2)[1]
    ref = O.lba_solve(prob)
    poses, points = d['lba_poses'][nP:2 * nP], d['lba_points'][nL:2 * nL]
    assert d['lba_poses'].shape == (2 * nP, 7) and d['lba_points'].shape == (2 * nL, 3) and len(d['lba_chi2']) == len(d['lba_depth_pos'])
    assert d['lba_stats'][1, 0] == ref['iters'] and d['lba_stats'][1, 1] == ref['stats'][3]
    assert np.abs(O.lba_residuals(prob, poses, points) - O.lba_residuals(prob, ref['poses'], ref['points'])).max() < bench.TOL_PX


def test_blurred_planes_equal_oracle(orb, bench):
    """a6: the 7x7 sigma-2 blur of every level, byte for byte (src/ORBextractor.cc:1132-1133)."""
    B = 3
    frames = bench.make_frames(B, 0)
    ex = orb.ORBextractor(1000, 1.2, 8, 20, 7, W, H, B)
    ex.extract_batch(frames, (0, 1000))
    oe = O.OracleExtractor(1000, 1.2, 8, 20, 7)
    for b in range(B):
        oe(frames[b], (0, 1000))
        for l in range(8):
            want = O.blur7(oe.level(l))
            got = ex.level(l, frame=b, blurred=True)
            assert got.shape == want.shape and np.array_equal(got, want), (b, l, int((got != want).sum()))
            assert np.array_equal(ex.level(l, frame=b), oe.level(l)), (b, l)

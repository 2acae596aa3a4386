"""CPU checks of bench.py's host-side pieces: the clock sampler's bookkeeping, and the reference arm's JSON contract
(`--impl reference`: the oracle on the host cores, one worker process per core)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_clock_sampler_reports_only_the_marked_region():
    import bench

    class FakeProc:
        stdout = iter(['1965, 1965, Not Active, Not Active, Not Active, Not Active\n'] * 4)

        def terminate(self):
            pass

        def wait(self, timeout=None):
            pass

    cs = bench.ClockSampler.__new__(bench.ClockSampler)
    cs.rows, cs.m0, cs.proc = [], 0, FakeProc()
    cs._read()
    assert cs.samples() == 4
    cs.mark()
    assert cs.samples() == 0
    cs.rows.append(['1830', '1965', 'Not Active', 'Not Active', 'Not Active', 'Active'])
    out = cs.stop()
    assert out == {'sm_mhz': 1830, 'sm_max_mhz': 1965, 'reasons': ['sw_power_cap'], 'samples': 1}


def test_reference_arm_json_contract():
    two = sorted(os.sched_getaffinity(0))[:2]
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                                  cwd=ROOT, preexec_fn=lambda: os.sched_setaffinity(0, two), timeout=600).decode().strip().splitlines()
    d = json.loads(out[-1])
    assert d['impl'] == 'reference' and d['unit'] == 'frames/s' and d['higher_is_better'] is True and d['value'] > 0
    have_ref = os.path.exists(os.path.join(ROOT, 'oracle', '_ref', 'libref_orb.so'))
    cb = d['cpu_baseline']
    assert cb['kind'] == ('reference' if have_ref else 'port') and cb['kind_per_stage']['lba'] == 'port'
    assert cb['cores'] == len(two) and cb['value'] == d['value'] and 0.4 <= cb["effective_cores_measured"] <= 2.6       # a timing ratio on a shared box: sanity bounds only
    assert cb['split']['extract_ms_per_frame'] > 1 and cb['split']['lba_ms_per_problem'] > 10
    assert d['e2e'] == {'value': d['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert d['metric'].startswith('frames/sec') and d['config']['workload'].startswith('configs[1]')


def test_host_cores_respects_affinity():
    import bench
    n, how = bench.host_cores()
    assert 1 <= n <= len(os.sched_getaffinity(0)) and isinstance(how, str)


def test_dump_outputs_writes_the_sampled_rows_as_float_arrays(tmp_path):
    """--dump-outputs on host tensors shaped like the device loop's: valid rows only, a seeded sample, float32 / float64 files."""
    import numpy as np
    import torch
    import bench
    from orb_slam3_modified_b200 import sharding
    gb, cap = [(0, 7), (7, 40)], 16
    slabs = [sharding.PackedSlab(b1 - b0, cap, 'cpu') for b0, b1 in gb]
    match, claimed, nmatch = [], [], []
    for g, (b0, b1) in enumerate(gb):
        S = slabs[g]
        for i, b in enumerate(range(b0, b1)):
            S.n[i], S.mono[i] = b % 5 + 3, b
            S.kps[i, :, :5] = b + torch.arange(cap, dtype=torch.float32)[:, None]
            S.kps[i].view(torch.int32)[:, 5:] = torch.arange(cap, dtype=torch.int32)[:, None]
            S.desc[i] = b
        match.append(torch.arange(b0, b1, dtype=torch.int32)[:, None].repeat(1, cap))
        claimed.append(torch.ones((b1 - b0, cap), dtype=torch.uint8))
        nmatch.append(torch.arange(b0, b1, dtype=torch.int32) + 100)
    lba_out = [dict(poses=np.full((3, 7), p, np.float64), points=np.full((5, 3), p, np.float64), chi2=np.full(4, p, np.float64),
                    depth_pos=np.ones(4, np.uint8), iters=p, trials=p + 1, lambda_=0.5, initial_chi2=2.0, final_chi2=1.0) for p in range(12)]
    out = str(tmp_path / 'dump')
    bench.dump_outputs(out, gb, slabs, match, claimed, nmatch, lba_out)
    d = {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}
    assert all(v.dtype in (np.float32, np.float64) for v in d.values())
    s = d['frame_streams'].astype(int)
    assert len(s) == bench.DUMP_STREAMS and len(set(s)) == len(s) and list(s) == sorted(s) and s.max() < 40
    n = s % 5 + 3
    assert np.array_equal(d['frame_n_keypoints'], n) and np.array_equal(d['frame_mono'], s) and np.array_equal(d['frame_n_matches'], s + 100)
    rows = np.concatenate([np.arange(k) for k in n])
    owner = np.repeat(s, n)
    assert d['frame_keypoints'].shape == (n.sum(), 7) and np.array_equal(d['frame_keypoints'][:, 0], owner + rows)
    assert np.array_equal(d['frame_keypoints'][:, 6], rows) and np.array_equal(d['frame_descriptors'], np.repeat(owner[:, None], 32, 1))
    assert np.array_equal(d['frame_match'], owner) and np.all(d['frame_claimed'] == 1)
    p = d['lba_problems'].astype(int)
    assert len(p) == bench.DUMP_LBAS and np.array_equal(d['lba_points'], np.repeat(p, 5)[:, None].repeat(3, 1))
    assert np.array_equal(d['lba_poses'], np.repeat(p, 3)[:, None].repeat(7, 1)) and np.array_equal(d['lba_chi2'], np.repeat(p, 4))
    assert np.array_equal(d['lba_stats'][:, :2], np.stack([p, p + 1], 1)) and d['lba_depth_pos'].shape == (4 * len(p),)
    again = str(tmp_path / 'again')
    bench.dump_outputs(again, gb, slabs, match, claimed, nmatch, lba_out)
    assert all(np.array_equal(np.load(os.path.join(again, k + '.npy')), v) for k, v in d.items())


def test_reference_arm_other_ranks_do_nothing():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2'], cwd=ROOT, env=env, timeout=120)
    assert out.strip() == b''

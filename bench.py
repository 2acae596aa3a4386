#!/usr/bin/env python3
"""bench.py -- frames/sec of the ORB-SLAM3 hot path (BASELINE.json metric) on N B200s.

One "step" = ROUNDS rounds (default 16); in one round every one of the B synthetic 640x480 mono streams of a GPU (default 240)
advances by one frame:
  * ORBextractor::operator() + ORBmatcher::SearchByProjection(current, last frame) for every stream   (BASELINE configs[1]);
  * every KF_INTERVAL-th frame of a stream is a keyframe and triggers one LocalBundleAdjustment of the configs[3] size
    (20 keyframes x 5000 points x 40000 edges) on the mapping side -> exactly B / KF_INTERVAL LBAs per round, on both arms.
`value` is whole-job frames/s with all inputs already resident in HBM; `e2e` is the same metric through the reference-facing C-ABI
with HOST buffers (pinned), host<->device copies inside the timed region.  Before anything is printed, a sample of the buffers the
TIMED loops wrote (frames and bundle adjustments, both measurements) is compared with the CPU oracle; a mismatch aborts the run.
--impl reference times the CPU implementation of the path on the host cores: the reference's own ORBextractor / SearchByProjection
text (oracle/_ref, compiled from /root/reference against type stand-ins) + the oracle port of the g2o bundle adjustment.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'frames/sec (extract+match+LBA) 640x480 mono-inertial'
UNIT = 'frames/s'
W, H, NFEAT = 640, 480, 1000
KF_INTERVAL = 10     # one keyframe (-> one LBA) per 10 frames of a stream
LBA_CFG = dict(n_kf=20, n_pts=5000, obs_per_pt=8)   # BASELINE configs[3]
STAGES = ['extract', 'match(SearchByProjection last frame)', 'LBA(1 per %d frames)' % KF_INTERVAL]
WORKLOAD = 'configs[1]: 640x480 mono stream, 1000 feats/frame, extract+SearchByProjection, + configs[3]-sized LBA every %d frames' % KF_INTERVAL
# SURVEY.md 8d algorithmic bytes, 640x480, K = 1000 keypoints (S = 950,532 px over the 8 levels, A0 = 307,200, A7 = 23,986)
ALG = {'pyramid': 926546 + 643332, 'blur': 2 * 950532, 'fast_cells': 950532, 'quadtree_orient': 749 * 1000, 'assemble': 60 * 1000,
       'brief': 512 * 1000 + 32 * 1000}
ALG_BYTES_EXTRACT = 5742474
ALG_BYTES_MATCH = 552000
ALG_BYTES_LBA_PER_TRIAL = 13.6e6
DISTINCT = 32        # distinct synthetic streams; larger batches replicate them (separate buffers, same content)
TH_PROJ = 15.0       # SearchByProjection window for mono tracking (reference src/Tracking.cc:2884-2889)
TOL_PX = 1e-4        # LBA parity bar (BASELINE.json north_star): reprojection residuals within 1e-4 px of the oracle's


def _peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return json.load(open(p))['hbm_gbs'], 'measured'
    return 6650.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows, self.proc, self.m0 = [], None, 0
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(index), '--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
                 'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap',
                 '--format=csv,noheader,nounits', '-lms', '50'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def mark(self):
        """Start of the region of interest: only samples taken from here on are reported."""
        self.m0 = len(self.rows)

    def samples(self):
        return len(self.rows) - self.m0

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = self.rows[self.m0:]
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith('active')})
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
# synthetic workload
# ------------------------------------------------------------------------------------------------
def stream_time(s, k):
    """Frame index of distinct stream s at parity k (consecutive frames t, t+1)."""
    return 5 * s + k


def make_frames(n, k, rank=0):
    from orb_slam3_modified_b200 import synth
    import numpy as np
    d = min(n, DISTINCT)
    base = np.stack([synth.frame(stream_time(s, k), W, H, seed=s % 4 + 4 * rank) for s in range(d)])
    return np.ascontiguousarray(np.concatenate([base] * ((n + d - 1) // d))[:n])


def stream_pose(s, k, rank=0, noise=0.003):
    """Motion-model prior of Tcw for stream s at parity k: the exact synthetic pose plus a seeded perturbation."""
    from orb_slam3_modified_b200 import synth
    import numpy as np
    d = s % DISTINCT
    rng = np.random.default_rng(1000 * rank + 2 * d + k)
    T = synth.pose(stream_time(d, k), seed=d % 4 + 4 * rank)
    T[4:] += rng.normal(0, noise, 3)
    return T.astype(np.float32)


def last_frame_slabs(kps_list, desc_list, k_last, cap, rank=0):
    """Map points of the 'last frame' (parity k_last) of every stream as fixed-capacity host slabs."""
    from orb_slam3_modified_b200 import synth
    import numpy as np
    B = len(kps_list)
    out = dict(nM=np.zeros(B, np.int32), valid=np.zeros((B, cap), np.uint8), xyz=np.zeros((B, cap, 3), np.float32),
               octave=np.zeros((B, cap), np.int32), angle=np.zeros((B, cap), np.float32), hasObs=np.zeros((B, cap), np.uint8),
               mpDesc=np.zeros((B, cap, 32), np.uint8))
    for b in range(B):
        k, d = kps_list[b], desc_list[b]
        m = len(k)
        sd = b % DISTINCT
        out['nM'][b] = m
        out['valid'][b, :m] = 1
        out['xyz'][b, :m] = synth.backproject(np.stack([k['x'], k['y']], 1), stream_time(sd, k_last), sd % 4 + 4 * rank, W, H)
        out['octave'][b, :m] = k['octave']
        out['angle'][b, :m] = k['angle']
        out['hasObs'][b, :m] = 1
        out['mpDesc'][b, :m] = d
    return out


def lba_problems(n, rank=0):
    from orb_slam3_modified_b200 import synth
    base = [synth.lba_problem(seed=100 * rank + i, **LBA_CFG) for i in range(min(n, 4))]
    return [base[i % len(base)] for i in range(n)]


# ------------------------------------------------------------------------------------------------
# CPU side: the reference's own text where it compiles here (oracle/_ref), the oracle port elsewhere
# ------------------------------------------------------------------------------------------------
def _cpu_impl():
    """(extractor class, last-frame matcher, LBA solver, kind dict).  oracle/_ref is /root/reference/src/ORBextractor.cc and the
    SearchByProjection body of src/ORBmatcher.cc compiled verbatim (oracle/Makefile); g2o needs Eigen and is the oracle port."""
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import oracle_lib as O
    if os.path.exists(os.path.join(ROOT, 'oracle', '_ref', 'libref_orb.so')):
        import ref_lib as R
        return R.RefExtractor, R.search_last_frame, O.lba_solve, {'extract': 'reference', 'match': 'reference', 'lba': 'port'}
    return O.OracleExtractor, O.search_last_frame, O.lba_solve, {'extract': 'port', 'match': 'port', 'lba': 'port'}


def host_cores():
    """(cores this process may use, how that was determined): the affinity mask, capped by the cgroup CPU quota -- a container with 128
    visible CPUs and a quota of 12 runs 128 workers no faster than 12."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    how = 'sched_getaffinity'
    quota = None
    try:
        q, p = open('/sys/fs/cgroup/cpu.max').read().split()[:2]           # cgroup v2
        if q != 'max':
            quota = float(q) / float(p)
    except (OSError, ValueError):
        try:                                                                # cgroup v1
            q = float(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            p = float(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    if quota is not None and quota < n:
        n, how = max(1, int(quota + 0.5)), 'cgroup cpu quota %.1f' % quota
    return n, how


def _spin(n):
    x = 0
    for i in range(n):
        x += i * i
    return x


def measured_parallelism(workers, pool):
    """How many cores the pool really gets: aggregate rate of `workers` identical CPU-bound tasks over the single-task rate
    (catches quotas that neither the affinity mask nor the cgroup files show)."""
    n = 2_000_000
    _spin(n // 10)
    t0 = time.perf_counter(); _spin(n); t1 = time.perf_counter() - t0
    t0 = time.perf_counter(); pool.map(_spin, [n] * workers, chunksize=1); tp = time.perf_counter() - t0
    return workers * t1 / tp


def cpu_info():
    model = None
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                model = line.split(':', 1)[1].strip()
                break
    except OSError:
        pass
    return {'model': model, 'nproc': os.cpu_count()}


def cv2_orb_ms(frames, n=12):
    """Single-thread OpenCV ORB (SIMD build) on the same frames, next to the scalar CPU arm (SURVEY.md 8d: note the gap explicitly)."""
    try:
        import cv2
        cv2.setNumThreads(1)
        orb = cv2.ORB_create(NFEAT, 1.2, 8)
        orb.detectAndCompute(frames[0], None)
        t0 = time.perf_counter()
        for i in range(n):
            orb.detectAndCompute(frames[i % len(frames)], None)
        return 1e3 * (time.perf_counter() - t0) / n
    except Exception:
        return None


_REF = {}


def _ref_init(nsrc):
    """Worker-process initialiser of the CPU arm: extractor + the untimed 'last frame' of every source stream."""
    import numpy as np
    from orb_slam3_modified_b200 import synth
    Ex, search, lba, kind = _cpu_impl()
    ex = Ex(NFEAT, 1.2, 8, 20, 7)
    f0, f1 = make_frames(nsrc, 0), make_frames(nsrc, 1)
    last = []
    for s in range(nsrc):
        _, k, d = ex(f0[s], (0, 1000))
        last.append(dict(valid=np.ones(len(k), np.uint8), xyz=synth.backproject(np.stack([k['x'], k['y']], 1), stream_time(s, 0), s % 4, W, H).astype(np.float32),
                         octave=k['octave'].astype(np.int32), angle=k['angle'].astype(np.float32), hasObs=np.ones(len(k), np.uint8), descriptors=d))
    _REF.update(ex=ex, search=search, lba=lba, f1=f1, last=last, sf=ex.tables()['scale'], cam=synth.camera(W, H),
                poses=[stream_pose(s, 1) for s in range(nsrc)], prob=lba_problems(1)[0], nsrc=nsrc)
    return True


def _ref_work(job):
    """One worker's share: frames first .. n by stride (extract + SearchByProjection), then its share of the LBAs (1 per 10 frames)."""
    import numpy as np
    first, stride, n_frames, n_lba = job
    R = _REF
    t_ex = t_mt = t_lba = 0.0
    for i in range(first, n_frames, stride):
        s = i % R['nsrc']
        t0 = time.perf_counter()
        _, k, d = R['ex'](R['f1'][s], (0, 1000))
        t1 = time.perf_counter()
        match = np.full(len(k), -1, np.int32)
        claimed = np.zeros(len(k), np.uint8)
        R['search'](k, d, (0.0, 0.0, float(W), float(H)), R['sf'], R['poses'][s], R['cam'], R['last'][s], TH_PROJ, True, match, claimed)
        t2 = time.perf_counter()
        t_ex += t1 - t0; t_mt += t2 - t1
    for i in range(first, n_lba, stride):
        t0 = time.perf_counter()
        R['lba'](R['prob'])
        t_lba += time.perf_counter() - t0
    return t_ex, t_mt, t_lba


def run_cpu_arm(workers, steps, warmup, per_worker_frames):
    """Runs the CPU arm on `workers` processes; returns (frames/s, seconds, sample string, split dict)."""
    import multiprocessing as mp
    nsrc = 16
    n_frames = per_worker_frames * workers
    n_lba = n_frames // KF_INTERVAL
    if workers == 1:      # in this process (the GPU arm calls this after CUDA is up: no fork)
        _ref_init(nsrc)
        for _ in range(max(warmup, 1)):
            _ref_work((0, 1, KF_INTERVAL, 1))
        t0 = time.perf_counter()
        acc = [0.0, 0.0, 0.0]
        for _ in range(steps):
            r = _ref_work((0, 1, n_frames, n_lba))
            for i in range(3):
                acc[i] += r[i]
        t_all = time.perf_counter() - t0
        fps = n_frames * steps / t_all
        split = {'extract_ms_per_frame': 1e3 * acc[0] / (n_frames * steps), 'match_ms_per_frame': 1e3 * acc[1] / (n_frames * steps),
                 'lba_ms_per_problem': 1e3 * acc[2] / max(n_lba * steps, 1)}
        return fps, t_all, '%d frames (extract+SearchByProjection) + %d LBAs (20 KF x 5000 pts x 40k edges), 1 thread' % (n_frames * steps, n_lba * steps), split, 1.0
    ctx = mp.get_context('fork')
    with ctx.Pool(workers, initializer=_ref_init, initargs=(nsrc,)) as pool:
        jobs = [(w, workers, n_frames, n_lba) for w in range(workers)]
        warm = [(w, workers, KF_INTERVAL * workers, workers) for w in range(workers)]
        for _ in range(max(warmup, 1)):
            pool.map(_ref_work, warm, chunksize=1)                  # the first one also waits for every worker's initialiser
        eff = measured_parallelism(workers, pool) if workers > 1 else 1.0
        t_all, acc = 0.0, [0.0, 0.0, 0.0]
        for _ in range(steps):
            t0 = time.perf_counter()
            res = pool.map(_ref_work, jobs, chunksize=1)
            t_all += time.perf_counter() - t0
            for r in res:
                for i in range(3):
                    acc[i] += r[i]
    fps = n_frames * steps / t_all
    split = {'extract_ms_per_frame': 1e3 * acc[0] / (n_frames * steps), 'match_ms_per_frame': 1e3 * acc[1] / (n_frames * steps),
             'lba_ms_per_problem': 1e3 * acc[2] / max(n_lba * steps, 1)}
    sample = '%d frames (extract+SearchByProjection) + %d LBAs (20 KF x 5000 pts x 40k edges) per step on %d worker process%s' % (
        n_frames, n_lba, workers, '' if workers == 1 else 'es')
    return fps, t_all, sample, split, eff


def run_reference(args):
    """Reference arm: the CPU implementation of the path on all host cores the process really has -- one worker PROCESS per core."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    cores, how = host_cores()
    kind = _cpu_impl()[3]
    fps, t_all, sample, split, eff = run_cpu_arm(cores, args.steps, args.warmup, 4 * KF_INTERVAL)   # 40 frames + 4 LBAs per worker and step: ~1 s
    cv2ms = cv2_orb_ms(make_frames(4, 1))
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * t_all / max(args.steps, 1), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'u8 (extract/match), f64 (LBA)', 'data': 'synthetic', 'config': {'workload': WORKLOAD, 'stages': STAGES},
        'cpu_baseline': {'value': fps, 'unit': UNIT, 'cores': cores, 'kind': 'reference' if kind['extract'] == 'reference' else 'port',
                         'kind_per_stage': kind, 'sample': sample, 'host': cpu_info(), 'cores_from': how,
                         'effective_cores_measured': round(eff, 1), 'split': split,
                         'build': 'oracle/_ref: the reference\'s sources, -O3 -march=x86-64-v3 (the reference\'s -march=native spelt portably), scalar '
                                  'OpenCV primitives; LBA: oracle port of g2o, -O3 -march=x86-64-v3 -ffp-contract=off',
                         'cv2_orb_simd_ms_per_frame_1thread': cv2ms,
                         'note': 'OpenCV\'s own SIMD ORB (cv2.ORB_create(1000,1.2,8).detectAndCompute, different keypoint selection) on one thread of this '
                                 'box next to the scalar extract_ms_per_frame above: the CPU arm is about that factor slower than a SIMD OpenCV build would be'},
        'e2e': {'value': fps, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(index):
    """Run this process on the CPUs the GPU is attached to (sysfs local_cpulist), so that pinned host memory is NUMA-local."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)
        bus = '%04x:%02x:%02x.0' % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        cpus = set()
        for tok in open('/sys/bus/pci/devices/%s/local_cpulist' % bus).read().strip().split(','):
            a, _, b = tok.partition('-')
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return '%s: %d cpus' % (bus, len(cpus))
    except (OSError, ValueError, AttributeError):
        pass
    return None


class ParityError(SystemExit):
    pass


def check_frames_against_oracle(tag, frames, kps, desc, n, match, nmatch, last, poses, sf, cam, idx):
    """The buffers a TIMED loop wrote (slab rows `idx`) against the CPU oracle: keypoints and descriptors bit for bit, match arrays equal."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import oracle_lib as O
    oe = O.OracleExtractor(NFEAT, 1.2, 8, 20, 7)
    for b in idx:
        _, okps, odesc = oe(frames[b], (0, 1000))
        k = int(n[b])
        if k != len(okps) or kps[b, :k].tobytes() != okps.tobytes() or not np.array_equal(desc[b, :k], odesc):
            raise ParityError('PARITY FAILURE (%s): extraction of stream %d differs from the oracle' % (tag, b))
        m = int(last['nM'][b])
        L = dict(valid=last['valid'][b, :m], xyz=last['xyz'][b, :m], octave=last['octave'][b, :m], angle=last['angle'][b, :m],
                 hasObs=last['hasObs'][b, :m], descriptors=last['mpDesc'][b, :m])
        om = np.full(k, -1, np.int32); oc = np.zeros(k, np.uint8)
        on = O.search_last_frame(okps, odesc, (0.0, 0.0, float(W), float(H)), sf, poses[b], cam, L, TH_PROJ, True, om, oc)
        if on != int(nmatch[b]) or not np.array_equal(match[b, :k], om):
            raise ParityError('PARITY FAILURE (%s): SearchByProjection of stream %d differs from the oracle' % (tag, b))
    return len(idx)


def check_lba_against_oracle(tag, prob, out):
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import oracle_lib as O
    ref = O.lba_solve(prob)
    d = np.abs(O.lba_residuals(prob, ref['poses'], ref['points']) - O.lba_residuals(prob, out['poses'], out['points'])).max()
    if out['iters'] != ref['iters'] or out['trials'] != int(ref['stats'][3]) or not d < TOL_PX:
        raise ParityError('PARITY FAILURE (%s): LBA differs from the oracle (iterations %s vs %s, residual diff %.3g px)' % (tag, out['iters'], ref['iters'], d))
    return float(d)


DUMP_STREAMS, DUMP_LBAS = 32, 8    # --dump-outputs sample: a few MB whatever --batch is (the bound is 64 MB)


def dump_outputs(out_dir, gb, slabs, match, claimed, nmatch, lba_out):
    """Writes what the device-resident loop computed in its last timed round as out_dir/<name>.npy (float32 / float64): for a fixed,
    seeded sample of the streams, the keypoint rows (x, y, size, angle, response, octave, class_id), descriptors, mono counts, match and
    claimed arrays of SearchByProjection; for a seeded sample of the bundle adjustments, poses, points, per-edge chi2 / depth flags and
    (iterations, LM trials, lambda, initial chi2, final chi2).  Rows are concatenated over the sampled streams / problems in index order."""
    import numpy as np
    B, P = gb[-1][1], len(lba_out)
    rng = np.random.default_rng(0)
    streams = np.sort(rng.choice(B, min(B, DUMP_STREAMS), replace=False))
    probs = np.sort(rng.choice(P, min(P, DUMP_LBAS), replace=False))
    cols = {k: [] for k in ('keypoints', 'descriptors', 'match', 'claimed')}
    n_kp, mono, n_match = [], [], []
    for b in streams:
        g = next(g for g, (b0, b1) in enumerate(gb) if b0 <= b < b1)
        i = int(b - gb[g][0])
        k = int(slabs[g].n[i])
        kp = slabs[g].kps[i, :k].cpu().numpy()
        cols['keypoints'].append(np.concatenate([kp[:, :5], kp.view(np.int32)[:, 5:].astype(np.float32)], 1))
        cols['descriptors'].append(slabs[g].desc[i, :k].cpu().numpy().astype(np.float32))
        cols['match'].append(match[g][i, :k].cpu().numpy().astype(np.float32))
        cols['claimed'].append(claimed[g][i, :k].cpu().numpy().astype(np.float32))
        n_kp.append(k); mono.append(int(slabs[g].mono[i])); n_match.append(int(nmatch[g][i]))
    out = {'frame_streams': streams.astype(np.float64), 'frame_n_keypoints': np.array(n_kp, np.float64), 'frame_mono': np.array(mono, np.float64),
           'frame_n_matches': np.array(n_match, np.float64)}
    out.update({'frame_' + k: np.concatenate(v) for k, v in cols.items()})
    lba = [lba_out[p] for p in probs]
    out['lba_problems'] = probs.astype(np.float64)
    for k in ('poses', 'points', 'chi2'):
        out['lba_' + k] = np.concatenate([o[k] for o in lba]).astype(np.float64)
    out['lba_depth_pos'] = np.concatenate([o['depth_pos'] for o in lba]).astype(np.float32)
    out['lba_stats'] = np.array([[o['iters'], o['trials'], o['lambda_'], o['initial_chi2'], o['final_chi2']] for o in lba], np.float64)
    total = sum(v.nbytes for v in out.values())
    if total > 64 << 20:
        raise SystemExit('--dump-outputs: %d bytes exceed 64 MB' % total)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + '.npy'), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=240, help='streams (frames per round) per GPU; a multiple of %d' % KF_INTERVAL)
    ap.add_argument('--rounds', type=int, default=18, help='rounds (frames per stream) per step: sizes the timed region (20 steps ~ 2 s)')
    ap.add_argument('--lba-rounds', type=int, default=3, help='the keyframes of this many rounds are bundle-adjusted by one persistent-kernel launch')
    ap.add_argument('--lba-concurrent', action='store_true', help='let the LBA kernel compete with the frame kernels for SMs instead of running between rounds')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the BASELINE configs[0] / configs[2] latency lines')
    ap.add_argument('--dev-groups', type=int, default=2, help='stream groups (own handles + CUDA stream) in the device-resident measurement')
    ap.add_argument('--e2e-groups', type=int, default=3, help='stream groups (host threads with their own handles) in flight in the e2e measurement')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the device-resident loop computed in its last timed round (a seeded sample of '
                    'the streams and bundle adjustments) as DIR/<name>.npy, for comparing two builds output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)

    import numpy as np
    import torch
    import orb_slam3_modified_b200 as orb
    from orb_slam3_modified_b200 import sharding, synth

    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (there is no CPU path in the product)')
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)     # pinned buffers (ours and the library's) land on the GPU's socket: ~53 vs ~20 GB/s over PCIe
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    B, R = args.batch, args.rounds
    if B % KF_INTERVAL:
        raise SystemExit('--batch must be a multiple of %d (exactly one LBA per %d frames)' % (KF_INTERVAL, KF_INTERVAL))
    NLBA = B // KF_INTERVAL
    LR = max(1, args.lba_rounds)
    if R % LR:
        raise SystemExit('--rounds must be a multiple of --lba-rounds')
    dev = torch.device('cuda', local)
    ex = orb.ORBextractor(NFEAT, 1.2, 8, 20, 7, W, H, B, local)
    cap = ex.max_keypoints
    matcher = orb.ORBmatcher(0.9, True, max_batch=B, max_keypoints=cap, max_mappoints=cap, device=local)
    opt = orb.Optimizer(max_poses=LBA_CFG['n_kf'], max_points=LBA_CFG['n_pts'], max_edges=LBA_CFG['n_pts'] * LBA_CFG['obs_per_pt'],
                        max_batch=NLBA * LR, device=local)
    sf = ex.GetScaleFactors()
    cam = [float(c) for c in synth.camera(W, H)]
    bounds = (0.0, 0.0, float(W), float(H))

    # ---- inputs: two alternating sets (consecutive frames t / t+1 of every stream); round i extracts set i&1 and matches it
    # against the map points of set (i+1)&1.  2 x B x 307 KB (147 MB at B=240) > 126 MB L2, per-round working set > 1 GB.
    host_sets = [torch.from_numpy(make_frames(B, k, rank)).pin_memory() for k in range(2)]
    dev_sets = [h.to(dev) for h in host_sets]
    poses_h = [np.stack([stream_pose(s, k, rank) for s in range(B)]) for k in range(2)]
    # untimed set-up: features of both sets -> last-frame map points (the map state the tracker would already hold)
    last_h, last_d = [], []
    for k in range(2):
        monos, kl, dl = ex.extract_batch(host_sets[k].numpy(), (0, 1000))
        slabs = last_frame_slabs(kl, dl, k, cap, rank)
        slabs = {n: torch.from_numpy(v).pin_memory().numpy() for n, v in slabs.items()}     # the tracker's map state: pinned, like every per-round host input
        last_h.append(slabs)
        last_d.append({n: torch.from_numpy(v).to(dev) for n, v in slabs.items()})
    d_sf = torch.from_numpy(sf).to(dev)
    d_Tcw = [torch.from_numpy(p).to(dev) for p in poses_h]
    probs = lba_problems(NLBA * LR, rank)   # the keyframes of LR rounds: one LocalBundleAdjustment each, solved by ONE kernel launch
    opt.upload(probs)                      # flattened graphs resident in HBM for the `value` measurement
    stream = torch.cuda.current_stream()
    lba_stream = torch.cuda.Stream(device=dev)      # LocalMapping runs beside Tracking in the reference (src/System.cc:197)
    ev_fork, ev_join = torch.cuda.Event(), torch.cuda.Event()

    # The B streams are served as DG groups, each with its own extractor / matcher handles on its own CUDA stream: the latency-bound
    # kernels of one group (quadtree) overlap the throughput-bound ones of another (FAST, blur).  Every group writes packed slabs
    # (two sets, alternating per round) so that the multi-GPU exchange is one collective per group and round with no rank-wide join.
    DG = max(1, min(args.dev_groups, B))
    gb = [(g * B // DG, (g + 1) * B // DG) for g in range(DG)]
    g_ex = [orb.ORBextractor(NFEAT, 1.2, 8, 20, 7, W, H, b1 - b0, local) for b0, b1 in gb]
    g_mt = [orb.ORBmatcher(0.9, True, max_batch=b1 - b0, max_keypoints=cap, max_mappoints=cap, device=local) for b0, b1 in gb]
    g_st = [torch.cuda.Stream(device=dev) for _ in gb]
    g_ev = [torch.cuda.Event() for _ in gb]
    g_slab = [[sharding.PackedSlab(b1 - b0, cap, dev) for _ in range(2)] for b0, b1 in gb]
    g_match = [torch.full((b1 - b0, cap), -1, dtype=torch.int32, device=dev) for b0, b1 in gb]
    g_claimed = [torch.zeros((b1 - b0, cap), dtype=torch.uint8, device=dev) for b0, b1 in gb]
    g_nmatch = [torch.zeros(b1 - b0, dtype=torch.int32, device=dev) for b0, b1 in gb]
    gather = sharding.GroupSlabGather(dist, world, g_slab) if world > 1 and os.environ.get('BENCH_DIAG', '') != 'nogather' else None

    EXCL = not args.lba_concurrent
    ev_lba = torch.cuda.Event()
    DIAG = os.environ.get('BENCH_DIAG', '')     # diagnosis only ('nolba' / 'noframes': half of the work skipped -> the line is marked invalid)

    def match_args(i, S, b0, b1):
        cur, lst = i & 1, (i + 1) & 1
        L = last_d[lst]
        return dict(batch=b1 - b0, kcap=cap, mcap=cap, nlevels=8, kps=S.kps, desc=S.desc, nK=S.n, scaleFactors=d_sf,
                    nM=L['nM'][b0:b1], valid=L['valid'][b0:b1], xyz=L['xyz'][b0:b1], octave=L['octave'][b0:b1], angle=L['angle'][b0:b1],
                    hasObs=L['hasObs'][b0:b1], mpDesc=L['mpDesc'][b0:b1], Tcw7=d_Tcw[cur][b0:b1], bounds=bounds, cam=cam, reset=1)

    def round_device(i):
        # LocalMapping is asynchronous to Tracking in the reference (own thread, src/System.cc:197): the bundle adjustments are
        # enqueued on their own stream and only joined at the end of the timed region (all of them finish inside it).  The B / 10
        # keyframes of each of LR consecutive rounds are solved by one persistent-kernel launch (more problems per launch = smaller
        # clusters = no CTA idling through another CTA's LDL^T; 72 problems x 2 CTAs is 27 % faster per problem than 24 x 5).
        d = i & 1
        for g, (b0, b1) in enumerate(gb if DIAG != 'noframes' else []):
            st = g_st[g]
            S = g_slab[g][d]
            if gather:
                with torch.cuda.stream(st):
                    gather.wait(g, d)                                # the gather of round i-2 read this slab set
            g_ex[g].extract_batch_device(dev_sets[d][b0:b1], S.kps, S.desc, S.n, S.mono, (0, 1000), st.cuda_stream)
            g_mt[g].search_last_frame_batch_device(match_args(i, S, b0, b1), TH_PROJ, g_match[g], g_claimed[g], g_nmatch[g], st.cuda_stream)
            if gather:   # shared-map exchange (SURVEY.md 8e): this group's packed slab, right behind its kernels, on its own communicator
                with torch.cuda.stream(st):
                    gather.gather(g, d)
        if i % LR == LR - 1 and DIAG != 'nolba':
            # The persistent LBA kernel (512 threads x 128 registers per CTA = a whole SM's register file) does not share SMs: run
            # beside the frame kernels it stretches both (measured 6.5 ms per round against 3.4 + 2.35 one after the other), so it gets
            # the GPU to itself between two rounds -- the mapping stream waits for the groups, and the groups for the mapping stream.
            if EXCL:
                for g, st in enumerate(g_st):
                    if gather:     # the collectives in flight finish first: an NCCL kernel starved of SMs by the LBA kernel stalls its peer rank too
                        with torch.cuda.stream(st):
                            gather.wait(g, 0)
                            gather.wait(g, 1)
                    g_ev[g].record(st)
                    lba_stream.wait_event(g_ev[g])
            opt.run_device(lba_stream.cuda_stream)
            if EXCL:
                ev_lba.record(lba_stream)
                for st in g_st:
                    st.wait_event(ev_lba)

    def fork_groups():
        ev_fork.record(stream)
        for st in g_st:
            st.wait_event(ev_fork)
        lba_stream.wait_event(ev_fork)

    def join_all():
        for g, st in enumerate(g_st):
            if gather:
                with torch.cuda.stream(st):
                    for d in range(2):
                        gather.wait(g, d)
            g_ev[g].record(st)
            stream.wait_event(g_ev[g])
        ev_join.record(lba_stream)
        stream.wait_event(ev_join)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (`value`) ----------------
    clocks = ClockSampler(local) if rank == 0 else None      # started before the warm-up: nvidia-smi needs ~0.2 s to deliver its first row
    fork_groups()
    for i in range(args.warmup * R):
        round_device(i)
    join_all()
    barrier()
    if clocks:
        clocks.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fork_groups()
    n_rounds = args.steps * R
    for i in range(n_rounds):
        round_device(i)
    join_all()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = (sum(e.last_launch_count() for e in g_ex) + sum(m_.last_launch_count() for m_ in g_mt)) * n_rounds + n_rounds // LR
    ms = sharding.max_over_ranks(dist, ms, dev)
    clk = clocks.stop() if clocks else None
    value = world * B * n_rounds / (ms * 1e-3)

    if DIAG:
        if rank == 0:
            print(json.dumps({'INVALID_diagnostic_run': DIAG, 'ms_per_round': ms / n_rounds}))
        if world > 1:
            dist.destroy_process_group()
        return
    # ---------------- parity gate 1: what the timed loop left in the slabs, against the CPU oracle ----------------
    i_last = n_rounds - 1
    d_last = i_last & 1
    n_checked = 0
    for g, (b0, b1) in enumerate(gb):
        S = g_slab[g][d_last]
        nb = b1 - b0
        kps_np = S.kps.cpu().numpy().view(np.uint8).reshape(nb, cap, 28).view(orb.KP_DTYPE).reshape(nb, cap)
        L = {k: v[b0:b1] for k, v in last_h[(i_last + 1) & 1].items()}
        n_checked += check_frames_against_oracle('device-resident loop', host_sets[d_last].numpy()[b0:b1], kps_np, S.desc.cpu().numpy(), S.n.cpu().numpy(),
                                                 g_match[g].cpu().numpy(), g_nmatch[g].cpu().numpy(), L, poses_h[d_last][b0:b1], sf, cam, [0, nb - 1])
    lba_out = opt.download()
    lba_diff = check_lba_against_oracle('device-resident loop', probs[0], lba_out[0])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gb, [g_slab[g][d_last] for g in range(DG)], g_match, g_claimed, g_nmatch, lba_out)
    mean_trials = float(np.mean([o['trials'] for o in lba_out]))
    mean_kp = float(np.mean([float(g_slab[g][d_last].n.float().mean().item()) for g in range(DG)]))
    mean_matches = float(np.mean([float(g_nmatch[g].float().mean().item()) for g in range(DG)]))
    parity = {'device_loop': {'frames_checked': n_checked, 'lba_checked': 1, 'lba_max_residual_diff_px': lba_diff, 'ok': True}}

    # ---------------- per-stage split (events on the launching stream) + rooflines ----------------
    stage = {}
    if rank == 0:
        d_kps = torch.zeros((B, cap, 7), dtype=torch.float32, device=dev)
        d_desc = torch.zeros((B, cap, 32), dtype=torch.uint8, device=dev)
        d_n = torch.zeros(B, dtype=torch.int32, device=dev); d_mono = torch.zeros(B, dtype=torch.int32, device=dev)
        d_match = torch.full((B, cap), -1, dtype=torch.int32, device=dev); d_claimed = torch.zeros((B, cap), dtype=torch.uint8, device=dev)
        d_nmatch = torch.zeros(B, dtype=torch.int32, device=dev)

        class _S:
            kps, desc, n = d_kps, d_desc, d_n
        ex.set_profiling(True)
        acc = {}
        reps = 3
        for i in range(reps):
            ex.extract_batch_device(dev_sets[i & 1], d_kps, d_desc, d_n, d_mono, (0, 1000), stream.cuda_stream)
            for k, v in ex.stage_ms().items():
                acc[k] = acc.get(k, 0.0) + v / reps
        ex.set_profiling(False)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for i in range(reps):
            matcher.search_last_frame_batch_device(match_args(i, _S, 0, B), TH_PROJ, d_match, d_claimed, d_nmatch, stream.cuda_stream)
        a1.record(stream)
        b0_, b1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0_.record(stream)
        for i in range(reps):
            opt.run_device(stream.cuda_stream)
        b1_.record(stream)
        torch.cuda.synchronize()
        stage = dict(acc)
        stage['match_frame_kernel'] = a0.elapsed_time(a1) / reps
        lba_launch_ms = b0_.elapsed_time(b1_) / reps
        stage['lba_cluster_kernel'] = lba_launch_ms / LR      # per round: one launch serves LR rounds
        del d_kps, d_desc, d_match, d_claimed
    torch.cuda.synchronize()

    # ---------------- end to end through the host C-ABI (`e2e`) ----------------
    # Host buffers in, host buffers out, every round.  The B streams are served as G groups, each by its own host thread with its own
    # extractor / matcher handles (the batch calls are synchronous, so two groups in flight let one group's PCIe copies overlap the
    # other's kernels), and the local maps' bundle adjustments by G mapping threads (the LocalMapping thread of the reference,
    # src/System.cc:197), one round behind the frames.  The matcher reads the current frame from the extractor handle's resident slabs
    # (orbx_resident_slabs): the keypoints go to the host once and never back.
    e2e, e2e_steps, h2d, d2h, e2e_err = None, 0, 0, 0, None
    if not args.no_e2e:
        try:
            from concurrent.futures import ThreadPoolExecutor
            G = max(1, min(args.e2e_groups, B))
            pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
            kps_h = pin((B, cap, 7), torch.float32).view(np.uint8).reshape(B, cap, 28).view(orb.KP_DTYPE).reshape(B, cap)
            desc_h = pin((B, cap, 32), torch.uint8)
            nK_h, mono_h, nmatch_h = pin((B,), torch.int32), pin((B,), torch.int32), pin((B,), torch.int32)
            match_h, claimed_h = pin((B, cap), torch.int32), pin((B, cap), torch.uint8)
            hb = [(g * B // G, (g + 1) * B // G) for g in range(G)]
            exs = [orb.ORBextractor(NFEAT, 1.2, 8, 20, 7, W, H, b1 - b0, local) for b0, b1 in hb]
            mts = [orb.ORBmatcher(0.9, True, max_batch=b1 - b0, max_keypoints=cap, max_mappoints=cap, device=local) for b0, b1 in hb]
            pool = ThreadPoolExecutor(G + 2)

            def frames_job(g, i):
                cur, lst = i & 1, (i + 1) & 1
                b0, b1 = hb[g]
                exs[g].extract_batch_slabs(host_sets[cur].numpy()[b0:b1], kps_h[b0:b1], desc_h[b0:b1], nK_h[b0:b1], mono_h[b0:b1], (0, 1000))
                L = last_h[lst]
                d = dict(batch=b1 - b0, kcap=cap, mcap=cap, nlevels=8, scaleFactors=sf, nM=L['nM'][b0:b1], valid=L['valid'][b0:b1], xyz=L['xyz'][b0:b1],
                         octave=L['octave'][b0:b1], angle=L['angle'][b0:b1], hasObs=L['hasObs'][b0:b1], mpDesc=L['mpDesc'][b0:b1],
                         Tcw7=poses_h[cur][b0:b1], bounds=bounds, cam=cam, reset=1)
                mts[g].search_last_frame_batch(d, TH_PROJ, match_h[b0:b1], claimed_h[b0:b1], nmatch_h[b0:b1], resident=exs[g].resident_slabs())
                return int(nK_h[b0:b1].sum())

            # Mapping side: the graphs of a batch are uploaded and the results of the previous one downloaded by a mapping thread WHILE the frames
            # of the following rounds run; two handles alternate.  Here the persistent kernel shares the GPU with the frame kernels: the loop is
            # bound by the sum of the two kernel loads (about 5.6 ms of GPU time per round) whichever way they are interleaved -- gating the frame
            # calls while a bundle-adjustment launch runs, splitting the launch into halves that own half of the SMs each, and a high-priority
            # mapping stream were all measured and none was faster (tools/run_e2e_var.sh, DESIGN.md 6).
            opt_pair = [opt, orb.Optimizer(max_poses=LBA_CFG['n_kf'], max_points=LBA_CFG['n_pts'], max_edges=LBA_CFG['n_pts'] * LBA_CFG['obs_per_pt'],
                                           max_batch=NLBA * LR, device=local)]
            up = [None, None]       # upload future per handle
            down = [None, None]     # download future per handle
            # Streams are independent SLAM instances: every group's host thread free-runs through its rounds (no join between rounds, so one
            # group's PCIe copies always overlap another group's kernels); the mapping thread waits only for the keyframes it optimises.
            import threading
            # A host thread coming back from a C-ABI call must re-take the interpreter lock; with CPython's default 5 ms switch interval it can
            # wait that long behind another thread's Python glue (GPU idle meanwhile).  Hand the lock over promptly instead.
            sys.setswitchinterval(float(os.environ.get('BENCH_SWITCH_INTERVAL', '5e-5')))
            cv = threading.Condition()
            done = [0] * G                                          # rounds finished per group (absolute round counter)
            state = {'outs': None, 'nbatch': 0, 'err': None}

            def group_loop(g, r0, r1):
                try:
                    for i in range(r0, r1):
                        frames_job(g, i)
                        with cv:
                            done[g] = i + 1
                            cv.notify_all()
                except BaseException as exc:                       # surfaced by the main thread
                    with cv:
                        state['err'] = exc
                        done[g] = 1 << 60
                        cv.notify_all()

            def mapping_loop(r0, r1):
                try:
                    for i in range(r0, r1):
                        if i % LR == 0:                             # graphs of this batch's keyframes: uploaded while their frames run
                            k = state['nbatch'] & 1
                            if down[k] is not None:
                                state['outs'] = down[k].result()    # the handle's previous results are out before it is reused
                                down[k] = None
                            up[k] = pool.submit(opt_pair[k].upload, probs)
                        if i % LR == LR - 1:
                            with cv:
                                cv.wait_for(lambda: min(done) >= i + 1)     # the batch's keyframes exist
                            k = state['nbatch'] & 1
                            up[k].result()
                            opt_pair[k].run_device(lba_stream.cuda_stream)
                            down[k] = pool.submit(opt_pair[k].download)     # waits for the kernel on the device (event inside the library)
                            state['nbatch'] += 1
                except BaseException as exc:
                    with cv:
                        state['err'] = exc

            def run_rounds(r0, r1):
                ediag = os.environ.get('BENCH_E2E_DIAG', '')          # diagnosis only: 'nolba' / 'noframes' (half of the work skipped -> line marked invalid)
                th = [threading.Thread(target=group_loop, args=(g, r0, r1)) for g in range(G)] if ediag != 'noframes' else []
                if ediag == 'noframes':
                    with cv:
                        for g in range(G):
                            done[g] = 1 << 60
                if ediag != 'nolba':
                    th.append(threading.Thread(target=mapping_loop, args=(r0, r1)))
                for t in th:
                    t.start()
                for t in th:
                    t.join()
                if state['err'] is not None:
                    raise state['err']

            run_rounds(0, 2 * LR)
            torch.cuda.synchronize()
            barrier()
            e2e_steps = args.steps
            nr = e2e_steps * R
            t0 = time.perf_counter()
            run_rounds(2 * LR, 2 * LR + nr)                         # 2 LR is even: the input sets alternate as in the warm-up
            torch.cuda.synchronize()
            # every LR rounds of the timed region uploaded, solved and started to download one batch of bundle adjustments; the last
            # download may complete just outside the timed region (its kernel ran inside)
            dt = time.perf_counter() - t0
            outs = state['outs']
            tail = [d.result() for d in down if d is not None]
            tail = tail[-1] if tail else None
            dt = sharding.max_over_ranks(dist, dt, dev)
            e2e = world * B * nr / dt
            if os.environ.get('BENCH_E2E_DIAG'):
                if rank == 0:
                    print(json.dumps({'INVALID_diagnostic_run': 'e2e ' + os.environ['BENCH_E2E_DIAG'], 'groups': G, 'e2e_frames_per_s_equiv': e2e, 'ms_per_round': 1e3 * dt / nr}))
                os._exit(0)
            # parity gate 2: the host buffers of the last timed round
            cur = (nr - 1) & 1
            L = last_h[(nr) & 1]
            nchk = check_frames_against_oracle('e2e loop', host_sets[cur].numpy(), kps_h, desc_h, nK_h, match_h, nmatch_h, L, poses_h[cur], sf, cam,
                                               [0, B // 2 - 1, B // 2, B - 1])
            dl = check_lba_against_oracle('e2e loop', probs[0], (tail or outs)[0])
            parity['e2e_loop'] = {'frames_checked': nchk, 'lba_checked': 1, 'lba_max_residual_diff_px': dl, 'ok': True}
            p0 = probs[0]
            lba_h2d = NLBA * (p0['poses'].nbytes + p0['points'].nbytes + p0['obs'].nbytes + 3 * 4 * len(p0['edge_point']) + p0['cam'].nbytes)
            lba_d2h = NLBA * (p0['poses'].nbytes + p0['points'].nbytes + 9 * len(p0['edge_point']))
            per_round_h2d = B * W * H + sum(v.nbytes for v in last_h[0].values()) + B * 28 + lba_h2d      # frames, last-frame map points, poses, graphs
            per_round_d2h = B * cap * 60 + 12 * B + B * cap * 5 + lba_d2h                                   # slabs, counts, match + claimed, LBA results
            h2d, d2h = per_round_h2d * R, per_round_d2h * R
            pool.shutdown()
        except ParityError:
            raise
        except Exception as exc:     # the device-resident result is still reported (single GPU); with several ranks a failure must stay fatal
            if world > 1:
                raise
            e2e, e2e_err = None, repr(exc)[:300]

    if rank == 0:
        peak, how = _peaks()
        traffic_tab = {}
        for name in ('r2_traffic.json', 'r1_traffic.json'):
            try:
                traffic_tab = json.load(open(os.path.join(ROOT, 'profiles', name)))
                break
            except (OSError, ValueError):
                pass

        def alg_of(k):
            if k == 'lba_cluster_kernel':
                return ALG_BYTES_LBA_PER_TRIAL * mean_trials * NLBA, 'LBA, per round: %.1f LM trials x 13.6 MB x %d problems (one launch solves %d, %.3f ms)' % (mean_trials, NLBA, NLBA * LR, lba_launch_ms)
            if k.startswith('match'):
                return ALG_BYTES_MATCH * B, '552,000 B/frame x %d frames' % B
            return ALG[k] * B, '%d B/frame x %d frames' % (ALG[k], B)

        def traffic_of(k):
            t = traffic_tab.get(k)
            if not t:     # ncu DRAM bytes per launch, scaled from the launch size of the capture to this run's
                return None
            return t['bytes'] * ((NLBA / float(t.get('problems', 25))) if k == 'lba_cluster_kernel' else B / float(t.get('frames', 256)))

        per_kernel = {}
        for k in stage:
            ab, _ = alg_of(k)
            per_kernel[k] = {'ms': stage[k], 'achieved': ab / (stage[k] * 1e-3) / 1e9, 'frac': ab / (stage[k] * 1e-3) / 1e9 / peak, 'traffic': traffic_of(k)}
        top = max(stage, key=stage.get)
        alg_bytes, per = alg_of(top)
        ach = alg_bytes / (stage[top] * 1e-3) / 1e9
        em_ms = sum(v for k, v in stage.items() if k != 'lba_cluster_kernel')
        em_ach = (ALG_BYTES_EXTRACT + ALG_BYTES_MATCH) * B / (em_ms * 1e-3) / 1e9
        out = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'u8 (extract/match), f64 (LBA)', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'stages': STAGES, 'streams_per_gpu': B, 'rounds_per_step': R, 'frames_per_gpu_per_step': B * R,
                       'lba_per_gpu_per_step': NLBA * R, 'lba_problems_per_launch': NLBA * LR, 'timed_region_s': ms * 1e-3,
                       'l2': 'inputs alternate between two %d-frame sets (2 x %.0f MB) > 126 MB L2; per-round working set > 1 GB' % (B, B * W * H / 1e6),
                       'mean_keypoints_per_frame': mean_kp, 'mean_matches_per_frame': mean_matches, 'lba_cluster_size': opt.last_cluster_size(),
                       'lba_mean_trials': mean_trials, 'host_numa_binding': numa, 'device_stream_groups': DG,
                       'multi_gpu_exchange': None if world == 1 else 'one NCCL all-gather of the packed slab per stream group and round (%d B per rank), own communicator per group, slab sets double-buffered' % sum(s[0].nbytes for s in g_slab)},
            'clocks': clk, 'gpu_launches': launches, 'parity': parity,
            'stage_ms_per_round': stage,
            'roofline': {'bound': 'hbm', 'kernel': top, 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': traffic_of(top),
                         'traffic_source': (traffic_tab.get(top) or {}).get('source'),
                         'peak_source': how, 'algorithmic_bytes_per_launch': alg_bytes, 'per': per, 'launch_ms': stage[top],
                         'note': 'FP64 LM solver bound by L1 look-ups of per-lane gathers and by cluster barriers, not by DRAM (DESIGN.md 5); frac is against the HBM copy peak as the contract asks',
                         'per_kernel': per_kernel,
                         'whole_step_frac': (ALG_BYTES_EXTRACT + ALG_BYTES_MATCH + ALG_BYTES_LBA_PER_TRIAL * mean_trials / KF_INTERVAL) * (value / world) / 1e9 / peak},
            'roofline_extract_match': {'bound': 'hbm', 'achieved': em_ach, 'peak': peak, 'unit': 'GB/s', 'frac': em_ach / peak,
                                       'per': '(5,742,474 + 552,000) B/frame x %d frames / %.3f ms (sum of the extract + match kernels of one round, measured alone)' % (B, em_ms)},
        }
        if e2e_err:
            out['e2e'], out['e2e_error'] = None, e2e_err
        if e2e is not None:
            out['e2e'] = {'value': e2e, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h), 'steps': e2e_steps,
                          'stream_groups': max(1, min(args.e2e_groups, B))}
        if world == 1 and not args.no_extra:
            try:
                sys.path.insert(0, os.path.join(ROOT, 'tools'))
                import extra_configs
                out['configs'] = extra_configs.measure(orb, synth, local)
            except Exception as exc:
                out['configs'] = {'error': repr(exc)[:300]}
        if world == 1 and not args.no_cpu_baseline:
            try:
                kind = _cpu_impl()[3]
                fps1, dt1, sample, split, _ = run_cpu_arm(1, 1, 1, 24 * KF_INTERVAL)     # 240 frames + 24 LBAs: ~8 s of single-thread CPU work
                try:      # the oracle port of Optimizer::LocalInertialBA on the map extra_configs times on the GPU (single thread, 3 runs)
                    import numpy as np
                    import oracle_lib as O
                    from orb_slam3_modified_b200 import synth
                    lpr = synth.local_inertial_ba_problem(n_opt=10, n_cov_fixed=6, n_pts=2500, seed=12)
                    lP = O.liba_preints(lpr)
                    ts = []
                    for _ in range(3):
                        t0 = time.perf_counter(); O.local_inertial_ba(lpr, lP); ts.append(time.perf_counter() - t0)
                    split['local_inertial_ba_ms_per_map'] = 1e3 * float(np.median(ts))
                except Exception as exc:
                    split['local_inertial_ba_error'] = repr(exc)[:120]
                out['cpu_baseline'] = {'value': fps1, 'unit': UNIT, 'cores': 1, 'kind': 'reference' if kind['extract'] == 'reference' else 'port',
                                       'kind_per_stage': kind, 'host': cpu_info(), 'sample': sample + ' (%.1f s)' % dt1, 'split': split}
            except Exception as exc:
                out['cpu_baseline'] = None
                out['cpu_baseline_error'] = repr(exc)[:300]
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()

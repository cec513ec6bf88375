#!/usr/bin/env python
"""bench.py -- audio-hours/sec of the inaSpeechSegmenter hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One step = one pass of the whole hot path (K1 log-mel/energy -> energy Viterbi
-> smn CNN -> Viterbi -> gender CNN -> Viterbi -> segment list on the host) over
one batch of synthetic 16 kHz mono int16 audio: BASELINE.json configs[1]
("smn+gender on 10 h synthetic, 1xB200").  With N > 1 ranks (torchrun) ONE recording
of N x 10 h is time-sharded over the ranks (inaspeechsegmenter_b200/shard.py:
34-frame halo, NCCL all-gathers of loge and of the CNN posteriors, BASELINE
configs[4]) => weak scaling (per-GPU work fixed); the timed region is bracketed
by barrier + synchronize and the max over ranks is reported.

The same JSON line carries, all measured in this run and outside the timed region:
  parity        GPU result vs the CPU oracle at benchmark scale: per-patch softmax and
                Viterbi labels of both CNNs on randomly placed 60 s windows of the 10 h
                recording, log-mel rows of the same windows, the whole-file energy track
                (N = 1); the sharded segment list vs a single-GPU run of the whole
                recording on rank 0 (N > 1)
  roofline      the dominant kernel (conv/dense layer with most FLOPs), CUDA events per launch
  configs2      BASELINE configs[2]: sm+gender on 100 h, with roofline_k1 (feature kernel, HBM)
  configs3      BASELINE configs[3]: VBx features + ResNet101 x-vectors, with roofline_k5 (tensor)
  cpu_baseline  the reference's CPU path (oracle port) on all host cores, process-parallel

`--impl reference` times the reference's CPU path (numpy front-end + torch-CPU CNN
restatement + C Viterbi: TensorFlow and the .hdf5 networks are not installable here) the way the
reference scales out (one worker process per file chunk, scripts/ina_speech_segmenter_pyro_client.py:64-74):
host_cores/16 workers x 16 threads on disjoint 10-minute chunks.

`--dump-outputs DIR` writes the segment list the last timed step returned (b200 arm, rank 0) to
DIR/segments.npy: float64 [n, 3], one row (index into SEGMENT_LABELS, start s, stop s) per segment.
The synthetic input is seeded, so two builds run with the same arguments can be compared row for row.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'audio-hours/sec segmented (16 kHz mono)'
UNIT = 'audio-hours/s'
SR = 16000
SEGMENT_LABELS = ('noEnergy', 'energy', 'speech', 'music', 'noise', 'female', 'male')


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError('must be at least 1, got %d' % v)
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=positive_int, default=3, help='timed steps')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--hours', type=float, default=10.0, help='audio hours per GPU per step')
    ap.add_argument('--fft', default='fp64', choices=['fp64', 'fp32'])
    ap.add_argument('--cpu-chunk-sec', type=float, default=None,
                    help='seconds of audio per CPU worker and step (default 600 for --impl reference, 120 for the cpu_baseline leg)')
    ap.add_argument('--cpu-workers', type=int, default=0, help='CPU worker processes (0 = host_cores / 16)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip parity / configs2 / configs3 (profiling runs)')
    ap.add_argument('--parity-windows', type=int, default=10)
    ap.add_argument('--k1-hours', type=float, default=100.0, help='BASELINE configs[2] size')
    ap.add_argument('--vbx-hours', type=float, default=50.0, help='BASELINE configs[3] size (1 h files)')
    ap.add_argument('--vbx-max-sec', type=float, default=60.0, help='stop the VBx leg after this many seconds (bounded sample)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the segment list of the last timed step to DIR/segments.npy')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    return args


def dump_outputs(out_dir, segs):
    """[(label, start s, stop s)] -> DIR/segments.npy, float64 [n, 3] (label as its index in SEGMENT_LABELS)."""
    rows = np.array([(SEGMENT_LABELS.index(lab), a, b) for lab, a, b in segs], dtype=np.float64).reshape(-1, 3)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'segments.npy'), rows)


# ----------------------------------------------------------------------------- synthetic audio
def synth_block_torch(torch, block, seconds, device):
    """One block of the SURVEY 8(d) generator on the device: spans of exact
    silence, white noise, a harmonic 'speech-like' source with 4 Hz AM and
    multi-tone 'music' (5-30 s, plus a few spans < 0.68 s), quantised to int16."""
    g = torch.Generator(device='cpu')
    g.manual_seed(20260922 + block)
    n = int(seconds * SR)
    out = torch.zeros(n, dtype=torch.float32, device=device)
    gd = torch.Generator(device=device)
    gd.manual_seed(977 * (20260922 + block) + 1)
    pos = 0
    while pos < n:
        u = torch.rand(8, generator=g)
        dur = int((0.3 + 0.35 * u[0].item()) * SR) if u[1].item() < 0.08 else int((5 + 25 * u[0].item()) * SR)
        kind = int(u[2].item() * 4)
        end = min(n, pos + dur)
        m = end - pos
        t = torch.arange(m, device=device, dtype=torch.float32) / SR
        if kind == 1:
            out[pos:end] = torch.randn(m, generator=gd, device=device) * (1e-3 + 0.3 * u[3].item())
        elif kind == 2:
            f0 = 100 + 150 * u[3].item()
            s = torch.zeros(m, device=device)
            for h in range(1, 12):
                s += torch.sin(2 * np.pi * f0 * h * t + 6.28 * u[4].item() * h) / h
            out[pos:end] = 0.08 * s * (0.6 + 0.4 * torch.sin(2 * np.pi * 4 * t)) + torch.randn(m, generator=gd, device=device) * 2e-3
        elif kind == 3:
            s = torch.zeros(m, device=device)
            for q in range(5):
                s += torch.sin(2 * np.pi * (200 + 2800 * ((u[3].item() * (q + 1) * 0.618) % 1.0)) * t)
            out[pos:end] = 0.05 * s + torch.randn(m, generator=gd, device=device) * 1e-3
        pos = end
    return torch.clamp(torch.round(out * 32768), -32768, 32767).to(torch.int16)


BLOCK_SEC = 600.0


def synth_range(torch, sa, sb, device):
    """Samples [sa, sb) of the (arbitrarily long) synthetic recording made of 10-minute blocks."""
    bl = int(BLOCK_SEC * SR)
    parts = []
    for b in range(sa // bl, (sb - 1) // bl + 1):
        blk = synth_block_torch(torch, b, BLOCK_SEC, device)
        parts.append(blk[max(sa - b * bl, 0):min(sb - b * bl, bl)])
    return torch.cat(parts)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(gpu_index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                       '-lms', '200'], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(',')]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for nme, v in zip(names, c[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(nme)
        self.f.close()
        os.unlink(self.f.name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ----------------------------------------------------------------------------- CPU (reference-port) leg
def cpu_reference_pass(sample_f32, mods, threads, vad_engine='smn'):
    """The reference's CPU path restated (oracle): numpy front-end, numpy patch
    materialisation, torch-CPU CNNs, C Viterbi."""
    import warnings
    from oracle import cnn_oracle, segmenter_oracle as so
    t0 = time.perf_counter()
    mspec, loge, difflen = so.media2feats(sample_f32)
    v = so.DnnSegmenterOracle(cnn_oracle.KerasLikeModel(*mods['vad'], threads=threads), **(so.VAD_SMN if vad_engine == 'smn' else so.VAD_SM))
    g = so.DnnSegmenterOracle(cnn_oracle.KerasLikeModel(*mods['gender'], threads=threads), **so.GENDER)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        segs = so.segment_feats(mspec, loge, difflen, 0, v, g)
    return time.perf_counter() - t0, segs


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def make_models(vad_classes=3):
    from inaspeechsegmenter_b200 import models
    return {'vad': models.synthetic_keras_cnn(21, vad_classes, seed=11), 'gender': models.synthetic_keras_cnn(24, 2, seed=13)}


def _cpu_worker(conn, wid, threads, chunk_sec):
    """One worker process of the CPU arm = one 'file server' of the reference's Pyro farm: it owns one chunk
    of the synthetic recording (a file of its own) and segments it with `threads` torch threads."""
    try:
        import torch
        torch.set_num_threads(threads)
        from oracle import viterbi_oracle
        viterbi_oracle.build()
        mods = make_models()
        n = int(chunk_sec * SR)
        s16 = synth_range(torch, wid * n, (wid + 1) * n, 'cpu').numpy()
        sample = s16.astype(np.float32) / np.float32(32768)
        cpu_reference_pass(sample[:SR * 5], mods, threads)               # import / allocator warm-up
        conn.send(('ready', 0.0))
        while True:
            msg = conn.recv()
            if msg == 'stop':
                break
            t, segs = cpu_reference_pass(sample, mods, threads)
            conn.send(('done', t, len(segs)))
    except Exception as e:                                               # surface worker failures in the parent
        conn.send(('error', repr(e)))


class CpuFarm:
    """W worker processes x T threads.  The torch-CPU convolutions of the port stop scaling near 16 threads
    (measured on the GPU box in round 1: 16 threads 0.0086, 128 threads 0.0015 audio-hours/s in ONE process), so
    the host is filled the way the reference does it -- process-level, one chunk (file) per worker."""

    def __init__(self, chunk_sec, workers=0):
        import multiprocessing as mp
        cores = host_cores()
        self.threads = min(16, cores)
        self.workers = workers or max(1, cores // self.threads)
        self.chunk_sec = chunk_sec
        ctx = mp.get_context('spawn')
        self.procs, self.conns = [], []
        for w in range(self.workers):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(b, w, self.threads, chunk_sec), daemon=True)
            p.start()
            self.procs.append(p); self.conns.append(a)
        for c in self.conns:
            m = c.recv()
            if m[0] != 'ready':
                raise RuntimeError('CPU worker failed: %r' % (m,))

    def step(self):
        t0 = time.perf_counter()
        for c in self.conns:
            c.send('go')
        for c in self.conns:
            m = c.recv()
            if m[0] != 'done':
                raise RuntimeError('CPU worker failed: %r' % (m,))
        return time.perf_counter() - t0

    def close(self):
        for c in self.conns:
            try:
                c.send('stop')
            except Exception:
                pass
        for p in self.procs:
            p.join(timeout=10)

    @property
    def audio_hours_per_step(self):
        return self.workers * self.chunk_sec / 3600.0

    def describe(self):
        return ('%d worker processes x %d torch threads (the reference scales out per file, pyro_client.py:64-74), each segmenting its own '
                '%g s chunk of the synthetic recording per step: reference-numpy front-end + torch-CPU restatement of the CNNs + C Viterbi '
                '(TensorFlow absent)' % (self.workers, self.threads, self.chunk_sec))


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    chunk = args.cpu_chunk_sec or 600.0
    farm = CpuFarm(chunk, args.cpu_workers)
    for _ in range(args.warmup):
        pass                                                             # workers warmed themselves up on a 5 s slice (a full extra pass would only add minutes)
    ts = [farm.step() for _ in range(args.steps)]
    farm.close()
    t = float(np.mean(ts))
    val = farm.audio_hours_per_step / t
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': t * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'smn+gender on %g h synthetic 16 kHz mono (bounded sample: %d chunks of %g s per step)' % (args.hours, farm.workers, chunk),
                   'networks': 'synthetic-weight stand-ins (release .hdf5 absent)'},
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': farm.workers * farm.threads, 'kind': 'port', 'host_cores': host_cores(),
                         'sample': farm.describe()},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- parity at benchmark scale
def _rows_of(ranges):
    """ranges [(a, b)] -> (starts, stops, row offset of each range in the concatenated probability matrix)."""
    st = np.array([a for a, _ in ranges], dtype=np.int64)
    sp = np.array([b for _, b in ranges], dtype=np.int64)
    off = np.concatenate(([0], np.cumsum(sp - st)))
    return st, sp, off


def _track(lseg, P, names):
    """Segment list in patch units -> int8 label per patch (index into `names`, -1 elsewhere)."""
    out = np.full(P, -1, dtype=np.int8)
    for lab, a, b in lseg:
        if lab in names:
            out[a:b] = names.index(lab)
    return out


def parity_block(torch, seg, pcm, mods, n_windows, seed=20260923):
    """GPU vs CPU oracle on the benchmark recording (outside the timed region).  Whole file: energy track
    (threshold = np.mean of the float32 loge, segmenter.py:70, + the 2-state Viterbi).  Windows of 60 s
    placed on randomly chosen CNN input segments: log-mel rows, per-patch softmax of both CNNs (every evaluated
    patch of the window), Viterbi labels of every segment that lies wholly inside the window."""
    import warnings
    from inaspeechsegmenter_b200.segmenter import feats_from_signal
    from oracle import cnn_oracle, segmenter_oracle as so, sidekit_oracle as sk
    t_start = time.perf_counter()
    mspec, loge, difflen = feats_from_signal(pcm, seg.device, seg.fft_precision, 'main')
    L = loge.numel()
    P = (L + 1) // 2
    lseg_e = seg.energy_segments(loge)
    # ---- whole-file energy track
    loge_h = loge.cpu().numpy()
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        ref_e = so.energy_segments(loge_h, seg.energy_ratio)
    energy_equal = (ref_e == lseg_e)
    lseg_v = seg.vad(mspec, lseg_e, difflen)
    probs_v = seg.vad.last_probs
    lseg_g = seg.gender(mspec, lseg_v, difflen)
    probs_g = seg.gender.last_probs
    torch.cuda.synchronize()
    host = pcm.cpu().numpy() if pcm.is_cuda else pcm.numpy()
    rng = np.random.default_rng(seed)
    WINP = 3000                                                          # 60 s of patches
    res = {'softmax_max_abs': 0.0, 'labels_equal': True, 'energy_equal': bool(energy_equal), 'mspec_max_abs': 0.0,
           'inf_pattern_equal': True, 'windows': 0, 'patches_compared': 0, 'segments_compared': 0, 'energy_frames': int(L)}
    nets = [('vad', seg.vad, lseg_e, lseg_v, probs_v, so.VAD_SMN if len(seg.vad.outlabels) == 3 else so.VAD_SM),
            ('gender', seg.gender, lseg_v, lseg_g, probs_g, so.GENDER)]
    per_net = {}
    for name, dnn, lin, lout, probs, okw in nets:
        ranges = [(a, b) for lab, a, b in lin if lab == dnn.inlabel]
        st, sp, off = _rows_of(ranges)
        track_out = _track(lout, P, list(dnn.outlabels))
        cand = [i for i, (a, b) in enumerate(ranges) if 50 <= b - a <= 2500 and a >= 40 and b <= P - 40]
        if not cand:                                                     # no short segment: clipped ranges only (softmax still compared)
            cand = [i for i, (a, b) in enumerate(ranges) if a >= 40 and b <= P - 40]
        if not cand:
            continue
        pick = rng.choice(cand, size=min(n_windows, len(cand)), replace=False)
        oracle_net = so.DnnSegmenterOracle(cnn_oracle.KerasLikeModel(*mods[name], threads=min(32, host_cores())), **okw)
        worst, nseg, npatch = 0.0, 0, 0
        for i in pick:
            a0 = int(st[i])
            p0 = max(17, a0 - int(rng.integers(0, 200)))                 # window start (padded patch index)
            p1 = min(p0 + WINP, P - 17 - 1)
            f0 = 2 * (p0 - 17)
            nfr = 2 * (p1 - p0 - 1) + 68
            sig = host[160 * f0:160 * (f0 + nfr - 1) + 400].astype(np.float32) / np.float32(32768)
            m_ref, _ = sk.logmel_loge(sig)
            m_gpu = mspec[f0:f0 + nfr].cpu().numpy()
            fin = np.isfinite(m_ref)
            res['inf_pattern_equal'] &= bool(np.array_equal(fin, np.isfinite(m_gpu)))
            if fin.any():
                res['mspec_max_abs'] = max(res['mspec_max_abs'], float(np.abs(m_ref[fin] - m_gpu[fin]).max()))
            # local padded index = global - p0 + 17 (the local un-replicated window j' is patch p0 + j')
            loc, rows, whole = [], [], []
            for k in range(len(ranges)):
                a, b = int(st[k]), int(sp[k])
                if b <= p0 or a >= p1:
                    continue
                a2, b2 = max(a, p0), min(b, p1)
                loc.append((dnn.inlabel, a2 - p0 + 17, b2 - p0 + 17))
                rows.append((int(off[k]) + a2 - a, int(off[k]) + b2 - a, a2, b2))
                whole.append(a2 == a and b2 == b)
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                out_ref = oracle_net(m_ref, loc, 0)
            ref_p = oracle_net.last_probs
            got_p = torch.cat([probs[r0:r1] for r0, r1, _, _ in rows]).cpu().numpy()
            worst = max(worst, float(np.abs(got_p - ref_p).max()))
            npatch += len(got_p)
            ref_track = _track([(lab, a + p0 - 17, b + p0 - 17) for lab, a, b in out_ref], P, list(dnn.outlabels))
            for (r0, r1, a2, b2), w in zip(rows, whole):
                if w:
                    nseg += 1
                    if not np.array_equal(ref_track[a2:b2], track_out[a2:b2]):
                        res['labels_equal'] = False
            res['windows'] += 1
        per_net[name] = {'softmax_max_abs': worst, 'patches': npatch, 'whole_segments': nseg}
        res['softmax_max_abs'] = max(res['softmax_max_abs'], worst)
        res['patches_compared'] += npatch
        res['segments_compared'] += nseg
    res['per_network'] = per_net
    res['tolerance'] = {'softmax_max_abs': 1e-4, 'mspec_max_abs': 2e-5, 'labels': 'identical', 'energy': 'identical'}
    res['ok'] = bool(res['softmax_max_abs'] <= 1e-4 and res['labels_equal'] and res['energy_equal'] and
                     res['mspec_max_abs'] <= 2e-5 and res['inf_pattern_equal'] and res['windows'] > 0)
    res['oracle'] = 'oracle/ (numpy front-end pinned bit-for-bit to sidekit_mfcc.py; torch-CPU fp32 Keras interpreter: CNN parity vs TensorFlow unpinned)'
    res['seconds'] = time.perf_counter() - t_start
    return res


# ----------------------------------------------------------------------------- configs[2]: 100 h sm+gender, K1 roofline
def config2_block(torch, args, dev, peaks, fft):
    from inaspeechsegmenter_b200 import Segmenter, _lib
    from inaspeechsegmenter_b200.segmenter import feats_from_signal
    lib = _lib.load()
    hours = args.k1_hours
    n = int(hours * 3600 * SR)
    t0 = time.perf_counter()
    pcm = synth_range(torch, 0, n, dev)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    mods = make_models(vad_classes=2)
    seg = Segmenter(vad_engine='sm', detect_gender=True, ffmpeg=None, models=mods, device=dev.index, fft_precision=fft)
    seg.segment_signal(pcm[:SR * 600])                                   # warm-up on the first 10 minutes
    # ---- K1 alone: events around the feature call (the kernel + its 2-launch statistics tail)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    feats_from_signal(pcm, dev.index, seg.fft_precision, 'main')
    torch.cuda.synchronize()
    reps = 3
    l0 = lib.iss_launch_count()
    ev[0].record()
    for _ in range(reps):
        mspec, loge, _ = feats_from_signal(pcm, dev.index, seg.fft_precision, 'main')
    ev[1].record()
    ev[1].synchronize()
    k1_launches = (lib.iss_launch_count() - l0) // reps
    ms_k1 = ev[0].elapsed_time(ev[1]) / reps
    L = loge.numel()
    bytes_alg = 420.0 * L                                                # SURVEY 8(d): 320 B int16 in + 100 B out per frame
    gbs = bytes_alg / (ms_k1 * 1e-3) / 1e9
    peak_gbs = peaks.get('hbm_gbs') or 6650.0
    del mspec, loge
    # ---- the whole sm+gender pass, device-resident and from pinned host memory
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    segs = seg.segment_signal(pcm)
    e1.record(); e1.synchronize()
    ms_dev = e0.elapsed_time(e1)
    host = torch.empty(pcm.shape, dtype=torch.int16, pin_memory=True)
    host.copy_(pcm)
    torch.cuda.synchronize()
    del pcm
    torch.cuda.empty_cache()
    e0.record()
    segs2 = seg.segment_signal(host)
    e1.record(); e1.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    out = {
        'workload': "vad_engine='sm' + gender on %g h synthetic 16 kHz mono int16, 1xB200 (BASELINE configs[2]); one pass each, after a 10-minute warm-up" % hours,
        'value': hours / (ms_dev * 1e-3), 'unit': UNIT, 'ms': ms_dev,
        'e2e': {'value': hours / (ms_e2e * 1e-3), 'unit': UNIT, 'ms': ms_e2e, 'h2d_bytes': int(n * 2), 'd2h_bytes': int(3 * ((L + 1) // 2)),
                'equal_to_device_run': bool(segs2 == segs)},
        'segments': len(segs), 'generate_seconds': t_gen,
        'roofline_k1': {'bound': 'hbm', 'kernel': 'sidekit_features_kernel (%s FFT) + loge statistics' % fft, 'achieved': gbs, 'peak': peak_gbs,
                        'unit': 'GB/s', 'frac': gbs / peak_gbs, 'traffic': None,
                        'peak_source': 'MEASURED_PEAKS.json hbm_gbs (of measured)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s (of fallback)',
                        'bytes_per_frame': 420, 'frames': int(L), 'ms': ms_k1, 'launches': int(k1_launches),
                        'x_real_time': hours * 3600 / (ms_k1 * 1e-3)},
    }
    del host
    return out


# ----------------------------------------------------------------------------- configs[3]: VBx x-vectors, K5 roofline
def config3_block(torch, args, dev, peaks):
    from inaspeechsegmenter_b200 import _lib, engine, vbx_segmenter as vb
    from oracle import vbx_oracle as vx
    lib = _lib.load()
    ctx = engine.Context(dev.index)
    sd = vx.synthetic_resnet101_state(seed=5)
    ext = vb.B200BackendExtractor(state_dict=sd, ctx=ctx)
    fe = vb.VbxFrontEnd(ctx)
    file_sec = 3600
    nfiles = max(1, int(round(args.vbx_hours)))

    def one_file(src, keep=None):
        """get_features + VBxExtractor.__call__ windows (vbx_segmenter.py:72-89,217-246) of one 1 h file -> embeddings on the host."""
        pcm = src if src.is_cuda else src.to(dev, non_blocking=True)
        fea = fe(pcm)
        plan = vb.window_plan(fea.shape[0])
        reg = [s for s, nn, tail in plan if not tail]
        emb = ext.embed_windows(fea, reg, vb.WINLEN)
        out = emb.cpu()
        for s, nn, tail in plan:
            if tail:
                ext.embed_windows(fea, [s], nn).cpu()
        if keep is not None:
            keep['fea'], keep['reg'], keep['emb'] = fea, reg, out
        return len(plan), out

    blocks = [synth_range(torch, f * file_sec * SR, (f + 1) * file_sec * SR, dev) for f in range(min(nfiles, 2))]
    one_file(blocks[0][:SR * 120])                                       # warm-up (2 minutes)
    torch.cuda.synchronize()
    done_files, nwin = 0, 0
    l0 = lib.iss_launch_count()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    while done_files < nfiles and (time.perf_counter() - t0) < args.vbx_max_sec:
        w, _ = one_file(blocks[done_files % len(blocks)])
        nwin += w
        done_files += 1
    e1.record(); e1.synchronize()
    ms = e0.elapsed_time(e1)
    launches = lib.iss_launch_count() - l0
    # e2e: the same files from pinned host memory
    host = torch.empty(blocks[0].shape, dtype=torch.int16, pin_memory=True)
    host.copy_(blocks[0])
    torch.cuda.synchronize()
    e0.record()
    nfile_e2e = max(1, min(done_files, 3))
    for _ in range(nfile_e2e):
        one_file(host)
    e1.record(); e1.synchronize()
    ms_e2e = e0.elapsed_time(e1)
    hours = done_files * file_sec / 3600.0
    tf = nwin * ext.flops_per_window / (ms * 1e-3) / 1e12
    peak_tf = peaks.get('bf16_tflops_sustained') or 1400.0
    # CPU: the reference's torch backend (resnet.py, vbx_segmenter.py:271-288) restated, all host cores, a bounded sample of windows
    torch.set_num_threads(host_cores())
    net = vx.ResNet101Oracle(sd)
    # the 32 CPU windows are REAL windows of the benchmark file, spread over all of its sweeps: their x-vectors double as the
    # benchmark-scale parity check of K5 (the GPU embeddings of the same windows come out of full 256-window sweeps)
    keep = {}
    k5_parity = None
    xw = torch.randn(32, 64, 144)
    pick = list(range(32))
    try:
        one_file(blocks[0], keep)
        reg = keep['reg']
        pick = sorted(set(int(i) for i in np.linspace(0, len(reg) - 1, 32)))
        xw = torch.stack([keep['fea'][reg[i]:reg[i] + vb.WINLEN].T.contiguous() for i in pick]).cpu()
    except Exception as e:                                               # (the timing below must survive a parity-plumbing error)
        k5_parity = {'error': repr(e)}
    net.forward(xw[:4])
    tc0 = time.perf_counter()
    yw = net.forward(xw)
    tcpu = time.perf_counter() - tc0
    cpu_win_s = len(pick) / tcpu
    if k5_parity is None:
        try:
            yw = np.asarray(yw.detach().cpu().numpy() if hasattr(yw, 'detach') else yw, dtype=np.float32).reshape(len(pick), -1)
            got = keep['emb'].numpy()[pick]
            k5_rel = float(np.abs(got - yw).max() / max(np.abs(yw).max(), 1e-30))
            k5_parity = {'windows': len(pick), 'max_rel_err': k5_rel, 'tolerance': 2e-4, 'ok': bool(k5_rel <= 2e-4),
                         'oracle': 'oracle/vbx_oracle.py ResNet101Oracle (bit-identical to the real resnet.py on seeded weights)'}
        except Exception as e:
            k5_parity = {'error': repr(e)}
    del keep
    win_per_hour = nwin / hours
    return {
        'workload': 'VBx x-vector path (features_vbx + resnet.py ResNet101) on %g h synthetic 16 kHz mono as 1 h files, 1xB200 (BASELINE configs[3] = 50 h)' % hours
                    + ('' if done_files == nfiles else ' -- BOUNDED SAMPLE: stopped after %g s' % args.vbx_max_sec),
        'value': hours / (ms * 1e-3), 'unit': UNIT, 'ms': ms, 'windows': int(nwin), 'windows_per_s': nwin / (ms * 1e-3),
        'x_real_time': hours * 3600 / (ms * 1e-3), 'gpu_launches': int(launches),
        'e2e': {'value': nfile_e2e * file_sec / 3600.0 / (ms_e2e * 1e-3), 'unit': UNIT, 'files': nfile_e2e,
                'h2d_bytes_per_file': int(file_sec * SR * 2), 'd2h_bytes_per_file': int(win_per_hour * 256 * 4)},
        'roofline_k5': {'bound': 'tensor', 'kernel': 'ResNet101 implicit-GEMM convolutions (iss_resnet_embed, 104 conv layers)', 'achieved': tf, 'peak': peak_tf,
                        'unit': 'TFLOP/s', 'frac': tf / peak_tf, 'traffic': None, 'flops_per_window': ext.flops_per_window,
                        'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained (of measured)' if 'bf16_tflops_sustained' in peaks else 'fallback 1.4 PFLOP/s (of fallback)',
                        'note': 'whole x-vector path time (features 0.2 %, ResNet 99 %)'},
        'cpu_baseline': {'value': cpu_win_s / win_per_hour, 'unit': UNIT, 'cores': host_cores(), 'kind': 'port',
                         'sample': '32 windows of 144 frames of the benchmark file through the torch-CPU restatement of resnet.py (the reference\'s own torch backend, vbx_segmenter.py:271-288), all host cores; %.1f windows/s' % cpu_win_s},
        'parity': k5_parity,
        'weights': 'seeded synthetic ResNet101 (final.onnx / raw_81.pth absent)',
    }


# ----------------------------------------------------------------------------- the B200 arm
def run_b200(args):
    import ctypes

    import torch
    import torch.distributed as dist
    from inaspeechsegmenter_b200 import Segmenter, _lib

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _lib.load()
    mods = make_models()
    seg = Segmenter(vad_engine='smn', detect_gender=True, ffmpeg=None, models=mods, device=local, fft_precision=args.fft)

    from inaspeechsegmenter_b200.shard import ShardPlan, segment_signal_sharded
    total = int(args.hours * world * 3600 * SR)            # ONE recording of world x hours, time-sharded
    plan = ShardPlan(total, world)
    sa, sb = plan.sample_range(rank)
    pcm = synth_range(torch, sa, sb, dev)                               # this rank's samples (+halo), resident in HBM
    host = torch.empty(pcm.shape, dtype=torch.int16, pin_memory=True)    # pinned copy for the e2e leg
    host.copy_(pcm)
    torch.cuda.synchronize()
    audio_h = total / SR / 3600.0 / world                             # per-rank share of the recording

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        e1.synchronize()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), out

    if world == 1:
        step_dev = lambda: seg.segment_signal(pcm)          # noqa: E731  inputs already in HBM
        step_e2e = lambda: seg.segment_signal(host)         # noqa: E731  pinned host -> device inside the call
    else:
        step_dev = lambda: segment_signal_sharded(seg, pcm, total)[0]     # noqa: E731
        step_e2e = lambda: segment_signal_sharded(seg, host, total)[0]    # noqa: E731

    warm = max(args.warmup, 3)
    for _ in range(warm):
        segs = step_dev()
    # dominant kernel = the conv/dense layer with the most FLOPs of the VAD network
    nl = lib.iss_cnn_num_layers(seg.vad.nn.handle)
    lf = [lib.iss_cnn_layer_flops(seg.vad.nn.handle, i) for i in range(nl)]
    dom = int(np.argmax(lf))
    _lib.check(lib.iss_cnn_profile(seg.vad.nn.handle, dom), 'iss_cnn_profile')

    clocks = ClockSampler(local)
    l0 = lib.iss_launch_count()
    ms, segs = timed(step_dev, args.steps)
    launches = lib.iss_launch_count() - l0
    clk = clocks.stop()
    tms, nlaunch, fl = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
    _lib.check(lib.iss_cnn_profile_read(seg.vad.nn.handle, ctypes.byref(tms), ctypes.byref(nlaunch), ctypes.byref(fl)), 'profile_read')
    _lib.check(lib.iss_cnn_profile(seg.vad.nn.handle, -1), 'iss_cnn_profile')

    ms_e2e, segs2 = timed(step_e2e, args.steps)
    e2e_equal = bool(segs2 == segs)
    d2h = int(seg_d2h_bytes(segs, pcm.numel()))

    # ---- N > 1: the sharded list against a single-GPU run of the WHOLE recording (rank 0, outside the timed region)
    sharded = None
    if world > 1:
        if rank == 0:
            t0 = time.perf_counter()
            whole = synth_range(torch, 0, total, dev)
            ref = seg.segment_signal(whole)
            torch.cuda.synchronize()
            del whole
            sharded = {'sharded_equals_single_gpu': bool(ref == segs), 'segments': len(ref), 'recording_hours': args.hours * world,
                       'seconds': time.perf_counter() - t0,
                       'what': 'complete (label, start, stop) list of the %d-rank time-sharded run == one-GPU run of the same %g h recording' % (world, args.hours * world)}
        barrier()

    value = audio_h * world * args.steps / (ms / 1e3)
    e2e = audio_h * world * args.steps / (ms_e2e / 1e3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, segs)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_tf = peaks.get('bf16_tflops_sustained') or 1400.0
    peak_src = 'MEASURED_PEAKS.json bf16_tflops_sustained (of measured)' if 'bf16_tflops_sustained' in peaks else 'fallback 1.4 PFLOP/s sustained (of fallback)'
    ach = (fl.value / max(nlaunch.value, 1)) / (tms.value / max(nlaunch.value, 1) * 1e-3) / 1e12 if tms.value > 0 else 0.0
    mode = lib.iss_get_gemm_mode()
    gemm = {0: 'fp32 CUDA cores', 2: 'tcgen05 kind::tf32, 3xTF32 split', 3: 'tcgen05 kind::f16 direct kernel (both operands from shared memory), fp16 hi/lo split (3 products), first layer fused into the operand fill'}.get(mode, 'engine %d' % mode)
    traffic, traffic_src = ncu_dram_bytes(dominant_profile(mode))
    roof = {'bound': 'tensor', 'kernel': 'conv_gemm %s (VAD layer %d: %s)' % (gemm, dom, layer_name(seg.vad.nn.lowered.descs[dom])),
            'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach / peak_tf, 'traffic': traffic, 'traffic_source': traffic_src,
            'peak_source': peak_src, 'launches': int(nlaunch.value), 'avg_launch_ms': tms.value / max(nlaunch.value, 1),
            'flops_per_launch': fl.value / max(nlaunch.value, 1), 'share_of_step': tms.value / ms,
            'note': 'useful fp32-equivalent FLOPs of the layer; the tensor pipe executes 3x as many (hi.hi + hi.lo + lo.hi) on 1/0.773 as many rows (tall-image slots), so the ceiling of this scheme is 0.257; the time includes the fused first layer'}

    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': warm,
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32' if mode == 0 else ('f32 (3xTF32 split on tcgen05, fp32 accumulate)' if mode == 2 else 'f32 (fp16 hi/lo split on tcgen05 kind::f16, fp32 accumulate; 22 significant bits)'),
        'data': 'synthetic',
        'config': {'workload': 'smn+gender on %g h synthetic 16 kHz mono int16 per GPU (BASELINE configs[1])' % args.hours,
                   'networks': 'synthetic-weight stand-ins of the ~1.4M-parameter CNN family (release .hdf5 absent)',
                   'fft': args.fft, 'l2': 'inputs larger than L2 (%.2f GB PCM per step)' % (pcm.numel() * 2 / 1e9),
                   'parallelism': ('single GPU' if world == 1 else
                                   'one %g h recording time-sharded over %d GPUs (34-frame halo); NCCL all-gathers of loge and of the CNN posteriors, Viterbi passes replicated (bit-identical to one GPU)' % (args.hours * world, world)),
                   'segments': len(segs),
                   'vad_flops_per_patch': seg.vad.nn.flops_per_patch, 'gender_flops_per_patch': seg.gender.nn.flops_per_patch},
        'clocks': clk,
        'e2e': {'value': e2e, 'unit': UNIT, 'h2d_bytes_per_step': int(pcm.numel() * 2), 'd2h_bytes_per_step': d2h,
                'ms_per_step': ms_e2e / args.steps, 'equal_to_device_run': e2e_equal},
        'gpu_launches': int(launches),
        'roofline': roof,
    }
    if sharded is not None:
        line['parity'] = sharded
    extras = not args.no_extras and world == 1
    if extras:
        for key, fn in (('parity', lambda: parity_block(torch, seg, pcm, mods, args.parity_windows)),):
            try:
                line[key] = fn()
            except Exception as e:                                       # a failed check must be visible, not fatal to the headline
                line[key] = {'ok': False, 'error': repr(e)}
    del pcm, host
    torch.cuda.empty_cache()
    if extras:
        for key, fn in (('configs2', lambda: config2_block(torch, args, dev, peaks, args.fft)),
                        ('configs3', lambda: config3_block(torch, args, dev, peaks))):
            try:
                line[key] = fn()
            except Exception as e:
                line[key] = {'error': repr(e)}
            torch.cuda.empty_cache()
    if not args.no_cpu_baseline and world == 1:
        chunk = args.cpu_chunk_sec or 120.0
        farm = CpuFarm(chunk, args.cpu_workers)
        t = farm.step()
        farm.close()
        line['cpu_baseline'] = {'value': farm.audio_hours_per_step / t, 'unit': UNIT, 'cores': farm.workers * farm.threads, 'kind': 'port',
                                'host_cores': host_cores(), 'sample': farm.describe()}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def dominant_profile(mode):
    """The committed `ncu --set full` summary of the dominant kernel for this engine (per-round file name)."""
    name = {3: 'r02_direct_tc4h_full.txt'}.get(mode)
    return os.path.join(ROOT, 'profiles', name) if name else None


def _strip_cxx_comments(src):
    """C++ source without comments and without white space: the text the compiler's result depends on."""
    out, i, n = [], 0, len(src)
    while i < n:
        c = src[i]
        if c == '"' or c == "'":                                          # string / character literal: copied verbatim
            j = i + 1
            while j < n and src[j] != c:
                j += 2 if src[j] == '\\' else 1
            out.append(src[i:j + 1]); i = j + 1
        elif src.startswith('//', i):
            j = src.find('\n', i)
            i = n if j < 0 else j
        elif src.startswith('/*', i):
            j = src.find('*/', i + 2)
            i = n if j < 0 else j + 2
        else:
            out.append(c); i += 1
    return ''.join(''.join(out).split())


def kernel_source_hash():
    """sha256 over the CODE (comments and white space stripped) of the dominant kernel's sources; tools/ncu_summary.py
    stamps it into the profile summary."""
    import hashlib
    h = hashlib.sha256()
    for f in ('conv_gemm_tc_f16d.cu', 'tc_common.cuh', 'conv_gemm.cuh'):
        with open(os.path.join(ROOT, 'inaspeechsegmenter_b200', 'csrc', f)) as fh:
            h.update(_strip_cxx_comments(fh.read()).encode())
    return h.hexdigest()


def ncu_dram_bytes(path):
    """dram__bytes_read.sum + dram__bytes_write.sum (bytes per launch) of the first kernel in a committed
    `ncu --set full` summary of the same 8192-patch launch (a profiler cannot run inside the timed process).
    The summary is stamped with the hash of the kernel sources it was captured from: if they changed since,
    the figure is withheld (None, 'stale ...') instead of silently going out of date."""
    if not path or not os.path.exists(path):
        return None, None
    try:
        tot, seen, stamp = 0.0, False, None
        for line in open(path):
            if line.startswith('# source_sha256:'):
                stamp = line.split(':', 1)[1].strip()
                continue
            if line.startswith('kernel:'):
                if seen:
                    break
                seen = True
            elif seen and ('dram__bytes_read.sum ' in line or 'dram__bytes_write.sum ' in line):
                val, unit = line.split()[-2:]
                tot += float(val) * {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}[unit]
        if stamp != kernel_source_hash():
            return None, 'stale: %s was captured from other kernel sources' % os.path.relpath(path, ROOT)
        if tot > 0:
            return tot, 'ncu --set full, %s (bytes per launch, cold cache; capture of an identical launch, not this run)' % os.path.relpath(path, ROOT)
    except Exception:
        pass
    return None, None


def layer_name(d):
    kind = {1: 'Conv2D', 2: 'Dense', 3: 'MaxPool'}[d['kind']]
    return '%s %dx%d %d->%d' % (kind, d['kh'], d['kw'], d['cin'], d['cout'])


def seg_d2h_bytes(segs, n_samples):
    """Bytes read back per step: the three uint8 label tracks (energy [P], VAD and gender tracks over evaluated patches)."""
    L = (n_samples - 400) // 160 + 1
    return 3 * ((L + 1) // 2)


if __name__ == '__main__':
    a = parse()
    sys.exit(run_reference(a) if a.impl == 'reference' else run_b200(a))

#!/usr/bin/env python3
"""Benchmark of the audio template-matching hot path (BASELINE.json metric: subtitle events/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload config3]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic subtitle events: broadcast of the two
normalised streams to every rank, stream preparation (running sums + the block spectra a rank's events
touch), every event's TM_SQDIFF_NORMED search at the configuration's full window, all-gather of the
per-event results.  One event = one search group = one find_substream query (SURVEY.md section 8d).

The default workload is BASELINE.json configs[2], the configuration north_star's target is quoted on
(10 000 events, 2 x 90-minute streams, +-120 s); it fits one GPU.  At N ranks the ONE event list is
sharded contiguously (strong scaling; `--scaling weak` multiplies the list by N instead).  The step is
sushi_b200.parallel.ShardedMatcher -- the product's own multi-GPU path over the library's NCCL
communicator; no PyTorch in this process.

Numbers printed (one JSON line, rank 0):
  value   events/s with the raw streams already resident in the root's HBM, device-timed (CUDA events on the
          library stream), maximum over ranks
  e2e     events/s through the public API from page-locked HOST buffers on the root: H2D of both streams and
          of the event list, planning, the step above, D2H of the gathered results -- all inside the timed region
  roofline       dominant kernel class against the measured HBM peak (algorithmic bytes, 8d), plus what ncu says
                 really limits it (issue slots / L2 -> SM traffic), from a capture of this very source
  cpu_baseline   the oracle port (reference find_substream over cv2.matchTemplate) on this box's host cores,
                 on a bounded sample of the same events (N=1, rank 0 only)
  load    the loader leg (N=1): 90 min of 48 kHz stereo PCM -> resident normalised stream (decode, resample,
          medians, normalise, running sums), per-kernel GB/s against the HBM peak, the oracle loader beside it

--impl reference times the CPU path as the reference arm.

--dump-outputs DIR writes what the last device-timed step computed, as find_batch returns it to a caller:
DIR/diffs.npy (float32, one per event) and DIR/times.npy (float64 seconds).  The inputs derive from fixed seeds,
so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from sushi_b200 import _hostmem, parallel, synth      # noqa: E402
from sushi_b200.wavstream import WavStream   # noqa: E402

_hostmem.keep_heap()

SAMPLE_RATE = 12000
WORKLOADS = {
    # BASELINE.json configs[0]: the reference's own CPU-runnable case
    'config1': dict(events=100, duration=60.0, window=10.0, min_len=1.0, max_len=4.0, shift=1.5,
                    text='100 events, 2x60 s 12 kHz streams, +1.5 s shift, +-10 s window'),
    # BASELINE.json configs[1]: the single-GPU configuration
    'config2': dict(events=2000, duration=1800.0, window=60.0, min_len=1.0, max_len=4.0, shift=1.5,
                    text='2000 events, 2x30 min 12 kHz streams, +-60 s window'),
    # BASELINE.json configs[2]: the configuration north_star's target is quoted on (default)
    'config3': dict(events=10000, duration=5400.0, window=120.0, min_len=1.0, max_len=4.0, shift=1.5,
                    text='10000 events, 2x90 min 12 kHz streams, +-120 s window, event-sharded'),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------
# inputs
# --------------------------------------------------------------------------------------
class HostStream(object):
    """A normalised stream on the host (what WavStream.data holds) without any GPU state."""

    def __init__(self, pcm, sample_type):
        s = object.__new__(WavStream)
        s._handle = None

        class _Mem(object):
            pass
        from sushi_b200.wavstream import decode_downmix
        raw = np.ascontiguousarray(pcm, '<i2').view(np.uint8)
        mem = _Mem()
        mem.framerate, mem.channels_count, mem.sample_width, mem.frame_size = SAMPLE_RATE, 1, 2, 2
        mem.frames_count = raw.size // 2
        pos = [0]

        def readframes(count):
            a = pos[0]
            b = min(a + count * 2, raw.size)
            pos[0] = b
            return decode_downmix(raw[a:b].tobytes(), 2, 1)
        mem.readframes = readframes
        s._load(mem, SAMPLE_RATE, sample_type)
        self.data, self.sample_count, self.padding_size = s.data, s.sample_count, s.padding_size
        self.sample_rate = SAMPLE_RATE
        self.sample_type = sample_type


def make_inputs(wl, sample_type, events, seed=2):
    t0 = time.time()
    src_pcm, dst_pcm = synth.make_pair(wl['duration'], seed, wl['shift'])
    src = HostStream(src_pcm, sample_type)
    dst = HostStream(dst_pcm, sample_type)
    starts, ends = synth.make_events(events, wl['duration'], seed, wl['min_len'], wl['max_len'])
    log('[bench] inputs ready in %.1f s' % (time.time() - t0))
    return src, dst, starts, ends


def algorithmic_bytes(tlen, nlags, bytes_per_sample):
    """SURVEY.md 8(d): one template read + one pass over the search span + (diff, idx) out."""
    tlen = np.asarray(tlen, np.float64)
    nlags = np.asarray(nlags, np.float64)
    return float(np.sum(bytes_per_sample * tlen + bytes_per_sample * (nlags + tlen - 1) + 16))


def workload_config(args, wl, events_total):
    """The `config` object: identical in both arms (it names the workload, not the implementation)."""
    return {'workload': args.workload + ': ' + wl['text'], 'events': events_total, 'sample_type': args.sample_type,
            'sample_rate': SAMPLE_RATE, 'window_s': wl['window'], 'stream_minutes': wl['duration'] / 60.0,
            'scaling': args.scaling, 'parallelism': 'events sharded over %d rank(s), contiguous shards' % args.gpus,
            'l2': 'inputs larger than L2: per stream %.0f MB running sums + up to %.0f MB block spectra, rebuilt every step'
                  % ((wl['duration'] + 20) * SAMPLE_RATE * 16 / 1e6, (wl['duration'] + 20) * SAMPLE_RATE * 8 / 1e6)}


# --------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores
# --------------------------------------------------------------------------------------
_CPU = {}


def _cpu_init():
    import cv2
    cv2.setNumThreads(1)       # matchTemplate does not scale with threads on 1-row images (SURVEY 8d)


def _cpu_run(chunk):
    src, dst = _CPU['src'], _CPU['dst']
    out = []
    for (a, b, c, w) in chunk:
        d, t = dst.find_substream(src.get_substream(a, b), c, w)
        out.append((float(d), t))
    return out


def effective_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    for path in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            txt = open(path).read().split()
            if path.endswith('cpu.max'):
                if txt[0] != 'max':
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                quota = float(txt[0])
                period = float(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
                if quota > 0:
                    n = min(n, max(1, int(quota / period)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def cpu_events_per_s(src, dst, starts, ends, window, budget_s, cores=None):
    """Throughput of the reference's CPU path on a bounded sample of the workload's events."""
    import multiprocessing as mp
    from oracle.ref_matcher import RefStream
    cores = cores or effective_cores()
    _CPU['src'] = RefStream(src.data, SAMPLE_RATE, src.padding_size, src.sample_count)
    _CPU['dst'] = RefStream(dst.data, SAMPLE_RATE, dst.padding_size, dst.sample_count)
    _cpu_init()
    order = np.linspace(0, len(starts) - 1, min(len(starts), 8)).astype(int)
    _cpu_run([(starts[order[0]], ends[order[0]], starts[order[0]], window)])       # warm-up
    t1 = time.perf_counter()
    _cpu_run([(starts[i], ends[i], starts[i], window) for i in order[1:3]])
    per_event = max((time.perf_counter() - t1) / 2, 1e-4)
    m = int(max(cores, min(len(starts), cores * budget_s / per_event)))
    m = min(m, len(starts))
    sel = np.linspace(0, len(starts) - 1, m).astype(int)
    items = [(starts[i], ends[i], starts[i], window) for i in sel]
    nchunk = min(len(items), cores * 4)
    chunks = [items[i::nchunk] for i in range(nchunk)]
    ctx = mp.get_context('fork')
    with ctx.Pool(cores, initializer=_cpu_init) as pool:
        pool.map(_cpu_run, [[items[0]]] * cores)                                   # spin the workers up
        t0 = time.perf_counter()
        res = pool.map(_cpu_run, chunks)
        wall = time.perf_counter() - t0
    first = res[0][0]
    return m / wall, cores, m, per_event, first


# --------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------
class ClockSampler(object):
    FIELDS = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
              'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(prefix='clocks_', suffix='.csv')
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '--query-gpu=' + self.FIELDS, '--format=csv,noheader,nounits', '-lms', '50',
                 '-i', str(gpu_index)], stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in open(self.path):
            p = [x.strip() for x in line.split(',')]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(names, p[5:9]):
                if v == 'Active':
                    reasons.add(name)
        try:
            os.remove(self.path)
        except OSError:
            pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# --------------------------------------------------------------------------------------
# evidence from ncu captures (profiles/traffic.json), valid only for the source it was taken from
# --------------------------------------------------------------------------------------
def _strip_comments(text):
    """C / C++ source without comments and without layout (string and character literals are kept intact)."""
    out, i, n = [], 0, len(text)
    while i < n:
        c = text[i]
        if c == '"' or c == "'":
            j = i + 1
            while j < n and text[j] != c:
                j += 2 if text[j] == '\\' else 1
            out.append(text[i:j + 1])
            i = j + 1
        elif text.startswith('//', i):
            j = text.find('\n', i)
            i = n if j < 0 else j
        elif text.startswith('/*', i):
            j = text.find('*/', i + 2)
            i = n if j < 0 else j + 2
        else:
            out.append(c)
            i += 1
    return ' '.join(''.join(out).split())


def kernel_source_hash():
    """Hash of the CUDA sources, comments and layout ignored: a capture is evidence for the code it was taken from,
    nothing else -- and rewording a comment does not change the code."""
    h = hashlib.sha1()
    csrc = os.path.join(ROOT, 'sushi_b200', 'csrc')
    for name in sorted(os.listdir(csrc)):
        if name.endswith(('.cu', '.cuh', '.h')):
            h.update(name.encode())
            h.update(_strip_comments(open(os.path.join(csrc, name), encoding='utf-8').read()).encode())
    return h.hexdigest()[:16]


def capture_for(key):
    """(entry, reason): the ncu capture recorded for `key`, or (None, why there is none that applies)."""
    try:
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
    except (OSError, ValueError):
        return None, 'no profiles/traffic.json'
    e = tr.get(key)
    if e is None:
        return None, 'no capture for ' + key
    if e.get('src_hash') != kernel_source_hash():
        return None, 'capture for %s is stale (taken from source %s, this is %s)' % (key, e.get('src_hash'), kernel_source_hash())
    return e, None


def read_peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except (OSError, ValueError):
        return {}


def profile_snapshot(lib):
    prof = {}
    for name in lib.sb_profile_names().decode().split(','):
        if not name:
            continue
        ms, n = ctypes.c_double(), ctypes.c_int64()
        lib.sb_profile_get(name.encode(), ctypes.byref(ms), ctypes.byref(n))
        if n.value or ms.value:
            prof[name] = (ms.value, n.value)
    return prof


# --------------------------------------------------------------------------------------
# loader leg
# --------------------------------------------------------------------------------------
def loader_leg(lib, peak, args):
    """PCM (48 kHz stereo int16, 90 min) -> resident normalised uint8 stream: sb_load_pcm + sb_normalise (which
    ends with the running sums).  Device time per kernel class from the library's event brackets; the PCM sits in
    page-locked host memory and its H2D copy is inside the wall-clock figure, not inside the kernel figures."""
    from sushi_b200 import _native
    minutes, rate, ch = args.load_minutes, 48000, 2
    frames = int(minutes * 60 * rate)
    t0 = time.time()
    unit = synth.programme_audio(rate * 20, 5, rate)                      # 20 s of programme audio, tiled (medians do not care)
    pcm = _native.pinned_empty((frames, ch), np.int16)
    for c in range(ch):
        reps = -(-frames // unit.size)
        pcm[:, c] = np.tile(np.roll(unit, 977 * c), reps)[:frames]
    log('[bench] loader input (%.0f MB PCM) ready in %.1f s' % (pcm.nbytes / 1e6, time.time() - t0))
    total_seconds = frames / float(rate)
    sample_count = int(np.ceil(total_seconds * SAMPLE_RATE))
    padding = 10 * rate
    total = int(20 * rate + sample_count)

    def once():
        raw, h = ctypes.c_void_p(), ctypes.c_void_p()
        lo, hi = ctypes.c_float(), ctypes.c_float()
        _native.check(lib.sb_load_pcm(pcm.ctypes.data_as(ctypes.c_void_p), frames, ch, 2, rate, SAMPLE_RATE, padding, total,
                                      ctypes.byref(raw)), 'sb_load_pcm')
        _native.check(lib.sb_normalise(raw, _native.SB_U8, ctypes.byref(h), ctypes.byref(lo), ctypes.byref(hi)), 'sb_normalise')
        lib.sb_stream_destroy(raw)
        _native.check(lib.sb_sync())
        lib.sb_stream_destroy(h)
    for _ in range(2):
        once()
    reps = 5
    lib.sb_profile_reset()
    lib.sb_profile_enable(1)
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    wall = (time.perf_counter() - t0) / reps
    lib.sb_profile_enable(0)
    prof = profile_snapshot(lib)
    # algorithmic bytes per kernel class for one load (DESIGN.md section 4)
    pcm_b, f32_b, u8_b, pfx_b = pcm.nbytes, 4.0 * total, 1.0 * total, 16.0 * (total + 1)
    alg = {'decode_resample_pad': pcm_b + f32_b, 'normalise_quantise': f32_b + u8_b,
           'median_select': f32_b, 'scan': u8_b + pfx_b}
    groups = {'decode_resample_pad': ['decode_resample_pad'], 'normalise_quantise': ['normalise_quantise'],
              'median_select': [k for k in prof if k.startswith('median_')],
              'scan': [k for k in prof if k.startswith('scan_')]}
    kernels = {}
    for g, names in groups.items():
        ms = sum(prof[n][0] for n in names if n in prof) / reps
        launches = sum(prof[n][1] for n in names if n in prof) / reps
        if ms > 0:
            gbs = alg[g] / (ms / 1e3) / 1e9
            kernels[g] = {'ms': round(ms, 4), 'launches': launches, 'algorithmic_bytes': alg[g],
                          'achieved_gbs': round(gbs, 1), 'frac_of_hbm_peak': round(gbs / peak, 4)}
    dev_ms = sum(k['ms'] for k in kernels.values())
    out = {'input': '%g min of %d Hz %d-channel int16 PCM (%.0f MB, page-locked host memory) -> %d samples uint8 + running sums'
                    % (minutes, rate, ch, pcm.nbytes / 1e6, total),
           'wall_ms_per_stream': round(wall * 1e3, 2), 'device_kernel_ms_per_stream': round(dev_ms, 3),
           'h2d_bytes': int(pcm.nbytes), 'kernels': kernels,
           'streams_per_s': round(1.0 / wall, 2)}
    if not args.no_cpu_baseline:
        # the oracle loader (reference WavStream.__init__ restated) on a bounded slice of the same PCM, one core
        from oracle import ref_loader
        sl_frames = int(min(frames, args.load_cpu_minutes * 60 * rate))
        raw = pcm[:sl_frames].reshape(-1).view(np.uint8)
        pos = [0]

        def read_raw(nframes):
            a = pos[0]
            b = min(a + nframes * 2 * ch, raw.size)
            pos[0] = b
            return raw[a:b].tobytes()
        t0 = time.perf_counter()
        ref_loader.load_stream(read_raw, sl_frames, rate, 2, ch, SAMPLE_RATE, 'uint8')
        cpu_s = time.perf_counter() - t0
        out['cpu_baseline'] = {'kind': 'port', 'cores': 1, 'sample': 'the first %g min of the same PCM through oracle/ref_loader.load_stream'
                               % (sl_frames / 60.0 / rate), 'seconds': round(cpu_s, 3),
                               'seconds_per_90min_stream': round(cpu_s * frames / sl_frames * 90.0 / minutes, 2)}
    return out


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def pinned_copy(arr):
    from sushi_b200 import _native
    out = _native.pinned_empty(arr.shape, arr.dtype)
    np.copyto(out, arr)
    return out


def run_b200(args):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('bench.py --gpus %d must be launched with torch.distributed.run (WORLD_SIZE=%d)' % (args.gpus, world))
    wl = WORKLOADS[args.workload]
    stype = args.sample_type
    bps = 1 if stype == 'uint8' else 4
    events_total = wl['events'] * (world if args.scaling == 'weak' else 1)
    root = rank == 0
    if args.load_only:              # the loader leg alone (profiler captures of the HBM-bound kernels)
        from sushi_b200 import _native
        peaks = read_peaks()
        print(json.dumps({'load': loader_leg(_native.lib(local_rank), float(peaks.get('hbm_gbs', 6650.0)), args)}), flush=True)
        return

    src_h = dst_h = starts = ends = None
    if root:
        src_h, dst_h, starts, ends = make_inputs(wl, stype, events_total)
        centers, windows = starts.copy(), np.full(len(starts), wl['window'])

    # ---- CPU baseline first (fork before CUDA is initialised in this process) -------
    cpu = None
    if root and world == 1 and not args.no_cpu_baseline:
        v, cores, m, per_event, _ = cpu_events_per_s(src_h, dst_h, starts, ends, wl['window'], args.cpu_budget)
        cpu = {'value': round(v, 3), 'unit': 'events/s', 'cores': cores, 'kind': 'port',
               'sample': '%d of the %d events of %s, evenly spaced, one process per core, cv2 threads=1; '
                         '1-core calibration %.1f ms/event' % (m, events_total, args.workload, per_event * 1e3)}
        log('[bench] cpu baseline: %.1f events/s on %d cores (%d events)' % (v, cores, m))

    from sushi_b200 import _native
    lib = _native.lib(local_rank)
    if args.block:
        _native.check(lib.sb_set_block_size(args.block))
    if args.engine >= 0:
        _native.check(lib.sb_set_engine(args.engine))
    if args.hop_mode >= 0:
        _native.check(lib.sb_set_hop_mode(args.hop_mode))
    if args.premac_mode >= 0:
        _native.check(lib.sb_set_premac_mode(args.premac_mode))
    if args.epilogue > 0:
        _native.check(lib.sb_set_epilogue(args.epilogue))

    backend = parallel.DeviceBackend(lib)
    comm = parallel.NcclComm(rank, world, lib) if world > 1 else parallel.SingleComm(backend)
    matcher = parallel.ShardedMatcher(comm, backend)

    if root:        # page-locked host copies (the e2e leg copies from these every step)
        src_h.data, dst_h.data = pinned_copy(src_h.data), pinned_copy(dst_h.data)
    matcher.set_streams(src_h, dst_h)                                   # raw streams resident on the root from here on
    plan = matcher.plan(*((starts, ends, centers, windows) if root else ()))
    count = plan['count']
    my_bytes = algorithmic_bytes(plan['shard'][1], plan['shard'][3], bps)
    step_bytes = algorithmic_bytes(plan['all'][1], plan['all'][3], bps)

    def barrier():
        comm.barrier()
        _native.check(lib.sb_sync())

    # ---- correctness of what is being timed: known shift recovered --------------------
    matcher.run_planned()
    diff, idx = matcher.gather_results()
    bad = checked = 0
    if root:
        shifts = plan['t0'] + idx / float(SAMPLE_RATE) - starts
        ok = (ends + wl['shift'] < wl['duration']) & (starts + wl['shift'] > 0)
        checked = int(ok.sum())
        bad = int(np.sum(np.abs(shifts[ok] - wl['shift']) > 1.0 / SAMPLE_RATE + 1e-9))
        if bad:
            log('[bench] WARNING: %d of %d events did not recover the known shift' % (bad, checked))

    # ---- warm-up, then the device-timed region --------------------------------------------
    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        matcher.run_planned()
    barrier()
    sampler = ClockSampler(local_rank) if root else None
    lib.sb_profile_reset()
    lib.sb_profile_enable(1)
    barrier()
    _native.check(lib.sb_timer_start())
    for _ in range(args.steps):
        matcher.run_planned()
    ms = ctypes.c_float()
    _native.check(lib.sb_timer_stop(ctypes.byref(ms)))
    barrier()
    lib.sb_profile_enable(0)
    clocks = sampler.stop() if sampler else None
    launches = int(lib.sb_launch_count())
    prof = profile_snapshot(lib)
    ms_total = comm.max_over_ranks([ms.value])[0]
    if root and args.dump_outputs:
        diff, idx = matcher.gather_results()
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, 'diffs.npy'), diff)
        np.save(os.path.join(args.dump_outputs, 'times.npy'), plan['t0'] + idx / float(SAMPLE_RATE))

    # ---- e2e: host buffers on the root, public API, results back on the host; wall clock bracketed by
    # barriers + device syncs, maximum over ranks
    def step_e2e():
        matcher.upload_streams(src_h, dst_h)                                  # H2D of both streams (root)
        matcher.find_batch(*((starts, ends, centers, windows) if root else ()))   # H2D events, plan, step, D2H results
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = comm.max_over_ranks([time.perf_counter() - t0])[0]

    if root:
        ms_step = ms_total / args.steps
        value = events_total / (ms_step / 1e3)
        peaks = read_peaks()
        peak = float(peaks.get('hbm_gbs', 6650.0))
        peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if peaks else 'fallback 6.65 TB/s (B200_PROFILING.md)'
        # dominant kernel class by accumulated device time inside the timed steps (this rank's launches)
        dom = max(prof.items(), key=lambda kv: kv[1][0]) if prof else (None, (0.0, 0))
        dom_name, (dom_ms, dom_n) = dom
        dom_ms_step = dom_ms / args.steps
        achieved = my_bytes / (dom_ms_step / 1e3) / 1e9 if dom_ms_step > 0 else 0.0
        key = '%s/%s/%s/N%d' % (args.workload, stype, dom_name, world)
        cap, why = capture_for(key)
        if cap is None and world > 1:        # ncu never wraps a multi-rank command: the 1-GPU capture's bytes per CTA serve every N
            cap, why = capture_for('%s/%s/%s/N1' % (args.workload, stype, dom_name))
        # DRAM traffic per launch of the class: the capture holds ONE launch of the match kernel (launches are cut at
        # 524 288 pairs of lag blocks), so its bytes per pair are scaled to this rank's pairs per step
        B = lib.sb_get_block_size()
        lag0_s, nlags_s = plan['shard'][2], plan['shard'][3]
        nk = (lag0_s + nlags_s - 1) // B - lag0_s // B + 1
        ctas_step = int(np.sum((nk + 1) // 2))
        traffic = None
        if cap and cap.get('dram_bytes_per_pair') and dom_n:
            traffic = cap['dram_bytes_per_pair'] * ctas_step * args.steps / dom_n
        roof = {'bound': 'hbm', 'kernel': dom_name, 'achieved': round(achieved, 2), 'peak': peak, 'unit': 'GB/s',
                'frac': round(achieved / peak, 5), 'traffic': traffic,
                'peak_source': peak_src,
                'launches_per_step': dom_n / args.steps, 'avg_launch_ms': round(dom_ms / max(dom_n, 1), 5),
                'algorithmic_bytes_per_launch': my_bytes * args.steps / max(dom_n, 1),
                'algorithmic_bytes_per_step_this_rank': my_bytes, 'algorithmic_bytes_per_step_all_ranks': step_bytes,
                'whole_step': {'achieved': round(step_bytes / (ms_step / 1e3) / 1e9, 2),
                               'frac': round(step_bytes / (ms_step / 1e3) / 1e9 / peak / world, 5)},
                'kernel_ms_per_step': {k: round(v[0] / args.steps, 4) for k, v in sorted(prof.items())}}
        if cap:
            m = cap.get('metrics', {})
            roof['traffic_basis'] = ('ncu dram__bytes_read+write of one captured launch (%d pairs of lag blocks) / pair x %d pairs of this rank per step / %g launches per step'
                                     % (int(cap.get('pairs_in_launch', 0)), ctas_step, dom_n / args.steps))
            roof['limiter'] = {'note': 'the kernel keeps the correlation on chip and is not HBM-bound; what ncu shows it waits on',
                               'issue_slots_active_pct': m.get('smsp__issue_active.avg.pct_of_peak_sustained_active'),
                               'warps_active_pct': m.get('sm__warps_active.avg.pct_of_peak_sustained_active'),
                               'l2_throughput_pct': m.get('lts__throughput.avg.pct_of_peak_sustained_elapsed'),
                               'l2_hit_rate_pct': m.get('lts__t_sector_hit_rate.pct'),
                               'fma_pipe_pct': m.get('sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active'),
                               'source': 'profiles/' + cap.get('report', '?')}
        else:
            roof['traffic_reason'] = why
        h2d = int(src_h.data.nbytes + dst_h.data.nbytes + count * 32)
        d2h = int(12 * plan['cap'] * world)
        e2e_value = events_total * args.steps / e2e_s
        line = {
            'metric': 'subtitle_events_per_s', 'value': round(value, 2), 'unit': 'events/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': warmup,
            'ms_per_step': round(ms_step, 4), 'ms_per_event': round(ms_step * world / events_total, 6),
            'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args, wl, events_total),
            'implementation': {'events_on_rank0': int(plan['hi'] - plan['lo']), 'lag_block': lib.sb_get_block_size(),
                               'kernel_body': lib.sb_get_epilogue(), 'spectrum_rows': 'f32',
                               'engine': {0: 'cufft', 1: 'fused', 2: 'fused_packed', 4: 'fused_packed_pair', 5: 'fused_packed_single'}[lib.sb_get_engine()],
                               'step': 'stream broadcast + running sums + block spectra of the shard + all queries + all-gather'
                                       if world > 1 else 'running sums + block spectra + all queries',
                               'collectives': 'library-owned NCCL %d (no PyTorch in the process)' % lib.sb_comm_nccl_version() if world > 1 else 'none',
                               'kernel_source_hash': kernel_source_hash()},
            'roofline': roof,
            'e2e': {'value': round(e2e_value, 2), 'unit': 'events/s', 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h, 'ms_per_step': round(e2e_s / args.steps * 1e3, 3)},
            'gpu_launches': launches,
            'clocks': clocks,
            'shift_check': {'events_checked': checked, 'mismatches': bad},
        }
        if cpu is not None:
            line['cpu_baseline'] = cpu
        if world == 1 and not args.no_load_leg:
            try:
                line['load'] = loader_leg(lib, peak, args)
            except Exception as e:                      # the loader leg must never cost the headline line
                line['load'] = {'error': str(e)}
        print(json.dumps(line), flush=True)
    barrier()
    comm.close()


# --------------------------------------------------------------------------------------
# reference arm
# --------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    world = args.gpus
    events_total = wl['events'] * (world if args.scaling == 'weak' else 1)
    src_h, dst_h, starts, ends = make_inputs(wl, args.sample_type, events_total)
    vals = []
    budget = max(2.0, min(args.cpu_budget, 60.0 / max(args.steps + args.warmup, 1)))
    cores = m = 0
    for i in range(args.warmup + args.steps):
        v, cores, m, per_event, _ = cpu_events_per_s(src_h, dst_h, starts, ends, wl['window'], budget)
        if i >= args.warmup:
            vals.append(v)
    value = float(np.mean(vals))
    line = {
        'impl': 'reference', 'metric': 'subtitle_events_per_s', 'value': round(value, 3), 'unit': 'events/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': round(m / value * 1e3, 3), 'higher_is_better': True, 'scaling': args.scaling,
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, wl, events_total),
        'cpu_baseline': {'value': round(value, 3), 'unit': 'events/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d of the %d events per step, evenly spaced, one process per core, cv2 threads=1'
                                   % (m, events_total)},
        'e2e': {'value': round(value, 3), 'unit': 'events/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='config3', choices=sorted(WORKLOADS))
    ap.add_argument('--scaling', default='strong', choices=['strong', 'weak'],
                    help='strong (default): one event list sharded over the ranks; weak: the list grows with the ranks')
    ap.add_argument('--sample-type', default='uint8', choices=['uint8', 'float32'])
    ap.add_argument('--cpu-budget', type=float, default=12.0, help='seconds of wall clock for the CPU baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-load-leg', action='store_true')
    ap.add_argument('--load-only', action='store_true', help='run the loader leg alone')
    ap.add_argument('--load-minutes', type=float, default=90.0, help='length of the PCM the loader leg loads')
    ap.add_argument('--load-cpu-minutes', type=float, default=10.0, help='slice of it the oracle loader is timed on')
    ap.add_argument('--block', type=int, default=0, help='lag-block size override')
    ap.add_argument('--premac-mode', type=int, default=-1, help='blocked multiply kernel: 0 by template length (default), 1 never, 2 always')
    ap.add_argument('--hop-mode', type=int, default=-1, help='fused engine geometry: 1 hop B (default), 2 hop B/2, 0 cost rule per batch')
    ap.add_argument('--epilogue', type=int, default=0, help='body variant of the packed kernels on uint8 streams: 3 run-level bounds + k_finish_runs (default), 1 first version')
    ap.add_argument('--engine', type=int, default=-1, help='0: cuFFT pipeline, 1: fused kernel, 2: packed fused kernels (default), 4 / 5: always / never pairs of lag blocks')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the results of the last timed step to DIR/*.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl == 'reference' or args.load_only):
        ap.error('--dump-outputs needs the timed matcher steps (--impl b200 without --load-only)')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()

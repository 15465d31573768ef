#!/usr/bin/env python3
"""Generate tests/golden/*.npz by running THE REFERENCE ITSELF (a read-only checkout of tp7/Sushi)
under Python 3.  TEST INFRASTRUCTURE ONLY: the tests never need the reference, the frozen outputs
stand in for it.  Seeded inputs are stored as CRC-32s (oracle/golden_inputs.py regenerates them).

What runs unmodified from the reference:
  * wav.WavStream.get_substream / find_substream / _get_sample_for_time / duration_seconds
    (wav.py:164-188) on instances built by the reference's own WavStream.__init__ (wav.py:108-162)
  * wav.WavStream.__init__ + DownmixedWavFile (wav.py:15-162) behind a bytes/str shim for the
    py2 string literals (wav.py:23,25,38,41) and np.fromstring -> np.frombuffer (wav.py:69);
    the int24 branch (wav.py:71-74) divides two ints for an array length (`len(data) / 3`, an int under
    Python 2): the module sees a numpy proxy whose zeros() accepts that float when it is a whole number
    (gen_loader24 -> loader24.npz).
  * sushi.prepare_search_groups / calculate_shifts (sushi.py:319-508) after an in-memory, purely
    mechanical py2->py3 text transform listed in PY3_EDITS below (no reference source is copied
    into this repository; the transformed text only lives in memory).

Usage:  python oracle/gen_golden.py REFERENCE_DIR [loader|loader24|matcher|shifts ...]
        (writes tests/golden/*.npz)
"""
import functools
import io
import os
import sys
import types
import wave
import zlib

import numpy as np

if len(sys.argv) < 2 or not os.path.isfile(os.path.join(sys.argv[1], 'wav.py')):
    sys.exit(__doc__)
REF = os.path.abspath(sys.argv[1])
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, 'tests', 'golden')
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

import chunk as _chunk      # noqa: E402  (stdlib, still present in 3.12)
import wav as refwav        # noqa: E402  the reference module
import subs as refsubs      # noqa: E402

from oracle import golden_inputs   # noqa: E402  seeded inputs
from sushi_b200 import synth       # noqa: E402  seeded PCM generator (inputs only)


class _Py2Str(bytes):
    """bytes that compare equal to the py2 str literals the reference uses for chunk ids."""
    def __eq__(self, other):
        return bytes(self) == (other.encode('latin1') if isinstance(other, str) else other)

    def __ne__(self, other):
        return not self.__eq__(other)
    __hash__ = bytes.__hash__


class _ChunkCompat(_chunk.Chunk):
    def getname(self):
        return _Py2Str(super().getname())

    def read(self, size=-1):
        return _Py2Str(super().read(size))


refwav.Chunk = _ChunkCompat
refwav.xrange = range
refwav.reduce = functools.reduce
np.fromstring = lambda data, dtype=float: np.frombuffer(bytes(data), dtype=dtype)   # wav.py:69


class _NpPy2Division(object):
    """numpy as wav.py sees it: identical, except that zeros() takes the float that `len(data) / 3` (wav.py:72) yields
    under Python 3 -- under Python 2 that expression is an int; frames are whole, so the division is exact."""
    def __getattr__(self, name):
        return getattr(np, name)

    @staticmethod
    def zeros(shape, dtype=float):
        if isinstance(shape, float):
            assert shape.is_integer(), shape
            shape = int(shape)
        return np.zeros(shape, dtype)


refwav.np = _NpPy2Division()

PY3_EDITS = [
    ('from itertools import takewhile, izip, chain', 'from itertools import takewhile, chain\nizip = zip'),
    ('xrange(', 'range('),
    ('.iteritems()', '.items()'),
    ('groups = filter(None, groups)', 'groups = list(filter(None, groups))'),
    ('len(tv_audio[0])/2', 'len(tv_audio[0])//2'),
    ('unicode(', 'str('),
    ('xp=map(operator.itemgetter(0), data_list)', 'xp=list(map(operator.itemgetter(0), data_list))'),
    ('fp=map(operator.itemgetter(1), data_list)', 'fp=list(map(operator.itemgetter(1), data_list))'),
]


def load_reference_sushi():
    text = open(os.path.join(REF, 'sushi.py')).read()
    for old, new in PY3_EDITS:
        assert old in text, old
        text = text.replace(old, new)
    mod = types.ModuleType('ref_sushi_py3')
    mod.__file__ = os.path.join(REF, 'sushi.py')
    exec(compile(text, mod.__file__, 'exec'), mod.__dict__)
    return mod


def write_wav(path, pcm, framerate, channels):
    with wave.open(path, 'wb') as w:
        w.setnchannels(channels)
        w.setsampwidth(2)
        w.setframerate(framerate)
        w.writeframes(np.ascontiguousarray(pcm, '<i2').tobytes())


def ref_load(pcm, framerate, channels, sample_rate, sample_type, tmp='/tmp/_golden.wav'):
    write_wav(tmp, pcm, framerate, channels)
    s = refwav.WavStream(tmp, sample_rate=sample_rate, sample_type=sample_type)
    os.remove(tmp)
    return s


def gen_loader():
    """Loader golden: PCM in -> reference WavStream.data out, several rate/channel combinations."""
    cases = {}
    inputs = golden_inputs.loader_inputs()
    specs = golden_inputs.LOADER_SPECS
    for name, fr, ch, secs, sr in specs:
        frames = int(round(secs * fr))
        # the reference reads UNINITIALISED memory (np.empty, wav.py:119) when
        # ceil(total_seconds*sample_rate) exceeds the samples its chunk loop writes (float error in
        # wav.py:113-116); golden cases are chosen gap-free so that they are well defined
        import math
        written = sum(int(round(min(fr, frames - a) * (sr / float(fr)))) for a in range(0, frames, fr))
        assert written == math.ceil(frames / float(fr) * sr), (name, written)
        pcm = inputs[name + '_pcm']
        for st in ('uint8', 'float32'):
            s = ref_load(pcm, fr, ch, sr, st)
            cases['{0}_{1}_data'.format(name, st)] = s.data
            cases['{0}_{1}_meta'.format(name, st)] = np.array([s.sample_rate, s.sample_count, s.padding_size], np.int64)
        cases['{0}_pcm_crc'.format(name)] = golden_inputs.crc(pcm)
        cases['{0}_spec'.format(name)] = np.array([fr, ch, sr], np.int64)
    np.savez_compressed(os.path.join(OUT, 'loader.npz'), **cases)
    print('loader.npz:', len(specs), 'cases')


def gen_loader24():
    """24-bit PCM through the reference's own readframes branch (wav.py:71-74: the top 16 bits of every sample):
    the reference's WavStream.data of the seeded WAV files for both sample types."""
    cases = {}
    inputs = golden_inputs.loader24_inputs()
    for name, *_ in golden_inputs.LOADER24_SPECS:
        tmp = '/tmp/_golden24.wav'
        open(tmp, 'wb').write(inputs[name + '_wav'].tobytes())
        cases[name + '_wav_crc'] = golden_inputs.crc(inputs[name + '_wav'])
        for st in ('uint8', 'float32'):
            s = refwav.WavStream(tmp, sample_rate=12000, sample_type=st)
            cases['{0}_{1}_data'.format(name, st)] = s.data
            cases['{0}_{1}_meta'.format(name, st)] = np.array([s.sample_rate, s.sample_count, s.padding_size], np.int64)
        os.remove(tmp)
    np.savez_compressed(os.path.join(OUT, 'loader24.npz'), **cases)
    print('loader24.npz:', len(golden_inputs.LOADER24_SPECS), 'cases')


def gen_matcher():
    """Matcher golden: reference find_substream outputs on reference-loaded streams."""
    inputs = golden_inputs.matcher_inputs()
    src_pcm, dst_pcm = inputs['src_pcm'], inputs['dst_pcm']
    out = {'src_pcm_crc': golden_inputs.crc(src_pcm), 'dst_pcm_crc': golden_inputs.crc(dst_pcm)}
    # (start, end, center, window) -- centre given as absolute time, like sushi.py:432,450-452
    queries = [
        (2.00, 4.50, 3.50, 1.5),      # small-window fast path (sushi.py:432)
        (2.00, 4.50, 2.00, 10.0),     # window clipped at -PADDING (wav.py:178)
        (6.10, 7.05, 7.60, 10.0),
        (6.10, 6.575, 7.60, 10.0),    # left half (sushi.py:445,451)
        (6.575, 7.05, 8.075, 10.0),   # right half with offset (sushi.py:452)
        (10.0, 13.7, 11.5, 30.0),     # max_window, clipped both sides
        (18.0, 21.0, 19.5, 10.0),     # window reaches past the end (wav.py:179)
        (20.5, 23.9, 22.0, 1.5),      # pattern runs into the tail padding
        (0.00, 0.60, 1.50, 5.0),      # pattern at the very start
        (12.0, 12.04, 13.5, 2.0),     # very short pattern (480 samples)
        (3.0, 15.0, 4.5, 10.0),       # 12 s pattern
        (23.0, 24.0, 40.0, 10.0),     # centre far beyond the end: start clipped to duration
    ]
    out['queries'] = np.array(queries, np.float64)
    for st in ('uint8', 'float32'):
        src = ref_load(src_pcm, 12000, 1, 12000, st)
        dst = ref_load(dst_pcm, 12000, 1, 12000, st)
        out['src_{0}_crc'.format(st)] = np.array([zlib.crc32(src.data.tobytes())], np.int64)
        out['dst_{0}_crc'.format(st)] = np.array([zlib.crc32(dst.data.tobytes())], np.int64)
        diffs, times = [], []
        for (a, b, c, w) in queries:
            pat = src.get_substream(a, b)
            d, t = dst.find_substream(pat, c, w)
            assert isinstance(d, np.float32)
            diffs.append(d)
            times.append(t)
        out['diff_{0}'.format(st)] = np.array(diffs, np.float32)
        out['time_{0}'.format(st)] = np.array(times, np.float64)
        # two whole curves (cv2 output of the same call, wav.py:185)
        import cv2
        for qi, stride in ((0, 1), (2, 7)):           # second curve kept every 7th lag to stay small
            a, b, c, w = queries[qi]
            pat = src.get_substream(a, b)
            st_t = refwav.clip(c - w, -dst.PADDING_SECONDS, dst.duration_seconds)
            en_t = refwav.clip(c + w, 0, dst.duration_seconds + dst.PADDING_SECONDS)
            s0 = dst._get_sample_for_time(st_t)
            s1 = dst._get_sample_for_time(en_t) + len(pat[0])
            out['curve{0}_{1}'.format(qi, st)] = cv2.matchTemplate(dst.data[:, s0:s1], pat, cv2.TM_SQDIFF_NORMED)[0][::stride]
            out['curve{0}_{1}_s0'.format(qi, st)] = np.array([s0, s1, stride], np.int64)
        out['meta_{0}'.format(st)] = np.array([dst.sample_rate, dst.sample_count, dst.padding_size], np.int64)
    # degenerate inputs straight through cv2 the way find_substream would see them (SURVEY appendix A)
    import cv2
    z = np.zeros((1, 64), np.uint8)
    seven = np.full((1, 8), 7, np.uint8)
    nine = np.full((1, 64), 9, np.uint8)
    ramp = (np.arange(64) % 8).astype(np.uint8)[None, :]
    out['deg_zero_window'] = cv2.matchTemplate(z, seven, cv2.TM_SQDIFF_NORMED)[0]
    out['deg_zero_template'] = cv2.matchTemplate(nine, z[:, :8], cv2.TM_SQDIFF_NORMED)[0]
    out['deg_const_7_vs_9'] = cv2.matchTemplate(nine, seven, cv2.TM_SQDIFF_NORMED)[0]
    out['deg_periodic'] = cv2.matchTemplate(ramp, ramp[:, :16], cv2.TM_SQDIFF_NORMED)[0]
    np.savez_compressed(os.path.join(OUT, 'matcher.npz'), **out)
    print('matcher.npz:', len(queries), 'queries x 2 sample types')


class _Event(refsubs.ScriptEventBase):
    is_comment = False


def gen_shifts():
    """calculate_shifts golden: the (transformed) reference state machine on reference streams."""
    sushi = load_reference_sushi()
    import logging
    logging.disable(logging.CRITICAL)
    out = {}
    scenarios = {
        # constant shift: fast path only (BASELINE config 1 in miniature)
        'const': dict(dur=40.0, seed=21, shift=1.5, count=14, window=10, max_window=30),
        # shift jumps at t=30: uncommitted states, triple check, back-fill (sushi.py:445-493)
        'jump': dict(dur=60.0, seed=22, shift=[(0.0, 0.75), (30.0, -2.5)], count=22, window=10, max_window=30),
        # jump larger than the normal window: rewind to max_window (sushi.py:473-478)
        'rewind': dict(dur=70.0, seed=23, shift=[(0.0, 0.3), (28.0, 14.0)], count=26, window=10, max_window=30),
    }
    for name, sc in scenarios.items():
        src_pcm, dst_pcm = synth.make_pair(sc['dur'], sc['seed'], sc['shift'])
        starts, ends = synth.make_events(sc['count'], sc['dur'] - 16.0, sc['seed'], 0.8, 2.6, 1.0)
        # inputs are regenerated from the seed by the tests; the CRCs catch generator drift
        out[name + '_pcm_crc'] = np.array([zlib.crc32(src_pcm.tobytes()), zlib.crc32(dst_pcm.tobytes())], np.int64)
        out[name + '_gen'] = np.array([sc['dur'], sc['seed'], sc['count']], np.float64)
        out[name + '_shift'] = np.array(sc['shift'] if not np.isscalar(sc['shift']) else [(0.0, sc['shift'])], np.float64)
        out[name + '_events'] = np.stack([starts, ends], 1)
        out[name + '_params'] = np.array([sc['window'], sc['max_window'], 5], np.float64)
        for st in ('uint8', 'float32'):
            src = ref_load(src_pcm, 12000, 1, 12000, st)
            dst = ref_load(dst_pcm, 12000, 1, 12000, st)
            events = [_Event(i, float(a), float(b), '') for i, (a, b) in enumerate(zip(starts, ends))]
            calls = []
            orig = dst.find_substream

            def traced(pattern, center, window, _orig=orig, _calls=calls, _src=src):
                d, t = _orig(pattern, center, window)
                off = (pattern.__array_interface__['data'][0] - _src.data.__array_interface__['data'][0]) // _src.data.itemsize
                _calls.append((off, len(pattern[0]), center, window, float(d), t))
                return d, t
            dst.find_substream = traced
            groups = sushi.prepare_search_groups(events, src.duration_seconds, [], 0.417, 0.417)
            sushi.calculate_shifts(src, dst, groups, sc['window'], sc['max_window'], 5)
            res = np.array([[e.shift, e.diff, (e._linked_event.source_index if e.linked else -1)] for e in events], np.float64)
            out['{0}_{1}_result'.format(name, st)] = res
            out['{0}_{1}_calls'.format(name, st)] = np.array(calls, np.float64)
            out['{0}_{1}_groups'.format(name, st)] = np.array([[g[0].source_index, g[-1].source_index] for g in groups], np.int64)
            print(name, st, 'groups', len(groups), 'calls', len(calls), 'shifts', np.unique(np.round(res[:, 0], 2)))
    np.savez_compressed(os.path.join(OUT, 'shifts.npz'), **out)


if __name__ == '__main__':
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[2:] or ['loader', 'loader24', 'matcher', 'shifts']
    if 'loader' in which:
        gen_loader()
    if 'loader24' in which:
        gen_loader24()
    if 'matcher' in which:
        gen_matcher()
    if 'shifts' in which:
        gen_shifts()

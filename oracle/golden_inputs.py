"""Seeded inputs of the golden cases in tests/golden/ -- TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

loader.npz, loader24.npz and matcher.npz hold what the reference computed and a CRC-32 of every input it was
given.  The inputs themselves (PCM, 24-bit WAV files) are most of the bytes and derive from fixed seeds, so they
are regenerated here; load() checks each against its CRC before a test sees it, so a generator that no longer
reproduces them fails loudly instead of comparing the reference's outputs with the wrong inputs.
"""
import io
import wave
import zlib

import numpy as np

from sushi_b200 import synth

# name, framerate, channels, seconds, sample_rate
LOADER_SPECS = [
    ('mono12k', 12000, 1, 2.5, 12000),
    ('stereo48k', 48000, 2, 1.25, 12000),
    ('mono44k1', 44100, 1, 2.0, 12000),
    ('stereo22k05', 22050, 2, 2.0, 12000),
    ('mono8k_up', 8000, 1, 1.5, 12000),
    ('six48k', 48000, 6, 0.6, 12000),
]
# name, framerate, channels, seconds (sample_rate 12000)
LOADER24_SPECS = [('stereo48k_24', 48000, 2, 1.25), ('mono44k1_24', 44100, 1, 2.0), ('six48k_24', 48000, 6, 0.6)]


def matcher_inputs():
    src_pcm, dst_pcm = synth.make_pair(24.0, 3, 1.5)
    return {'src_pcm': src_pcm, 'dst_pcm': dst_pcm}


def loader_inputs():
    """{name}_pcm: int16 (frames, channels) per LOADER_SPECS case."""
    rng = np.random.default_rng(11)
    out = {}
    for i, (name, fr, ch, secs, sr) in enumerate(LOADER_SPECS):
        frames = int(round(secs * fr))
        base = synth.programme_audio(frames, 100 + 6 * i, rate=fr)
        pcm = np.empty((frames, ch), np.int16)
        for c in range(ch):
            pcm[:, c] = np.clip(base.astype(np.int32) * (c + 2) // (ch + 1) + rng.integers(-300, 300, frames), -32768, 32767)
        out[name + '_pcm'] = pcm
    return out


def wav24_bytes(values, framerate, channels):
    """values: int array (frames, channels) of signed 24-bit samples -> RIFF/WAVE PCM file with 3-byte samples."""
    v = np.ascontiguousarray(values, np.int64) & 0xFFFFFF
    raw = np.empty(v.shape + (3,), np.uint8)
    raw[..., 0], raw[..., 1], raw[..., 2] = v & 0xFF, (v >> 8) & 0xFF, (v >> 16) & 0xFF
    f = io.BytesIO()
    with wave.open(f, 'wb') as w:
        w.setnchannels(channels)
        w.setsampwidth(3)
        w.setframerate(framerate)
        w.writeframes(raw.tobytes())
    return f.getvalue()


def loader24_inputs():
    """{name}_wav: uint8 bytes of a 24-bit WAV file per LOADER24_SPECS case."""
    rng = np.random.default_rng(24)
    out = {}
    for i, (name, fr, ch, secs) in enumerate(LOADER24_SPECS):
        frames = int(round(secs * fr))
        base = synth.programme_audio(frames, 240 + 5 * i, rate=fr).astype(np.int64)
        vals = np.empty((frames, ch), np.int64)
        for c in range(ch):
            vals[:, c] = np.clip(base * 256 * (c + 2) // (ch + 1) + rng.integers(-70000, 70000, frames), -2 ** 23, 2 ** 23 - 1)
        out[name + '_wav'] = np.frombuffer(wav24_bytes(vals, fr, ch), np.uint8)
    return out


INPUTS = {'loader': loader_inputs, 'loader24': loader24_inputs, 'matcher': matcher_inputs}


def crc(a):
    return np.array([zlib.crc32(np.ascontiguousarray(a).tobytes())], np.int64)


def load(path, kind):
    """The arrays of a golden file, with the seeded inputs of `kind` (a key of INPUTS) added after their CRC check."""
    with np.load(path) as z:
        g = {k: z[k] for k in z.files}
    for key, value in INPUTS[kind]().items():
        assert int(crc(value)[0]) == int(g[key + '_crc'][0]), \
            '%s: the seeded generator no longer reproduces the input the golden outputs were computed from' % key
        g[key] = value
    return g

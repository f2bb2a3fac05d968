"""Deterministic synthetic QRSS / DFCW test streams (SURVEY.md section 8d).

Host-generated so the CPU oracle and the GPU see identical samples: a sum of weak
steady carriers, a QRSS-keyed carrier and a DFCW pair over Gaussian noise, quantised to
int16 and converted exactly as the reference's WAV reader does (`(float)s / 32768`,
wav_fmt.c:113).  Keying follows the reference transmitter's timing rules (dot = dot_time,
dash = 3 dots, element gap = 1 dot, character gap: qrs.c:467-486,510-557; DFCW dot/dash
tones 800/810 Hz: glfer.c:261-262)."""
from __future__ import annotations

import numpy as np

_MORSE = {"G": "--.", "L": ".-..", "F": "..-.", "E": ".", "R": ".-.", " ": " "}


def _keying(message: str, nsamp: int, fs: int, dot_s: float) -> tuple[np.ndarray, np.ndarray]:
    """on/off gate for QRSS and a dot(0)/dash(1) selector for DFCW, one value per sample."""
    gate = []
    sel = []
    for ch in message:
        if ch == " ":
            gate += [0] * 4
            sel += [0] * 4
            continue
        for el in _MORSE[ch]:
            k = 1 if el == "." else 3
            gate += [1] * k + [0]
            sel += [0 if el == "." else 1] * (k + 1)
        gate += [0] * 2
        sel += [0] * 2
    gate = np.array(gate, dtype=np.float32)
    sel = np.array(sel, dtype=np.float32)
    dot_n = max(1, int(dot_s * fs))
    reps = int(np.ceil(nsamp / (len(gate) * dot_n)))
    g = np.tile(np.repeat(gate, dot_n), reps)[:nsamp]
    s = np.tile(np.repeat(sel, dot_n), reps)[:nsamp]
    return g, s


def qrss_stream_int16(nsamples: int, fs: int = 48000, seed: int = 0x5EED, dot_s: float = 3.0,
                      noise_sigma: float = 0.03) -> np.ndarray:
    rng = np.random.Generator(np.random.Philox(seed))
    t = np.arange(nsamples, dtype=np.float64) / fs
    x = noise_sigma * rng.standard_normal(nsamples)
    gate, sel = _keying("GLFER ", nsamples, fs, dot_s)
    # QRSS carrier (on/off keyed), scaled to the band so small sample rates keep it in band
    f0 = 800.0 if fs >= 4000 else fs * 0.1
    x += 0.02 * gate * np.sin(2 * np.pi * f0 * t + 0.3)
    # DFCW pair: dot tone f0+100, dash tone f0+110 (10 Hz shift as glfer.c:261-262)
    fd = f0 + 100.0 + 10.0 * sel
    x += 0.01 * np.sin(2 * np.pi * np.cumsum(fd) / fs + 1.1)
    # steady weak carriers
    for fc, amp, ph in ((f0 * 0.5, 0.003, 0.0), (f0 * 1.3, 0.01, 0.7), (f0 * 1.45, 0.03, 2.1)):
        x += amp * np.sin(2 * np.pi * fc * t + ph)
    x += 0.002  # small DC offset so mean removal has something to do
    return np.clip(np.rint(x * 32768.0), -32768, 32767).astype(np.int16)


def pcm16_to_float(pcm: np.ndarray) -> np.ndarray:
    """wav_fmt.c:113: buff[i] = (float) buf16[i] / 32768"""
    return pcm.astype(np.float32) / np.float32(32768)


def qrss_stream(nsamples: int, fs: int = 48000, seed: int = 0x5EED, dot_s: float = 3.0,
                noise_sigma: float = 0.03) -> np.ndarray:
    return pcm16_to_float(qrss_stream_int16(nsamples, fs, seed, dot_s, noise_sigma))


def tiled_stream(nsamples: int, fs: int = 48000, block_s: float = 60.0, seed: int = 0x5EED) -> np.ndarray:
    """A long stream for timing: one generated block of block_s seconds tiled to length
    (the bench says so in its `data` field)."""
    nb = int(block_s * fs)
    blk = qrss_stream(min(nb, nsamples), fs, seed, dot_s=1.0)
    reps = -(-nsamples // len(blk))
    return np.tile(blk, reps)[:nsamples]


def iq_stream_int16(nsamples: int, fs: int = 48000, seed: int = 0x5EED, dot_s: float = 3.0,
                    noise_sigma: float = 0.03) -> np.ndarray:
    """A complex (I/Q) QRSS-like recording centred on the dial frequency, [nsamples, 2] int16 (I, Q): a keyed QRSS
    carrier at -300 Hz below the dial, a DFCW pair at +400 / +410 Hz above it, steady weak carriers on both sides
    (-1000, +150, +1200 Hz), a small LO-leakage offset at DC and complex Gaussian noise.  Offsets scale with fs
    below 4 kHz so the tones stay in band."""
    rng = np.random.Generator(np.random.Philox(seed))
    t = np.arange(nsamples, dtype=np.float64) / fs
    sc = 1.0 if fs >= 4000 else fs / 4000.0
    z = noise_sigma / np.sqrt(2.0) * (rng.standard_normal(nsamples) + 1j * rng.standard_normal(nsamples))
    gate, sel = _keying("GLFER ", nsamples, fs, dot_s)
    z += 0.02 * gate * np.exp(1j * (2 * np.pi * (-300.0 * sc) * t + 0.3))
    fd = (400.0 + 10.0 * sel) * sc
    z += 0.01 * np.exp(1j * (2 * np.pi * np.cumsum(fd) / fs + 1.1))
    for fc, amp, ph in ((-1000.0, 0.003, 0.0), (150.0, 0.01, 0.7), (1200.0, 0.03, 2.1)):
        z += amp * np.exp(1j * (2 * np.pi * fc * sc * t + ph))
    z += 0.002 - 0.001j
    pcm = np.stack([z.real, z.imag], axis=1)
    return np.clip(np.rint(pcm * 32768.0), -32768, 32767).astype(np.int16)


def iq_stream(nsamples: int, fs: int = 48000, seed: int = 0x5EED, dot_s: float = 3.0,
              noise_sigma: float = 0.03) -> np.ndarray:
    """iq_stream_int16 as complex64 [nsamples] (I + iQ, each (float) s / 32768)"""
    pcm = pcm16_to_float(iq_stream_int16(nsamples, fs, seed, dot_s, noise_sigma))
    return np.ascontiguousarray(pcm).view(np.complex64)[:, 0]


def write_wav16(path: str, pcm: np.ndarray, fs: int, channels: int = 1) -> None:
    """Canonical 44-byte-header 16-bit PCM WAV (the layout wav_fmt.h:34-52 describes); pcm is the interleaved
    sample stream ([frames][channels] flattened)."""
    import struct
    data = pcm.astype("<i2").tobytes()
    with open(path, "wb") as fh:
        fh.write(b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVE")
        fh.write(b"fmt " + struct.pack("<IHHIIHH", 16, 1, channels, fs, fs * 2 * channels, 2 * channels, 16))
        fh.write(b"data" + struct.pack("<I", len(data)))
        fh.write(data)

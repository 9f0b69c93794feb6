"""Synthetic IQ captures for the PMR446 receive chain (SURVEY.md §8d "concrete synthetic inputs").

The reference has no recorded captures or fixtures (SURVEY.md §4), so tests and the benchmark
use seeded synthetic captures: narrow-band FM carriers on the 12.5 kHz PMR446 grid
(/root/reference/src/sdr_pmr446.c:22-28) with an audio tone plus a CTCSS sub-tone
(tone table :138-141), complex AWGN and a DC offset, quantised to RTL-SDR style cu8 with the
inverse of the SoapyRTLSDR conversion (u8 - 127.4)/128, or to signed cs16 / cs8 (x 32768 / x 128).

All phases are closed-form in the absolute sample index, so a capture generated in pieces
(`start=`) is identical to one generated in one go (noise aside, which is drawn per call).
"""
from dataclasses import dataclass, field, replace
from typing import Sequence

import numpy as np

CHANNEL_WIDTH_HZ = 12500.0


@dataclass
class Carrier:
    channel: int            # 1-based PMR channel number (1..M)
    amplitude: float
    audio_hz: float
    ctcss_hz: float
    audio_dev_hz: float = 2500.0
    ctcss_dev_hz: float = 500.0
    phase0: float = 0.0
    t_on: float = 0.0       # the carrier is keyed on during [t_on, t_off) seconds (squelch / selector tests)
    t_off: float = float("inf")


@dataclass
class CaptureSpec:
    fs: float = 1024000.0
    num_channels: int = 16
    carriers: Sequence[Carrier] = field(default_factory=lambda: CFG1_CARRIERS)
    noise_sigma: float = 0.01
    dc: complex = 0.02 - 0.015j
    offset_hz: float = 0.0   # extra frequency offset applied to every carrier (dsd_in: single carrier at 0 Hz)


CFG1_CARRIERS = (
    Carrier(2, 0.20, 1000.0, 67.0),
    Carrier(7, 0.10, 600.0, 88.5),
    Carrier(8, 0.15, 1700.0, 123.0),
    Carrier(15, 0.05, 2400.0, 250.3),
)


def rotated_carriers(stream_id: int, num_channels: int = 16, base=CFG1_CARRIERS):
    """cfg3/cfg5: channel set rotated by stream_id mod M."""
    r = stream_id % num_channels
    return tuple(replace(c, channel=((c.channel - 1 + r) % num_channels) + 1) for c in base)


def channel_offset_hz(channel_1based: int, num_channels: int = 16) -> float:
    """Baseband centre of a PMR channel when the SDR is tuned to the band centre (:28)."""
    return (channel_1based - (num_channels + 1) / 2.0) * CHANNEL_WIDTH_HZ


def make_cf64(spec: CaptureSpec, n: int, seed: int = 446, start: int = 0) -> np.ndarray:
    """Complex baseband capture (float64 complex), before quantisation."""
    t = (np.arange(n, dtype=np.float64) + float(start)) / spec.fs
    x = np.zeros(n, dtype=np.complex128)
    for c in spec.carriers:
        f0 = channel_offset_hz(c.channel, spec.num_channels) + spec.offset_hz
        ph = 2.0 * np.pi * f0 * t + c.phase0
        if c.audio_hz > 0:
            ph -= (c.audio_dev_hz / c.audio_hz) * np.cos(2.0 * np.pi * c.audio_hz * t)
        if c.ctcss_hz > 0:
            ph -= (c.ctcss_dev_hz / c.ctcss_hz) * np.cos(2.0 * np.pi * c.ctcss_hz * t)
        keyed = c.amplitude * np.exp(1j * ph)
        if c.t_on > 0.0 or c.t_off != float("inf"):
            keyed = np.where((t >= c.t_on) & (t < c.t_off), keyed, 0.0)
        x += keyed
    if spec.noise_sigma > 0:
        rng = np.random.Generator(np.random.PCG64(seed))
        x += spec.noise_sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    x += spec.dc
    return x


def to_cu8(x: np.ndarray) -> np.ndarray:
    """Interleaved I,Q uint8: u8 = clip(round(127.4 + 128 x), 0, 255)."""
    out = np.empty(2 * x.shape[0], dtype=np.uint8)
    out[0::2] = np.clip(np.rint(127.4 + 128.0 * x.real), 0, 255).astype(np.uint8)
    out[1::2] = np.clip(np.rint(127.4 + 128.0 * x.imag), 0, 255).astype(np.uint8)
    return out


def make_cu8(spec: CaptureSpec, n: int, seed: int = 446, start: int = 0) -> np.ndarray:
    return to_cu8(make_cf64(spec, n, seed, start))


def _to_signed(x: np.ndarray, bits: int, dtype) -> np.ndarray:
    full = float(1 << (bits - 1))
    out = np.empty(2 * x.shape[0], dtype=dtype)
    out[0::2] = np.clip(np.rint(full * x.real), -full, full - 1).astype(dtype)
    out[1::2] = np.clip(np.rint(full * x.imag), -full, full - 1).astype(dtype)
    return out


def to_cs16(x: np.ndarray) -> np.ndarray:
    """Interleaved I,Q int16 (Airspy, SDRplay, LimeSDR, USRP, PlutoSDR): clip(round(32768 x), -32768, 32767)."""
    return _to_signed(x, 16, np.int16)


def to_cs8(x: np.ndarray) -> np.ndarray:
    """Interleaved I,Q int8 (HackRF): clip(round(128 x), -128, 127)."""
    return _to_signed(x, 8, np.int8)


def make_cf32(spec: CaptureSpec, n: int, seed: int = 446, start: int = 0) -> np.ndarray:
    return make_cf64(spec, n, seed, start).astype(np.complex64)


def make_cs16(spec: CaptureSpec, n: int, seed: int = 446, start: int = 0) -> np.ndarray:
    return to_cs16(make_cf64(spec, n, seed, start))


def make_cs8(spec: CaptureSpec, n: int, seed: int = 446, start: int = 0) -> np.ndarray:
    return to_cs8(make_cf64(spec, n, seed, start))


def cfg1_capture(n: int = 10_240_000, fs: float = 1024000.0, seed: int = 446, stream_id: int = 0) -> np.ndarray:
    """BASELINE cfg1/cfg3 capture as cu8: four FM carriers (+CTCSS) at PMR channels {2,7,8,15}, rotated by stream."""
    spec = CaptureSpec(fs=fs, carriers=rotated_carriers(stream_id))
    return make_cu8(spec, n, seed + stream_id)


def cfg2_capture(n: int = 24_000_000, fs: float = 2400000.0, seed: int = 446) -> np.ndarray:
    """BASELINE cfg2 capture as cu8: one FM carrier at 0 Hz offset with a 1 kHz tone, +-2.5 kHz deviation."""
    spec = CaptureSpec(fs=fs, carriers=(Carrier(1, 0.3, 1000.0, 0.0),), offset_hz=-channel_offset_hz(1))
    return make_cu8(spec, n, seed)

"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the per-frame radio metrics (include/snoutrx.h snrx_frame_rf_t).

Evaluated the slow, obvious way: wideband channel samples from the channelizer's direct form (oracle.pfb, pfb_oracle_direct),
narrow-band ones straight from the input, reference phase increments from the modulators of snout_b200.synth."""
from __future__ import annotations

import math

import numpy as np

from snout_b200 import _abi, chanplan, synth

from . import pfb

FS = 4.0e6
BLE_REF_ORIGIN = -39            # first sample of the reference GFSK burst relative to sample_index
RF_POWER, RF_NOISE, RF_CFO = 1, 2, 4


def windows(proto: int, s: int):
    """((signal a, b), (noise a, b)), half-open, capture-relative channel indices."""
    if proto == _abi.PROTO_BLE:
        return (s - 24, s + 120), (s - 104, s - 40)
    return (s - 392, s - 136), (s - 720, s - 656)


def ble_known_bits(aa: int) -> np.ndarray:
    pre = 0x55 if aa & 1 else 0xAA
    return synth.bytes_to_bits_lsb(bytes([pre]) + int(aa).to_bytes(4, "little"))


def ble_theta0(aa: int) -> float:
    """arg sum exp(j dtheta_ref[m]) over the BLE signal window: the GFSK burst of the 40 known bits, first sample at s - 39."""
    w = synth.gfsk_modulate(ble_known_bits(aa))
    d = np.angle(w[1:] * np.conj(w[:-1]))            # d[i - 1] = increment into burst sample i
    i = np.arange(-24 - BLE_REF_ORIGIN, 120 - BLE_REF_ORIGIN)
    return float(np.angle(np.exp(1j * d[i - 1]).sum()))


def zb_theta0() -> float:
    """The same over whole periods of the 802.15.4 preamble (periodic in 64 samples): a constant."""
    w = synth.oqpsk_modulate(bytes([0, 0, 0, 0, 0xA7, 0]))
    d = np.angle(w[1:] * np.conj(w[:-1]))
    return float(np.angle(np.exp(1j * d[127:127 + 256]).sum()))   # samples 128 .. 383: inside the 512-sample preamble


def channel_bin(proto: int, channel: int) -> int:
    return chanplan.ble_channel_bin(channel) if proto == _abi.PROTO_BLE else chanplan.zigbee_channel_bin(channel)


def channel_samples(x: np.ndarray, m0: int, m1: int, proto: int, channel: int, taps=None) -> np.ndarray:
    """y[m0:m1] (buffer-local) of one capture: the channelizer's direct form for the frame's bin when `taps` is given
    (wideband), else the input itself."""
    if taps is None:
        return np.asarray(x[m0:m1], dtype=np.complex128)
    return pfb(x, taps, [channel_bin(proto, channel)], m0, m1)[0].astype(np.complex128)


def db(mean_power: float) -> float:
    return -200.0 if mean_power < 1e-20 else 10.0 * math.log10(mean_power)


def wrap(a: float) -> float:
    return (a + math.pi) % (2 * math.pi) - math.pi


def frame_rf(x, frames, taps_ble=None, taps_zb=None, origin: int = 0, first_capture: int = 0) -> np.ndarray:
    """Metrics of every record.  x: [captures, n] or [n] input (cf32 values; sc8 as q / 128); taps_*: the prototypes in
    wideband modes (None: narrow band); origin: capture-relative channel index of buffer sample 0."""
    x = np.atleast_2d(np.asarray(x))
    wb = taps_ble is not None or taps_zb is not None
    n_out = x.shape[1] // (chanplan.WB_DECIM if wb else 1)
    out = np.zeros(len(frames), dtype=_abi.RF_DTYPE)
    th_zb = zb_theta0()
    for i, f in enumerate(frames):
        proto, s, ch = int(f["proto"]), int(f["sample_index"]), int(f["channel"])
        r = out[i]
        for k in ("sample_index", "capture_id", "channel", "proto"):
            r[k] = f[k]
        r["frame"] = i
        xc = x[int(f["capture_id"]) - first_capture]
        taps = (taps_ble if proto == _abi.PROTO_BLE else taps_zb) if wb else None
        (sa, sb), (na, nb) = windows(proto, s)
        sig_ok = sa - 1 >= 0 and sa - 1 - origin >= 0 and sb - origin <= n_out
        noise_ok = na >= 0 and na - origin >= 0 and nb - origin <= n_out
        nan = float("nan")
        r["power_dbfs"] = r["noise_dbfs"] = r["snr_db"] = r["cfo_hz"] = nan
        if sig_ok:
            y = channel_samples(xc, sa - 1 - origin, sb - origin, proto, ch, taps)
            r["power_dbfs"] = db(float(np.mean(np.abs(y[1:]) ** 2)))
            theta0 = ble_theta0(int(f["access_addr"])) if proto == _abi.PROTO_BLE else th_zb
            lag = np.sum(y[1:] * np.conj(y[:-1]))
            r["cfo_hz"] = FS / (2 * math.pi) * wrap(math.atan2(lag.imag, lag.real) - theta0)
        if noise_ok:
            y = channel_samples(xc, na - origin, nb - origin, proto, ch, taps)
            r["noise_dbfs"] = db(float(np.mean(np.abs(y) ** 2)))
        if sig_ok and noise_ok:
            r["snr_db"] = float(r["power_dbfs"]) - float(r["noise_dbfs"])
        r["valid"] = (RF_POWER | RF_CFO if sig_ok else 0) | (RF_NOISE if noise_ok else 0)
    return out

"""The two rules every check of the BLE front end states its expectation with (DESIGN.md 4: the link between the channel
streams of S1 and the quantised streams S2 is stated on).

* Quantiser: q8 = clamp(rint(y * S), -128, 127), ties to even.  The wideband kernel evaluates it as one FFMA.SAT and one
  rounding add (csrc/pfb.cuh quant_pair), whose extra roundings may move a value that lies within EDGE of a step boundary
  k + 1/2; everywhere else the result is exact.
* Slicer: bit n of a channel's stream is I[n] Q[n+1] - I[n+1] Q[n] > 0 on q8, with the successor of the last sample 0;
  the stream is kBitsLeadWords zero words, the decisions (bit n & 31 of word n >> 5), then zero words up to
  kBitsTailWords past the capture (csrc/common.cuh BitsLayout)."""
import numpy as np

EDGE = 1e-4              # of a quantiser step
LEAD_WORDS, TAIL_WORDS = 4, 64


def quantize(v):
    return np.clip(np.rint(v), -128, 127)


def _components(y):
    y = np.asarray(y)
    return np.stack([y.real, y.imag], -1).astype(np.float64)


def _tie_distance(v):
    return np.abs(v - np.floor(v) - 0.5)


def check_q8(q8, y, yd, scale, what="", max_excluded=0.005):
    """q8 [..., n, 2] int8 against the engine's own channel streams y and the float64 definition yd ([..., n] complex).
    Returns the share of components excluded from the comparison against yd and the mean of q8 - clamp(rint(yd S));
    the mean is held to 1e-3 (no constant bias) where there are enough components for it to say so."""
    q = np.asarray(q8).astype(np.int64)
    v = _components(y) * scale
    bad = (_tie_distance(v) > EDGE) & (q != quantize(v))
    assert not bad.any(), (f"{what}: q8 != clamp(rint(y S)) at {np.argwhere(bad)[:5].tolist()}: "
                           f"{q[bad][:5].tolist()} vs y S = {v[bad][:5].tolist()}")
    vd = _components(yd) * scale
    margin = scale * float(np.abs(np.asarray(y).astype(np.complex128) - yd).max()) + EDGE
    far = _tie_distance(vd) > margin
    excluded = 1.0 - float(far.mean())
    assert excluded < max_excluded or (~far).sum() <= 2, \
        f"{what}: {excluded:.2%} of the components lie within {margin:.2e} of a step boundary"
    qd = quantize(vd)
    bad = far & (q != qd)
    assert not bad.any(), (f"{what}: q8 != clamp(rint(yd S)) at {np.argwhere(bad)[:5].tolist()}: "
                           f"{q[bad][:5].tolist()} vs yd S = {vd[bad][:5].tolist()}")
    bias = float(np.mean(q - qd))
    assert q.size < 100_000 or abs(bias) < 1e-3, f"{what}: mean(q8 - clamp(rint(yd S))) = {bias:.2e}: the quantiser is biased"
    return excluded, bias


def slicer_words(q8):
    """Expected bit stream words [..., LEAD_WORDS + ceil(n / 32) + TAIL_WORDS] (uint32) of q8 [..., n, 2]."""
    q = np.asarray(q8).astype(np.int64)
    i, qq = q[..., 0], q[..., 1]
    pad = np.zeros(i.shape[:-1] + (1,), np.int64)
    i1 = np.concatenate([i[..., 1:], pad], -1)
    q1 = np.concatenate([qq[..., 1:], pad], -1)
    b = (i * q1 - i1 * qq) > 0
    n = b.shape[-1]
    nw = (n + 31) // 32
    full = np.zeros(b.shape[:-1] + ((LEAD_WORDS + nw + TAIL_WORDS) * 32,), bool)
    full[..., LEAD_WORDS * 32: LEAD_WORDS * 32 + n] = b
    return np.packbits(full, axis=-1, bitorder="little").view("<u4")

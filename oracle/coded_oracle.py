"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the BLE Long Range contract (include/snoutrx.h above snrx_ble_coded_t,
DESIGN.md section 4): from a batch's slicer bit words (SNRX_STAGE_BLE_BITS layout) to the list snrx_ble_coded returns, field
for field.

The contract, restated (b[m] = slicer decision of channel sample m; decision m is usable when m + 1 < n_out):
* Encoder (Core Vol 6 Part B 3.3.1): rate 1/2, K = 4, state D1 | D2 << 1 | D3 << 2 (D1 = the most recent input bit),
  a0 = u ^ D1 ^ D2 ^ D3, a1 = u ^ D2 ^ D3, a0 sent first.  Pattern mapper (3.3.2): S=8 maps 0 -> 0011 and 1 -> 1100, S=2 is
  the identity.  Each symbol is 4 channel samples.
* Packet: 80 symbols of preamble, FEC block 1 (S=8, from state 0): AA 32 | CI 2 (LSB first) | TERM1 3 zeros, FEC block 2
  (from state 0, S=8 if CI = 0, S=2 if CI = 1): whitened PDU | CRC-24 | TERM2 3 zeros.
* d(n) = #{j in 0..1023 : b[n + j] != P[j]}, P[j] = c[j >> 2], c = the coded, mapped access address; defined when n + 1023
  is usable.
* Primaries (channels 37..39): d(n) <= T = 400, d(n) < d(m) for m in [n - 16, n), d(n) <= d(m) for m in (n, n + 16]; in a
  shard only n inside the body.
* CI: the v in 0..3 whose pattern on [n + 1024, n + 1184) differs least (lower v on ties); v >= 2 is RESERVED_CI.
* Viterbi from n + 1184, coded bit k on L = 16 (S=8) or 4 (S=2) decisions, branch metric = differing decisions, ties keep
  the predecessor with D3 = 0.  Header run: 40 steps, traced back from the lowest-metric state (lowest index on ties);
  full run: 8 len + 43 steps, traced back from state 0.
* Pointer rounds as oracle/aux_oracle.py, with the window shifted by the preamble lengths (P = 32 at 1M / 2M, 320 Coded),
  Coded targets taking the n of the window with the smallest d(n) <= T (earliest on ties), depth limit 16.
Plain numpy, no engine.
"""
from __future__ import annotations

import numpy as np

from oracle import aux_oracle as ao

ADV_AA = ao.ADV_AA
T = 400
HALF = 16                      # the local-minimum neighbourhood on each side
AA_SAMPLES = 1024              # 256 coded symbols at 4 samples
CI_SAMPLES = 160               # CI + TERM1: 5 bits, 10 coded bits, 16 decisions each
BLOCK2 = AA_SAMPLES + CI_SAMPLES
PREAMBLE = {ao.PHY_1M: 32, ao.PHY_2M: 32, ao.PHY_CODED: 320}
MAX_DEPTH = ao.MAX_DEPTH + 1   # primaries are depth 0, the packet they point at depth 1
INF = 1 << 20                  # path metric of an unreached state
NO_PARENT = 0xFFFFFFFF
OK, NOT_FOUND, OUTSIDE, TRUNCATED, UNSUPPORTED_PHY, BAD_CHANNEL, DEPTH_LIMIT = range(7)
RESERVED_CI = 7
PRIMARY_CHANNELS = (37, 38, 39)

CODED_DTYPE = np.dtype([("sample_index", "<i8"), ("win_lo", "<i8"), ("win_hi", "<i8"), ("capture_id", "<u4"), ("parent", "<u4"),
                        ("first", "<u4"), ("depth", "u1"), ("channel", "u1"), ("phy", "u1"), ("phase", "u1"), ("status", "u1"),
                        ("crc_ok", "u1"), ("len", "<u2"), ("ci", "u1"), ("reserved0", "u1"), ("aa_errors", "<u2"),
                        ("metric", "<u4"), ("bytes", "u1", (ao.MAX_BYTES,)), ("reserved", "u1", (8,))], align=True)
assert CODED_DTYPE.itemsize == 320


# ------------------------------------------------------------------------------------------------ the PHY definitions
def encode(bits, state: int = 0) -> tuple[list[int], int]:
    """Coded bits a0 a1 per input bit, and the final state."""
    out = []
    for u in bits:
        d1, d2, d3 = state & 1, (state >> 1) & 1, (state >> 2) & 1
        out += [u ^ d1 ^ d2 ^ d3, u ^ d2 ^ d3]
        state = ((state << 1) | u) & 7
    return out, state


def map_symbols(coded, s: int) -> np.ndarray:
    coded = np.asarray(coded, dtype=np.uint8)
    if s == 2:
        return coded
    return np.stack([coded, coded, 1 - coded, 1 - coded], axis=1).reshape(-1)      # 0 -> 0011, 1 -> 1100


def samples(symbols) -> np.ndarray:
    return np.repeat(np.asarray(symbols, dtype=np.uint8), 4)


def lsb_bits(value: int, n: int) -> list[int]:
    return [(value >> i) & 1 for i in range(n)]


AA_CODED, AA_STATE = encode(lsb_bits(ADV_AA, 32))
PATTERN = samples(map_symbols(AA_CODED, 8))                      # P[j], j = 0..1023
assert len(PATTERN) == AA_SAMPLES


def ci_pattern(v: int) -> np.ndarray:
    coded, _ = encode(lsb_bits(v, 2) + [0, 0, 0], AA_STATE)
    return samples(map_symbols(coded, 8))


CI_PATTERNS = np.stack([ci_pattern(v) for v in range(4)])


# ------------------------------------------------------------------------------------------------ distance and search
def distances(b: np.ndarray, n_out: int) -> np.ndarray:
    """d(n) for n = 0..n_out - 1, with d = INF where n + 1023 is not usable."""
    from scipy.signal import fftconvolve
    d = np.full(n_out, INF, dtype=np.int64)
    m = n_out - AA_SAMPLES                      # positions 0..m - 1 are defined (n + 1023 <= n_out - 2)
    if m <= 0:
        return d
    x = b[: m + AA_SAMPLES - 1].astype(np.float64)
    cross = np.rint(fftconvolve(x, PATTERN[::-1].astype(np.float64), mode="valid")).astype(np.int64)[:m]
    cs = np.concatenate([[0], np.cumsum(b[: m + AA_SAMPLES - 1], dtype=np.int64)])
    ones = cs[AA_SAMPLES:AA_SAMPLES + m] - cs[:m]
    d[:m] = ones + int(PATTERN.sum()) - 2 * cross
    return d


def primaries(d: np.ndarray, body: tuple[int, int]) -> list[int]:
    out = []
    for n in np.nonzero(d <= T)[0]:
        n = int(n)
        if not body[0] <= n < body[1]:
            continue
        before = d[max(0, n - HALF):n]
        after = d[n + 1:n + 1 + HALF]
        if (before > d[n]).all() and (after >= d[n]).all():
            out.append(n)
    return out


def window_min(d: np.ndarray, lo: int, hi: int) -> int:
    seg = d[lo:hi + 1]
    k = int(np.argmin(seg))
    return lo + k if seg[k] <= T else -1


# ------------------------------------------------------------------------------------------------ decode
def branch_metrics(b: np.ndarray, start: int, n_coded: int, s: int) -> np.ndarray:
    """[k, x]: decisions of coded bit k that differ from its pattern if it were x."""
    L = 16 if s == 8 else 4
    seg = b[start:start + n_coded * L].reshape(n_coded, L).astype(np.int64)
    p0 = samples(map_symbols([0], s))
    bm0 = (seg != p0[None, :]).sum(axis=1)
    return np.stack([bm0, L - bm0], axis=1)


_PRED = [((sp >> 1), (sp >> 1) | 4) for sp in range(8)]
_OUT = [[(((sp & 1) ^ (p & 1) ^ ((p >> 1) & 1) ^ ((p >> 2) & 1)), ((sp & 1) ^ ((p >> 1) & 1) ^ ((p >> 2) & 1))) for p in _PRED[sp]]
        for sp in range(8)]


def viterbi(bm: np.ndarray, steps: int, pm=None, surv=None, t0: int = 0):
    """ACS from step t0 to `steps`; returns (path metrics after the last step, survivors [step][state] = took D3 = 1)."""
    pm = [0] + [INF] * 7 if pm is None else list(pm)
    surv = [] if surv is None else surv
    bml = bm.tolist()
    for t in range(t0, steps):
        A, B = bml[2 * t], bml[2 * t + 1]
        new, sv = [0] * 8, [0] * 8
        for sp in range(8):
            (p0, p1), ((a00, a10), (a01, a11)) = _PRED[sp], _OUT[sp]
            m0 = pm[p0] + A[a00] + B[a10]
            m1 = pm[p1] + A[a01] + B[a11]
            if m1 < m0:
                new[sp], sv[sp] = m1, 1
            else:
                new[sp] = m0
        pm = new
        surv.append(sv)
    return pm, surv


def traceback(surv, steps: int, state: int) -> list[int]:
    bits = [0] * steps
    for t in range(steps - 1, -1, -1):
        bits[t] = state & 1
        state = (state >> 1) | (surv[t][state] << 2)
    return bits


def pack(bits) -> np.ndarray:
    return np.packbits(np.asarray(bits, dtype=np.uint8).reshape(-1, 8), axis=1, bitorder="little").reshape(-1)


def decode(r, b: np.ndarray, n: int, n_out: int) -> None:
    """CI, both Viterbi runs, de-whitening and CRC of the packet whose coded AA starts at local sample n; fills r."""
    last = n_out - 2
    r["status"] = TRUNCATED
    if n + BLOCK2 - 1 > last:
        return
    seg = b[n + AA_SAMPLES:n + BLOCK2]
    ci = int(np.argmin((CI_PATTERNS != seg[None, :]).sum(axis=1)))
    r["ci"] = ci
    if ci >= 2:
        r["status"] = RESERVED_CI
        return
    s = 8 if ci == 0 else 2
    L = 16 if s == 8 else 4
    start = n + BLOCK2
    if start + 80 * L - 1 > last:
        return
    bm = branch_metrics(b, start, 80, s)
    pm, surv = viterbi(bm, 40)
    best = min(range(8), key=lambda q: (pm[q], q))
    hdr = pack(traceback(surv, 40, best)[:16])
    wh = ao.whitening(int(r["channel"]), ao.MAX_BYTES)
    length = int(hdr[1] ^ wh[1])
    N = 8 * length + 43
    if start + 2 * N * L - 1 > last:
        return
    bm = branch_metrics(b, start, 2 * N, s)
    pm, surv = viterbi(bm, N, pm, surv, 40)
    nb = length + 5
    data = pack(traceback(surv, N, 0)[: 8 * nb]) ^ wh[:nb]
    r["status"], r["len"], r["metric"] = OK, nb, pm[0]
    r["bytes"][:nb] = data
    r["crc_ok"] = int(ao.crc24_ok(bytes(data[: nb - 3]), bytes(data[nb - 3:])))


# ------------------------------------------------------------------------------------------------ the list
class _Streams(ao._Streams):
    def __init__(self, words, n_out):
        super().__init__(words, n_out)
        self.dcache = {}

    def d(self, cap: int, ch: int) -> np.ndarray:
        key = (cap, ch)
        if key not in self.dcache:
            self.dcache[key] = distances(self.bits(cap, ch), self.n_out)
        return self.dcache[key]


def _blank(k: int) -> np.void:
    r = np.zeros(1, CODED_DTYPE)[0]
    r["sample_index"], r["first"], r["ci"] = -1, k, 0xFF
    return r


def _found(r, base: int, n: int, d: int) -> None:
    r["sample_index"], r["phase"], r["aa_errors"] = base + n, (base + n) % 4, d


def _pointer(src_at: int, src_phy: int, cap_id: int, parent: int, depth: int, ptr, k: int, geo, streams) -> np.void:
    ch, ca, units, off, phy = ptr
    base, n_out, first_capture = geo
    r = _blank(k)
    lo, hi = ao.window(units, off, ca)
    shift = -PREAMBLE[src_phy] + PREAMBLE.get(phy, 32)
    r["win_lo"], r["win_hi"] = src_at + shift + lo, src_at + shift + hi
    r["capture_id"], r["parent"], r["depth"], r["channel"], r["phy"] = cap_id, parent, depth, ch, phy
    if depth > MAX_DEPTH:
        r["status"] = DEPTH_LIMIT
        return r
    if ch > 36:
        r["status"] = BAD_CHANNEL
        return r
    if phy > ao.PHY_CODED:
        r["status"] = UNSUPPORTED_PHY
        return r
    last = n_out - 2
    l_lo, l_hi = int(r["win_lo"]) - base, int(r["win_hi"]) - base
    span = AA_SAMPLES - 1 if phy == ao.PHY_CODED else 31 * (2 if phy == ao.PHY_2M else 4)
    if l_lo < 0 or l_hi + span > last:
        r["status"] = OUTSIDE
        return r
    b = streams.bits(cap_id - first_capture, ch)
    if phy == ao.PHY_CODED:
        d = streams.d(cap_id - first_capture, ch)
        n = window_min(d, l_lo, l_hi)
        if n < 0:
            r["status"] = NOT_FOUND
            return r
        _found(r, base, n, int(d[n]))
        decode(r, b, n, n_out)
        return r
    # LE 1M / 2M: exactly aux_oracle's search and decode
    a = ao._entry(src_at + shift, cap_id, parent, 0, (ch, ca, units, off, phy), k, geo, streams)
    for f in ("sample_index", "phase", "status", "crc_ok", "len", "bytes"):
        r[f] = a[f]
    return r


def _same(o, r) -> bool:
    return (o["status"] in (OK, TRUNCATED) and o["sample_index"] == r["sample_index"] and o["channel"] == r["channel"]
            and o["capture_id"] == r["capture_id"] and o["phy"] == r["phy"])


def coded_list(words: np.ndarray, n_out: int, first_window: int = 0, pre_out: int = 0, first_capture: int = 0,
               n_windows: int | None = None) -> np.ndarray:
    """The snrx_ble_coded list of a batch.  words: uint32 [captures, 40, words] (SNRX_STAGE_BLE_BITS); n_out: channel samples
    per capture in the buffer; first_window / pre_out / n_windows / first_capture: the shard (defaults: whole captures)."""
    words = np.asarray(words, dtype=np.uint32)
    streams = _Streams(words, n_out)
    base = first_window * 8192 - pre_out
    geo = (base, n_out, first_capture)
    if n_windows is None:
        n_windows = -(-n_out // 8192)
    body = (pre_out, pre_out + n_windows * 8192)
    out: list = []
    for cap in range(words.shape[0]):
        for ch in PRIMARY_CHANNELS:
            d = streams.d(cap, ch)
            for n in primaries(d, body):
                r = _blank(len(out))
                r["win_lo"] = r["win_hi"] = base + n
                r["capture_id"], r["parent"], r["channel"], r["phy"] = first_capture + cap, NO_PARENT, ch, ao.PHY_CODED
                _found(r, base, n, int(d[n]))
                decode(r, streams.bits(cap, ch), n, n_out)
                out.append(r)
    k0, depth = 0, 1
    while depth <= MAX_DEPTH + 1:
        src = [k for k in range(k0, len(out)) if out[k]["status"] == OK and out[k]["crc_ok"] and out[k]["first"] == k
               and out[k]["len"] >= 5]
        k1 = len(out)
        for k in src:
            s = out[k]
            ptr = ao.parse_aux_ptr(bytes(s["bytes"][: int(s["len"])]), int(s["len"]) - 5)
            if ptr is not None:
                out.append(_pointer(int(s["sample_index"]), int(s["phy"]), int(s["capture_id"]), k, depth, ptr, len(out), geo,
                                    streams))
        if len(out) == k1:
            break
        for k in range(k1, len(out)):
            r = out[k]
            if r["status"] in (OK, TRUNCATED):
                for j in range(k):
                    if _same(out[j], r):
                        r["first"] = j
                        break
        k0, depth = k1, depth + 1
    return np.array(out, dtype=CODED_DTYPE) if out else np.zeros(0, CODED_DTYPE)

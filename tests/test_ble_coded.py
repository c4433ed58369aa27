"""BLE Long Range (snrx_ble_coded): the contract's restatement (oracle/coded_oracle.py) on constructed multi-channel bit
streams, the PHY definitions against synth's independent statement, the receive chain's sensitivity through the numpy GFSK
-> AWGN -> int8 -> slicer model, and the host side (messages, lines, pcap, CLI).  No GPU."""
import io
import struct

import numpy as np
import pytest

from fake_engine import RecordingEngine
from oracle import aux_oracle as ao
from oracle import coded_oracle as co
from snout_b200 import _abi, btle_cli, formats, messages, synth
from test_ble_aux import Batch, aux_pdu, aux_symbols, plant_stride


# ------------------------------------------------------------------------------------------------ construction
def coded_decisions(pdu: bytes, channel: int, s: int, ci: int | None = None) -> np.ndarray:
    """Slicer decisions of a noise-free LE Coded packet from its coded AA on (synth's statement, 4 samples per symbol)."""
    return np.repeat(synth.ble_phy_bits_coded(pdu, channel, s, ci=ci)[80:], 4)


def plant(b: np.ndarray, n: int, dec) -> None:
    dec = np.asarray(dec, dtype=np.uint8)
    m = min(len(dec), len(b) - n)
    b[n:n + m] = dec[:m]


def run(bt: Batch, **kw):
    return co.coded_list(bt.words(), bt.n, **kw)


def prim_pdu(rng, ptr: bytes | None = None, extra: int = 0) -> bytes:
    return synth.ext_pdu(synth.ext_header(0, bytes(rng.integers(0, 256, 6, dtype=np.uint8)), 0, int(rng.integers(0, 1 << 16)), ptr),
                         bytes(rng.integers(0, 256, extra, dtype=np.uint8)))


def check(r, channel, pdu, ci=0, crc_ok=True):
    want = pdu + synth.ble_crc24(pdu)
    assert r["status"] == co.OK and r["channel"] == channel and r["ci"] == ci
    assert r["len"] == len(want) and bool(r["crc_ok"]) == crc_ok
    if crc_ok:
        assert bytes(r["bytes"][: len(want)]) == want
    assert not r["bytes"][len(want):].any()


def planted(got, spots):
    """The primaries at the planted positions and every pointed entry.  An S=8 packet's own coded body holds positions with
    d <= T (at coded-bit alignment d has a deviation of 64 there, not 16): those false primaries decode with a failed CRC
    or a reserved CI and start no chain, so the tests look past them."""
    keep = (got["depth"] > 0) | np.isin(got["sample_index"], list(spots))
    return got[keep], np.nonzero(keep)[0]


def packet_end(n: int, length: int, s: int) -> int:
    """The last decision of a packet of `length` payload bytes whose coded AA starts at n."""
    return n + co.BLOCK2 + 2 * (8 * length + 43) * (16 if s == 8 else 4) - 1


# ------------------------------------------------------------------------------------------------ the definitions
def test_encoder_mapper_and_patterns_agree_with_synth():
    rng = np.random.default_rng(0)
    for _ in range(50):
        bits = [int(x) for x in rng.integers(0, 2, 40)]
        assert co.encode(bits)[0] == synth.coded_fec(bits)
    assert list(co.map_symbols([0, 1], 8)) == synth.coded_map([0, 1], 8) == [0, 0, 1, 1, 1, 1, 0, 0]
    assert list(co.map_symbols([0, 1], 2)) == synth.coded_map([0, 1], 2) == [0, 1]
    sym = synth.ble_phy_bits_coded(b"\x07\x00", 37, 8)
    assert list(sym[:80]) == [0, 0, 1, 1, 1, 1, 0, 0] * 10
    assert np.array_equal(np.repeat(sym[80:80 + 256], 4), co.PATTERN)
    for v in range(4):
        dec = np.repeat(synth.ble_phy_bits_coded(b"\x07\x00", 37, 8, ci=v)[80:], 4)
        assert np.array_equal(dec[co.AA_SAMPLES:co.BLOCK2], co.CI_PATTERNS[v])
    # G0 = 1 + x + x^2 + x^3, G1 = 1 + x^2 + x^3: the impulse responses
    assert synth.coded_fec([1, 0, 0, 0]) == [1, 1, 1, 0, 1, 1, 1, 1]
    assert co.encode([1, 0, 0, 0])[0] == [1, 1, 1, 0, 1, 1, 1, 1]


@pytest.mark.parametrize("s", [8, 2])
def test_noise_free_round_trips_every_length(s):
    rng = np.random.default_rng(s)
    step = 4 if s == 8 else 1          # S=8 bodies hold many false primaries (see DESIGN 4), each decoded: every 4th length
    for lo in range(0, 256, 64):
        lengths = list(range(lo, lo + 64, step)) + ([255] if lo == 192 and step > 1 else [])
        ends = [0]
        for ln in lengths:
            ends.append(packet_end(ends[-1] + 300, ln, s) + 40)
        bt = Batch(ends[-1] + 2000, seed=lo + s)
        want = []
        for ln, n0 in zip(lengths, ends[:-1]):
            pdu = bytes([int(rng.integers(0, 256)) & 0xEF, ln]) + bytes(rng.integers(0, 256, ln, dtype=np.uint8))
            plant(bt.b[37], n0 + 300, coded_decisions(pdu, 37, s))
            want.append((n0 + 300, pdu))
        got = run(bt)
        ok = got[(got["status"] == co.OK) & (got["crc_ok"] == 1)]
        assert [int(r["sample_index"]) for r in ok] == [n for n, _ in want]
        for r, (n, pdu) in zip(ok, want):
            check(r, 37, pdu, ci=0 if s == 8 else 1)
            assert r["aa_errors"] == 0 and r["metric"] == 0 and r["phase"] == n % 4 and r["parent"] == co.NO_PARENT


# ------------------------------------------------------------------------------------------------ the threshold and the minimum rule
@pytest.mark.parametrize("extra", [0, 1])
def test_distance_exactly_at_threshold(extra):
    """A clean pattern with T (found) or T + 1 (not found) decisions flipped, on a zero background far from anything."""
    rng = np.random.default_rng(3)
    bt = Batch(8000, seed=3)
    for c in (37, 38, 39):
        bt.b[c] &= 0
    n = 3000
    clean = coded_decisions(prim_pdu(rng), 37, 8)
    for seed in range(200):                                        # flips that leave every neighbour above 401
        dec = clean.copy()
        dec[np.random.default_rng(seed).choice(co.AA_SAMPLES, 400 + extra, replace=False)] ^= 1   # T = 400 (include/snoutrx.h)
        plant(bt.b[37], n, dec)
        d = co.distances(bt.b[37], bt.n)
        if (np.r_[d[n - 16:n], d[n + 1:n + 17]] > 401).all():
            break
    assert d[n] == 400 + extra
    got = run(bt)
    hits = [int(r["sample_index"]) for r in got if r["channel"] == 37]
    assert (n in hits) == (extra == 0)


def tie_stream(seed: int):
    """Two overlapping copies of the pattern at n and n + k whose disagreements are split evenly, so d(n) == d(n + k) <= T;
    (n, k, b) such that d(n) is below every other d in [n - 16, n + 16]."""
    rng = np.random.default_rng(seed)
    P = co.PATTERN
    for k in rng.permutation(np.arange(1, 17)):
        k = int(k)
        n, N = 500, 3000
        b = rng.integers(0, 2, N).astype(np.uint8)
        b[n:n + co.AA_SAMPLES] = P
        b[n + co.AA_SAMPLES:n + co.AA_SAMPLES + k] = P[co.AA_SAMPLES - k:]
        dis = np.nonzero(P[k:] != P[:-k])[0] + k                # offsets from n where the two copies disagree
        if len(dis) % 2:
            continue
        take_b = rng.permutation(dis)[: len(dis) // 2]
        b[n + take_b] = P[take_b - k]
        d = co.distances(b, N)
        if d[n] != d[n + k] or d[n] > co.T:
            continue
        around = np.concatenate([d[n - 16:n], d[n + 1:n + k], d[n + k + 1:n + k + 17]])
        if (around > d[n]).all():
            return n, k, b
    raise AssertionError("no construction")


@pytest.mark.parametrize("seed", range(4))
def test_minimum_rule_ties_on_both_sides(seed):
    """d(n) == d(n + k), k <= 16: n is the packet (the earliest wins: <= on the right), n + k is not (< on the left)."""
    n, k, b = tie_stream(seed)
    bt = Batch(len(b), seed=seed)
    bt.b[38] = b
    got = run(bt)
    hits = [int(r["sample_index"]) for r in got if r["channel"] == 38]
    assert n in hits and n + k not in hits
    assert got[hits.index(n)]["aa_errors"] == co.distances(b, len(b))[n]
    # the same tie 17 samples apart is two packets
    assert co.primaries(np.r_[np.full(10, co.INF), [300], np.full(16, co.INF), [300], np.full(20, co.INF)], (0, 100)) == [10, 27]


def test_random_streams_give_no_packet():
    bt = Batch(400_000, seed=77)
    for c in (37, 38, 39):
        bt.b[c]
    assert len(run(bt)) == 0
    assert co.distances(bt.b[37], bt.n)[: bt.n - 1100].min() > co.T


# ------------------------------------------------------------------------------------------------ CI and Viterbi ties
def ref_viterbi(bm, steps, end_state=None):
    """Independent statement: transitions (p, u) -> ((p << 1) | u) & 7, their coded bits from synth's encoder fed with the
    register's history, ties to the predecessor with D3 = 0; returns the decoded bits."""
    out = {}
    for p in range(8):
        for u in (0, 1):
            c = synth.coded_fec([(p >> 2) & 1, (p >> 1) & 1, p & 1, u])[-2:]
            out[(p, u)] = c
    pm = {0: 0}
    hist = []
    for t in range(steps):
        new, back = {}, {}
        for s in range(8):
            u = s & 1
            best = None
            for p in ((s >> 1), (s >> 1) | 4):                    # D3 = 0 first: kept on ties
                if p not in pm:
                    continue
                a0, a1 = out[(p, u)]
                m = pm[p] + int(bm[2 * t][a0]) + int(bm[2 * t + 1][a1])
                if best is None or m < best[0]:
                    best = (m, p)
            if best is not None:
                new[s], back[s] = best
        pm = new
        hist.append(back)
    s = min(pm, key=lambda q: (pm[q], q)) if end_state is None else end_state
    bits = []
    for t in range(steps - 1, -1, -1):
        bits.append(s & 1)
        s = hist[t][s]
    return bits[::-1], pm


@pytest.mark.parametrize("s", [8, 2])
def test_viterbi_ties_follow_the_d3_rule(s):
    """Coded bits whose decisions are half their pattern and half its complement tie every branch: the decoded bytes are
    what the tie rule makes them."""
    rng = np.random.default_rng(11 + s)
    L = 16 if s == 8 else 4
    pdu = prim_pdu(rng, extra=10)
    dec = coded_decisions(pdu, 37, s).copy()
    start = co.BLOCK2
    for k in list(range(40, 56)) + list(range(150, 152)) + [230]:   # header-run-safe, then inside the payload
        seg = dec[start + k * L:start + (k + 1) * L]
        half = np.r_[np.ones(L // 2), np.zeros(L // 2)].astype(np.uint8) if s == 2 else np.tile([0, 1], L // 2).astype(np.uint8)
        seg[:] = half
    bt = Batch(40000, seed=5)
    for c in (37, 38, 39):
        bt.b[c] &= 0
    plant(bt.b[37], 1000, dec)
    got = run(bt)
    (r,) = got[got["sample_index"] == 1000]
    ln = pdu[1]
    N = 8 * ln + 43
    bm = co.branch_metrics(bt.b[37], 1000 + start, 2 * N, s)
    hdr_bits, _ = ref_viterbi(bm, 40)
    bits, pm = ref_viterbi(bm, N, end_state=0)
    data = np.packbits(np.array(bits[: 8 * (ln + 5)], np.uint8).reshape(-1, 8), axis=1, bitorder="little").reshape(-1)
    data ^= ao.whitening(37, ln + 5)
    assert r["status"] == co.OK and r["len"] == ln + 5 and r["metric"] == pm[0]
    assert bytes(r["bytes"][: ln + 5]) == bytes(data)
    assert bytes(r["bytes"][: ln + 5]) != pdu + synth.ble_crc24(pdu)      # the ties did change bits


def test_ci_ties_and_reserved_values():
    rng = np.random.default_rng(4)
    pdu = prim_pdu(rng)
    bt = Batch(60000, seed=4)
    for c in (37, 38, 39):
        bt.b[c] &= 0
    for j, v in enumerate(range(4)):
        plant(bt.b[37], 1000 + 12000 * j, coded_decisions(pdu, 37, 8, ci=v))
    got, _ = planted(run(bt), [1000 + 12000 * j for j in range(4)])
    assert list(got["ci"]) == [0, 1, 2, 3]
    assert list(got["status"]) == [co.OK, co.OK, co.RESERVED_CI, co.RESERVED_CI]
    assert got[1]["crc_ok"] == 0 and got[2]["len"] == 0 and got[3]["metric"] == 0
    # a CI field exactly between two values goes to the lower one
    for a, b_ in ((0, 1), (1, 3), (2, 3), (0, 2)):
        dec = coded_decisions(pdu, 37, 8, ci=a).copy()
        pa, pb = co.CI_PATTERNS[a], co.CI_PATTERNS[b_]
        diff = np.nonzero(pa != pb)[0]
        dec[co.AA_SAMPLES + diff[: len(diff) // 2]] = pb[diff[: len(diff) // 2]]
        bt2 = Batch(30000, seed=a)
        for c in (37, 38, 39):
            bt2.b[c] &= 0
        plant(bt2.b[37], 1000, dec)
        assert int(planted(run(bt2), [1000])[0][0]["ci"]) == min(a, b_)


# ------------------------------------------------------------------------------------------------ buffer end
@pytest.mark.parametrize("s", [8, 2])
def test_truncation_at_every_residue(s):
    """The three edges of a packet, each at 16 buffer ends around it (usable decisions end at n_out - 2): the CI field's last
    decision (before it: TRUNCATED with no CI; from it on: the CI is read), the header run's (the packet stays TRUNCATED: its
    full run is longer still) and the full run's (TRUNCATED before, OK from it on)."""
    rng = np.random.default_rng(s + 20)
    pdu = prim_pdu(rng, extra=5)
    ln = pdu[1]
    L = 16 if s == 8 else 4
    ci = 0 if s == 8 else 1
    n = 600
    ci_last = n + co.BLOCK2 - 1
    hdr_last = n + co.BLOCK2 + 80 * L - 1
    full_last = packet_end(n, ln, s)
    assert ci_last < hdr_last < full_last
    for edge, last in (("ci", ci_last), ("hdr", hdr_last), ("full", full_last)):
        for r in range(16):
            n_out = last + 2 - 8 + r
            bt = Batch(n_out, seed=r)
            for c in (37, 38, 39):
                bt.b[c] &= 0
            plant(bt.b[37], n, coded_decisions(pdu, 37, s))
            got, _ = planted(run(bt), [n])
            assert len(got) == 1 and got[0]["sample_index"] == n
            g = got[0]
            usable = n_out - 2 >= last
            if edge == "ci":
                assert g["status"] == co.TRUNCATED and g["ci"] == (ci if usable else 0xFF), (s, r)
            elif edge == "hdr":
                assert g["status"] == co.TRUNCATED and g["ci"] == ci and g["len"] == 0, (s, r)
            else:
                assert g["status"] == (co.OK if usable else co.TRUNCATED) and g["ci"] == ci, (s, r)
                assert g["len"] == (ln + 5 if usable else 0)


def test_last_defined_position():
    """d(n) is defined while n + 1023 is usable, i.e. n <= n_out - 1025: a clean pattern there is a (TRUNCATED) primary, one
    sample later it is none; a Coded pointer whose win_hi is the last defined position finds a packet there."""
    rng = np.random.default_rng(30)
    pdu = prim_pdu(rng)
    n = 5000
    for n_out, found in ((n + co.AA_SAMPLES + 1, True), (n + co.AA_SAMPLES, False)):
        bt = Batch(n_out, seed=1)
        for c in (37, 38, 39):
            bt.b[c] &= 0
        plant(bt.b[37], n, coded_decisions(pdu, 37, 8))
        d = co.distances(bt.b[37], bt.n)
        assert (d[n] == 0) == found
        got = run(bt)
        assert (n in got["sample_index"]) == found             # (n - 1, one sample off the pattern, may be one instead)
        if found:
            assert len(got) == 1 and got[0]["status"] == co.TRUNCATED and got[0]["ci"] == 0xFF
    units, off, ca = 30, 40, 1
    lo, hi = ao.window(units, off, ca)
    src = 1000
    win_hi = src + hi
    for extra, status in ((0, co.TRUNCATED), (-1, co.OUTSIDE)):
        n_out = win_hi + co.AA_SAMPLES + 1 + extra
        bt = Batch(n_out, seed=2)
        for c in (37, 38, 39, 9):
            bt.b[c] &= 0
        coded_primary_with_ptr(rng, bt, src, synth.aux_ptr_bytes(9, ca, units, off, 2))
        plant(bt.b[9], win_hi, coded_decisions(aux_pdu(rng, 20), 9, 8))
        got, _ = planted(run(bt), [src])
        assert len(got) == 2 and got[1]["win_hi"] == win_hi and got[1]["status"] == status
        if status == co.TRUNCATED:
            assert got[1]["sample_index"] == win_hi and got[1]["aa_errors"] == 0


# ------------------------------------------------------------------------------------------------ pointers
def coded_primary_with_ptr(rng, bt, n, ptr, channel=37, s=8):
    pdu = prim_pdu(rng, ptr)
    plant(bt.b[channel], n, coded_decisions(pdu, channel, s))
    return pdu


@pytest.mark.parametrize("where", ["lo", "hi", "lo-1", "hi+1"])
@pytest.mark.parametrize("dst_phy", [0, 1, 2])
def test_windows_with_the_preamble_shift(where, dst_phy):
    """Coded primary -> 1M / 2M / Coded target exactly at either edge of s - 320 + P(dst) + [lo, hi], and one outside."""
    rng = np.random.default_rng(hash((where, dst_phy)) & 0xFFFF)
    units, off, ca = 30, 40, 1
    lo, hi = ao.window(units, off, ca)
    n = 2000
    shift = -320 + co.PREAMBLE[dst_phy]
    at = n + shift + {"lo": lo, "hi": hi, "lo-1": lo - 1, "hi+1": hi + 1}[where]
    bt = Batch(n + hi + 40000, seed=dst_phy)
    for c in (37, 38, 39, 9):
        bt.b[c] &= 0
    coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(9, ca, units, off, dst_phy))
    target = aux_pdu(rng, 30)
    if dst_phy == 2:
        plant(bt.b[9], at, coded_decisions(target, 9, 2))
    else:
        plant_stride(bt.b[9], at, aux_symbols(9, target), 2 if dst_phy == 1 else 4)
    got, idx = planted(run(bt), [n])
    assert len(got) == 2 and got[1]["parent"] == idx[0] and got[1]["depth"] == 1
    assert (got[1]["win_lo"], got[1]["win_hi"]) == (n + shift + lo, n + shift + hi)
    if where in ("lo", "hi"):
        check(got[1], 9, target, ci=1 if dst_phy == 2 else 0xFF)
        assert got[1]["sample_index"] == at and got[1]["aa_errors"] == 0
    elif dst_phy == 2:                          # the smallest d inside the window: the edge, one sample off the packet
        edge = got[1]["win_lo"] if where == "lo-1" else got[1]["win_hi"]
        assert got[1]["sample_index"] == edge and 0 < got[1]["aa_errors"] <= co.T
    else:
        assert got[1]["status"] == co.NOT_FOUND


@pytest.mark.parametrize("src_phy", [0, 1])
def test_uncoded_source_to_coded_target(src_phy):
    """Coded -> 1M / 2M -> Coded: the second link's window is s - 32 + 320 + [lo, hi]."""
    rng = np.random.default_rng(src_phy + 40)
    bt = Batch(80000, seed=src_phy)
    for c in (37, 38, 39, 4, 21):
        bt.b[c] &= 0
    n, a1 = 1000, 20000
    lo1, _ = ao.window(30, 100, 1)
    off1 = 100
    a1 = n - 320 + 32 + lo1 + 50 if src_phy == 0 else n - 320 + 32 + lo1 + 50
    lo2, hi2 = ao.window(30, 60, 1)
    a2 = a1 - 32 + 320 + hi2                                    # the second target at the far edge
    link = aux_pdu(rng, 20, synth.aux_ptr_bytes(21, 1, 30, 60, 2))
    plant_stride(bt.b[4], a1, aux_symbols(4, link), 2 if src_phy else 4)
    coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(4, 1, 30, off1, src_phy))
    last = aux_pdu(rng, 12)
    plant(bt.b[21], a2, coded_decisions(last, 21, 8))
    got, idx = planted(run(bt), [n])
    assert len(got) == 3
    check(got[1], 4, link, ci=0xFF)
    check(got[2], 21, last, ci=0)
    assert got[2]["sample_index"] == a2 and got[2]["win_hi"] == a2 and got[2]["depth"] == 2 and got[2]["parent"] == idx[1]


def test_three_primaries_one_packet_and_outside():
    rng = np.random.default_rng(8)
    bt = Batch(120000, seed=8)
    for c in (37, 38, 39, 17):
        bt.b[c] &= 0
    target_at = 60000
    target = aux_pdu(rng, 25)
    plant(bt.b[17], target_at, coded_decisions(target, 17, 2))
    for j, n in enumerate((2000, 20000, 38000)):
        coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(17, 1, 30, (target_at - n) // 120, 2), channel=37 + j)
    bt.b[37][100_000:] = 0
    coded_primary_with_ptr(rng, bt, 100_000, synth.aux_ptr_bytes(17, 1, 300, 8000, 2))   # window beyond the buffer
    got, idx = planted(run(bt), [2000, 20000, 38000, 100_000])
    assert list(got["depth"]) == [0, 0, 0, 0, 1, 1, 1, 1]
    assert list(got["channel"][:4]) == [37, 37, 38, 39] and list(got["sample_index"][:4]) == [2000, 100_000, 20000, 38000]
    assert list(got["parent"][4:]) == list(idx[:4])                  # (capture, channel, sample) order
    assert got[4]["status"] == co.OK and list(got["first"][4:]) == [idx[4], idx[5], idx[4], idx[4]]
    assert got[5]["status"] == co.OUTSIDE
    for r in got[[4, 6, 7]]:
        check(r, 17, target, ci=1)


def test_depth_limit():
    """A Coded primary and a chain of 1M links: 16 pointed packets are followed, the 17th pointer is DEPTH_LIMIT."""
    rng = np.random.default_rng(12)
    links = 17
    bt = Batch(2000 + 3000 * (links + 3), seed=12)
    for c in (37, 38, 39):
        bt.b[c] &= 0
    starts = [4000 + 3000 * k for k in range(links)]
    n = 500
    coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(3, 1, 30, (starts[0] - (n - 320 + 32)) // 120, 0))
    for k in range(links):
        ptr = synth.aux_ptr_bytes(3 + (k + 1) % 30, 1, 30, (starts[k + 1] - starts[k]) // 120, 0) if k + 1 < links else None
        plant_stride(bt.b[3 + k % 30], starts[k], aux_symbols(3 + k % 30, aux_pdu(rng, 20, ptr)), 4)
    got, _ = planted(run(bt), [n])
    assert len(got) == 1 + co.MAX_DEPTH + 1
    assert all(got[d]["status"] == co.OK and got[d]["crc_ok"] for d in range(1, co.MAX_DEPTH + 1))
    assert got[-1]["status"] == co.DEPTH_LIMIT and got[-1]["depth"] == co.MAX_DEPTH + 1


def test_shards_against_the_whole_stream():
    rng = np.random.default_rng(13)
    whole = Batch(8192 * 12, seed=13)
    for c in (37, 38, 39):
        whole.b[c] &= 0
    spots = [100, 8192 * 3 - 30, 8192 * 3 + 5, 8192 * 6 - 1100, 8192 * 9 + 17]
    for k, n in enumerate(spots):
        plant(whole.b[37 + k % 3], n, coded_decisions(prim_pdu(rng), 37 + k % 3, 8 if k % 2 else 2))
    want = run(whole)
    assert all(planted(want, spots)[0]["crc_ok"]) and len(planted(want, spots)[0]) == len(spots)
    got_all = []
    for w0, w1 in ((0, 3), (3, 6), (6, 9), (9, 12)):
        pre = 128 if w0 else 0
        a, b = 8192 * w0 - pre, min(whole.n, 8192 * w1 + 9000)
        sh = Batch(b - a)
        for c in list(whole.b):
            sh.b[c] = whole.b[c][a:b]
        got = run(sh, first_window=w0, pre_out=pre, n_windows=w1 - w0)
        assert all(8192 * w0 <= int(r["sample_index"]) < 8192 * w1 for r in got)
        got_all += list(planted(got, spots)[0])
    want = planted(want, spots)[0]
    key = ("sample_index", "channel", "status", "ci", "len", "crc_ok", "aa_errors", "metric", "bytes")
    assert sorted(tuple(np.asarray(r[k]).tobytes() for k in key) for r in got_all) == \
        sorted(tuple(np.asarray(r[k]).tobytes() for k in key) for r in want)


# ------------------------------------------------------------------------------------------------ sensitivity (numpy model)
def chain_recall(esn0_db: float, phy: str, n_pkts: int, seed: int) -> float:
    """GFSK (synth) -> AWGN at Es/N0 (synth's definition, 4 samples per symbol) -> int8 (scale 100 / peak of the clean
    signal) -> the slicer -> the coded oracle (Coded) or an uncoded decode at the known position (1M).  20-byte PDUs."""
    rng = np.random.default_rng(seed)
    ok = 0
    for _ in range(n_pkts):
        pdu = bytes([0x07, 18]) + bytes(rng.integers(0, 256, 18, dtype=np.uint8))
        if phy == "1m":
            sym = synth.ble_phy_bits(pdu, 37)
        else:
            sym = synth.ble_phy_bits_coded(pdu, 37, 8 if phy == "s8" else 2)
        pad = 400
        wave = np.r_[np.zeros(pad), synth.gfsk_modulate(sym), np.zeros(pad)]
        sigma2 = 4.0 / (10 ** (esn0_db / 10.0))                  # Es = 4 samples of unit power, as synth's captures
        x = wave * np.exp(1j * rng.uniform(0, 2 * np.pi)) + synth._awgn(len(wave), rng, sigma2)
        q = np.clip(np.rint(np.c_[x.real, x.imag] * 100.0), -128, 127).astype(np.int64)
        nxt = np.vstack([q[1:], np.zeros((1, 2), np.int64)])
        b = (q[:, 0] * nxt[:, 1] - nxt[:, 0] * q[:, 1] > 0).astype(np.uint8)
        b = np.r_[b, np.zeros(64, np.uint8)]
        if phy == "1m":
            at = pad + 8 * 4 + 8                                  # AA bit 0 with the Gaussian filter's delay
            best = None
            for s in range(at - 2, at + 3):
                pos = s + 4 * np.arange(len(sym) - 8)
                got = np.packbits(b[pos[32:]].reshape(-1, 8), axis=1, bitorder="little").reshape(-1) ^ synth.ble_whitening(37, 23)
                if bytes(got) == pdu + synth.ble_crc24(pdu):
                    best = s
            ok += best is not None
        else:
            d = co.distances(b, len(b))
            n = co.window_min(d, pad + 320, pad + 320 + 16)
            if n >= 0:
                r = np.zeros(1, co.CODED_DTYPE)[0]
                r["channel"] = 37
                co.decode(r, b, n, len(b))
                ok += r["status"] == co.OK and r["crc_ok"] and bytes(r["bytes"][:23]) == pdu + synth.ble_crc24(pdu)
    return ok / n_pkts


# Measured with this model (20 packets per point, seed 5), recall of S=8 / S=2 / uncoded 1M:
#   Es/N0  6 dB: 0.00 / 0.00 / 0.00     8 dB: 0.90 / 0.00 / 0.00    10 dB: 1.00 / 0.00 / 0.00
#         12 dB: 1.00 / 0.15 / 0.00    16 dB: 1.00 / 1.00 / 0.00
def test_sensitivity_coded_beats_uncoded():
    s8, one_m = chain_recall(10.0, "s8", 20, 5), chain_recall(10.0, "1m", 20, 5)
    assert s8 >= 0.9 and one_m <= 0.1, (s8, one_m)


# ------------------------------------------------------------------------------------------------ host side
def _coded_list():
    rng = np.random.default_rng(21)
    bt = Batch(90000, seed=21)
    for c in (37, 38, 39, 17, 5):
        bt.b[c] &= 0
    t1, t2 = 40000, 60000
    lo2, _ = ao.window(30, 30, 1)
    chain = aux_pdu(rng, 14)
    head = aux_pdu(rng, 30, synth.aux_ptr_bytes(5, 1, 30, (t2 - t1) // 120, 1))
    plant(bt.b[17], t1, coded_decisions(head, 17, 8))
    plant_stride(bt.b[5], t2 - 320 + 32 + 0, aux_symbols(5, chain), 2)
    pdus = []
    for j, n in enumerate((2000, 20000)):
        off = (t1 - n) // 120
        pdus.append(coded_primary_with_ptr(rng, bt, n, synth.aux_ptr_bytes(17, 1, 30, off, 2), channel=37 + j, s=8 if j else 2))
    got, _ = planted(run(bt), [2000, 20000])
    lst = np.array(got).astype(_abi.CODED_DTYPE)
    lst["first"] = np.arange(len(lst))                              # re-indexed: the list without the false primaries
    lst["first"][3] = 2
    lst["parent"][2:] = [0, 1, 2]
    return lst, pdus, head, chain


def test_messages_lines_and_pcap():
    lst, pdus, head, chain = _coded_list()
    assert list(lst["depth"]) == [0, 0, 1, 1, 2] and list(lst["first"]) == [0, 1, 2, 2, 4]
    msgs = messages.ble_coded_adv(lst)
    assert [m["index"] for m in msgs] == [0, 1, 2, 4]
    assert [m["phy"] for m in msgs] == ["Coded", "Coded", "Coded", "2M"] and [m.get("s") for m in msgs[:3]] == [2, 8, 8]
    assert msgs[2]["chain"] == [2, 4] and msgs[2]["complete"]
    assert msgs[2]["chain_data"] == b"".join(p[3 + (p[2] & 0x3F):] for p in (head, chain))
    assert messages.ble_ext_adv(lst)[0]["phy"] == "Coded"
    line = formats.coded_line(msgs[0])
    m = msgs[0]
    assert line == f"CODED Ch37 S2 AdvA:{m['adv_a']} ADI:{m['did']:03x}/{m['sid']:x} PloadL{m['pload_len']} CRC0 AAerr0\n"
    assert len(line.split()) == 8 and not line[0].isdigit()
    assert formats.aux_line(msgs[2]).startswith("AUX Ch17 PHYCoded ") and " Depth1 " in formats.aux_line(msgs[2])
    blob = formats.ble_pcap_coded_block(lst)
    at, recs = 0, []
    while at < len(blob):
        n = struct.unpack(">i", blob[at + 8:at + 12])[0]
        assert struct.unpack(">i", blob[at + 12:at + 16])[0] == n
        recs.append(blob[at + 16:at + 16 + n])
        at += 16 + n
    assert len(recs) == 4
    for k, rec in zip((0, 1, 2, 4), recs):
        r = lst[k]
        flags = struct.unpack("<H", rec[8:10])[0]
        pdu_type = 0 if r["depth"] == 0 else 1
        assert rec[0] == r["channel"] and flags == 0x0001 | (pdu_type << 7) | (int(r["phy"]) << 14)
        assert struct.unpack("<I", rec[10:14])[0] == ao.ADV_AA
        body = rec[14:]
        if r["phy"] == _abi.AUX_PHY_CODED:
            assert body[0] == r["ci"]
            body = body[1:]
        assert body == bytes(r["bytes"][: int(r["len"]) - 3])


class CodedEngine(RecordingEngine):
    lst = None

    def ble_coded(self):
        return self.lst


def test_cli_coded(tmp_path):
    lst, *_ = _coded_list()
    bad = lst[:1].copy()                                  # a primary whose CRC fails: neither printed nor written
    bad["crc_ok"], bad["first"], bad["sample_index"] = 0, len(lst), 70000
    lst = np.concatenate([lst, bad])
    out = io.StringIO()
    assert btle_cli.run(btle_cli.parse_commandline(["--coded", "--iq", "-"], out=out), out=out) == 1
    assert "--coded needs --wideband" in out.getvalue()
    pcap = tmp_path / "x.pcap"
    CodedEngine.lst = lst
    out = io.StringIO()
    o = btle_cli.parse_commandline(["--wideband", "--coded", "-s", str(pcap)], out=out)
    rc = btle_cli.run(o, out=out, engine_factory=lambda mode, **kw: CodedEngine(mode, **{k: v for k, v in kw.items() if k == "max_samples"}),
                      blocks=[np.zeros(24 * 8192, np.complex64)])
    assert rc == 0
    lines = out.getvalue().splitlines()
    assert sum(ln.startswith("CODED ") for ln in lines) == 2 and sum(ln.startswith("AUX ") for ln in lines) == 2
    data = pcap.read_bytes()
    blk = formats.ble_pcap_coded_block(lst, crc_failed_primaries=False)
    assert data.startswith(formats.PCAP_HDR_BLE) and data.endswith(blk) and blk != formats.ble_pcap_coded_block(lst)

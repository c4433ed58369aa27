"""Constructed 802.15.4 chip streams: IQ whose receive chain decides a chosen chip stream.

The 802.15.4 back end (DC tracker, Mueller-Mueller clock recovery, packet sink) sees the discriminator output
f[n] = arg(x[n] conj(x[n-1])).  The packet sink compares hard chips with the discriminator-domain chip words
(synth.zb_chip_mapping(): bit 31-k is chip k; bits 31 and 0 are never compared).  A capture whose phase steps by
+pi/4 on both samples of a '1' chip and by -pi/4 on both samples of a '0' chip,

    x = exp(j cumsum(d)),   d[s0 + 2i] = d[s0 + 2i + 1] = (2 c[i] - 1) pi/4,

has f = d exactly, and a chain that starts on an even sample reads chip i between samples p + 3 and p + 4 with
p = 2i when s0 = 3.  A chip-rate offset eps samples the same piecewise-linear phase at t = n / (1 + eps): a chip then
lasts 2 (1 + eps) samples.  The clock recovery does not stay on the even grid (DC and mu drift), so positions are
always read from the oracle's chain (oracle.zb_chain(..., want_chips=True)), never computed as 2i.

Frames are built from synth.fcs16 (the definition), not from the oracle.  Plain numpy; no engine.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Callable

import numpy as np

from snout_b200 import synth

WORDS = synth.zb_chip_mapping()
M0 = int(WORDS[0])
MASK = 0x7FFFFFFE
SEGMENT, PREHALO = 4096, 2048         # include/snoutrx.h defaults
SINK_LEAD = 1024                      # csrc/zb.cuh kZbSinkLead
POST_HALO = 16448                     # csrc/zb.cuh kZbPostHalo
MIN_SYNC_CHIPS = 193                  # PHR (64) + one byte (64) + one chip to re-lock + 7 (32) + 10 (32)
FILLER = np.array([0, 1], np.uint8)   # 0101...: 14 chips from symbol 0 at every shift, DC free
CHANNEL = 11


def slots_bound(body: int) -> int:
    """Records a chain body of `body` samples can hold: syncs >= 193 chips apart, every chip advances >= 1 sample."""
    return (body - 1) // MIN_SYNC_CHIPS + 1


def word_chips(w: int) -> np.ndarray:
    return ((int(w) >> (31 - np.arange(32))) & 1).astype(np.uint8)


def dist(reg: int, s: int) -> int:
    return bin((reg & MASK) ^ int(WORDS[s])).count("1")


def relock_k(thr: int) -> int:
    """Chips after a reset (empty register) that lock the unlocked search on the tail of symbol 0."""
    return next(k for k in range(1, 33) if bin(M0 & ~((1 << k) - 1) & 0xFFFFFFFF).count("1") < thr)


def flip_positions(s: int, d: int, floor: int = 0) -> np.ndarray:
    """d compared chip positions (1..30) of symbol s to invert so that every other symbol stays more than max(d, floor)
    away: the register is then exactly d from s and decides nothing else.  Deterministic."""
    rng = np.random.default_rng(33 * s + d)
    for _ in range(50000):
        pos = np.sort(rng.choice(np.arange(1, 31), d, replace=False))
        reg = int(WORDS[s]) ^ int(sum(1 << (31 - int(p)) for p in pos))
        if min(dist(reg, t) for t in range(16) if t != s) > max(d, floor):
            return pos
    raise AssertionError(f"no flip set of {d} for symbol {s}")


def sym_chips(s: int, flips=()) -> np.ndarray:
    c = word_chips(int(WORDS[s])).copy()
    for p in flips:
        c[int(p)] ^= 1
    return c


def nibbles(data: bytes) -> list[int]:
    out = []
    for b in data:
        out += [b & 15, b >> 4]
    return out


def with_fcs(mpdu: bytes) -> bytes:
    return bytes(mpdu) + synth.fcs16(bytes(mpdu)).to_bytes(2, "little")


def frame_syms(psdu: bytes, phr: int | None = None, preamble: int = 4) -> list[int]:
    """SHR (preamble symbols 0, SFD 0xA7 low nibble first), PHR, PSDU nibbles.  A PHR of 0 still needs one byte to
    complete the frame; give it in `psdu`."""
    phr = len(psdu) if phr is None else phr
    return [0] * preamble + [7, 10, phr & 15, phr >> 4] + nibbles(psdu)


def chips_of(syms, flips: dict | None = None) -> np.ndarray:
    """Chips of a symbol list; flips = {index in syms: chip positions to invert}."""
    flips = flips or {}
    return np.concatenate([sym_chips(s, flips.get(i, ())) for i, s in enumerate(syms)]) if syms else np.zeros(0, np.uint8)


def frame(psdu: bytes, phr: int | None = None, preamble: int = 4, flips: dict | None = None) -> np.ndarray:
    return chips_of(frame_syms(psdu, phr, preamble), flips)


def filler(n: int, phase: int = 0) -> np.ndarray:
    return np.resize(np.roll(FILLER, phase), n).astype(np.uint8)


def tail0(k: int) -> np.ndarray:
    """The last k chips of symbol 0: after a reset they lock the search exactly when k >= relock_k(thr)."""
    return word_chips(M0)[32 - k:] if k else np.zeros(0, np.uint8)


def dense_run(thr: int, n_frames: int, k: int | None = None) -> np.ndarray:
    """Back-to-back len-0 frames (PHR 0, one byte), each re-locked by the k-chip tail of symbol 0 right after the
    previous one ends: SFD-completing chips 192 + k chips apart.  The first frame has a full symbol 0 in front."""
    k = relock_k(thr) if k is None else k
    one = chips_of([7, 10, 0, 0, 0, 0])
    return np.concatenate([sym_chips(0), one] + [np.concatenate([tail0(k), one]) for _ in range(n_frames - 1)])


def chips_to_iq(chips, n: int, s0: int = 3, eps: float = 0.0, amp: float = 1.0) -> np.ndarray:
    """complex64 [n]: chip i on samples s0 + 2i, s0 + 2i + 1 (at eps = 0); samples past the chips carry FILLER."""
    chips = np.asarray(chips, np.uint8)
    n_chips = max((int(np.ceil(n / (1.0 + eps))) + 4 - s0) // 2 + 2, len(chips))
    c = np.concatenate([chips, filler(n_chips - len(chips), len(chips) & 1)])
    d = np.zeros(s0 + 2 * n_chips, np.float64)
    step = (2.0 * c.astype(np.float64) - 1.0) * (np.pi / 4)
    d[s0::2] = step
    d[s0 + 1::2] = step
    phi = np.cumsum(d)
    phi[0] = 0.0
    if eps == 0.0:
        ph = phi[:n]
    else:
        t = np.arange(n, dtype=np.float64) / (1.0 + eps)
        ph = np.interp(t, np.arange(len(phi), dtype=np.float64), phi)
    return (amp * np.exp(1j * ph)).astype(np.complex64)


def place(target: int, syms_before_sync: int, chips, n: int, eps: float = 0.0, **kw) -> np.ndarray:
    """IQ [n] with `chips` after filler, shifted so that the chip completing the SFD (index syms_before_sync * 32 - 1 of
    `chips`) sits at sample `target`: s0 = 3 puts chip i at position 2i, s0 = 4 at 2i + 1 (observed on the oracle;
    Case.check states the position it needs)."""
    s0 = 3 + (target & 1)
    i0 = int(round((target - (s0 - 3)) / (1.0 + eps) / 2.0)) - (32 * syms_before_sync - 1)
    return chips_to_iq(np.concatenate([filler(i0), chips]), n, s0=s0, eps=eps, **kw)


def tie_register(a: int, b: int) -> np.ndarray | None:
    """Chips of a register exactly as far from symbols a and b and farther from every other symbol, or None."""
    wa, wb = int(WORDS[a]), int(WORDS[b])
    diff = [p for p in range(1, 31) if ((wa ^ wb) >> (31 - p)) & 1]
    if len(diff) % 2:
        return None
    reg = wa
    for p in diff[: len(diff) // 2]:
        reg ^= 1 << (31 - p)
    h = len(diff) // 2
    if dist(reg, a) != h or dist(reg, b) != h or min(dist(reg, t) for t in range(16) if t not in (a, b)) <= h:
        return None
    return word_chips(reg)


@dataclass
class Case:
    """One constructed input and the edge it is meant to hit.  iq: complex64 [n] or [captures, n].  check(oracle, case,
    frames) runs on the oracle's records (every capture, capture_id set) and asserts that the edge fires."""
    name: str
    iq: np.ndarray
    check: Callable
    edge: str
    threshold: int = 10
    segment: int = SEGMENT
    prehalo: int = PREHALO
    chips: list = field(default_factory=list)       # the constructed chip stream of every capture, from sample 0 on
    eps: float = 0.0

    @property
    def captures(self) -> np.ndarray:
        return self.iq if self.iq.ndim == 2 else self.iq[None]


def oracle_frames(oracle, case: Case) -> np.ndarray:
    """What the receiver must report for the case: zb_receive of every capture, capture ids 0, 1, ..."""
    out = []
    for i, x in enumerate(case.captures):
        f = oracle.zb_receive(x, CHANNEL, threshold=case.threshold, segment=case.segment, prehalo=case.prehalo)
        f["capture_id"] = i
        out.append(f)
    return np.concatenate(out)


def _ok_tags(frames) -> set:
    return {int(f["bytes"][0]) for f in frames if f["crc_ok"]}


def _threshold_case(thr: int, role: str) -> Case:
    """Three frames whose symbol in `role` is thr - 1, thr and thr + 1 chips from its word (every other word farther)."""
    pre = 1 if role == "search" else 2
    idx = {"search": 0, "preamble": 1, "sfd7": pre, "sfd10": pre + 1, "decode": pre + 4}[role]
    parts, want = [filler(600)], set()
    for j, d in enumerate(range(thr - 1, thr + 2)):
        tag = 0x21 + 0x11 * j
        syms = frame_syms(with_fcs(bytes([tag, 0x5A])), preamble=pre)
        if d >= 0:
            parts += [chips_of(syms, {idx: flip_positions(syms[idx], d, thr)}), filler(400)]
            if (d < thr) if role in ("search", "decode") else (d <= thr):
                want.add(tag)
    chips = np.concatenate(parts)

    def check(oracle, case, frames):
        assert _ok_tags(frames) == want, (sorted(_ok_tags(frames)), sorted(want))
    rule = "<" if role in ("search", "decode") else "<="
    return Case(f"thr{thr}_{role}", chips_to_iq(chips, 16384), check, f"{role} accepts distance {rule} {thr}", thr,
                chips=[chips])


def _tie_case() -> Case:
    """PSDU nibbles whose register is as far from two symbols a < b as from nothing else: decode_chips keeps the first
    minimum, a.  The FCS is that of the bytes with a, so a decoder that picks b fails the CRC."""
    pairs = [(a, b) for a in range(16) for b in range(a + 1, 16) if tie_register(a, b) is not None]
    parts, want, k = [filler(600)], set(), 0
    for a, b in pairs[:6]:
        tag = 0x30 + k
        psdu = with_fcs(bytes([tag, a | (a << 4)]))
        syms = frame_syms(psdu)
        c = chips_of(syms)
        for ni in (6, 7):                                   # both nibbles of the second byte
            p0 = 32 * (4 + 2 + 2 + 2 + (ni - 6))
            c[p0:p0 + 32] = tie_register(a, b)
        parts += [c, filler(400)]
        want.add(tag)
        k += 1
    chips = np.concatenate(parts)

    def check(oracle, case, frames):
        assert len(pairs) >= 6 and _ok_tags(frames) == want
    return Case("decode_ties", chips_to_iq(chips, 2 * len(chips) + 400), check, "decode ties go to the lower symbol",
                chips=[chips])


def _phr_case() -> Case:
    """PHR 0, 1, 2 (00 00), 127 and 128 in one stream; LQI saturates at 255 on a full frame, uses 4 symbols on len 1."""
    rng = np.random.default_rng(127)
    psdus = [(0, b"\x00"), (1, b"\x33"), (2, b"\x00\x00"), (127, with_fcs(bytes(rng.integers(0, 256, 125, dtype=np.uint8)))),
             (128, bytes([0x55] * 128))]
    parts = [filler(600)]
    for phr, p in psdus:
        parts += [frame(p, phr=phr), filler(400)]
    chips = np.concatenate(parts)

    def check(oracle, case, frames):
        got = [(int(f["len"]), int(f["crc_ok"]), int(f["lqi"])) for f in frames]
        assert got == [(1, 0, 128), (1, 0, 128), (2, 1, 192), (127, 1, 255)], got
        assert bytes(frames[3]["bytes"][:127]) == psdus[3][1]
    return Case("phr_edges", chips_to_iq(chips, 2 * len(chips) + 400), check,
                "PHR 127 accepted, 128 rejected; crc_ok needs 2 bytes; LQI of 4 and of 8 symbols", chips=[chips])


def _dense_cases() -> list[Case]:
    out = []
    chips10 = np.concatenate([filler(64), dense_run(10, 230)])
    x10 = chips_to_iq(chips10, 65536 + POST_HALO + 4096)
    for seg in (2048, 4096, 16384, 65536):
        def check(oracle, case, frames, seg=seg):
            per = np.bincount(frames["window"])
            d = np.diff(frames["sample_index"])
            assert per.max() <= slots_bound(seg) and (d >= 2 * (192 + relock_k(10)) - 4).all()
            if seg >= 16384:                        # more records than the former segment / 448 + 2 slots
                assert per.max() > seg // 448 + 2, (per.max(), seg // 448 + 2)
        out.append(Case(f"dense_thr10_seg{seg}", x10, check, "back-to-back len-0 frames re-locked after 14 chips",
                        10, seg, chips=[chips10]))
    # threshold 12 (k = 11): the first sync on the first sample of chain 1's body fills it to the former slot count
    run = dense_run(12, 30)
    x12 = place(4096, 3, run, 4096 + 4096 + POST_HALO + 2048)

    def check12(oracle, case, frames):
        one = frames[frames["window"] == 1]
        assert one["sample_index"][0] == 4096 and len(one) == 4096 // 448 + 2 == 11, one["sample_index"]
    out.append(Case("dense_thr12_sync_on_body_start", x12, check12, "a sync on the body's first sample", 12, 4096))
    # every threshold whose sink can decode the plain run (SFD 7 is farther than thr from symbol 0 up to 12)
    for thr in (2, 4, 8, 12):
        chips = np.concatenate([filler(64), dense_run(thr, 48)])

        def check_thr(oracle, case, frames, thr=thr):
            k = relock_k(thr)
            assert len(frames) == 48 and (np.abs(np.diff(frames["sample_index"]) - 2 * (192 + k)) <= 2).all()
        out.append(Case(f"dense_thr{thr}", chips_to_iq(chips, 2 * len(chips) + 512), check_thr,
                        f"re-lock {relock_k(thr)} chips after a reset", thr, 65536, chips=[chips]))
    # a batch of three such captures
    xs = np.stack([chips_to_iq(np.concatenate([filler(64 + 2 * i), dense_run(12, 100)]), 16384 + POST_HALO) for i in range(3)])

    def check_batch(oracle, case, frames):
        for i in range(3):
            per = np.bincount(frames["window"][frames["capture_id"] == i])
            assert per.max() > 16384 // 448 + 2
    out.append(Case("dense_batch3", xs, check_batch, "three captures with chains past the former slot count", 12, 16384))
    return out


def _segment_edge_case() -> Case:
    """Captures whose frame syncs at lo - 1, lo, hi - 1, hi of body [8192, 12288), and one whose 40-symbol preamble
    straddles the sink start lo - 1024 of that chain."""
    fr = frame(with_fcs(b"\x41\x88\x07"), preamble=4)
    targets = (8191, 8192, 12287, 12288)
    xs = [place(t, 6, fr, 32768) for t in targets]
    xs.append(place(8192 + 100, 42, frame(with_fcs(b"\x41\x88\x08"), preamble=40), 32768))

    def check(oracle, case, frames):
        assert [int(f["sample_index"]) for f in frames] == list(targets) + [8293]
        assert [int(f["window"]) for f in frames] == [1, 2, 2, 3, 2] and frames["crc_ok"].all()
    return Case("segment_edges", np.stack(xs), check, "syncs at lo - 1, lo, hi - 1, hi; preamble across the sink start")


def _halo_cases() -> list[Case]:
    """A len-127 frame syncing at hi - 1 = 8191 finishes inside the post halo; 0.4 % slower chips push its end past it
    (the unsegmented chain still decodes it; at 0.5 % this construction no longer decodes at all)."""
    rng = np.random.default_rng(128)
    fr = frame(with_fcs(bytes(rng.integers(0, 256, 125, dtype=np.uint8))))
    out = []
    for eps in (0.0, 0.004):
        x = place(8191, 6, fr, 8192 + POST_HALO + 4096, eps=eps)

        def check(oracle, case, frames, eps=eps):
            z = oracle.zb_dc_remove(oracle.zb_quad_demod(case.iq))
            whole, _, _ = oracle.zb_chain(z, 0, len(z), 0, len(z))
            s = int(whole["sample_index"][0])
            assert len(whole) == 1 and 8192 - 26 <= s < 8192, s
            if eps == 0.0:
                assert len(frames) == 1 and frames["window"][0] == 1 and frames["len"][0] == 127 and frames["crc_ok"][0]
            else:
                assert len(frames) == 0                # would end more than 16448 samples past hi: no chain reports it
        out.append(Case(f"post_halo_eps{eps}", x, check, "a len-127 frame from hi - 1 against the post halo", eps=eps))
    # capture end: the second frame is cut
    chips = np.concatenate([filler(600), fr, filler(300), fr])
    x = chips_to_iq(chips, 2 * (600 + len(fr) + 300) + len(fr))

    def check_end(oracle, case, frames):
        assert len(frames) == 1 and frames["crc_ok"][0]
    out.append(Case("capture_end", x, check_end, "a frame cut off by the capture end"))
    return out


def _drift_cases() -> list[Case]:
    """Chip-rate offsets over chains of 65536: the clock recovery drifts against the tracker's two samples per step, so
    k_zb_rx catches up (lead < 44) and pauses (lead > 84).  Frames every 3000 chips keep the sink busy."""
    rng = np.random.default_rng(9)
    parts = [filler(300)]
    for i in range(40):
        parts += [frame(with_fcs(bytes(rng.integers(0, 256, 20, dtype=np.uint8)))), filler(2000)]
    chips = np.concatenate(parts)
    out = []
    for eps in (1e-3, -1e-3, 3e-3, -3e-3):
        def check(oracle, case, frames):
            s = lead_schedule(oracle, case, (64, 44, 84))
            assert s["catch_up"] > 0 and s["pause"] > 0 and s["min_read_lead"] >= 8
        out.append(Case(f"drift_{eps:+g}", chips_to_iq(chips, 65536 + 2 * 65536 // 2, eps=eps), check,
                        "catch-up and pause windows of the tracker", 10, 65536, 4096, chips=[chips], eps=eps))
    return out


def solve_fcs(mpdu: bytes, free: tuple, target: int) -> bytes:
    """mpdu with the two bytes at `free` chosen so that its FCS is `target`.  The FCS has init 0 and no final xor, so it is
    linear over GF(2) in the bytes: eliminate over the FCS of the 16 single free bits."""
    m = bytearray(mpdu)
    for i in free:
        m[i] = 0
    basis = {}
    for j in range(16):
        e = bytearray(len(m))
        e[free[j // 8]] = 1 << (j % 8)
        v, tag = synth.fcs16(bytes(e)), 1 << j
        for bit in range(15, -1, -1):
            if (v >> bit) & 1:
                if bit not in basis:
                    basis[bit] = (v, tag)
                    break
                v, tag = v ^ basis[bit][0], tag ^ basis[bit][1]
    x, w = 0, synth.fcs16(bytes(m)) ^ target
    for bit in range(15, -1, -1):
        if (w >> bit) & 1:
            w, x = w ^ basis[bit][0], x ^ basis[bit][1]
    for k, i in enumerate(free):
        m[i] = (x >> (8 * k)) & 0xFF
    assert synth.fcs16(bytes(m)) == target
    return bytes(m)


def _span_case() -> Case:
    """The span filter (k_zb_span_filter) at its two edges, segment 2048, lookback 9.  A CRC-ok len-127 frame syncs at
    4292 (chain 2) and spans up to good_end = 4292 + 256 * 64 = 20676.  Its MPDU ends in zero bytes, and two free bytes
    are solved so that its FCS itself plants an inner SFD; an inner PHR 3 and three bytes (bad FCS) follow the frame.  Chain
    10 -- lookback - 1 chains after the frame's chain -- starts its sink inside those zeros and reports the inner record:
      capture 0: FCS bytes 70 3A, the inner sync at good_end - 64: inside the span, dropped;
      capture 1: FCS bytes 00 A7, the inner sync at exactly good_end: kept."""
    rng = np.random.default_rng(5)
    base = bytearray(rng.integers(0, 256, 125, dtype=np.uint8))
    base[-16:] = bytes(16)
    xs = []
    for target, after in ((0x3A70, [0]), (0xA700, [3, 0])):
        mpdu = solve_fcs(bytes(base), (10, 11), target)
        chips = np.concatenate([frame(mpdu + target.to_bytes(2, "little")), chips_of(after + nibbles(b"\x11\x22\x33"))])
        xs.append(place(4292, 6, chips, 24576))

    def check(oracle, case, frames):
        good_end = 4292 + 256 * 64
        for i, (inner, kept) in enumerate(((good_end - 64, False), (good_end, True))):
            f = frames[frames["capture_id"] == i]
            assert f["sample_index"][0] == 4292 and f["window"][0] == 2 and f["crc_ok"][0] and f["len"][0] == 127
            z = oracle.zb_dc_remove(oracle.zb_quad_demod(case.captures[i]))
            lo = 10 * 2048                               # chain 2 + 8 = lookback - 1 chains after the frame's chain
            raw, _, _ = oracle.zb_chain(z, lo - 2048, min(len(z), lo + 2048 + POST_HALO), lo, lo + 2048, threshold=10,
                                        hold=lo - SINK_LEAD)
            assert len(raw) == 1 and raw["sample_index"][0] == inner and raw["len"][0] == 3 and not raw["crc_ok"][0]
            assert len(f) == (2 if kept else 1)
            if kept:
                assert f["sample_index"][1] == good_end and f["window"][1] == 10
    return Case("span_filter_edges", np.stack(xs), check, "span filter: a CRC-failed record at good_end - 64 is dropped "
                "lookback - 1 chains on, one at good_end is kept", 10, 2048, 2048)


SHARD_B0, SHARD_BODY, SHARD_PRE = 13 * 8192, 16384, 102400     # stream.shard_geometry(0, 1): 48 tracker blocks + prehalo


def shard_edge_captures():
    """Four captures whose frame syncs at b0 - 1, b0, b1 - 1 and b1 of a time shard's body [b0, b1) = [106496, 122880), and
    the shard that cuts them out (pre halo, body, post halo; first capture id 5).  Returns (iq [4, n], targets, shard, lo)."""
    fr = frame(with_fcs(b"\x41\x88\x09"), preamble=4)
    b0, b1 = SHARD_B0, SHARD_B0 + SHARD_BODY
    targets = (b0 - 1, b0, b1 - 1, b1)
    n = b1 + POST_HALO + 2048
    xs = np.stack([place(t, 6, fr, n) for t in targets])
    shard = dict(pre_samples=SHARD_PRE, body_samples=SHARD_BODY, first_window=b0 // 8192, first_capture_id=5)
    return xs, targets, shard, b0 - SHARD_PRE


def chain_geometry(n: int, segment: int, prehalo: int):
    """(lo, hi, begin, end) of every chain of a capture of n samples (the engine's zb_chain_init)."""
    for lo in range(0, n, segment):
        hi = min(lo + segment, n)
        yield lo, hi, max(0, lo - prehalo), min(n, hi + POST_HALO)


def lead_schedule(oracle, case: Case, lead: tuple) -> dict:
    """k_zb_rx's tracker pacing restated over the oracle's chip positions, with lead = (kZbLead, kZbLeadMin, kZbLeadMax) as
    the build has them (64, 44, 84): a chain starts with conv = kZbLead samples converted ahead of its first position;
    before each 32-step window, four bursts (+64) while the lead conv - (ii - begin) is below kZbLeadMin, and the tracker
    pauses for the window when it is above kZbLeadMax; an enabled window converts two samples before each step's read of
    z[ii, ii + 8).  Returns the number of catch-ups and pauses, the smallest lead at a read (all windows
    and paused windows) and the largest."""
    res = dict(catch_up=0, pause=0, min_read_lead=1 << 30, min_paused_lead=1 << 30, max_read_lead=0, windows=0)
    for x in case.captures:
        z = oracle.zb_dc_remove(oracle.zb_quad_demod(x))
        for lo, hi, begin, end in chain_geometry(len(z), case.segment, case.prehalo):
            _, ck, pos = oracle.zb_chain(z, begin, end, lo, hi, threshold=case.threshold, want_chips=True,
                                         hold=lo - SINK_LEAD)
            schedule_of(pos - begin, res, lead)
    return res


def schedule_of(rel_pos, res: dict, lead: tuple) -> dict:
    lead0, lead_min, lead_max = lead
    conv = lead0
    for w0 in range(0, len(rel_pos), 32):
        p = rel_pos[w0:w0 + 32]
        ahead = conv - int(p[0])
        while ahead < lead_min:
            conv += 64
            ahead += 64
            res["catch_up"] += 1
        enabled = ahead <= lead_max
        res["pause"] += 0 if enabled else 1
        res["windows"] += 1
        steps = np.arange(1, len(p) + 1)
        read = (conv + 2 * steps if enabled else np.full(len(p), conv)) - p.astype(np.int64) - 8
        res["min_read_lead"] = min(res["min_read_lead"], int(read.min()) + 8)
        res["max_read_lead"] = max(res["max_read_lead"], int(read.max()) + 8)
        if not enabled:
            res["min_paused_lead"] = min(res["min_paused_lead"], int(read.min()) + 8)
        conv += 64 if enabled else 0
    return res


def cases() -> list[Case]:
    out = [_threshold_case(thr, role) for thr in (1, 10) for role in ("search", "preamble", "sfd7", "sfd10", "decode")]
    chips31 = np.concatenate([filler(600), frame(with_fcs(b"\x01\x02"))])

    def check31(oracle, case, frames):
        assert len(frames) == 0
    out.append(Case("thr31_sfd_is_preamble", chips_to_iq(chips31, 8192), check31,
                    "at threshold 31 every register is within thr of symbol 0: no SFD is ever seen", 31, chips=[chips31]))
    out += [_tie_case(), _phr_case()]
    out += _dense_cases()
    out.append(_segment_edge_case())
    out += _halo_cases()
    out.append(_span_case())
    out += _drift_cases()
    return out

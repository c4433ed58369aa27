"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the BLE periodic-advertising contract (include/snoutrx.h above
snrx_ble_sync_t, DESIGN.md section 4): from a batch's slicer bit words (SNRX_STAGE_BLE_BITS layout) and the list
snrx_ble_aux returns for it to the list snrx_ble_periodic returns, field for field.

The contract, restated:
* Train sources.  The aux entries with status OK, crc_ok, first == own index and a PDU of type 7 whose extended header has
  the SyncInfo flag (0x20) and room for the fields in front of it (AdvA 6, TargetA 6, CTEInfo 1, ADI 2, AuxPtr 3, each if
  flagged) and the 18-byte SyncInfo.  Not a source: offset 0, Interval < 6, fewer than 2 used channels.  One train per
  (capture_id, AA), sourced by the candidate with the smallest sample_index (lower list index on ties); trains in source order.
* SyncInfo: offset 13 bits | units << 13 (30 / 300 us) | adjust << 14 (+2 457 600 us); Interval; ChM 37 bits | SCA << 37;
  AA; CRCInit (crc_init = c0 << 16 | c1 << 8 | c2, transmit order); paEventCounter.
* Event k: counter (paEventCounter + k) mod 2^16, channel CSA#2(counter), the source's PHY, window
  [s + early(O + k I') - 8, s + late(O + U + k I') + 8] with early / late the floor / ceiling of 4 D (10^6 -+ p) / 10^6.
* Listed: every k with width <= 2500 Interval and [win_lo, win_hi + 31 sps] meeting the usable decisions, ascending.
* Search and decode as aux_oracle, with the train's AA and crc_init.

CSA#2 and the windows are written here from their definitions, not from the kernels.  Plain numpy, no engine.
"""
from __future__ import annotations

import numpy as np

from . import aux_oracle as ao

OK, NOT_FOUND, OUTSIDE, TRUNCATED = ao.OK, ao.NOT_FOUND, ao.OUTSIDE, ao.TRUNCATED
GUARD = 8
MIN_INTERVAL = 6
OFFSET_ADJUST_US = 2_457_600
SCA_PPM = (500, 250, 150, 100, 75, 50, 30, 20)

SYNC_DTYPE = np.dtype([("sample_index", "<i8"), ("win_lo", "<i8"), ("win_hi", "<i8"), ("capture_id", "<u4"), ("source", "<u4"),
                       ("access_addr", "<u4"), ("crc_init", "<u4"), ("event", "<i4"), ("event_counter", "<u2"), ("interval", "<u2"),
                       ("channel", "u1"), ("phy", "u1"), ("phase", "u1"), ("status", "u1"), ("crc_ok", "u1"), ("sca", "u1"),
                       ("len", "<u2"), ("bytes", "u1", (ao.MAX_BYTES,)), ("reserved", "u1", (4,))], align=True)
assert SYNC_DTYPE.itemsize == 320


class SyncInfo:
    __slots__ = ("offset", "units_us", "adjust", "interval", "chm", "sca", "aa", "crc_init", "pa_counter")

    def __init__(self, b: bytes):
        o = b[0] | (b[1] << 8)
        self.offset, self.units_us, self.adjust = o & 0x1FFF, (300 if o & 0x2000 else 30), (o >> 14) & 1
        self.interval = b[2] | (b[3] << 8)
        v = int.from_bytes(bytes(b[4:9]), "little")
        self.chm, self.sca = v & ((1 << 37) - 1), (v >> 37) & 7
        self.aa = int.from_bytes(bytes(b[9:13]), "little")
        self.crc_init = (b[13] << 16) | (b[14] << 8) | b[15]
        self.pa_counter = b[16] | (b[17] << 8)

    @property
    def used(self) -> list[int]:
        return [c for c in range(37) if self.chm >> c & 1]

    @property
    def ppm(self) -> int:
        return SCA_PPM[self.sca]

    @property
    def o_us(self) -> int:
        return self.offset * self.units_us + (OFFSET_ADJUST_US if self.adjust else 0)

    def valid(self) -> bool:
        return self.offset != 0 and self.interval >= MIN_INTERVAL and len(self.used) >= 2


def parse_sync_info(pdu: bytes, n_payload: int) -> SyncInfo | None:
    """The SyncInfo of a PDU of type 7 (header | payload...), or None."""
    if len(pdu) < 2 or (pdu[0] & 0x0F) != 7 or n_payload < 2:
        return None
    p = pdu[2:]
    hlen = p[0] & 0x3F
    if hlen < 1 or 1 + hlen > n_payload:
        return None
    flags = p[1]
    if not flags & 0x20:
        return None
    off = 2 + sum(size for bit, size in ((0, 6), (1, 6), (2, 1), (3, 2), (4, 3)) if flags >> bit & 1)
    if off + 18 > 1 + hlen:
        return None
    return SyncInfo(bytes(p[off:off + 18]))


def csa2(counter: int, aa: int, used: list[int]) -> int:
    """Channel Selection Algorithm #2 (Core Vol 6 Part B 4.5.8.3)."""
    cid = ((aa >> 16) ^ aa) & 0xFFFF
    u = (counter ^ cid) & 0xFFFF
    for _ in range(3):
        u = int(f"{u & 0xFF:08b}"[::-1], 2) | (int(f"{u >> 8:08b}"[::-1], 2) << 8)     # PERM
        u = (17 * u + cid) & 0xFFFF                                                    # MAM
    prn_e = u ^ cid
    if prn_e % 37 in used:
        return prn_e % 37
    return used[(len(used) * prn_e) >> 16]


def early(d: int, ppm: int) -> int:
    """floor(4 d (10^6 - ppm) / 10^6) for d >= 0, floor(4 d (10^6 + ppm) / 10^6) for d < 0 (Python's // is the floor)."""
    return (4 * d * (10**6 - ppm if d >= 0 else 10**6 + ppm)) // 10**6


def late(d: int, ppm: int) -> int:
    """ceil(4 d (10^6 + ppm) / 10^6) for d >= 0, ceil(4 d (10^6 - ppm) / 10^6) for d < 0."""
    return -((-4 * d * (10**6 + ppm if d >= 0 else 10**6 - ppm)) // 10**6)


def window(si: SyncInfo, k: int) -> tuple[int, int]:
    """[lo, hi] of AA bit 0 positions of event k, relative to the source's AA bit 0."""
    d_lo = si.o_us + k * 1250 * si.interval
    return early(d_lo, si.ppm) - GUARD, late(d_lo + si.units_us, si.ppm) + GUARD


def rule_a(si: SyncInfo, k: int) -> bool:
    lo, hi = window(si, k)
    return hi - lo + 1 <= 2500 * si.interval


def listed_range(si: SyncInfo, s: int, sps: int, base: int, n_out: int) -> range:
    """The listed k: rule (a) on the range around D = 0 (walked out from it one event at a time), rule (b) inside it."""
    kc = -(si.o_us // (1250 * si.interval))          # ceil(-O / I')
    hi_a = kc
    while rule_a(si, hi_a + 1):
        hi_a += 1
    lo_a = kc - 1
    while rule_a(si, lo_a - 1):
        lo_a -= 1
    last = base + n_out - 2
    ks = []
    for k in range(lo_a, hi_a + 1):
        lo, hi = window(si, k)
        if s + lo <= last and s + hi + 31 * sps >= base:
            ks.append(k)
    assert ks == list(range(ks[0], ks[-1] + 1)) if ks else True, "listed events not contiguous"
    return range(ks[0], ks[-1] + 1) if ks else range(0)


def _search(b: np.ndarray, lo: int, hi: int, sps: int, aa: int) -> int:
    n = np.arange(lo, hi + 1)
    idx = n[:, None] + sps * np.arange(32)[None, :]
    want = ((aa >> np.arange(32)) & 1).astype(np.uint8)
    hit = np.nonzero(np.all(b[idx] == want[None, :], axis=1))[0]
    return int(n[hit[0]]) if len(hit) else -1


def sources(aux: np.ndarray) -> list[tuple[int, SyncInfo]]:
    """(aux index, SyncInfo) of every train's source, in source order."""
    cand = []
    for i, r in enumerate(aux):
        if int(r["status"]) != OK or not int(r["crc_ok"]) or int(r["first"]) != i or int(r["len"]) < 5:
            continue
        si = parse_sync_info(bytes(r["bytes"][: int(r["len"])]), int(r["len"]) - 5)
        if si is not None and si.valid():
            cand.append((i, si))
    best: dict = {}
    for i, si in cand:
        key = (int(aux[i]["capture_id"]), si.aa)
        if key not in best or int(aux[i]["sample_index"]) < int(aux[best[key][0]]["sample_index"]):
            best[key] = (i, si)
    return sorted(best.values(), key=lambda t: t[0])


def sync_list(words: np.ndarray, aux: np.ndarray, n_out: int, first_window: int = 0, pre_out: int = 0,
              first_capture: int = 0) -> np.ndarray:
    """The snrx_ble_periodic list of a batch.  words: uint32 [captures, 40, words] (SNRX_STAGE_BLE_BITS); aux: the batch's
    snrx_ble_aux list; n_out: channel samples per capture in the buffer; first_window / pre_out / first_capture: the shard."""
    streams = ao._Streams(words, n_out)
    base = first_window * 8192 - pre_out
    last_usable = n_out - 2
    out = []
    for src, si in sources(aux):
        a = aux[src]
        s, cap_id, phy = int(a["sample_index"]), int(a["capture_id"]), int(a["phy"])
        sps = 2 if phy == ao.PHY_2M else 4
        used = si.used
        for k in listed_range(si, s, sps, base, n_out):
            r = np.zeros(1, SYNC_DTYPE)[0]
            lo, hi = window(si, k)
            counter = (si.pa_counter + k) % 65536
            ch = csa2(counter, si.aa, used)
            r["sample_index"], r["win_lo"], r["win_hi"] = -1, s + lo, s + hi
            r["capture_id"], r["source"], r["access_addr"], r["crc_init"] = cap_id, src, si.aa, si.crc_init
            r["event"], r["event_counter"], r["interval"] = k, counter, si.interval
            r["channel"], r["phy"], r["sca"] = ch, phy, si.sca
            out.append(r)
            l_lo, l_hi = s + lo - base, s + hi - base
            if l_lo < 0 or l_hi + 31 * sps > last_usable:
                r["status"] = OUTSIDE
                continue
            b = streams.bits(cap_id - first_capture, ch)
            n = _search(b, l_lo, l_hi, sps, si.aa)
            if n < 0:
                r["status"] = NOT_FOUND
                continue
            r["sample_index"], r["phase"], r["status"] = base + n, (base + n) % sps, TRUNCATED
            if n + 47 * sps > last_usable:
                continue
            wh = ao.whitening(ch, ao.MAX_BYTES)
            nb = int(ao._read_bytes(b, n, 2, sps)[1] ^ wh[1]) + 5
            if n + (32 + 8 * nb - 1) * sps > last_usable:
                continue
            data = ao._read_bytes(b, n, nb, sps) ^ wh[:nb]
            r["status"], r["len"] = OK, nb
            r["bytes"][:nb] = data
            r["crc_ok"] = int(ao.crc24_ok(bytes(data[: nb - 3]), bytes(data[nb - 3:]), si.crc_init))
    return np.array(out, dtype=SYNC_DTYPE) if out else np.zeros(0, SYNC_DTYPE)

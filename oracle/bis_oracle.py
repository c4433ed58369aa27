"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the BLE broadcast-isochronous-stream contract (include/snoutrx.h above
snrx_ble_bis_t, DESIGN.md section 4): from a batch's slicer bit words (SNRX_STAGE_BLE_BITS layout) and the list
snrx_ble_periodic returns for it to the list snrx_ble_bis returns, field for field.

The contract, restated:
* Carriers.  Periodic entries with status OK, crc_ok and a PDU of type 7 whose extended header (L >= 1, 1 + L <= payload)
  holds its flagged fields (AdvA 6, TargetA 6, CTEInfo 1, ADI 2, AuxPtr 3, SyncInfo 18, TxPower 1); the rest of the header
  is the ACAD, walked as AD structures up to a length-0 or overrunning one; its first structure of type 0x2C must have
  length byte 34 or 58 and hold a valid BIGInfo.  One BIG per (capture_id, SAA), sourced by the earliest carrier (lower
  list index on ties); BIGs in source order.
* BIGInfo bit fields as tabled in include/snoutrx.h; valid: Num_BIS, BN, NSE >= 1, NSE mod BN = 0, 1 <= IRC <= NSE / BN,
  ISO_Interval >= 4, PHY 1M or 2M, >= 2 used channels, the last subevent starts inside the interval, S_min > 0.
* BIS n: AA_n = SAA ^ DW_n (D = (35 n + 42) mod 128, DW bits 31..16 = D0 x6, D1, D6, D1, 0, D5, D4, 0, D3, D2, 0);
  crc_init_n = n << 16 | (Base & 0xFF) << 8 | Base >> 8; AA_n = 0: NOT_FOUND, not searched.
* Event k: counter (bisPayloadCount // BN + k) mod 2^16; subevent (n, se) at D_lo = O + 1250 k ISO + (n-1) BIS_Spacing +
  se Sub_Interval, window [s + early(D_lo) - 8, s + late(D_lo + U) + 8] with the train's ppm; channel CSA#2 for se = 0,
  the subevent mapping for se >= 1; payload number ((P // BN + k + (g < IRC ? 0 : PTO (g - IRC + 1))) mod 2^39) BN + i.
* Listed: every k for which every window of every event from k to k_c is at most 2 S_min samples (k_c: the first k with
  D_lo(1, 0) >= 0) and [win_lo(1, 0), win_hi(Num_BIS, NSE - 1) + 31 sps] meets the usable decisions; all Num_BIS x NSE
  entries of a listed event, ascending k, then n, then se.
* Search and decode as periodic_oracle, with AA_n, crc_init_n and the subevent's channel.

The listed range is found by brute force over k (every window of every event tested), not by the kernels' stepping.  Plain
numpy, no engine.
"""
from __future__ import annotations

import numpy as np

from . import aux_oracle as ao
from . import periodic_oracle as po

OK, NOT_FOUND, OUTSIDE, TRUNCATED = ao.OK, ao.NOT_FOUND, ao.OUTSIDE, ao.TRUNCATED
GUARD = 8
AD_BIGINFO = 0x2C
ENCRYPTED, FRAMED = 0x01, 0x02

BIS_DTYPE = np.dtype([("sample_index", "<i8"), ("win_lo", "<i8"), ("win_hi", "<i8"), ("payload_number", "<u8"), ("capture_id", "<u4"),
                      ("source", "<u4"), ("access_addr", "<u4"), ("crc_init", "<u4"), ("event", "<i4"), ("event_counter", "<u2"),
                      ("bis", "u1"), ("subevent", "u1"), ("channel", "u1"), ("phy", "u1"), ("phase", "u1"), ("status", "u1"),
                      ("crc_ok", "u1"), ("flags", "u1"), ("len", "<u2"), ("bytes", "u1", (ao.MAX_BYTES,)), ("reserved", "u1", (12,))],
                     align=True)
assert BIS_DTYPE.itemsize == 336


def _bits(v: int, lo: int, n: int) -> int:
    return (v >> lo) & ((1 << n) - 1)


class BigInfo:
    __slots__ = ("offset", "units_us", "iso_interval", "num_bis", "nse", "bn", "sub_interval", "pto", "bis_spacing", "irc",
                 "max_pdu", "saa", "sdu_interval", "max_sdu", "base_crc", "chm", "phy", "payload_count", "framing", "encrypted")

    def __init__(self, b: bytes):
        assert len(b) in (33, 57)
        w = [int.from_bytes(bytes(b[a:a + n]), "little") for a, n in ((0, 4), (4, 4), (8, 4), (17, 4), (23, 5), (28, 5))]
        self.offset, self.units_us = _bits(w[0], 0, 14), (300 if _bits(w[0], 14, 1) else 30)
        self.iso_interval, self.num_bis = _bits(w[0], 15, 12), _bits(w[0], 27, 5)
        self.nse, self.bn, self.sub_interval, self.pto = _bits(w[1], 0, 5), _bits(w[1], 5, 3), _bits(w[1], 8, 20), _bits(w[1], 28, 4)
        self.bis_spacing, self.irc, self.max_pdu = _bits(w[2], 0, 20), _bits(w[2], 20, 4), _bits(w[2], 24, 8)
        self.saa = int.from_bytes(bytes(b[13:17]), "little")
        self.sdu_interval, self.max_sdu = _bits(w[3], 0, 20), _bits(w[3], 20, 12)
        self.base_crc = int.from_bytes(bytes(b[21:23]), "little")
        self.chm, self.phy = _bits(w[4], 0, 37), _bits(w[4], 37, 3)
        self.payload_count, self.framing = _bits(w[5], 0, 39), _bits(w[5], 39, 1)
        self.encrypted = len(b) == 57

    @property
    def used(self) -> list[int]:
        return [c for c in range(37) if self.chm >> c & 1]

    @property
    def interval_us(self) -> int:
        return 1250 * self.iso_interval

    @property
    def s_min(self) -> int:
        if self.nse == 1:
            return self.interval_us
        return min(self.sub_interval, self.interval_us - (self.nse - 1) * self.sub_interval)

    @property
    def sps(self) -> int:
        return 2 if self.phy == ao.PHY_2M else 4

    def valid(self) -> bool:
        return (self.num_bis >= 1 and self.bn >= 1 and self.nse >= 1 and self.nse % self.bn == 0 and 1 <= self.irc <= self.nse // self.bn
                and self.iso_interval >= 4 and self.phy in (0, 1) and len(self.used) >= 2
                and (self.num_bis - 1) * self.bis_spacing + (self.nse - 1) * self.sub_interval < self.interval_us and self.s_min > 0)


def ad_structures(data: bytes) -> list[tuple[int, bytes]]:
    """(type, value) of the AD structures of `data`, up to a length-0 structure or one that overruns it."""
    out, at = [], 0
    while at < len(data) and data[at] != 0 and at + 1 + data[at] <= len(data):
        out.append((data[at + 1], bytes(data[at + 2:at + 1 + data[at]])))
        at += 1 + data[at]
    return out


def acad_of(pdu: bytes, n_payload: int) -> bytes | None:
    """The ACAD of a PDU of type 7 (header | payload...): the extended header's bytes past its flagged fields, or None."""
    if len(pdu) < 2 or (pdu[0] & 0x0F) != 7 or n_payload < 2:
        return None
    p = pdu[2:]
    hlen = p[0] & 0x3F
    if hlen < 1 or 1 + hlen > n_payload:
        return None
    flags = p[1]
    off = 2 + sum(size for bit, size in ((0, 6), (1, 6), (2, 1), (3, 2), (4, 3), (5, 18), (6, 1)) if flags >> bit & 1)
    return bytes(p[off:1 + hlen])


def find_big_info(pdu: bytes, n_payload: int) -> BigInfo | None:
    """The BIGInfo of the first AD structure of type 0x2C in the ACAD, if it has 33 or 57 bytes."""
    acad = acad_of(pdu, n_payload)
    if acad is None:
        return None
    for t, v in ad_structures(acad):
        if t == AD_BIGINFO:
            return BigInfo(v) if len(v) in (33, 57) else None
    return None


def access_address(saa: int, n: int) -> int:
    d = (35 * n + 42) % 128
    b = [(d >> i) & 1 for i in range(7)]
    hi16 = [b[0]] * 6 + [b[1], b[6], b[1], 0, b[5], b[4], 0, b[3], b[2], 0]       # bit 31 first
    return saa ^ (int("".join(map(str, hi16)), 2) << 16)


def crc_init(base: int, n: int) -> int:
    """crc_init (c0 << 16 | c1 << 8 | c2, transmit order) of the 24-bit CRCInit base << 8 | n sent least significant byte first."""
    c = ((base << 8) | n).to_bytes(3, "little")
    return (c[0] << 16) | (c[1] << 8) | c[2]


def _perm_mam(u: int, cid: int) -> int:
    u = int(f"{u & 0xFF:08b}"[::-1], 2) | (int(f"{u >> 8:08b}"[::-1], 2) << 8)
    return (17 * u + cid) & 0xFFFF


def subevent_channels(counter: int, aa: int, used: list[int], nse: int) -> list[int]:
    """The channels of subevents 0..nse-1 of the event with counter `counter`."""
    cid = ((aa >> 16) ^ aa) & 0xFFFF
    prn_s = counter ^ cid
    for _ in range(3):
        prn_s = _perm_mam(prn_s, cid)
    ch0 = po.csa2(counter, aa, used)
    out, idx, lu = [ch0], used.index(ch0), prn_s
    n = len(used)
    d = max(1, max(min(3, n - 5), min(11, (n - 10) // 2)))
    for _ in range(1, nse):
        lu = _perm_mam(lu, cid)
        idx = (idx + d + (((lu ^ cid) * (n - 2 * d + 1)) >> 16)) % n
        out.append(used[idx])
    return out


def payload_number(bi: BigInfo, k: int, se: int) -> int:
    g, i = divmod(se, bi.bn)
    e = bi.payload_count // bi.bn + k + (0 if g < bi.irc else bi.pto * (g - bi.irc + 1))
    return (e % (1 << 39)) * bi.bn + i


def d_lo(bi: BigInfo, k: int, n: int, se: int) -> int:
    return bi.offset * bi.units_us + k * bi.interval_us + (n - 1) * bi.bis_spacing + se * bi.sub_interval


def window(bi: BigInfo, ppm: int, k: int, n: int, se: int) -> tuple[int, int]:
    """[lo, hi] of AA bit 0 positions of subevent (n, se) of event k, relative to the source's AA bit 0."""
    d = d_lo(bi, k, n, se)
    return po.early(d, ppm) - GUARD, po.late(d + bi.units_us, ppm) + GUARD


def event_ok(bi: BigInfo, ppm: int, k: int) -> bool:
    """Every subevent window of event k is at most 2 S_min samples long."""
    for n in range(1, bi.num_bis + 1):
        for se in range(bi.nse):
            lo, hi = window(bi, ppm, k, n, se)
            if hi - lo + 1 > 2 * bi.s_min:
                return False
    return True


def k_c(bi: BigInfo) -> int:
    return -((bi.offset * bi.units_us) // bi.interval_us)          # ceil(-O / I)


def rule_a_range(bi: BigInfo, ppm: int) -> range:
    """The k for which every event from k to k_c passes: walked out from k_c one event at a time."""
    kc = k_c(bi)
    if not event_ok(bi, ppm, kc):
        return range(kc, kc)
    hi = kc
    while event_ok(bi, ppm, hi + 1):
        hi += 1
    lo = kc
    while event_ok(bi, ppm, lo - 1):
        lo -= 1
    return range(lo, hi + 1)


def listed_range(bi: BigInfo, ppm: int, s: int, base: int, n_out: int) -> range:
    """The listed k: rule (a) by brute force, rule (b) tested at every k inside it."""
    last = base + n_out - 2
    ks = []
    for k in rule_a_range(bi, ppm):
        lo = window(bi, ppm, k, 1, 0)[0]
        hi = window(bi, ppm, k, bi.num_bis, bi.nse - 1)[1]
        if s + lo <= last and s + hi + 31 * bi.sps >= base:
            ks.append(k)
    assert ks == list(range(ks[0], ks[-1] + 1)) if ks else True, "listed events not contiguous"
    return range(ks[0], ks[-1] + 1) if ks else range(0)


def sources(sync: np.ndarray) -> list[tuple[int, BigInfo]]:
    """(periodic list index, BIGInfo) of every BIG's source, in source order."""
    cand = []
    for i, r in enumerate(sync):
        if int(r["status"]) != OK or not int(r["crc_ok"]) or int(r["len"]) < 5:
            continue
        bi = find_big_info(bytes(r["bytes"][: int(r["len"])]), int(r["len"]) - 5)
        if bi is not None and bi.valid():
            cand.append((i, bi))
    best: dict = {}
    for i, bi in cand:
        key = (int(sync[i]["capture_id"]), bi.saa)
        if key not in best or int(sync[i]["sample_index"]) < int(sync[best[key][0]]["sample_index"]):
            best[key] = (i, bi)
    return sorted(best.values(), key=lambda t: t[0])


def bis_list(words: np.ndarray, sync: np.ndarray, n_out: int, first_window: int = 0, pre_out: int = 0,
             first_capture: int = 0) -> np.ndarray:
    """The snrx_ble_bis list of a batch.  words: uint32 [captures, 40, words] (SNRX_STAGE_BLE_BITS); sync: the batch's
    snrx_ble_periodic list; n_out: channel samples per capture in the buffer; first_window / pre_out / first_capture: the
    shard."""
    streams = ao._Streams(words, n_out)
    base = first_window * 8192 - pre_out
    last_usable = n_out - 2
    out = []
    for src, bi in sources(sync):
        c = sync[src]
        s, cap_id, ppm = int(c["sample_index"]), int(c["capture_id"]), po.SCA_PPM[int(c["sca"])]
        sps, used = bi.sps, bi.used
        flags = (ENCRYPTED if bi.encrypted else 0) | (FRAMED if bi.framing else 0)
        for k in listed_range(bi, ppm, s, base, n_out):
            counter = (bi.payload_count // bi.bn + k) % 65536
            for n in range(1, bi.num_bis + 1):
                aa = access_address(bi.saa, n)
                ci = crc_init(bi.base_crc, n)
                chans = subevent_channels(counter, aa, used, bi.nse)
                for se in range(bi.nse):
                    r = np.zeros(1, BIS_DTYPE)[0]
                    lo, hi = window(bi, ppm, k, n, se)
                    ch = chans[se]
                    r["sample_index"], r["win_lo"], r["win_hi"] = -1, s + lo, s + hi
                    r["payload_number"] = payload_number(bi, k, se)
                    r["capture_id"], r["source"], r["access_addr"], r["crc_init"] = cap_id, src, aa, ci
                    r["event"], r["event_counter"], r["bis"], r["subevent"] = k, counter, n, se
                    r["channel"], r["phy"], r["flags"] = ch, bi.phy, flags
                    out.append(r)
                    l_lo, l_hi = s + lo - base, s + hi - base
                    if l_lo < 0 or l_hi + 31 * sps > last_usable:
                        r["status"] = OUTSIDE
                        continue
                    if aa == 0:
                        r["status"] = NOT_FOUND
                        continue
                    b = streams.bits(cap_id - first_capture, ch)
                    m = po._search(b, l_lo, l_hi, sps, aa)
                    if m < 0:
                        r["status"] = NOT_FOUND
                        continue
                    r["sample_index"], r["phase"], r["status"] = base + m, (base + m) % sps, TRUNCATED
                    if m + 47 * sps > last_usable:
                        continue
                    wh = ao.whitening(ch, ao.MAX_BYTES)
                    nb = int(ao._read_bytes(b, m, 2, sps)[1] ^ wh[1]) + 5
                    if m + (32 + 8 * nb - 1) * sps > last_usable:
                        continue
                    data = ao._read_bytes(b, m, nb, sps) ^ wh[:nb]
                    r["status"], r["len"] = OK, nb
                    r["bytes"][:nb] = data
                    r["crc_ok"] = int(ao.crc24_ok(bytes(data[: nb - 3]), bytes(data[nb - 3:]), ci))
    return np.array(out, dtype=BIS_DTYPE) if out else np.zeros(0, BIS_DTYPE)

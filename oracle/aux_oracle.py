"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the BLE 5 extended-advertising contract (include/snoutrx.h above
snrx_ble_aux_t, DESIGN.md section 4): from a batch's slicer bit words (SNRX_STAGE_BLE_BITS layout) and its frame records to
the list snrx_ble_aux returns, field for field.

The contract, restated:
* Pointer sources.  Depth 0: the records with proto BLE, channel 37..39, crc_ok, access address 0x8E89BED6, PDU type 7, an
  extended header of length L >= 1 with 1 + L <= the payload length, the AuxPtr flag (0x10) set, and room in the header for
  the fields in front of the AuxPtr (AdvA 6, TargetA 6, CTEInfo 1, ADI 2 bytes, each if flagged) and the AuxPtr.  Depth d > 0:
  the entries of depth d - 1 with status OK, crc_ok, first == their own index and the same AuxPtr conditions.
* AuxPtr bytes a0 a1 a2: channel a0 & 0x3F, CA (a0 >> 6) & 1, units 30 / 300 us (a0 >> 7), offset a1 | (a2 & 0x1F) << 8,
  PHY a2 >> 5.
* Window of AA bit 0 positions: [s + floor(4 O (10^6 - ppm) / 10^6) - 8, s + ceil(4 (O + U)(10^6 + ppm) / 10^6) + 8],
  O = offset * U, ppm = 50 if CA else 500.
* Search: the earliest n whose decisions b[n + k sps], k = 0..31, equal the advertising access address LSB first (sps 4 at
  1M, 2 at 2M).  Decision m is usable when m + 1 < n_out.
* Decode: byte j bit i = b[n + (32 + 8 j + i) sps]; len = header byte 1; 2 + len + 3 bytes; de-whitened with the channel's
  LFSR; CRC-24 (init 0x555555) over 2 + len bytes.
* Statuses with their precedence, order by depth then parent, `first` = the earliest entry that found the same (capture,
  channel, sample, PHY), chains from entries with first == self, depth limit 15.

The LFSR and the CRC are built here from their definitions (Bluetooth Core Vol 6 Part B 3.1.1 and 3.2), not from the
kernels' tables.  Plain numpy, no engine.
"""
from __future__ import annotations

import numpy as np

ADV_AA = 0x8E89BED6
LEAD_WORDS = 4
GUARD = 8
MAX_DEPTH = 15
MAX_BYTES = 260
OK, NOT_FOUND, OUTSIDE, TRUNCATED, UNSUPPORTED_PHY, BAD_CHANNEL, DEPTH_LIMIT = range(7)
PHY_1M, PHY_2M, PHY_CODED = 0, 1, 2

AUX_DTYPE = np.dtype([("sample_index", "<i8"), ("win_lo", "<i8"), ("win_hi", "<i8"), ("capture_id", "<u4"), ("parent", "<u4"),
                      ("first", "<u4"), ("depth", "u1"), ("channel", "u1"), ("phy", "u1"), ("phase", "u1"), ("status", "u1"),
                      ("crc_ok", "u1"), ("len", "<u2"), ("bytes", "u1", (MAX_BYTES,))], align=True)
assert AUX_DTYPE.itemsize == 304


def whitening(channel: int, n: int) -> np.ndarray:
    """x^7 + x^4 + 1, position 0 = 1 and positions 1..6 = the channel index MSB first; output bit = position 6, which is fed
    back into position 0 and XOR-ed into position 4 (Core Vol 6 Part B 3.2)."""
    pos = [1] + [(channel >> (5 - k)) & 1 for k in range(6)]
    out = np.zeros(n, dtype=np.uint8)
    for i in range(n):
        v = 0
        for b in range(8):
            o = pos[6]
            v |= o << b
            pos = [o, pos[0], pos[1], pos[2], pos[3] ^ o, pos[4], pos[5]]
        out[i] = v
    return out


def crc24_ok(data: bytes, crc_bytes: bytes, init: int = 0x555555) -> bool:
    """CRC-24 x^24 + x^10 + x^9 + x^6 + x^4 + x^3 + x + 1, bits in transmit order (LSB first).  The register is seeded as
    btle_rx's crc_init_reorder maps the `-k` value (byte swap, then 24-bit reversal); register bit 0 is transmitted first."""
    swapped = ((init & 0xFF) << 16) | (init & 0xFF00) | ((init >> 16) & 0xFF)
    reg = int(f"{swapped:024b}"[::-1], 2)
    for byte in data:
        for i in range(8):
            fb = (reg ^ (byte >> i)) & 1
            reg >>= 1
            if fb:
                reg ^= 0xDA6000          # the polynomial's low terms x^10 x^9 x^6 x^4 x^3 x^1 x^0, bit-reversed into 24 bits
    return reg == (crc_bytes[0] | (crc_bytes[1] << 8) | (crc_bytes[2] << 16))


def parse_aux_ptr(pdu: bytes, n_payload: int):
    """(channel, ca, units_us, offset, phy) of a PDU of type 7 with an AuxPtr, else None.  pdu = header | payload..."""
    if len(pdu) < 2 or (pdu[0] & 0x0F) != 7 or n_payload < 2:
        return None
    p = pdu[2:]
    hlen = p[0] & 0x3F
    if hlen < 1 or 1 + hlen > n_payload:
        return None
    flags = p[1]
    if not flags & 0x10:
        return None
    off = 2 + (6 if flags & 1 else 0) + (6 if flags & 2 else 0) + (1 if flags & 4 else 0) + (2 if flags & 8 else 0)
    if off + 3 > 1 + hlen:
        return None
    a0, a1, a2 = p[off], p[off + 1], p[off + 2]
    return a0 & 0x3F, (a0 >> 6) & 1, 300 if a0 & 0x80 else 30, a1 | ((a2 & 0x1F) << 8), a2 >> 5


def window(units_us: int, offset: int, ca: int) -> tuple[int, int]:
    U, ppm = units_us, (50 if ca else 500)
    O = offset * U
    lo = (4 * O * (1_000_000 - ppm)) // 1_000_000 - GUARD
    hi = -((-4 * (O + U) * (1_000_000 + ppm)) // 1_000_000) + GUARD
    return lo, hi


class _Streams:
    """Decisions of every (capture, channel) of the batch, unpacked from the bit words on first use."""

    def __init__(self, words: np.ndarray, n_out: int):
        self.words, self.n_out, self.cache = np.asarray(words, dtype=np.uint32), n_out, {}

    def bits(self, cap: int, ch: int) -> np.ndarray:
        key = (cap, ch)
        if key not in self.cache:
            w = np.ascontiguousarray(self.words[cap, ch, LEAD_WORDS:])
            self.cache[key] = np.unpackbits(w.view(np.uint8), bitorder="little")[: self.n_out]
        return self.cache[key]


def _search(b: np.ndarray, lo: int, hi: int, sps: int) -> int:
    n = np.arange(lo, hi + 1)
    idx = n[:, None] + sps * np.arange(32)[None, :]
    want = ((ADV_AA >> np.arange(32)) & 1).astype(np.uint8)
    hit = np.nonzero(np.all(b[idx] == want[None, :], axis=1))[0]
    return int(n[hit[0]]) if len(hit) else -1


def _read_bytes(b: np.ndarray, n: int, count: int, sps: int) -> np.ndarray:
    pos = n + sps * (32 + np.arange(8 * count))
    return np.packbits(b[pos].reshape(count, 8), axis=1, bitorder="little").reshape(count)


def _entry(src_at: int, cap_id: int, parent: int, depth: int, ptr, k: int, geo, streams) -> np.void:
    ch, ca, units, off, phy = ptr
    r = np.zeros(1, AUX_DTYPE)[0]
    lo, hi = window(units, off, ca)
    r["sample_index"] = -1
    r["win_lo"], r["win_hi"] = src_at + lo, src_at + hi
    r["capture_id"], r["parent"], r["first"], r["depth"], r["channel"], r["phy"] = cap_id, parent, k, depth, ch, phy
    base, n_out, first_capture = geo
    if depth > MAX_DEPTH:
        r["status"] = DEPTH_LIMIT
        return r
    if ch > 36:
        r["status"] = BAD_CHANNEL
        return r
    if phy > PHY_2M:
        r["status"] = UNSUPPORTED_PHY
        return r
    sps = 2 if phy == PHY_2M else 4
    l_lo, l_hi = int(r["win_lo"]) - base, int(r["win_hi"]) - base
    last_usable = n_out - 2
    if l_lo < 0 or l_hi + 31 * sps > last_usable:
        r["status"] = OUTSIDE
        return r
    b = streams.bits(cap_id - first_capture, ch)
    n = _search(b, l_lo, l_hi, sps)
    if n < 0:
        r["status"] = NOT_FOUND
        return r
    r["sample_index"] = base + n
    r["phase"] = (base + n) % sps
    r["status"] = TRUNCATED
    if n + 47 * sps > last_usable:
        return r
    wh = whitening(ch, MAX_BYTES)
    length = int(_read_bytes(b, n, 2, sps)[1] ^ wh[1])
    nb = length + 5
    if n + (32 + 8 * nb - 1) * sps > last_usable:
        return r
    data = _read_bytes(b, n, nb, sps) ^ wh[:nb]
    r["status"], r["len"] = OK, nb
    r["bytes"][:nb] = data
    r["crc_ok"] = int(crc24_ok(bytes(data[: nb - 3]), bytes(data[nb - 3:])))
    return r


def aux_list(words: np.ndarray, frames: np.ndarray, n_out: int, first_window: int = 0, pre_out: int = 0,
             first_capture: int = 0) -> np.ndarray:
    """The snrx_ble_aux list of a batch.  words: uint32 [captures, 40, words] (SNRX_STAGE_BLE_BITS); frames: the batch's
    records; n_out: channel samples per capture in the buffer; first_window / pre_out / first_capture: the shard (0 for
    whole captures)."""
    streams = _Streams(words, n_out)
    geo = (first_window * 8192 - pre_out, n_out, first_capture)
    out: list = []
    # depth 0: (source index, AA bit 0, capture id, PDU bytes, payload length)
    src = []
    for i, f in enumerate(frames):
        if (int(f["proto"]) != 3 or not int(f["crc_ok"]) or not 37 <= int(f["channel"]) <= 39
                or int(f["access_addr"]) != ADV_AA or int(f["len"]) < 5):
            continue
        src.append((i, int(f["sample_index"]), int(f["capture_id"]), bytes(f["bytes"][: int(f["len"])]), int(f["len"]) - 5))
    depth = 0
    while src and depth <= MAX_DEPTH + 1:
        k0 = len(out)
        for parent, at, cap_id, pdu, n_payload in src:
            ptr = parse_aux_ptr(pdu, n_payload)
            if ptr is not None:
                out.append(_entry(at, cap_id, parent, depth, ptr, len(out), geo, streams))
        for k in range(k0, len(out)):
            r = out[k]
            if r["status"] not in (OK, TRUNCATED):
                continue
            for j in range(k):
                o = out[j]
                if (o["status"] in (OK, TRUNCATED) and o["sample_index"] == r["sample_index"] and o["channel"] == r["channel"]
                        and o["capture_id"] == r["capture_id"] and o["phy"] == r["phy"]):
                    r["first"] = j
                    break
        src = [(k, int(out[k]["sample_index"]), int(out[k]["capture_id"]), bytes(out[k]["bytes"][: int(out[k]["len"])]),
                int(out[k]["len"]) - 5)
               for k in range(k0, len(out))
               if out[k]["status"] == OK and out[k]["crc_ok"] and out[k]["first"] == k and out[k]["len"] >= 5]
        depth += 1
    return np.array(out, dtype=AUX_DTYPE) if out else np.zeros(0, AUX_DTYPE)

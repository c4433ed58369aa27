"""Wire and text formats on the output side of the receive path.

Frame records (``_abi.FRAME_DTYPE``, filled by the CUDA engine) are rendered here into exactly what
Snout's two boundaries expect, byte for byte:

* the ``btle_rx`` stdout line that ``snout/core/pcontroller.py:115-131`` reads and
  ``BtleMessage.fromraw`` (``snout/core/message.py:205-237``) splits -- restated from
  ``vendor/BTLE/host/btle-tools/src/btle_rx.c``: line prefix 2137, ADV part 2140 +
  ``print_adv_pdu_payload`` 1962-2017 (field order of ``parse_adv_pdu_payload_byte`` 1423-1571),
  data-channel part 2147 + ``print_ll_pdu_payload`` 1850-1958 (``parse_ll_pdu_payload_byte``
  1573-1769);
* the pcap file ``btle_rx -s`` writes (``btle_rx.c:126-170``: big-endian magic, linktype 256,
  10-byte LE-LL pseudo header, access address, PDU without CRC);
* the RFtap datagram the Zigbee flowgraph sends to UDP 127.0.0.1:52002
  (``snout/modulations/Zigbee/hackrf/Zigbee_rx/top_block.py:53,71`` with
  ``epy_block_0.py:19-23``; dissector ``scapy-radio/scapy/scapy/layers/rftap.py:31-108``; fixture
  ``scapy-radio/scapy/test/rftap.pcap``);
* the 8-byte GnuradioPacket header of the older flowgraphs
  (``scapy-radio/scapy/scapy/layers/gnuradio.py:19-25``;
  ``scapy-radio/gnuradio/gr-zigbee/lib/packet_sink_scapy_impl.cc:333-349``);
* a DLT 195 pcap as scapy's ``wrpcap`` of ``Dot15d4FCS`` packets produces
  (``snout/util/zigbee.py:194-202``, ``scapy/layers/dot15d4.py:454``).

Nothing here touches samples: this is record -> bytes only.
"""
from __future__ import annotations

import struct
import time
from typing import BinaryIO, Iterable

import numpy as np

from ._abi import AUX_OK, AUX_PHY_CODED, PROTO_BLE, PROTO_ZIGBEE, RF_CFO, RF_NOISE, RF_POWER

# ---------------------------------------------------------------------------------- BLE text line
ADV_PDU_TYPE_STR = (      # btle_rx.c:1081-1098
    "ADV_IND", "ADV_DIRECT_IND", "ADV_NONCONN_IND", "SCAN_REQ", "SCAN_RSP", "CONNECT_REQ", "ADV_SCAN_IND",
    "RESERVED0", "RESERVED1", "RESERVED2", "RESERVED3", "RESERVED4", "RESERVED5", "RESERVED6", "RESERVED7", "RESERVED8",
)
LL_PDU_TYPE_STR = ("LL_RESERVED", "LL_DATA1", "LL_DATA2", "LL_CTRL")      # btle_rx.c:958-963
LL_CTRL_STR = (           # btle_rx.c:987-1003
    "LL_CONNECTION_UPDATE_REQ", "LL_CHANNEL_MAP_REQ", "LL_TERMINATE_IND", "LL_ENC_REQ", "LL_ENC_RSP", "LL_START_ENC_REQ",
    "LL_START_ENC_RSP", "LL_UNKNOWN_RSP", "LL_FEATURE_REQ", "LL_FEATURE_RSP", "LL_PAUSE_ENC_REQ", "LL_PAUSE_ENC_RSP",
    "LL_VERSION_IND", "LL_REJECT_IND", "LL_RESERVED",
)
_LL_CTRL_LEN = {0: 12, 1: 8, 2: 2, 7: 2, 13: 2, 3: 23, 4: 13, 5: 1, 6: 1, 10: 1, 11: 1, 8: 9, 9: 9, 12: 6}


def _hx(b: bytes) -> str:
    return b.hex()


def _rev(b: bytes) -> str:
    return b[::-1].hex()


def _le16(b: bytes, i: int) -> int:
    return b[i] | (b[i + 1] << 8)


def _adv_body(pdu_type: int, p: bytes) -> tuple[str, bool]:
    """Text after 'PloadL%d ' for an advertising-channel PDU.  Returns (text, complete):
    complete=False reproduces the reference's early `continue` after an Error line
    (btle_rx.c:1453-1455, 1477-1479, 2142-2144) -- no ' CRC%d' follows."""
    n = len(p)
    if n < 6:                                                             # btle_rx.c:1428-1432
        return f"Error: Payload Too Short (only {n} bytes)!\n", False
    if pdu_type in (0, 2, 4, 6):                                          # AdvA reversed, then AdvData
        return f"AdvA:{_rev(p[:6])} Data:{_hx(p[6:])}", True
    if pdu_type in (1, 3):
        if n != 12:
            return f"Error: Payload length {n} bytes. Need to be 12 for PDU Type {ADV_PDU_TYPE_STR[pdu_type]}!\n", False
        return f"A0:{_rev(p[:6])} A1:{_rev(p[6:12])}", True
    if pdu_type == 5:
        if n != 34:
            return f"Error: Payload length {n} bytes. Need to be 34 for PDU Type {ADV_PDU_TYPE_STR[pdu_type]}!\n", False
        crc_init = (p[16] << 16) | (p[17] << 8) | p[18]
        return (f"InitA:{_rev(p[:6])} AdvA:{_rev(p[6:12])} AA:{_rev(p[12:16])} CRCInit:{crc_init:06x} WSize:{p[19]:02x} "
                f"WOffset:{_le16(p, 20):04x} Itrvl:{_le16(p, 22):04x} Ltncy:{_le16(p, 24):04x} Timot:{_le16(p, 26):04x} "
                f"ChM:{_rev(p[28:33])} Hop:{p[33] & 0x1F} SCA:{(p[33] >> 5) & 7}"), True
    return f"Byte:{_hx(p)}", True


def _ll_body(llid: int, p: bytes) -> tuple[str, bool]:
    """Text after 'PloadL%d ' for a data-channel PDU (print_ll_pdu_payload, btle_rx.c:1850-1958).
    The ' CRC%d' suffix is appended by the caller; an empty payload prints 'CRC%d' directly after
    the prefix (1864-1867)."""
    n = len(p)
    if n == 0:
        if llid in (2, 3):                                                # btle_rx.c:1587-1594
            return f"Error: LL PDU TYPE{llid}({LL_PDU_TYPE_STR[llid]}) should not have payload length 0!\n", False
        return "", True
    if llid != 3:
        return f"LL_Data:{_hx(p)}", True
    op = p[0]
    if op in _LL_CTRL_LEN and n != _LL_CTRL_LEN[op]:
        return f"Error: LL CTRL PDU TYPE{op}({LL_CTRL_STR[op]}) should have payload length {_LL_CTRL_LEN[op]}!\n", False
    name = LL_CTRL_STR[op if op <= 13 else 14]
    head = f"Op{op:02x}({name})"
    if op == 0:
        return (f"{head} WSize:{p[1]:02x} WOffset:{_le16(p, 2):04x} Itrvl:{_le16(p, 4):04x} Ltncy:{_le16(p, 6):04x} "
                f"Timot:{_le16(p, 8):04x} Inst:{_le16(p, 10):04x}"), True
    if op == 1:
        return f"{head} ChM:{_rev(p[1:6])} Inst:{_le16(p, 6):04x}", True
    if op in (2, 7, 13):
        return f"{head} Err:{p[1]:02x}", True
    if op == 3:
        return f"{head} Rand:{_rev(p[1:9])} EDIV:{_rev(p[9:11])} SKDm:{_rev(p[11:19])} IVm:{_rev(p[19:23])}", True
    if op == 4:
        return f"{head} SKDs:{_rev(p[1:9])} IVs:{_rev(p[9:13])}", True
    if op in (5, 6, 10, 11):
        return head, True
    if op in (8, 9):
        return f"{head} FteurSet:{_rev(p[1:9])}", True
    if op == 12:
        return f"{head} Ver:{p[1]:02x} CompId:{_le16(p, 2):04x} SubVer:{_le16(p, 4):04x}", True
    return f"{head} Byte:{_hx(p[1:])}", True


def btle_rx_line(frame, pkt_count: int, timestamp: tuple[int, int] | float | None = None) -> str:
    """One stdout line of ``btle_rx`` for a BLE frame record (including the trailing newline).

    `timestamp` is the (sec, usec) printed as token 0 -- the reference prints gettimeofday() at
    decode time (btle_rx.c:2130-2137), so it is not part of the parity contract; default = now.
    """
    if timestamp is None:
        timestamp = time.time()
    if isinstance(timestamp, (int, float)):
        sec = int(timestamp)
        usec = int(round((timestamp - sec) * 1e6)) % 1_000_000
    else:
        sec, usec = timestamp
    ch = int(frame["channel"])
    b = bytes(frame["bytes"][: int(frame["len"])])
    hdr, payload = b[:2], b[2:-3]
    crc_flag = 0 if int(frame["crc_ok"]) else 1
    out = f"{sec}.{usec:06d} Pkt{pkt_count} Ch{ch} AA:{int(frame['access_addr']):08x} "
    if ch in (37, 38, 39):                                                # adv_flag, btle_rx.c:2034
        t = hdr[0] & 0x0F
        plen = hdr[1] & 0x3F
        out += f"ADV_PDU_t{t}:{ADV_PDU_TYPE_STR[t]} T{int(bool(hdr[0] & 0x40))} R{int(bool(hdr[0] & 0x80))} PloadL{plen} "
        body, complete = _adv_body(t, payload)
        return out + body + (f" CRC{crc_flag}\n" if complete else "")
    llid = hdr[0] & 3
    plen = hdr[1] & 0x1F
    out += (f"LL_PDU_t{llid}:{LL_PDU_TYPE_STR[llid]} NESN{int(bool(hdr[0] & 4))} SN{int(bool(hdr[0] & 8))} "
            f"MD{int(bool(hdr[0] & 0x10))} PloadL{plen} ")
    body, complete = _ll_body(llid, payload)
    if not complete:
        return out + body
    return out + (f"{body} CRC{crc_flag}\n" if body else f"CRC{crc_flag}\n")


def btle_rx_lines(frames: np.ndarray, first_pkt: int = 1, timestamp=None) -> list[str]:
    """Lines for the BLE frames of one channel in record order; Pkt numbers count up from
    `first_pkt` across calls exactly like the reference's static pkt_count (btle_rx.c:2021,2126)."""
    return [btle_rx_line(f, first_pkt + i, timestamp) for i, f in enumerate(frames)]


BTLE_RX_BANNER = "BLE sniffer. Xianjun Jiao. putaoshu@msn.com\n\n"          # btle_rx.c:1186


def strip_timestamp(line: str) -> str:
    """Drop token 0 (wall-clock time) so lines can be compared across runs."""
    return line.split(" ", 1)[1] if " " in line else line


# ---------------------------------------------------------------------------------- BLE pcap (btle_rx -s)
PCAP_HDR_BLE = bytes.fromhex("a1b2c3d4" "0002" "0004" "00000000" "00000000" "000005dc" "00000100")   # btle_rx.c:129


# LINKTYPE_BLUETOOTH_LE_LL_WITH_PHDR flags: de-whitened, signal power valid, noise power valid
PHDR_DEWHITENED, PHDR_SIGNAL_VALID, PHDR_NOISE_VALID = 0x0001, 0x0002, 0x0004


def _dbm_i8(db, offset: float) -> np.ndarray:
    """int8(round(dB + offset)), clamped to the int8 range; NaN reads 0."""
    v = np.nan_to_num(np.asarray(db, dtype=np.float64) + offset, nan=0.0)
    return np.clip(np.rint(v), -128, 127).astype(np.int8).view(np.uint8)


def ble_pcap_record(frame, ts: tuple[int, int] = (0, 0), rf=None, dbm_offset: float = 0.0) -> bytes:
    """One record of the file btle_rx -s writes (btle_rx.c:150-163): 16-byte record header whose
    lengths are big-endian (htonl) -- sec/usec are uninitialised stack in the reference, here the
    caller's `ts` in native order as fwrite() of the struct would store them -- then the 10-byte
    LINKTYPE_BLUETOOTH_LE_LL_WITH_PHDR header {channel,0,0,0,0,0,0,0,1,0}, the access address as
    the host stores a uint32 (little endian), and header+payload (no CRC).
    `rf`: the frame's radio metrics (_abi.RF_DTYPE record): signal / noise power go into PHDR bytes 1 / 2 as
    int8(round(dBFS + dbm_offset)) and the flags gain 0x0002 / 0x0004 for the valid ones.  dBFS + an offset is not a
    calibrated dBm: the offset is the caller's estimate of the front end's gain."""
    b = bytes(frame["bytes"][: int(frame["len"]) - 3])
    n = 10 + 4 + len(b)
    rec = struct.pack("<ii", ts[0], ts[1]) + struct.pack(">ii", n, n)
    phdr = bytearray([int(frame["channel"]) & 0xFF, 0, 0, 0, 0, 0, 0, 0, 1, 0])
    if rf is not None:
        valid = int(rf["valid"])
        if valid & RF_POWER:
            phdr[1] = int(_dbm_i8(rf["power_dbfs"], dbm_offset))
            phdr[8] |= PHDR_SIGNAL_VALID
        if valid & RF_NOISE:
            phdr[2] = int(_dbm_i8(rf["noise_dbfs"], dbm_offset))
            phdr[8] |= PHDR_NOISE_VALID
    return rec + bytes(phdr) + struct.pack("<I", int(frame["access_addr"])) + b


def _pack_records(prefix: np.ndarray, payload: np.ndarray, lens: np.ndarray, plens: np.ndarray | None = None) -> bytes:
    """Concatenation of [prefix[i, :plens[i]] | payload[i, :lens[i]]] over all i (plens None: whole prefix rows), built
    with numpy only (no per-record Python objects): the batch form of the record writers below (SURVEY 8f N2: at
    10^5..10^7 frames per second a Python object per packet is the bottleneck of the pcap / RFtap consumers)."""
    n, P = prefix.shape
    if n == 0:
        return b""
    lens = lens.astype(np.int64)
    pl = np.full(n, P, dtype=np.int64) if plens is None else plens.astype(np.int64)
    rec = pl + lens
    start = np.concatenate(([0], np.cumsum(rec)[:-1]))
    out = np.empty(int(rec.sum()), dtype=np.uint8)
    keep = np.arange(P)[None, :] < pl[:, None]
    out[(start[:, None] + np.arange(P)[None, :])[keep]] = prefix[keep]
    rows = np.repeat(np.arange(n), lens)
    cols = np.arange(int(lens.sum())) - np.repeat(np.cumsum(lens) - lens, lens)
    out[np.repeat(start + pl, lens) + cols] = payload[rows, cols]
    return out.tobytes()


def ble_pcap_block(frames: np.ndarray, ts: tuple[int, int] = (0, 0), rf=None, dbm_offset: float = 0.0) -> bytes:
    """All BLE records of `frames` as btle_rx -s writes them: byte-identical to b"".join(ble_pcap_record(f, ts, r)).
    `rf`: radio metrics aligned with `frames` (RxEngine.frame_rf())."""
    sel = frames["proto"] == PROTO_BLE
    f = frames[sel]
    n = len(f)
    lens = f["len"].astype(np.int64) - 3
    prefix = np.zeros((n, 16 + 10 + 4), dtype=np.uint8)
    prefix[:, 0:8] = np.frombuffer(struct.pack("<ii", ts[0], ts[1]), dtype=np.uint8)
    be = (10 + 4 + lens).astype(">i4").view(np.uint8).reshape(n, 4)
    prefix[:, 8:12], prefix[:, 12:16] = be, be
    prefix[:, 16] = f["channel"].astype(np.uint8)
    prefix[:, 24] = PHDR_DEWHITENED
    if rf is not None:
        r = np.asarray(rf)[sel]
        p_ok, n_ok = (r["valid"] & RF_POWER) != 0, (r["valid"] & RF_NOISE) != 0
        prefix[:, 17] = np.where(p_ok, _dbm_i8(r["power_dbfs"], dbm_offset), 0)
        prefix[:, 18] = np.where(n_ok, _dbm_i8(r["noise_dbfs"], dbm_offset), 0)
        prefix[:, 24] |= np.where(p_ok, PHDR_SIGNAL_VALID, 0).astype(np.uint8) | np.where(n_ok, PHDR_NOISE_VALID, 0).astype(np.uint8)
    prefix[:, 26:30] = f["access_addr"].astype("<u4").view(np.uint8).reshape(n, 4)
    return _pack_records(prefix, f["bytes"], lens)


# LINKTYPE_BLUETOOTH_LE_LL_WITH_PHDR flags bits 7..9: PDU type (1 = auxiliary advertising); bits 14..15: PHY (0 = LE 1M,
# 1 = LE 2M, 2 = LE Coded) -- the link-type definition published by tcpdump.org
PHDR_PDU_TYPE_SHIFT, PHDR_PDU_AUX_ADV, PHDR_PHY_SHIFT = 7, 1, 14


def ble_pcap_aux_block(aux: np.ndarray, ts: tuple[int, int] = (0, 0)) -> bytes:
    """The auxiliary packets of RxEngine.ble_aux() that were decoded (status OK) by the first entry to find them, as records
    of the file btle_rx -s writes (see ble_pcap_record): PHDR {channel, 0, 0, 0, 0, 0, 0, 0, flags}, flags = de-whitened |
    PDU type 1 (auxiliary advertising) << 7 | PHY << 14, then the advertising access address and header | payload (no
    CRC).  CRC-failed packets are written too, as btle_rx writes its CRC-failed frames."""
    sel = (aux["status"] == AUX_OK) & (aux["first"] == np.arange(len(aux)))
    a = aux[sel]
    n = len(a)
    lens = a["len"].astype(np.int64) - 3
    prefix = np.zeros((n, 16 + 10 + 4), dtype=np.uint8)
    prefix[:, 0:8] = np.frombuffer(struct.pack("<ii", ts[0], ts[1]), dtype=np.uint8)
    be = (10 + 4 + lens).astype(">i4").view(np.uint8).reshape(n, 4)
    prefix[:, 8:12], prefix[:, 12:16] = be, be
    prefix[:, 16] = a["channel"]
    flags = PHDR_DEWHITENED | (PHDR_PDU_AUX_ADV << PHDR_PDU_TYPE_SHIFT) | (a["phy"].astype(np.int64) << PHDR_PHY_SHIFT)
    prefix[:, 24:26] = flags.astype("<u2").view(np.uint8).reshape(n, 2)
    prefix[:, 26:30] = np.frombuffer(struct.pack("<I", 0x8E89BED6), dtype=np.uint8)
    return _pack_records(prefix, a["bytes"], lens)


PHDR_PDU_PRIMARY_ADV = 0


def ble_pcap_coded_block(lst: np.ndarray, ts: tuple[int, int] = (0, 0), crc_failed_primaries: bool = True) -> bytes:
    """The packets of RxEngine.ble_coded() that were decoded (status OK) by the first entry to find them, as records of the
    file btle_rx -s writes: PHDR {channel, 0 x 7, flags}, flags = de-whitened | PDU type << 7 (0 = primary advertising for
    the ADV_EXT_INDs of depth 0, 1 = auxiliary advertising) | PHY << 14, then the advertising access address, for LE Coded
    one Coding Indicator byte (0 = S=8, 1 = S=2), then header | payload (no CRC).  crc_failed_primaries=False leaves out the
    primaries whose CRC failed (most are positions inside an S=8 packet's own body: DESIGN 4)."""
    sel = (lst["status"] == AUX_OK) & (lst["first"] == np.arange(len(lst)))
    if not crc_failed_primaries:
        sel &= (lst["depth"] > 0) | (lst["crc_ok"] == 1)
    a = lst[sel]
    n = len(a)
    coded = a["phy"] == AUX_PHY_CODED
    lens = a["len"].astype(np.int64) - 3
    plens = 16 + 10 + 4 + coded.astype(np.int64)
    prefix = np.zeros((n, 16 + 10 + 4 + 1), dtype=np.uint8)
    prefix[:, 0:8] = np.frombuffer(struct.pack("<ii", ts[0], ts[1]), dtype=np.uint8)
    be = (plens - 16 + lens).astype(">i4").view(np.uint8).reshape(n, 4)
    prefix[:, 8:12], prefix[:, 12:16] = be, be
    prefix[:, 16] = a["channel"]
    pdu_type = np.where(a["depth"] == 0, PHDR_PDU_PRIMARY_ADV, PHDR_PDU_AUX_ADV).astype(np.int64)
    flags = PHDR_DEWHITENED | (pdu_type << PHDR_PDU_TYPE_SHIFT) | (a["phy"].astype(np.int64) << PHDR_PHY_SHIFT)
    prefix[:, 24:26] = flags.astype("<u2").view(np.uint8).reshape(n, 2)
    prefix[:, 26:30] = np.frombuffer(struct.pack("<I", 0x8E89BED6), dtype=np.uint8)
    prefix[:, 30] = a["ci"]
    return _pack_records(prefix, a["bytes"], lens, plens)


def ble_pcap_sync_block(sync: np.ndarray, ts: tuple[int, int] = (0, 0)) -> bytes:
    """The AUX_SYNC_INDs of RxEngine.ble_periodic() that were decoded (status OK), as records of the file btle_rx -s writes:
    PHDR {channel, 0 x 7, flags}, flags = de-whitened | PDU type 1 (auxiliary advertising) << 7 | PHY << 14, then the
    train's access address and header | payload (no CRC).  CRC-failed packets are written too."""
    a = sync[sync["status"] == AUX_OK]
    n = len(a)
    lens = a["len"].astype(np.int64) - 3
    prefix = np.zeros((n, 16 + 10 + 4), dtype=np.uint8)
    prefix[:, 0:8] = np.frombuffer(struct.pack("<ii", ts[0], ts[1]), dtype=np.uint8)
    be = (10 + 4 + lens).astype(">i4").view(np.uint8).reshape(n, 4)
    prefix[:, 8:12], prefix[:, 12:16] = be, be
    prefix[:, 16] = a["channel"]
    flags = PHDR_DEWHITENED | (PHDR_PDU_AUX_ADV << PHDR_PDU_TYPE_SHIFT) | (a["phy"].astype(np.int64) << PHDR_PHY_SHIFT)
    prefix[:, 24:26] = flags.astype("<u2").view(np.uint8).reshape(n, 2)
    prefix[:, 26:30] = a["access_addr"].astype("<u4").view(np.uint8).reshape(n, 4)
    return _pack_records(prefix, a["bytes"], lens)


def sync_line(train: dict, ev: dict) -> str:
    """btle_rx --periodic line of one decoded AUX_SYNC_IND (a train of messages.ble_periodic_adv and one of its events),
    8 tokens: SYNC Ch<ch> PHY<1M|2M> AA:<hex> Evt<counter> Int<interval> PloadL<len> CRC<0 ok|1 failed>."""
    return (f"SYNC Ch{ev['channel']} PHY{train['phy']} AA:{train['access_addr']:08x} Evt{ev['event_counter']} Int{train['interval']} "
            f"PloadL{ev['pload_len']} CRC{0 if ev['crc_ok'] else 1}\n")


# the LINKTYPE_BLUETOOTH_LE_LL_WITH_PHDR PDU type of broadcast isochronous PDUs, as read from the link-type page (not checked
# against a dissector here)
PHDR_PDU_BIS = 6


def ble_pcap_bis_block(bis: np.ndarray, ts: tuple[int, int] = (0, 0)) -> bytes:
    """The BIS PDUs of RxEngine.ble_bis() that were decoded (status OK), as records of the file btle_rx -s writes: PHDR
    {channel, 0 x 7, flags}, flags = de-whitened | PDU type 6 (broadcast isochronous) << 7 | PHY << 14, then the BIS's access
    address and header | payload (no CRC).  CRC-failed PDUs are written too; an encrypted payload is written as sent."""
    a = bis[bis["status"] == AUX_OK]
    n = len(a)
    lens = a["len"].astype(np.int64) - 3
    prefix = np.zeros((n, 16 + 10 + 4), dtype=np.uint8)
    prefix[:, 0:8] = np.frombuffer(struct.pack("<ii", ts[0], ts[1]), dtype=np.uint8)
    be = (10 + 4 + lens).astype(">i4").view(np.uint8).reshape(n, 4)
    prefix[:, 8:12], prefix[:, 12:16] = be, be
    prefix[:, 16] = a["channel"]
    flags = PHDR_DEWHITENED | (PHDR_PDU_BIS << PHDR_PDU_TYPE_SHIFT) | (a["phy"].astype(np.int64) << PHDR_PHY_SHIFT)
    prefix[:, 24:26] = flags.astype("<u2").view(np.uint8).reshape(n, 2)
    prefix[:, 26:30] = a["access_addr"].astype("<u4").view(np.uint8).reshape(n, 4)
    return _pack_records(prefix, a["bytes"], lens)


def bis_line(big: dict, stream: dict, pdu: dict) -> str:
    """btle_rx --bis line of one decoded BIS PDU (a BIG of messages.ble_broadcast_iso, one of its streams and one of its
    PDUs), 9 tokens: BIS Ch<ch> PHY<1M|2M> AA:<hex> BIS<n> Evt<counter> Se<subevent> PloadL<len> CRC<0 ok|1 failed>."""
    return (f"BIS Ch{pdu['channel']} PHY{big['phy']} AA:{stream['access_addr']:08x} BIS{stream['bis']} Evt{pdu['event_counter']} "
            f"Se{pdu['subevent']} PloadL{pdu['pload_len']} CRC{0 if pdu['crc_ok'] else 1}\n")


def coded_line(d: dict) -> str:
    """btle_rx --coded line of one primary LE Coded ADV_EXT_IND (a messages.ble_coded_adv dictionary of depth 0), 8 tokens:
    CODED Ch<37..39> S<8|2> AdvA:<address or -> ADI:<DID>/<SID> (hex, - if absent) PloadL<len> CRC<0 ok|1 failed> AAerr<d>."""
    adi = f"{d['did']:03x}/{d['sid']:x}" if d["adi"] is not None else "-/-"
    return (f"CODED Ch{d['channel']} S{d['s']} AdvA:{d['adv_a'] or '-'} ADI:{adi} PloadL{d['pload_len']} "
            f"CRC{0 if d['crc_ok'] else 1} AAerr{d['aa_errors']}\n")


def aux_line(d: dict) -> str:
    """btle_rx --aux line of one decoded auxiliary packet (a messages.ble_ext_adv dictionary), 8 tokens:
    AUX Ch<ch> PHY<1M|2M> AdvA:<address or -> ADI:<DID>/<SID> (hex, - if absent) Depth<d> PloadL<len> CRC<0 ok|1 failed>."""
    adi = f"{d['did']:03x}/{d['sid']:x}" if d["adi"] is not None else "-/-"
    return (f"AUX Ch{d['channel']} PHY{d['phy']} AdvA:{d['adv_a'] or '-'} ADI:{adi} Depth{d['depth']} "
            f"PloadL{d['pload_len']} CRC{0 if d['crc_ok'] else 1}\n")


def write_ble_pcap(fh: BinaryIO, frames: Iterable, header: bool = True, rf=None, dbm_offset: float = 0.0) -> int:
    if header:
        fh.write(PCAP_HDR_BLE)
    frames = np.asarray(frames)
    fh.write(ble_pcap_block(frames, rf=rf, dbm_offset=dbm_offset))
    return int((frames["proto"] == PROTO_BLE).sum())


# ---------------------------------------------------------------------------------- Zigbee datagrams
RFTAP_MAGIC = b"RFta"
DLT_IEEE802_15_4_WITHFCS = 195
DLT_RFTAP = 215


# RFtap flag bits of the fields written here (layers/rftap.py)
RFTAP_DLT, RFTAP_FREQOFS, RFTAP_POWER, RFTAP_NOISE, RFTAP_SNR, RFTAP_QUAL = 0x0100, 0x0800, 0x2000, 0x4000, 0x8000, 0x0001


def rftap_datagram(frame, rf=None, dbm_offset: float = 0.0) -> bytes:
    """RFtap header + PSDU: what rftap_encap(2, 195, '') emits for a PDU whose meta carries
    qual = lqi / 255.0 (epy_block_0.py:21).  16-byte header: magic, length32 = 4, flags = dlt | qual
    (0x0101), dlt = 195, qual as float32 -- equal to the records of scapy's test/rftap.pcap.
    `rf`: the frame's radio metrics (_abi.RF_DTYPE record): the valid ones are added as freqofs (float64, Hz), power and
    noise (float32, dBFS + dbm_offset) and snr (float32, dB), in RFtap field order, and length32 grows to match."""
    return _rftap_header(int(frame["lqi"]), rf, dbm_offset) + bytes(frame["bytes"][: int(frame["len"])])


def _rftap_header(lqi: int, rf, dbm_offset: float) -> bytes:
    flags, body = RFTAP_DLT | RFTAP_QUAL, struct.pack("<I", DLT_IEEE802_15_4_WITHFCS)
    if rf is not None:
        valid = int(rf["valid"])
        if valid & RF_CFO:
            flags |= RFTAP_FREQOFS
            body += struct.pack("<d", float(rf["cfo_hz"]))
        if valid & RF_POWER:
            flags |= RFTAP_POWER
            body += struct.pack("<f", float(rf["power_dbfs"]) + dbm_offset)
        if valid & RF_NOISE:
            flags |= RFTAP_NOISE
            body += struct.pack("<f", float(rf["noise_dbfs"]) + dbm_offset)
        if valid & RF_POWER and valid & RF_NOISE:
            flags |= RFTAP_SNR
            body += struct.pack("<f", float(rf["snr_db"]))
    body += struct.pack("<f", np.float32(lqi / 255.0))
    return RFTAP_MAGIC + struct.pack("<HH", 2 + len(body) // 4, flags) + body


def gnuradio_packet(frame) -> bytes:
    """8-byte GnuradioPacket header + payload (layers/gnuradio.py:19-25).  Zigbee: {2,0,0,0,0,0,0,0} +
    PSDU as packet_sink_scapy_impl.cc:333-349 publishes; BLE (proto 3): access address (LE) + PDU + CRC
    as gr-bt4le's sink lays it out (gr-bt4le/lib/packet_sink_impl.cc:102-108,332)."""
    proto = int(frame["proto"])
    body = bytes(frame["bytes"][: int(frame["len"])])
    if proto == PROTO_BLE:
        body = struct.pack("<I", int(frame["access_addr"])) + body
    return bytes([proto, 0, 0, 0, 0, 0, 0, 0]) + body


def parse_rftap(datagram: bytes) -> dict:
    """Minimal RFtap reader (layers/rftap.py field order) used by the tests and the pcap tools."""
    if datagram[:4] != RFTAP_MAGIC:
        raise ValueError("not an RFtap datagram")
    len32, flags = struct.unpack_from("<HH", datagram, 4)
    off = 8
    out = {"length32": len32, "flags": flags}
    if flags & 0x0100:
        out["dlt"] = struct.unpack_from("<I", datagram, off)[0]
        off += 4
    for bit, name in ((0x0200, "freq"), (0x0400, "nomfreq"), (0x0800, "freqofs")):
        if flags & bit:
            out[name] = struct.unpack_from("<d", datagram, off)[0]
            off += 8
    for bit, name in ((0x2000, "power"), (0x4000, "noise"), (0x8000, "snr"), (0x0001, "qual")):
        if flags & bit:
            out[name] = struct.unpack_from("<f", datagram, off)[0]
            off += 4
    out["payload"] = datagram[4 * len32:]
    return out


# ---------------------------------------------------------------------------------- Zigbee pcap (wrpcap)
def pcap_global_header(linktype: int, snaplen: int = 65535) -> bytes:
    """Little-endian classic pcap header as scapy's PcapWriter writes it (magic a1b2c3d4, v2.4)."""
    return struct.pack("<IHHiIII", 0xA1B2C3D4, 2, 4, 0, 0, snaplen, linktype)


def pcap_record(data: bytes, ts: float = 0.0) -> bytes:
    sec = int(ts)
    usec = int(round((ts - sec) * 1e6))
    return struct.pack("<IIII", sec, usec, len(data), len(data)) + data


def zigbee_pcap_block(frames: np.ndarray, ts=None, sample_rate: float = 4e6) -> bytes:
    """All 802.15.4 records of `frames` as DLT-195 pcap records: byte-identical to
    b"".join(pcap_record(psdu, base + sample_index / rate))."""
    f = frames[frames["proto"] == PROTO_ZIGBEE]
    n = len(f)
    lens = f["len"].astype(np.int64)
    t = float(ts or 0.0) + np.maximum(0, f["sample_index"].astype(np.int64)) / sample_rate
    sec = t.astype(np.int64)
    usec = np.rint((t - sec) * 1e6).astype(np.int64)
    prefix = np.stack([sec, usec, lens, lens], axis=1).astype("<u4").view(np.uint8).reshape(n, 16)
    return _pack_records(prefix, f["bytes"], lens)


def rftap_block(frames: np.ndarray, rf=None, dbm_offset: float = 0.0) -> tuple[bytes, np.ndarray]:
    """The RFtap datagrams (rftap_datagram) of all 802.15.4 records back to back + the offsets where each starts
    (n + 1 entries), for senders that batch their socket writes.  `rf`: radio metrics aligned with `frames`."""
    sel = frames["proto"] == PROTO_ZIGBEE
    f = frames[sel]
    n = len(f)
    lens = f["len"].astype(np.int64)
    if rf is not None:
        return _rftap_block_rf(f, np.asarray(rf)[sel], lens, dbm_offset)
    prefix = np.zeros((n, 16), dtype=np.uint8)
    prefix[:, 0:12] = np.frombuffer(RFTAP_MAGIC + struct.pack("<HHI", 4, 0x0101, DLT_IEEE802_15_4_WITHFCS), dtype=np.uint8)
    prefix[:, 12:16] = (f["lqi"].astype(np.int64) / 255.0).astype("<f4").view(np.uint8).reshape(n, 4)
    return _pack_records(prefix, f["bytes"], lens), np.concatenate(([0], np.cumsum(16 + lens)))


def _rftap_block_rf(f: np.ndarray, r: np.ndarray, lens: np.ndarray, dbm_offset: float) -> tuple[bytes, np.ndarray]:
    """rftap_block with radio metrics: the header of every record holds the fields its valid bits allow."""
    n = len(f)
    v = r["valid"].astype(np.int64)
    has_cfo, has_p, has_n = (v & RF_CFO) != 0, (v & RF_POWER) != 0, (v & RF_NOISE) != 0
    has_snr = has_p & has_n
    prefix = np.zeros((n, 40), dtype=np.uint8)
    col = np.full(n, 12, dtype=np.int64)                       # magic, length32, flags, dlt written below
    rows = np.arange(n)

    def put(mask, values: np.ndarray):
        b = values.view(np.uint8).reshape(n, -1)
        w = b.shape[1]
        idx = col[mask][:, None] + np.arange(w)[None, :]
        prefix[rows[mask][:, None], idx] = b[mask]
        col[mask] += w

    put(has_cfo, r["cfo_hz"].astype("<f8"))
    put(has_p, (r["power_dbfs"].astype(np.float64) + dbm_offset).astype("<f4"))
    put(has_n, (r["noise_dbfs"].astype(np.float64) + dbm_offset).astype("<f4"))
    put(has_snr, r["snr_db"].astype("<f4"))
    put(np.ones(n, dtype=bool), (f["lqi"].astype(np.int64) / 255.0).astype("<f4"))
    flags = (RFTAP_DLT | RFTAP_QUAL) + has_cfo * RFTAP_FREQOFS + has_p * RFTAP_POWER + has_n * RFTAP_NOISE + has_snr * RFTAP_SNR
    prefix[:, 0:4] = np.frombuffer(RFTAP_MAGIC, dtype=np.uint8)
    prefix[:, 4:6] = (col // 4).astype("<u2").view(np.uint8).reshape(n, 2)
    prefix[:, 6:8] = flags.astype("<u2").view(np.uint8).reshape(n, 2)
    prefix[:, 8:12] = np.frombuffer(struct.pack("<I", DLT_IEEE802_15_4_WITHFCS), dtype=np.uint8)
    return _pack_records(prefix, f["bytes"], lens, col), np.concatenate(([0], np.cumsum(col + lens)))


def write_zigbee_pcap(fh: BinaryIO, frames: Iterable, ts=None, sample_rate: float = 4e6, header: bool = True) -> int:
    """DLT 195 pcap of the PSDUs (FCS included).  Time stamps: capture-relative, from the frame's
    sample index, unless `ts` (a base epoch) is given."""
    if header:
        fh.write(pcap_global_header(DLT_IEEE802_15_4_WITHFCS))
    frames = np.asarray(frames)
    fh.write(zigbee_pcap_block(frames, ts, sample_rate))
    return int((frames["proto"] == PROTO_ZIGBEE).sum())


def read_pcap(data: bytes) -> tuple[int, list[tuple[float, bytes]]]:
    """(linktype, [(ts, bytes)]) of a classic pcap in either byte order."""
    magic = data[:4]
    if magic == b"\xd4\xc3\xb2\xa1":
        e = "<"
    elif magic == b"\xa1\xb2\xc3\xd4":
        e = ">"
    else:
        raise ValueError("not a pcap file")
    linktype = struct.unpack_from(e + "I", data, 20)[0]
    off, out = 24, []
    while off + 16 <= len(data):
        sec, usec, caplen, _ = struct.unpack_from(e + "IIII", data, off)
        out.append((sec + usec * 1e-6, data[off + 16: off + 16 + caplen]))
        off += 16 + caplen
    return linktype, out

"""Batch builders of Snout's per-packet message objects from GPU-decoded records (SURVEY 8(f) N2).

`snout zigbee scan` turns every datagram of the receive flowgraph into scapy objects one at a time
(snout/util/zigbee.py:194-202 handle_packet: RFtap(pkt), wrpcap(pkt.payload); snout/core/message.py:258-304
ZigbeeMessage.fromraw: sender = src_addr, receiver = dest_addr, seq_number = seqnum, pan = {src_panid, dest_panid},
rftap = the RFtap fields, vuln = {'zll': haslayer(ZLLScanResponse)}; snout/util/zigbee.py:176-192 collects the ZLL scan
responses of a touchlink scan).  Here the MAC headers of a whole batch are read on the GPU (RxEngine.zb_mac_summary ->
csrc/zb_mac.cuh) and the same dictionaries are built from the summary rows without any per-packet dissection."""
from __future__ import annotations

import numpy as np

from . import _abi


def _addr(value: int, mode: int):
    """An address the way scapy's dot15d4AddressField holds it: an int (16 or 64 bit), None when absent."""
    return int(value) if mode in (2, 3) else None


def zigbee_messages(frames: np.ndarray, mac: np.ndarray, timestamp: float | None = None) -> list[dict]:
    """One dictionary per 802.15.4 record with the keyword arguments ZigbeeMessage.fromraw (message.py:286-303) passes to
    ZigbeeMessage(...): sender, receiver, seq_number, timestamp, pan, rftap, vuln -- plus channel, crc_ok and the record index.
    `frames`: records of a batch (RxEngine.poll), `mac`: RxEngine.zb_mac_summary() of the same batch."""
    out = []
    P = _abi
    for f, m in zip(frames, mac):
        if m["present"] & P.ZBMAC_NOT_ZIGBEE:
            continue
        pr = int(m["present"])
        out.append(dict(
            sender=_addr(m["src_addr"], int(m["src_mode"])) if pr & P.ZBMAC_SRC_ADDR else None,
            receiver=_addr(m["dest_addr"], int(m["dest_mode"])) if pr & P.ZBMAC_DEST_ADDR else None,
            seq_number=int(m["seqnum"]),
            timestamp=timestamp,
            pan=dict(src_panid=int(m["src_panid"]) if pr & P.ZBMAC_SRC_PANID else None,
                     dest_panid=int(m["dest_panid"]) if pr & P.ZBMAC_DEST_PANID else None),
            rftap=dict(dlt=195, qual=float(f["lqi"]) / 255.0),                       # epy_block_0.py:21, rftap_encap(2, 195)
            vuln=dict(zll=bool(pr & P.ZBMAC_ZLL_SCAN_RESPONSE)),
            channel=int(f["channel"]), crc_ok=bool(f["crc_ok"]), frame_type=int(m["frame_type"]), record=int(m["frame"]),
        ))
    return out


def zll_scan_responses(frames: np.ndarray, mac: np.ndarray) -> list[dict]:
    """What ZigbeeZLLScan.handle_packet keeps (zigbee.py:176-192): {'pkt': the 802.15.4 frame, 'qual', 'channel'} for every
    record whose dissection holds a ZLLScanResponse."""
    sel = (mac["present"] & _abi.ZBMAC_ZLL_SCAN_RESPONSE) != 0
    return [dict(pkt=bytes(f["bytes"][: int(f["len"])]), qual=float(f["lqi"]) / 255.0, channel=int(f["channel"]))
            for f in frames[mac["frame"][sel]]]


# ----------------------------------------------------------------------------------------------------- SURVEY 8(f) N1
# A few well-known Bluetooth SIG company identifiers; a Snout installation passes its own table
# (snout.core.protocols.btle.assigned_numbers.company_ids) as `company_names`.
COMPANY_NAMES = {0x0006: "Microsoft", 0x004C: "Apple, Inc.", 0x0075: "Samsung Electronics Co. Ltd.", 0x00E0: "Google", 0x0087: "Garmin International, Inc.",
                 0x0059: "Nordic Semiconductor ASA"}
_OS_TEXT = {_abi.OS_NONE: "-", _abi.OS_UNDECIDED: "-", _abi.OS_IOS10: "iOS 10", _abi.OS_IOS11: "iOS 11", _abi.OS_IOS12: "iOS 12",
            _abi.OS_WINDOWS10: "Windows 10 >= v10.0.10240.0"}
_MODEL_TEXT = {_abi.MODEL_NONE: "-", _abi.MODEL_FITBIT_CHARGE: "Charge / Charge HR", _abi.MODEL_AIRPODS: "AirPods"}


def device_fingerprints(devices: np.ndarray, company_names: dict | None = None) -> list[dict]:
    """Device.vendor / .model / .os (snout/core/device.py:171-246) of every row of the GPU sender table (RxEngine.devices()):
    the three answers are decided on the GPU by each sender's FIRST deciding packet (csrc/ble_adv.cuh); this only renders the
    text.  Unknown company ids read '??' as in the reference (advertising.py:225)."""
    names = COMPANY_NAMES if company_names is None else company_names
    out = []
    for d in devices:
        kind = int(d["vendor_kind"])
        vendor = "-" if kind == _abi.VENDOR_NONE else "FitBit" if kind == _abi.VENDOR_FITBIT else names.get(int(d["vendor_company"]), "??")
        out.append(dict(address=bytes(d["adv_a"])[::-1].hex(), tx_add=int(d["tx_add"]), vendor=vendor, model=_MODEL_TEXT[int(d["model"])],
                        os=_OS_TEXT[int(d["os"])]))
    return out


# ----------------------------------------------------------------------------------------- BLE 5 extended advertising
def _ext_fields(pdu: bytes) -> dict:
    """Common extended advertising payload of a PDU of type 7 (header | payload | CRC): AdvMode and the flagged fields of the
    extended header in their order (Core Vol 6 Part B 2.3.4), then AdvData.  A field the header is too short for is None."""
    return _ext_walk(pdu)[0]


def _ext_walk(pdu: bytes) -> tuple[dict, bytes, bytes | None]:
    """(_ext_fields, the extended header bytes past its flagged fields -- the ACAD --, the 18-byte SyncInfo or None)."""
    n_payload = pdu[1]
    p = pdu[2:2 + n_payload]
    out = dict(adv_mode=None, adv_a=None, target_a=None, adi=None, did=None, sid=None, tx_power=None, aux_ptr=None, adv_data=b"")
    sync_info = None
    if not p:
        return out, b"", sync_info
    hlen, out["adv_mode"] = p[0] & 0x3F, p[0] >> 6
    hdr = p[1:1 + hlen]
    out["adv_data"] = bytes(p[1 + hlen:])
    if not hdr:
        return out, b"", sync_info
    flags, at = hdr[0], 1
    for bit, name, size in ((0, "adv_a", 6), (1, "target_a", 6), (2, "cte_info", 1), (3, "adi", 2), (4, "aux_ptr", 3),
                            (5, "sync_info", 18), (6, "tx_power", 1)):
        if not flags & (1 << bit):
            continue
        v = bytes(hdr[at:at + size])
        at += size
        if len(v) < size:
            break
        if name in ("adv_a", "target_a"):
            out[name] = v[::-1].hex()                         # printed most significant byte first, as btle_rx prints AdvA
        elif name == "adi":
            a = int.from_bytes(v, "little")
            out["adi"], out["did"], out["sid"] = a, a & 0x0FFF, a >> 12
        elif name == "tx_power":
            out["tx_power"] = v[0] - 256 if v[0] > 127 else v[0]
        elif name == "aux_ptr":
            out["aux_ptr"] = v
        elif name == "sync_info":
            sync_info = v
    return out, bytes(hdr[at:]), sync_info


_PHY_NAMES = {_abi.AUX_PHY_1M: "1M", _abi.AUX_PHY_2M: "2M", _abi.AUX_PHY_CODED: "Coded"}


def ble_ext_adv(aux: np.ndarray, head_depth: int = 0) -> list[dict]:
    """One dictionary per auxiliary packet of RxEngine.ble_aux() that was decoded (status OK) and is the first entry to have
    found it: index, channel, phy ('1M' / '2M' / 'Coded'), depth, crc_ok, tx_add, pload_len (header length field), adv_mode, adv_a, target_a, adi / did / sid, tx_power,
    adv_data.  The AUX_ADV_INDs (depth 0) also carry `chain` (the list indices of the chain from it) and `chain_data`: the
    AdvData of the whole chain reassembled in order, and `complete`: every link was received with a good CRC and the last
    one points nowhere.  head_depth: the depth of the AUX_ADV_INDs in the list (0 for RxEngine.ble_aux, 1 for
    RxEngine.ble_coded, whose primaries are depth 0)."""
    out, by_index = [], {}
    children = {int(r["parent"]): k for k, r in enumerate(aux) if int(r["depth"]) > head_depth}
    for k, r in enumerate(aux):
        if int(r["status"]) != _abi.AUX_OK or int(r["first"]) != k:
            continue
        pdu = bytes(r["bytes"][: int(r["len"])])
        d = dict(index=k, channel=int(r["channel"]), phy=_PHY_NAMES.get(int(r["phy"]), "1M"), depth=int(r["depth"]),
                 crc_ok=bool(r["crc_ok"]), tx_add=(pdu[0] >> 6) & 1, pload_len=pdu[1], sample_index=int(r["sample_index"]),
                 capture_id=int(r["capture_id"]), **_ext_fields(pdu))
        out.append(d)
        by_index[k] = d
    for d in out:
        if d["depth"] != head_depth:
            continue
        chain, data, k, complete = [d["index"]], d["adv_data"], d["index"], d["crc_ok"]
        while complete and by_index[k]["aux_ptr"] is not None:
            c = children.get(k)
            if c is None or c not in by_index or not by_index[c]["crc_ok"]:
                complete = False
                break
            chain.append(c)
            data += by_index[c]["adv_data"]
            k = c
        d["chain"], d["chain_data"], d["complete"] = chain, data, complete
    return out


def ble_coded_adv(lst: np.ndarray) -> list[dict]:
    """ble_ext_adv of RxEngine.ble_coded(): the primary ADV_EXT_INDs (depth 0) and the auxiliary packets (chains from the
    AUX_ADV_INDs at depth 1).  Coded packets also carry `s` (8 or 2, from the coding indicator) and `aa_errors` (d(n))."""
    out = ble_ext_adv(lst, head_depth=1)
    for d in out:
        r = lst[d["index"]]
        if int(r["phy"]) == _abi.AUX_PHY_CODED:
            d["s"], d["aa_errors"] = 8 if int(r["ci"]) == 0 else 2, int(r["aa_errors"])
    return out


# ----------------------------------------------------------------------------------------- BLE periodic advertising
SCA_PPM = (500, 250, 150, 100, 75, 50, 30, 20)
AD_BIGINFO = 0x2C


def sync_info_fields(b: bytes) -> dict:
    """The fields of an 18-byte SyncInfo (Core Vol 6 Part B 2.3.4.6 as read in include/snoutrx.h): offset_us (Sync Packet
    Offset x units, + 2 457 600 us with Offset Adjust), interval (1.25 ms units), used channels, sca / ppm, access_addr,
    crc_init (c0 << 16 | c1 << 8 | c2, the value RxEngine.follow takes) and pa_event_counter."""
    o = b[0] | (b[1] << 8)
    units = 300 if o & 0x2000 else 30
    v = int.from_bytes(bytes(b[4:9]), "little")
    sca = (v >> 37) & 7
    return dict(offset_us=(o & 0x1FFF) * units + (2_457_600 if o & 0x4000 else 0), offset_units_us=units,
                interval=b[2] | (b[3] << 8), channels=[c for c in range(37) if v >> c & 1], sca=sca, ppm=SCA_PPM[sca],
                access_addr=int.from_bytes(bytes(b[9:13]), "little"), crc_init=(b[13] << 16) | (b[14] << 8) | b[15],
                pa_event_counter=b[16] | (b[17] << 8))


def _ad_types(data: bytes) -> list[int]:
    """AD types of the AD structures of `data` (length | type | value), up to the first malformed one."""
    out, at = [], 0
    while at < len(data) and data[at] != 0 and at + 1 + data[at] <= len(data):
        out.append(data[at + 1])
        at += 1 + data[at]
    return out


def ble_periodic_adv(sync: np.ndarray, aux: np.ndarray | None = None) -> list[dict]:
    """One dictionary per train of RxEngine.ble_periodic() (in list order): source (aux list index), capture_id,
    access_addr, crc_init, interval (1.25 ms units) and interval_ms, channels (used), sca, ppm, phy ('1M' / '2M') and, when
    the aux list of the same batch is given, the source's adv_a / adi / did / sid.  `events` holds the train's decoded events
    (status OK), each with event (k), event_counter, channel, sample_index, crc_ok, pload_len, the extended-header fields of
    _ext_fields, adv_data, acad (the raw Additional Controller Advertising Data), big_info (an ACAD AD structure of type
    0x2C) and chained (the packet carries an AuxPtr to an AUX_CHAIN_IND, which is not followed)."""
    trains: dict = {}
    for r in sync:
        key = int(r["source"])
        if key not in trains:
            t = dict(source=key, capture_id=int(r["capture_id"]), access_addr=int(r["access_addr"]), crc_init=int(r["crc_init"]),
                     interval=int(r["interval"]), interval_ms=1.25 * int(r["interval"]), sca=int(r["sca"]), ppm=SCA_PPM[int(r["sca"])],
                     phy=_PHY_NAMES.get(int(r["phy"]), "1M"), channels=None, adv_a=None, adi=None, did=None, sid=None, events=[])
            if aux is not None and key < len(aux):
                a = aux[key]
                fields, _, si = _ext_walk(bytes(a["bytes"][: int(a["len"])]))
                t.update(adv_a=fields["adv_a"], adi=fields["adi"], did=fields["did"], sid=fields["sid"])
                if si is not None:
                    t["channels"] = sync_info_fields(si)["channels"]
            trains[key] = t
        if int(r["status"]) != _abi.AUX_OK:
            continue
        pdu = bytes(r["bytes"][: int(r["len"])])
        fields, acad, _ = _ext_walk(pdu)
        trains[key]["events"].append(dict(event=int(r["event"]), event_counter=int(r["event_counter"]), channel=int(r["channel"]),
                                          sample_index=int(r["sample_index"]), crc_ok=bool(r["crc_ok"]), pload_len=pdu[1],
                                          **fields, acad=acad, big_info=AD_BIGINFO in _ad_types(acad),
                                          chained=fields["aux_ptr"] is not None))
    return list(trains.values())


# ----------------------------------------------------------------------------------------- BLE broadcast isochronous streams
def big_info_fields(b: bytes) -> dict:
    """The fields of a 33-byte (or, encrypted, 57-byte) BIGInfo (Core Vol 6 Part B 2.3.4.8 as read in include/snoutrx.h):
    big_offset_us (BIG_Offset x units), iso_interval (1.25 ms units) and iso_interval_ms, num_bis, nse, bn, sub_interval_us,
    pto, bis_spacing_us, irc, max_pdu, seed_access_addr, sdu_interval_us, max_sdu, base_crc_init, channels (used), phy
    ('1M' / '2M' / 'Coded' / the raw value), payload_count, framed, encrypted and, when encrypted, giv and gskd."""
    def le(a, n):
        return int.from_bytes(bytes(b[a:a + n]), "little")
    w0, w1, w2, w5, w7, w8 = le(0, 4), le(4, 4), le(8, 4), le(17, 4), le(23, 5), le(28, 5)
    units = 300 if w0 >> 14 & 1 else 30
    iso = w0 >> 15 & 0xFFF
    phy = w7 >> 37 & 7
    d = dict(big_offset_us=(w0 & 0x3FFF) * units, big_offset_units_us=units, iso_interval=iso, iso_interval_ms=1.25 * iso,
             num_bis=w0 >> 27 & 0x1F, nse=w1 & 0x1F, bn=w1 >> 5 & 7, sub_interval_us=w1 >> 8 & 0xFFFFF, pto=w1 >> 28 & 0xF,
             bis_spacing_us=w2 & 0xFFFFF, irc=w2 >> 20 & 0xF, max_pdu=w2 >> 24 & 0xFF, seed_access_addr=le(13, 4),
             sdu_interval_us=w5 & 0xFFFFF, max_sdu=w5 >> 20 & 0xFFF, base_crc_init=le(21, 2),
             channels=[c for c in range(37) if w7 >> c & 1], phy=_PHY_NAMES.get(phy, phy), payload_count=w8 & ((1 << 39) - 1),
             framed=bool(w8 >> 39 & 1), encrypted=len(b) >= 57, giv=None, gskd=None)
    if d["encrypted"]:
        d["giv"], d["gskd"] = bytes(b[33:41]), bytes(b[41:57])
    return d


def _big_info_of(pdu: bytes) -> bytes | None:
    """The BIGInfo bytes of the first AD structure of type 0x2C in a PDU's ACAD (33 or 57 bytes), or None."""
    _, acad, _ = _ext_walk(pdu)
    at = 0
    while at < len(acad) and acad[at] != 0 and at + 1 + acad[at] <= len(acad):
        if acad[at + 1] == AD_BIGINFO:
            return bytes(acad[at + 2:at + 1 + acad[at]]) if acad[at] in (34, 58) else None
        at += 1 + acad[at]
    return None


def ble_broadcast_iso(bis: np.ndarray, sync: np.ndarray | None = None) -> list[dict]:
    """One dictionary per BIG of RxEngine.ble_bis() (in list order): source (periodic list index), capture_id, phy ('1M' /
    '2M'), encrypted, framed and, when the periodic list of the same batch is given, big_info (big_info_fields of the source's
    BIGInfo; None otherwise).  `streams` holds one dictionary per BIS (bis, access_addr, crc_init) with its decoded PDUs
    (status OK) in list order, each with event (k), event_counter, subevent, channel, sample_index, payload_number, llid,
    cssn, cstf, pload_len, payload (as sent: an encrypted payload keeps its MIC), crc_ok and encrypted."""
    bigs: dict = {}
    for r in bis:
        key = int(r["source"])
        if key not in bigs:
            flags = int(r["flags"])
            g = dict(source=key, capture_id=int(r["capture_id"]), phy=_PHY_NAMES.get(int(r["phy"]), "1M"),
                     encrypted=bool(flags & _abi.BIS_ENCRYPTED), framed=bool(flags & _abi.BIS_FRAMED), big_info=None, streams={})
            if sync is not None and key < len(sync):
                s = sync[key]
                b = _big_info_of(bytes(s["bytes"][: int(s["len"])]))
                if b is not None:
                    g["big_info"] = big_info_fields(b)
            bigs[key] = g
        g = bigs[key]
        n = int(r["bis"])
        if n not in g["streams"]:
            g["streams"][n] = dict(bis=n, access_addr=int(r["access_addr"]), crc_init=int(r["crc_init"]), pdus=[])
        if int(r["status"]) != _abi.AUX_OK:
            continue
        pdu = bytes(r["bytes"][: int(r["len"])])
        g["streams"][n]["pdus"].append(dict(event=int(r["event"]), event_counter=int(r["event_counter"]), subevent=int(r["subevent"]),
                                            channel=int(r["channel"]), sample_index=int(r["sample_index"]),
                                            payload_number=int(r["payload_number"]), llid=pdu[0] & 3, cssn=pdu[0] >> 2 & 7,
                                            cstf=pdu[0] >> 5 & 1, pload_len=pdu[1], payload=pdu[2:2 + pdu[1]],
                                            crc_ok=bool(r["crc_ok"]), encrypted=g["encrypted"]))
    out = []
    for g in bigs.values():
        g["streams"] = [g["streams"][n] for n in sorted(g["streams"])]
        out.append(g)
    return out

"""`btle_rx` -- drop-in for the BLE receive executable Snout spawns.

Snout runs `btle_rx -c <ch> -g 6 -a 8e89bed6 -k 555555` as a child process and parses its stdout
lines (snout/util/btle.py:53-76, snout/core/pcontroller.py:54,115, snout/core/message.py:205-237).
This module provides that executable on top of the CUDA engine:

* the option table of vendor/BTLE/host/btle-tools/src/btle_rx.c:1209-1294 (`-h -c -g -a -k -v -r -f
  -m -o -s` and their long forms), the same range checks and error texts (1295-1315), the same
  banner (1186), "Cmd line input" line (2303) and "Exit main loop ..." line (2396);
* one text line per frame in the reference format (snout_b200.formats.btle_rx_line), flushed after
  every processed shard as the reference flushes after every half buffer (2383);
* `-s FILE` writes the reference's LINKTYPE 256 pcap (126-170).

There is no SDR in the loop: IQ comes from `--iq FILE|-` (cf32 as in the BASELINE captures, or
sc8 = the HackRF's int8 stream), at 4 Msps for one channel or, with `--wideband`, at 96 Msps
centred on 2440 MHz, in which case all 40 channels are decoded at once and `-c` only selects
which channel is printed (`--all-channels` prints every channel; Pkt numbers then count per
channel as they do with one btle_rx process per channel).  `-g` and `-f` configure the radio in
the reference; here they are accepted, echoed and otherwise unused.  `-r` (raw mode) is outside
the receive path that Snout uses and is refused with a message.

`-o` (data channel tracking, receiver_controller btle_rx.c:2167-2282) works with `--wideband`: the
reference retunes its one channel on a wall-clock schedule after a CRC-ok CONNECT_REQ with a full
channel map; here every data channel is already channelized, so from the CONNECT_REQ on the batch's
bit streams are searched again with the connection's access address / CRC init (RxEngine.follow)
and every LL PDU of the connection is printed with the channel it was heard on -- no retuning, no
missed events.  The `Hop:` status lines of the reference are printed where it prints them.  With
one 4 Msps channel there is nothing to hop to and `-o` is refused.

`--aux` (with `--wideband`) also receives BLE 5 extended advertising: every ADV_EXT_IND's AuxPtr is followed to its
AUX_ADV_IND and down its AUX_CHAIN_INDs on the 1M and 2M PHYs (RxEngine.ble_aux), and every auxiliary packet found is
printed, whatever `-c` selects, as one line of 8 tokens (formats.aux_line):

    AUX Ch<ch> PHY<1M|2M> AdvA:<address or -> ADI:<DID hex>/<SID hex or -> Depth<d> PloadL<len> CRC<0|1>

It starts with AUX instead of a timestamp and a Pkt token, so a parser of the reference's lines does not take it for one.
With `-s` the packets also go to the pcap (formats.ble_pcap_aux_block).

`--coded` (with `--wideband`) also receives BLE Long Range advertising: the ADV_EXT_INDs sent on the LE Coded PHY on
channels 37..39 are found by their coded access address, Viterbi-decoded, and followed down their AuxPtrs on every PHY
(RxEngine.ble_coded).  Each primary with a good CRC is printed as one line of 8 tokens (formats.coded_line), each packet of
its chains as an AUX line (PHYCoded for LE Coded; its Depth counts from the primary, so the AUX_ADV_IND is Depth1).
Primaries whose CRC fails are left out of the lines and the pcap: most are positions inside an S=8 packet's own coded body
that come under the detection threshold (DESIGN.md 4).

    CODED Ch<37..39> S<8|2> AdvA:<address or -> ADI:<DID hex>/<SID hex or -> PloadL<len> CRC<0|1> AAerr<d>

With `-s` they also go to the pcap (formats.ble_pcap_coded_block).

`--periodic` (with `--wideband`) also receives BLE periodic advertising: the SyncInfo of every AUX_ADV_IND that ble_aux
finds describes a train of AUX_SYNC_INDs (its own access address and CRC init, a fixed interval, a CSA#2 channel per
event), and every event of the train inside the capture is searched for at its predicted place (RxEngine.ble_periodic).
Each AUX_SYNC_IND found is printed as one line of 8 tokens (formats.sync_line):

    SYNC Ch<ch> PHY<1M|2M> AA:<access address hex> Evt<paEventCounter> Int<interval, 1.25 ms units> PloadL<len> CRC<0|1>

With `-s` they also go to the pcap, with the train's access address (formats.ble_pcap_sync_block).

`--bis` (with `--wideband`) also receives BLE broadcast isochronous streams (LE Audio broadcast): the BIGInfo in the ACAD
of every AUX_SYNC_IND that ble_periodic finds describes a BIG (its BISes' access addresses and CRC inits, an ISO interval,
NSE subevents per BIS on CSA#2 subevent channels), and every subevent of the BIG inside the capture is searched for at its
predicted place (RxEngine.ble_bis).  Each BIS PDU found is printed as one line of 9 tokens (formats.bis_line):

    BIS Ch<ch> PHY<1M|2M> AA:<access address hex> BIS<n> Evt<BIG event counter> Se<subevent> PloadL<len> CRC<0|1>

Encrypted BISes are printed as sent (they are not decrypted).  With `-s` they also go to the pcap, with the BIS's access
address (formats.ble_pcap_bis_block).

There is no CPU path: without a usable GPU / libsnoutrx.so the program exits with an error.
"""
from __future__ import annotations

import getopt
import os
import sys

import numpy as np

from . import chanplan, formats, messages

DEFAULT_CHANNEL, DEFAULT_GAIN, MAX_GAIN, MAX_CHANNEL = 37, 6, 62, 39        # btle_rx.c:187,486,485,190
USAGE = """Usage:
    -h --help
      Print this help screen
    -c --chan
      Channel number. default 37. valid range 0~39
    -g --gain
      Rx gain in dB. Accepted for compatibility; the IQ source is a file or pipe
    -a --access
      Access address. 4 bytes. Hex format (like 89ABCDEF). Default 8e89bed6 for channel 37 38 39. For other channel you should pick correct value according to sniffed link setup procedure
    -k --crcinit
      CRC init value. 3 bytes. Hex format (like 555555). Default 555555 for channel 37 38 39. For other channel you should pick correct value according to sniffed link setup procedure
    -v --verbose
      Print more information when there is error
    -r --raw
      Raw mode (not supported by this engine)
    -f --freq_hz
      Accepted for compatibility (the capture is already tuned)
    -m --access_mask
      If a bit is 1 in this mask, corresponding bit in access address will be taken into packet existing decision
    -o --hop
      This will turn on data channel tracking (only with --wideband: all data channels are received at once)
    -s --filename
      Store packets to this pcap file (LINKTYPE_BLUETOOTH_LE_LL_WITH_PHDR)
    --iq FILE|-
      IQ source: interleaved samples from FILE or stdin (default: environment SNOUT_B200_IQ;
      SNOUT_B200_IQ_FORMAT and SNOUT_B200_WIDEBAND likewise preset --format / --wideband)
    --format cf32|sc8
      Sample format of the source (default cf32; sc8 = HackRF int8)
    --scale S
      Quantiser scale: q = clamp(rint(x * S), -128, 127) (default 128; 100 for --wideband)
    --wideband
      The source is a 96 Msps capture centred on 2440 MHz: decode all 40 channels at once
    --all-channels
      With --wideband: print frames of every channel, not just -c
    --device N
      CUDA device ordinal (default 0)
    --coded
      With --wideband: also receive BLE Long Range (LE Coded) ADV_EXT_INDs on 37..39 and their auxiliary packets
    --aux
      With --wideband: also follow BLE 5 extended advertising to its auxiliary packets (1M and 2M PHYs) and print them
    --periodic
      With --wideband: also follow the SyncInfo of every AUX_ADV_IND to its periodic advertising train (AUX_SYNC_IND)
    --bis
      With --wideband: also follow the BIGInfo of every AUX_SYNC_IND to its broadcast isochronous streams (BIS PDUs)
    --rf
      Measure signal power, noise floor and carrier offset of every frame; with -s the pcap's PHDR carries the
      signal and noise power (dBFS, flags 0x0002 / 0x0004).  Stdout lines are unchanged

See README for detailed information.
"""


class Options:
    chan = DEFAULT_CHANNEL
    gain = DEFAULT_GAIN
    access_addr = chanplan.BLE_ADV_AA
    crc_init = chanplan.BLE_ADV_CRC_INIT
    verbose = 0
    raw = 0
    freq_hz = 123                      # btle_rx.c:1201 sentinel
    access_mask = 0xFFFFFFFF
    hop = 0
    filename_pcap = None
    iq = None
    fmt = "cf32"
    scale = 0.0
    wideband = False
    all_channels = False
    device = 0
    shard_windows = 0
    rf = False
    aux = False
    coded = False
    periodic = False
    bis = False


def _strtol(text: str, base: int) -> int:
    """strtol() as the reference uses it: longest valid prefix, 0 if none."""
    t = text.strip().lower()
    sign = 1
    if t[:1] in "+-":
        sign = -1 if t[0] == "-" else 1
        t = t[1:]
    if base == 16 and t.startswith("0x"):
        t = t[2:]
    digits = "0123456789abcdef"[:base]
    n = 0
    while n < len(t) and t[n] in digits:
        n += 1
    return sign * int(t[:n], base) if n else 0


def parse_commandline(argv: list[str], out=sys.stdout) -> Options | None:
    """Mirror of parse_commandline(), btle_rx.c:1165-1315.  Returns None after printing the usage
    (the reference then exits with -1)."""
    o = Options()
    # Snout builds the argv itself (snout/util/btle.py:53), so the IQ source may also come from the environment
    o.iq = os.environ.get("SNOUT_B200_IQ")
    o.fmt = os.environ.get("SNOUT_B200_IQ_FORMAT", "cf32")
    o.wideband = bool(os.environ.get("SNOUT_B200_WIDEBAND"))
    out.write(formats.BTLE_RX_BANNER)
    try:
        opts, rest = getopt.getopt(argv, "hc:g:a:k:vrf:m:os:",
                                   ["help", "chan=", "gain=", "access=", "crcinit=", "verbose", "raw", "freq_hz=",
                                    "access_mask=", "hop", "filename=", "iq=", "format=", "scale=", "wideband",
                                    "all-channels", "device=", "shard-windows=", "rf", "aux", "coded", "periodic", "bis"])
    except getopt.GetoptError as e:
        out.write(f"btle_rx: {e}\n")
        out.write(USAGE)
        return None
    for k, v in opts:
        if k in ("-h", "--help"):
            out.write(USAGE)
            return None
        elif k in ("-c", "--chan"):
            o.chan = _strtol(v, 10)
        elif k in ("-g", "--gain"):
            o.gain = _strtol(v, 10)
        elif k in ("-a", "--access"):
            o.access_addr = _strtol(v, 16) & 0xFFFFFFFF
        elif k in ("-k", "--crcinit"):
            o.crc_init = _strtol(v, 16) & 0xFFFFFFFF
        elif k in ("-v", "--verbose"):
            o.verbose = 1
        elif k in ("-r", "--raw"):
            o.raw = 1
        elif k in ("-f", "--freq_hz"):
            o.freq_hz = _strtol(v, 10)
        elif k in ("-m", "--access_mask"):
            o.access_mask = _strtol(v, 16) & 0xFFFFFFFF
        elif k in ("-o", "--hop"):
            o.hop = 1
        elif k in ("-s", "--filename"):
            o.filename_pcap = v
        elif k == "--iq":
            o.iq = v
        elif k == "--format":
            o.fmt = v
        elif k == "--scale":
            o.scale = float(v)
        elif k == "--wideband":
            o.wideband = True
        elif k == "--all-channels":
            o.all_channels = True
        elif k == "--device":
            o.device = int(v)
        elif k == "--shard-windows":
            o.shard_windows = int(v)
        elif k == "--rf":
            o.rf = True
        elif k == "--aux":
            o.aux = True
        elif k == "--coded":
            o.coded = True
        elif k == "--periodic":
            o.periodic = True
        elif k == "--bis":
            o.bis = True
    if o.chan < 0 or o.chan > MAX_CHANNEL:
        out.write(f"channel number must be within 0~{MAX_CHANNEL}!\n")
        out.write(USAGE)
        return None
    if o.gain < 0 or o.gain > MAX_GAIN:
        out.write(f"rx gain must be within 0~{MAX_GAIN}!\n")
        out.write(USAGE)
        return None
    if rest:
        out.write("Error: unknown/extra arguments specified on command line!\n")
        out.write(USAGE)
        return None
    if o.fmt not in ("cf32", "sc8"):
        out.write("--format must be cf32 or sc8\n")
        out.write(USAGE)
        return None
    return o


def run(o: Options, out=sys.stdout, engine_factory=None, blocks=None) -> int:
    """The main loop of btle_rx.c:2288-2400 with the CUDA engine in place of receiver()."""
    freq_hz = o.freq_hz if o.freq_hz != 123 else chanplan.ble_channel_mhz(o.chan) * 1_000_000
    out.write(f"Cmd line input: chan {o.chan}, freq {freq_hz // 1000000}MHz, access addr {o.access_addr:08x}, "
              f"crc init {o.crc_init:06x} raw {o.raw} verbose {o.verbose} rx {o.gain}dB (B200) file={o.filename_pcap or '(null)'}\n")
    if o.raw:
        out.write("btle_rx (snout_b200): -r/--raw is not supported by the GPU receive engine\n")
        return 1
    if o.hop and not o.wideband:
        out.write("btle_rx (snout_b200): -o/--hop needs --wideband (a 4 Msps single-channel capture holds no data channel to hop to)\n")
        return 1
    if o.coded and not o.wideband:
        out.write("btle_rx (snout_b200): --coded needs --wideband (the Coded packets are found in the wideband bit streams)\n")
        return 1
    if o.aux and not o.wideband:
        out.write("btle_rx (snout_b200): --aux needs --wideband (auxiliary packets are sent on the data channels)\n")
        return 1
    if o.periodic and not o.wideband:
        out.write("btle_rx (snout_b200): --periodic needs --wideband (periodic advertising is sent on the data channels)\n")
        return 1
    if o.bis and not o.wideband:
        out.write("btle_rx (snout_b200): --bis needs --wideband (broadcast isochronous streams are sent on the data channels)\n")
        return 1
    if o.iq is None and blocks is None:
        out.write("btle_rx (snout_b200): no IQ source; pass --iq FILE (or - for stdin)\n")
        return 1
    fh_pcap = None
    if o.filename_pcap:
        out.write(f"will store packets to: {o.filename_pcap}\n")
        fh_pcap = open(o.filename_pcap, "wb")
        fh_pcap.write(formats.PCAP_HDR_BLE)
    out.flush()

    from .stream import ShardStreamer, iq_blocks, rf_of
    if engine_factory is None:
        from .engine import RxEngine
        engine_factory = RxEngine
    mode = "ble_wb40" if o.wideband else "ble_nb"
    decim = chanplan.WB_DECIM if o.wideband else 1
    windows = o.shard_windows or (64 if o.wideband else 512)          # 64 windows x 24 = 12.6 M input samples per shard
    max_samples = (windows * chanplan.BLE_WINDOW + 128 + 2048) * decim
    if o.access_mask == 0:
        # the reference's -m 0 lets EVERY sample position match (search_unique_bits compares nothing, btle_rx.c:1395-1401);
        # in snrx_config_t access_mask 0 means "default 0xFFFFFFFF", so the two must not be confused: refuse, loudly
        out.write("btle_rx (snout_b200): -m 0 (no access-address bit takes part in the match) is not supported\n")
        return 1
    try:
        eng = engine_factory(mode, channel=o.chan, device=o.device, max_samples=max_samples, access_addr=o.access_addr,
                             crc_init=o.crc_init, quant_scale=o.scale, access_mask=o.access_mask,
                             **({"rf_metrics": True} if o.rf else {}))
    except Exception as e:                                             # no GPU / no library: there is no CPU path
        out.write(f"btle_rx (snout_b200): cannot start the GPU receive engine: {e}\n")
        return 1
    pkt_count = {}
    rc = 0
    track = {"conn": None, "first": False}                             # -o: the connection being followed

    def lines(frames: np.ndarray, key=None, rf=None):
        if fh_pcap:
            fh_pcap.write(formats.ble_pcap_block(frames, rf=rf))       # the batch's records in one piece (same bytes)
        for f in frames:
            ch = int(f["channel"]) if key is None else key
            pkt_count[ch] = pkt_count.get(ch, 0) + 1                   # pkt_count++, btle_rx.c:2126
            out.write(formats.btle_rx_line(f, pkt_count[ch]))

    try:
        st = ShardStreamer(eng, units_per_shard=windows)

        def emit(frames: np.ndarray):
            rf = rf_of(frames, eng.frame_rf()) if o.rf else None
            if o.wideband and not o.all_channels:
                sel = frames["channel"] == o.chan
                frames, rf = frames[sel], (rf[sel] if rf is not None else None)
            if o.hop:
                follow(frames)
            else:
                lines(frames, rf=rf)
            if o.aux:
                aux = eng.ble_aux()
                if fh_pcap:
                    fh_pcap.write(formats.ble_pcap_aux_block(aux))
                for d in messages.ble_ext_adv(aux):
                    out.write(formats.aux_line(d))
            if o.coded:
                lst = eng.ble_coded()
                if fh_pcap:
                    fh_pcap.write(formats.ble_pcap_coded_block(lst, crc_failed_primaries=False))
                for d in messages.ble_coded_adv(lst):
                    if d["depth"] == 0 and not d["crc_ok"]:
                        continue                      # mostly positions inside an S=8 packet's own body (DESIGN 4)
                    out.write(formats.coded_line(d) if d["depth"] == 0 else formats.aux_line(d))
            if o.periodic:
                sync = eng.ble_periodic()
                if fh_pcap:
                    fh_pcap.write(formats.ble_pcap_sync_block(sync))
                for t in messages.ble_periodic_adv(sync):
                    for ev in t["events"]:
                        out.write(formats.sync_line(t, ev))
            if o.bis:
                bis = eng.ble_bis()
                if fh_pcap:
                    fh_pcap.write(formats.ble_pcap_bis_block(bis))
                for g in messages.ble_broadcast_iso(bis):
                    for st in g["streams"]:
                        for p in st["pdus"]:
                            out.write(formats.bis_line(g, st, p))
            out.flush()                                                # fflush(stdout), btle_rx.c:2383

        def follow(frames: np.ndarray):
            """receiver_controller (btle_rx.c:2167-2282) without a radio to retune.  State 0: advertising frames are printed
            until a CRC-ok CONNECT_REQ with a full channel map is heard on the listened channel (others: the reference's
            'Not full ChnMap' line, keep listening).  From there on the reference leaves the advertising channel, so only
            the connection's LL PDUs are printed: all of them, on whatever data channel they were sent."""
            c = track["conn"]
            if c is None:
                conns = eng.connections()
                if not o.all_channels:
                    conns = conns[conns["channel"] == o.chan]
                started = [k for k in conns if k["chm_full"]][:1]
                upto = int(started[0]["sample_index"]) if started else None
                heard = {(int(k["sample_index"]), int(k["channel"])): k for k in conns}
                for f in (frames if upto is None else frames[frames["sample_index"] <= upto]):
                    lines(np.asarray([f]))
                    k = heard.get((int(f["sample_index"]), int(f["channel"])))
                    if k is not None and not k["chm_full"]:            # btle_rx.c:2180-2184: stay on the advertising channel
                        out.write("Hop: Not full ChnMap 1FFFFFFFFF! (%s) Stay in ADV Chn\n" % bytes(k["chm"][::-1]).hex())
                if not started:
                    return
                c = track["conn"] = started[0].copy()
                ch0 = int(c["hop"]) % 37                               # hop_chan = (0 + hop) % 37, btle_rx.c:2194
                out.write("Hop: track start ...\n")
                out.write(f"Hop: next ch {ch0} freq {chanplan.ble_channel_mhz(ch0)}MHz access {int(c['access_addr']):08x} "
                          f"crcInit {int(c['crc_init']):06x}\n")
                out.write("Hop: next state 1\n")
            data = eng.follow(int(c["access_addr"]), int(c["crc_init"]))
            data = data[(data["channel"] < 37) & (data["sample_index"] > int(c["sample_index"]))]
            data = data[np.argsort(data["sample_index"], kind="stable")]    # records come channel by channel; print in air order
            for f in data:
                lines(np.asarray([f]), key=None if o.all_channels else o.chan)
                if not track["first"] and int(f["crc_ok"]):            # state 1 -> 2, btle_rx.c:2212-2217
                    track["first"] = True
                    out.write("Hop: 1st data pdu\nHop: next state 2\n")

        src = blocks if blocks is not None else iq_blocks(o.iq, o.fmt, scale=None)
        for block in src:
            for frames in st.feed(block):
                emit(frames)
        for frames in st.flush():
            emit(frames)
        st.close()
    except KeyboardInterrupt:
        pass
    except BrokenPipeError:
        rc = 0
    finally:
        eng.close()
        try:
            out.write("Exit main loop ...\n")                          # btle_rx.c:2396
            out.flush()
        except Exception:
            pass
        if fh_pcap:
            fh_pcap.close()
    return rc


def main(argv: list[str] | None = None) -> int:
    o = parse_commandline(sys.argv[1:] if argv is None else argv)
    if o is None:
        return 255                                                     # exit(-1), btle_rx.c:1314
    return run(o)


if __name__ == "__main__":
    sys.exit(main())

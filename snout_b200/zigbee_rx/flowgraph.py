"""Zigbee_rx -- drop-in for Snout's 802.15.4 receive flowgraph.

The reference receiver is the generated GNU Radio program
snout/modulations/Zigbee/hackrf/Zigbee_rx/top_block.py: class `top_block(channel=26)` with
`get_channel/set_channel`, `get_samp_rate/set_samp_rate`, `start/stop/wait` (29-103), an XMLRPC
server on localhost:8080 that exposes those methods (47-51), and a UDP client that sends one
RFtap-encapsulated PSDU per decoded frame to 127.0.0.1:52002 (53,71, epy_block_0.py:19-23).
scapy-radio launches it as a child process, waits for the XMLRPC port (wait_for_radio,
scapy/modules/gnuradio.py:342-381), retunes it with `set_channel` (323-338), reads the datagrams
(GnuradioSocket.recv, 67-73) and stops it by writing "\\r\\n" to its stdin (kill_process, 175-188).

This module keeps that interface and replaces the DSP blocks (quadrature_demod_cf, single_pole_iir,
sub_ff, clock_recovery_mm_ff, ieee802_15_4.packet_sink, rftap_encap) by the CUDA engine.  The IQ
source is a file or pipe instead of an osmosdr source:

* narrow band (4 Msps cf32 centred on the channel): `set_channel` re-labels the stream exactly as
  re-tuning the radio would (the samples are whatever the source delivers);
* `--wideband` (96 Msps centred on 2440 MHz): all 16 channels are decoded all the time and
  `set_channel` only selects which channel's frames are forwarded -- switching is instantaneous
  and nothing is lost while Snout sweeps channels 11..26 (snout/core/radio.py:415).

`--encap gnuradio` sends the 8-byte GnuradioPacket header + PSDU instead, which is what the older
flowgraphs under snout/util/.scapy emit (gr-zigbee packet_sink_scapy_impl.cc:333-349).
"""
from __future__ import annotations

import argparse
import os
import socket
import sys
import threading
import time
from xmlrpc.server import SimpleXMLRPCServer

import numpy as np

from .. import _abi, chanplan, formats

XMLRPC_ADDR = ("localhost", 8080)           # top_block.py:47
UDP_DEST = ("127.0.0.1", 52002)             # top_block.py:71


class top_block:
    """Same public surface as the generated flowgraph class (top_block.py:29-103)."""

    def __init__(self, channel: int = 26, iq: str | None = None, fmt: str = "cf32", wideband: bool = False,
                 encap: str = "rftap", device: int = 0, xmlrpc_addr=XMLRPC_ADDR, udp_dest=UDP_DEST,
                 realtime: bool = False, all_channels: bool = False, engine_factory=None, blocks=None,
                 segments_per_shard: int = 0, zb_segment: int = 0, serve_xmlrpc: bool = True, pcap: str | None = None,
                 rf: bool = False):
        self.channel = channel
        self.samp_rate = 4000000                                       # top_block.py:42
        self._iq, self._fmt, self._wideband, self._encap = iq, fmt, wideband, encap
        self._device, self._udp_dest = device, udp_dest
        self._realtime, self._all = realtime, all_channels
        self._engine_factory, self._blocks = engine_factory, blocks
        self._segments, self._zb_segment = segments_per_shard, zb_segment
        self._rf = rf                   # radio metrics: RFtap freqofs / power / noise / snr, and the pcap holds RFtap records
        self._stop = threading.Event()
        self._thread = None
        self._sock = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
        self._pcap = open(pcap, "wb") if pcap else None
        if self._pcap:
            self._pcap.write(formats.pcap_global_header(formats.DLT_RFTAP if rf else formats.DLT_IEEE802_15_4_WITHFCS))
        self.frames_sent = 0
        self.error = None
        self.xmlrpc_server_0 = None
        if serve_xmlrpc:
            self.xmlrpc_server_0 = SimpleXMLRPCServer(xmlrpc_addr, allow_none=True, logRequests=False)
            self.xmlrpc_server_0.register_instance(self)
            self.xmlrpc_server_0_thread = threading.Thread(target=self.xmlrpc_server_0.serve_forever, daemon=True)
            self.xmlrpc_server_0_thread.start()

    # ---- variables exposed over XMLRPC, same names as the reference -------------------------------
    def get_channel(self):
        return self.channel

    def set_channel(self, channel):
        if not 11 <= int(channel) <= 26:
            raise ValueError("802.15.4 channel 11..26")
        self.channel = int(channel)
        # reference: self.osmosdr_source_0.set_center_freq(1000000 * (2400 + 5 * (channel - 10)))  (top_block.py:94-96)

    def get_center_freq(self):
        return 1000000 * chanplan.zigbee_channel_mhz(self.channel)

    def get_samp_rate(self):
        return self.samp_rate

    def set_samp_rate(self, samp_rate):
        self.samp_rate = samp_rate

    # ---- life cycle ---------------------------------------------------------------------------
    def start(self):
        if self._thread is None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()

    def wait(self):
        if self._thread is not None:
            self._thread.join()
        if self.xmlrpc_server_0 is not None and threading.current_thread() is not self.xmlrpc_server_0_thread:
            self.xmlrpc_server_0.shutdown()
            self.xmlrpc_server_0.server_close()
            self.xmlrpc_server_0 = None
        if self._pcap:
            self._pcap.close()
            self._pcap = None

    # ---- data path ----------------------------------------------------------------------------
    def _emit(self, frames: np.ndarray, rf=None):
        for i, f in enumerate(frames):
            if self._wideband and not self._all and int(f["channel"]) != self.channel:
                continue
            if not self._wideband:
                f = f.copy()
                f["channel"] = self.channel
            r = rf[i] if rf is not None else None
            data = formats.rftap_datagram(f, r) if self._encap == "rftap" else formats.gnuradio_packet(f)
            self._sock.sendto(data, self._udp_dest)
            if self._pcap:
                rec = formats.rftap_datagram(f, r) if r is not None else bytes(f["bytes"][: int(f["len"])])
                self._pcap.write(formats.pcap_record(rec, time.time()))
            self.frames_sent += 1

    def _run(self):
        from ..stream import ShardStreamer, iq_blocks, rf_of, shard_geometry
        factory = self._engine_factory
        if factory is None:
            from ..engine import RxEngine
            factory = RxEngine
        mode = "zb_wb16" if self._wideband else "zb_nb"
        decim = chanplan.WB_DECIM if self._wideband else 1
        seg = self._zb_segment or _abi.ZB_SEGMENT_DEFAULT
        unit, pre, post = shard_geometry(0, 1, seg)                     # shard bodies: whole units of max(segment, 8192) samples
        nseg = self._segments or (262144 if self._wideband else 1048576) // unit
        try:
            eng = factory(mode, channel=self.channel, device=self._device, zb_segment=seg,
                          max_samples=(nseg * unit + pre + post) * decim, **({"rf_metrics": True} if self._rf else {}))
        except Exception as e:                                         # no GPU / no library: there is no CPU path
            self.error = e
            sys.stderr.write(f"Zigbee_rx (snout_b200): cannot start the GPU receive engine: {e}\n")
            return
        try:
            st = ShardStreamer(eng, units_per_shard=nseg)
            src = self._blocks if self._blocks is not None else iq_blocks(self._iq, self._fmt)
            rate = self.samp_rate * decim
            t0, done = time.time(), 0
            for block in src:
                if self._stop.is_set():
                    break
                for frames in st.feed(block):
                    self._emit(frames, rf_of(frames, eng.frame_rf()) if self._rf else None)
                done += len(block)
                if self._realtime:
                    lag = done / rate - (time.time() - t0)
                    if lag > 0:
                        time.sleep(lag)
            for frames in st.flush():
                self._emit(frames, rf_of(frames, eng.frame_rf()) if self._rf else None)
            st.close()
        except Exception as e:
            self.error = e
            sys.stderr.write(f"Zigbee_rx (snout_b200): {e}\n")
        finally:
            eng.close()


def argument_parser():
    p = argparse.ArgumentParser(prog="Zigbee_rx", description="B200 drop-in for Snout's Zigbee_rx flowgraph")
    p.add_argument("-c", "--channel", type=int, default=26, help="Set channel [default=26]")      # top_block.py:106-111
    p.add_argument("--iq", default=os.environ.get("SNOUT_B200_IQ"), help="IQ source: file, or - for stdin (env SNOUT_B200_IQ)")
    p.add_argument("--format", default=os.environ.get("SNOUT_B200_IQ_FORMAT", "cf32"), choices=["cf32", "sc8"])
    p.add_argument("--wideband", action="store_true", default=bool(os.environ.get("SNOUT_B200_WIDEBAND")),
                   help="source is 96 Msps centred on 2440 MHz: decode all 16 channels at once")
    p.add_argument("--all-channels", action="store_true", help="with --wideband: forward frames of every channel")
    p.add_argument("--encap", default="rftap", choices=["rftap", "gnuradio"])
    p.add_argument("--realtime", action="store_true", help="pace the source at its sample rate")
    p.add_argument("--device", type=int, default=0)
    p.add_argument("--pcap", default=None, help="also write the PSDUs to this DLT 195 pcap")
    p.add_argument("--no-stdin", action="store_true", help="do not wait for a newline on stdin; exit at end of the source")
    p.add_argument("--rf", action="store_true", help="measure signal power, noise floor and carrier offset of every frame: the "
                   "RFtap datagrams carry freqofs / power / noise / snr, and --pcap then holds RFtap records (LINKTYPE_RFTAP)")
    return p


def main(top_block_cls=top_block, argv=None):
    o = argument_parser().parse_args(argv)
    if not o.iq:
        sys.stderr.write("Zigbee_rx (snout_b200): no IQ source; pass --iq FILE or set SNOUT_B200_IQ\n")
        return 1
    stdin_is_source = (o.iq == "-")
    tb = top_block_cls(channel=o.channel, iq=o.iq, fmt=o.format, wideband=o.wideband, encap=o.encap, device=o.device,
                       realtime=o.realtime, all_channels=o.all_channels, pcap=o.pcap, rf=o.rf)
    tb.start()
    if o.no_stdin or stdin_is_source:
        tb._thread.join()
    else:
        try:
            sys.stdin.readline()                    # raw_input('Press Enter to quit: '), top_block.py:121-124
        except (EOFError, KeyboardInterrupt):
            pass
    tb.stop()
    tb.wait()
    return 1 if tb.error else 0


if __name__ == "__main__":
    sys.exit(main())

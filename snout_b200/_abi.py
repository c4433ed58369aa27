"""ctypes binding of libsnoutrx.so (include/snoutrx.h).

This is the only way Python reaches the receive path: no Triton, no torch ops, no CPU
implementation.  If the library is missing or no CUDA device is usable, the calls fail
loudly (SnrxError) -- they never fall back to anything else.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, byref, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint8, c_uint16, c_uint32, c_uint64, c_void_p

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libsnoutrx.so")
ABI_VERSION = 2

MODE_BLE_NB, MODE_ZB_NB, MODE_ZB_WB16, MODE_BLE_WB40, MODE_MIXED_WB56 = 0, 1, 2, 3, 4
F_KEEP_STREAMS = 1
F_RF_METRICS = 2               # include/snoutrx.h SNRX_F_RF_METRICS
ZB_SEGMENT_DEFAULT = 4096      # include/snoutrx.h SNRX_ZB_SEGMENT_DEFAULT / SNRX_ZB_PREHALO_DEFAULT
ZB_PREHALO_DEFAULT = 2048
ZB_IIR_BLOCK = 2048            # SNRX_ZB_IIR_BLOCK / SNRX_ZB_IIR_MEMORY_BLOCKS
ZB_IIR_MEMORY_BLOCKS = 48
STAGE_BLE_Q8, STAGE_BLE_BITS, STAGE_CHAN_CF32, STAGE_ZB_DISC, STAGE_ZB_CHIPS, STAGE_ZB_F, STAGE_ZB_NCHIPS = 1, 2, 3, 4, 5, 6, 7
PROTO_ZIGBEE, PROTO_BLE = 2, 3
XCHG_HANDLE_BYTES, XCHG_SLOTS, XCHG_MAX_WORLD = 64, 8, 16
# SURVEY 8(f) N3 record (include/snoutrx.h snrx_conn_t)
CONN_DTYPE = np.dtype([("sample_index", "<i8"), ("capture_id", "<u4"), ("frame", "<u4"), ("access_addr", "<u4"), ("crc_init", "<u4"),
                       ("init_a", "u1", (6,)), ("adv_a", "u1", (6,)), ("win_offset", "<u2"), ("interval", "<u2"), ("latency", "<u2"),
                       ("timeout", "<u2"), ("chm", "u1", (5,)), ("win_size", "u1"), ("hop", "u1"), ("sca", "u1"), ("channel", "u1"),
                       ("chm_full", "u1"), ("reserved", "u1", (2,))], align=True)
assert CONN_DTYPE.itemsize == 56
# SURVEY 8(f) N4 burst descriptor (include/snoutrx.h snrx_tx_burst_t)
TX_BURST_DTYPE = np.dtype([("start", "<i8"), ("data_offset", "<u4"), ("n_units", "<u4"), ("bin_slot", "<u2"), ("proto", "u1"),
                           ("reserved", "u1"), ("cfo_hz", "<f4"), ("phase0", "<f4"), ("amp", "<f4")], align=True)
assert TX_BURST_DTYPE.itemsize == 32
# SURVEY 8(f) N2 record (include/snoutrx.h snrx_zbmac_t)
(ZBMAC_SECURITY, ZBMAC_PENDING, ZBMAC_ACKREQ, ZBMAC_PANID_COMPRESS, ZBMAC_DEST_PANID, ZBMAC_DEST_ADDR, ZBMAC_SRC_PANID,
 ZBMAC_SRC_ADDR, ZBMAC_INTERPAN, ZBMAC_ZLL, ZBMAC_ZLL_SCAN_RESPONSE, ZBMAC_NO_ADDRESSING) = (1 << i for i in range(12))
ZBMAC_MALFORMED, ZBMAC_NOT_ZIGBEE = 0x4000, 0x8000
ZBMAC_DTYPE = np.dtype([
    ("dest_addr", "<u8"), ("src_addr", "<u8"), ("dest_panid", "<u2"), ("src_panid", "<u2"), ("fcf", "<u2"), ("present", "<u2"),
    ("seqnum", "u1"), ("frame_type", "u1"), ("dest_mode", "u1"), ("src_mode", "u1"), ("cmd_id", "u1"), ("payload_off", "u1"),
    ("zll_command", "u1"), ("reserved", "u1"), ("cluster", "<u2"), ("profile", "<u2"), ("frame", "<u4"),
], align=True)
assert ZBMAC_DTYPE.itemsize == 40

# per-frame radio metrics (include/snoutrx.h snrx_frame_rf_t)
RF_POWER, RF_NOISE, RF_CFO = 0x01, 0x02, 0x04
RF_ZB_THETA0 = 0.12435499454676144
RF_DTYPE = np.dtype([("sample_index", "<i8"), ("capture_id", "<u4"), ("frame", "<u4"), ("channel", "<u2"), ("proto", "u1"),
                     ("valid", "u1"), ("power_dbfs", "<f4"), ("noise_dbfs", "<f4"), ("snr_db", "<f4"), ("cfo_hz", "<f4"),
                     ("reserved", "<u4")], align=True)
assert RF_DTYPE.itemsize == 40

# BLE 5 extended advertising: one entry per AuxPtr (include/snoutrx.h snrx_ble_aux_t)
AUX_OK, AUX_NOT_FOUND, AUX_OUTSIDE, AUX_TRUNCATED, AUX_UNSUPPORTED_PHY, AUX_BAD_CHANNEL, AUX_DEPTH_LIMIT = range(7)
AUX_PHY_1M, AUX_PHY_2M, AUX_PHY_CODED = 0, 1, 2
AUX_MAX_DEPTH, AUX_MAX_BYTES = 15, 260
AUX_DTYPE = np.dtype([("sample_index", "<i8"), ("win_lo", "<i8"), ("win_hi", "<i8"), ("capture_id", "<u4"), ("parent", "<u4"),
                      ("first", "<u4"), ("depth", "u1"), ("channel", "u1"), ("phy", "u1"), ("phase", "u1"), ("status", "u1"),
                      ("crc_ok", "u1"), ("len", "<u2"), ("bytes", "u1", (AUX_MAX_BYTES,))], align=True)
assert AUX_DTYPE.itemsize == 304

# BLE Long Range: one entry per primary LE Coded packet or pointer (include/snoutrx.h snrx_ble_coded_t)
AUX_RESERVED_CI = 7
CODED_T, CODED_MAX_DEPTH = 400, 16
CODED_DTYPE = np.dtype([("sample_index", "<i8"), ("win_lo", "<i8"), ("win_hi", "<i8"), ("capture_id", "<u4"), ("parent", "<u4"),
                        ("first", "<u4"), ("depth", "u1"), ("channel", "u1"), ("phy", "u1"), ("phase", "u1"), ("status", "u1"),
                        ("crc_ok", "u1"), ("len", "<u2"), ("ci", "u1"), ("reserved0", "u1"), ("aa_errors", "<u2"),
                        ("metric", "<u4"), ("bytes", "u1", (AUX_MAX_BYTES,)), ("reserved", "u1", (8,))], align=True)
assert CODED_DTYPE.itemsize == 320

# BLE periodic advertising: one entry per listed event of an AUX_SYNC_IND train (include/snoutrx.h snrx_ble_sync_t)
SYNC_MIN_INTERVAL = 6
SYNC_DTYPE = np.dtype([("sample_index", "<i8"), ("win_lo", "<i8"), ("win_hi", "<i8"), ("capture_id", "<u4"), ("source", "<u4"),
                       ("access_addr", "<u4"), ("crc_init", "<u4"), ("event", "<i4"), ("event_counter", "<u2"), ("interval", "<u2"),
                       ("channel", "u1"), ("phy", "u1"), ("phase", "u1"), ("status", "u1"), ("crc_ok", "u1"), ("sca", "u1"),
                       ("len", "<u2"), ("bytes", "u1", (AUX_MAX_BYTES,)), ("reserved", "u1", (4,))], align=True)
assert SYNC_DTYPE.itemsize == 320

# BLE broadcast isochronous streams: one entry per subevent of a listed BIG event (include/snoutrx.h snrx_ble_bis_t)
BIS_ENCRYPTED, BIS_FRAMED = 0x01, 0x02
BIS_DTYPE = np.dtype([("sample_index", "<i8"), ("win_lo", "<i8"), ("win_hi", "<i8"), ("payload_number", "<u8"), ("capture_id", "<u4"),
                      ("source", "<u4"), ("access_addr", "<u4"), ("crc_init", "<u4"), ("event", "<i4"), ("event_counter", "<u2"),
                      ("bis", "u1"), ("subevent", "u1"), ("channel", "u1"), ("phy", "u1"), ("phase", "u1"), ("status", "u1"),
                      ("crc_ok", "u1"), ("flags", "u1"), ("len", "<u2"), ("bytes", "u1", (AUX_MAX_BYTES,)), ("reserved", "u1", (12,))],
                     align=True)
assert BIS_DTYPE.itemsize == 336

FRAME_DTYPE = np.dtype([
    ("sample_index", "<i8"), ("capture_id", "<u4"), ("window", "<u4"), ("channel", "<u2"),
    ("proto", "u1"), ("crc_ok", "u1"), ("lqi", "u1"), ("phase", "u1"), ("len", "<u2"),
    ("access_addr", "<u4"), ("bytes", "u1", (132,)),
], align=True)
assert FRAME_DTYPE.itemsize == 160


class Config(Structure):
    _fields_ = [
        ("abi_version", c_uint32), ("device", c_int32), ("mode", c_int32), ("channel", c_int32),
        ("access_addr", c_uint32), ("crc_init", c_uint32), ("zb_threshold", c_int32), ("quant_scale", c_float),
        ("max_samples", c_uint64), ("max_captures", c_uint32), ("max_frames", c_uint32),
        ("zb_segment", c_uint32), ("zb_prehalo", c_uint32), ("pfb_taps", c_uint32), ("flags", c_uint32),
        ("access_mask", c_uint32), ("reserved", c_uint32),
    ]


class Shard(Structure):
    _fields_ = [("pre_samples", c_uint64), ("body_samples", c_uint64), ("first_window", c_uint32),
                ("first_capture_id", c_uint32)]


class Stats(Structure):
    _fields_ = [
        ("samples_in", c_uint64), ("channel_samples", c_uint64), ("candidates", c_uint32), ("frames", c_uint32),
        ("frames_crc_ok", c_uint32), ("kernel_launches", c_uint32), ("gpu_ms", c_float), ("gpu_ms_frontend", c_float),
    ]


class SnrxError(RuntimeError):
    def __init__(self, code: int, what: str, detail: str = ""):
        self.code = code
        super().__init__(f"{what}: {detail}" if detail else what)


# every symbol include/snoutrx.h declares: (name, restype, argtypes)
# SURVEY 8(f) N1 records (include/snoutrx.h snrx_adv_t / snrx_device_t)
ADV_FLAGS, ADV_UUID128, ADV_OOB, ADV_SERVICE_DATA, ADV_MANUFACTURER, ADV_UNKNOWN, ADV_MALFORMED, ADV_SENDER = (1 << i for i in range(8))
ADV_DTYPE = np.dtype([
    ("adv_a", "u1", (6,)), ("pdu_type", "u1"), ("tx_add", "u1"), ("rx_add", "u1"), ("adv_len", "u1"), ("n_ad", "u1"),
    ("ad_flags", "u1"), ("present", "<u2"), ("company_id", "<u2"), ("service_uuid", "<u2"), ("unknown_type", "u1"),
    ("apple_action", "u1"), ("oob_flags", "u1"), ("hints", "u1"), ("apple_types", "<u4"), ("frame", "<u4"),
], align=True)
DEVICE_DTYPE = np.dtype([
    ("adv_a", "u1", (6,)), ("tx_add", "u1"), ("ad_flags", "u1"), ("packets", "<u4"), ("crc_ok", "<u4"), ("chan_mask", "<u8"),
    ("first_index", "<i8"), ("last_index", "<i8"), ("first_capture", "<u4"), ("last_capture", "<u4"), ("pdu_mask", "<u2"),
    ("present", "<u2"), ("company_id", "<u2"), ("vendor_company", "<u2"), ("apple_types", "<u4"), ("model", "u1"), ("os", "u1"),
    ("vendor_kind", "u1"), ("pad", "u1"),
], align=True)
assert ADV_DTYPE.itemsize == 32 and DEVICE_DTYPE.itemsize == 64
HINT_NEARBY_MASK, HINT_FITBIT = 0x0F, 0x10                    # snrx_adv_t.hints
MODEL_NONE, MODEL_FITBIT_CHARGE, MODEL_AIRPODS = 0, 1, 2       # snrx_device_t.model
OS_NONE, OS_UNDECIDED, OS_IOS10, OS_IOS11, OS_IOS12, OS_WINDOWS10 = range(6)
VENDOR_NONE, VENDOR_COMPANY, VENDOR_FITBIT = 0, 1, 2

SYMBOLS = [
    ("snrx_abi_version", c_int, []),
    ("snrx_strerror", c_char_p, [c_int]),
    ("snrx_last_error", c_char_p, [c_void_p]),
    ("snrx_device_count", c_int, [POINTER(c_int)]),
    ("snrx_create", c_int, [POINTER(c_void_p), POINTER(Config)]),
    ("snrx_destroy", None, [c_void_p]),
    ("snrx_process", c_int, [c_void_p, c_void_p, c_uint32, c_uint64, c_uint64, POINTER(Shard), c_int]),
    ("snrx_process_sc8", c_int, [c_void_p, c_void_p, c_uint32, c_uint64, c_uint64, POINTER(Shard), c_int]),
    ("snrx_poll", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_poll_view", c_int, [c_void_p, POINTER(c_void_p), POINTER(c_uint32)]),
    ("snrx_frames_device", c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p)]),
    ("snrx_polled_frames_device", c_int, [c_void_p, POINTER(c_void_p), POINTER(c_uint32)]),
    ("snrx_ble_adv_summary", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_ble_devices", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32), c_int]),
    ("snrx_ble_connections", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_ble_follow", c_int, [c_void_p, c_uint32, c_uint32, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_ble_aux", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_ble_coded", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_ble_periodic", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_ble_bis", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_zb_mac_summary", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_frame_rf", c_int, [c_void_p, c_void_p, c_uint32, POINTER(c_uint32)]),
    ("snrx_exchange_create", c_int, [c_void_p, c_uint32, c_uint32, c_uint32, c_void_p]),
    ("snrx_exchange_connect", c_int, [c_void_p, c_void_p]),
    ("snrx_allgather", c_int, [c_void_p, c_uint64, c_void_p, c_uint32, POINTER(c_uint32), POINTER(c_uint32), c_uint32]),
    ("snrx_synth_wideband", c_int, [c_int, c_void_p, c_uint32, c_void_p, c_uint64, c_void_p, c_uint32, c_void_p, c_void_p, c_uint64,
                             c_float, c_uint64, c_void_p, c_int]),
    ("snrx_set_channel", c_int, [c_void_p, c_int]),
    ("snrx_set_stream", c_int, [c_void_p, c_void_p]),
    ("snrx_sync", c_int, [c_void_p]),
    ("snrx_stats", c_int, [c_void_p, POINTER(Stats)]),
    ("snrx_debug_stage", c_int, [c_void_p, c_int, c_void_p, c_uint64, POINTER(c_uint64)]),
    ("snrx_debug_process_bits", c_int, [c_void_p, c_void_p, c_uint32, c_uint64, POINTER(Shard)]),
    ("snrx_pfb_prototype", c_int, [c_int, c_uint32, POINTER(c_double)]),
    ("snrx_host_alloc", c_int, [POINTER(c_void_p), c_uint64]),
    ("snrx_host_free", c_int, [c_void_p]),
    ("snrx_ble_channel_mhz", c_int, [c_int]),
    ("snrx_zigbee_channel_mhz", c_int, [c_int]),
    ("snrx_ble_channel_bin", c_int, [c_int]),
    ("snrx_zigbee_channel_bin", c_int, [c_int]),
]

_lib = None


def load() -> ctypes.CDLL:
    """Load libsnoutrx.so and bind every exported symbol.  Raises if the library is absent:
    the product path has no substitute for it."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("SNRX_LIB", LIB_PATH)          # SNRX_LIB: another build of the same library (kernel A/B runs)
    if not os.path.exists(path):
        raise SnrxError(-2, "libsnoutrx.so is not built",
                        f"{path} missing -- run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = ctypes.CDLL(path)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)          # AttributeError here = ABI symbol missing
        fn.restype = res
        fn.argtypes = args
    if lib.snrx_abi_version() != ABI_VERSION:
        raise SnrxError(-1, "libsnoutrx.so ABI version mismatch")
    _lib = lib
    return lib


def check(code: int, handle=None):
    if code == 0:
        return
    lib = load()
    what = lib.snrx_strerror(code).decode()
    detail = lib.snrx_last_error(handle).decode() if True else ""
    raise SnrxError(code, what, detail)


def device_count() -> int:
    n = c_int(0)
    load().snrx_device_count(byref(n))
    return n.value


def pfb_prototype(mode: int, taps: int = 384) -> np.ndarray:
    out = np.zeros(taps, dtype=np.float64)
    check(load().snrx_pfb_prototype(mode, taps, out.ctypes.data_as(POINTER(c_double))))
    return out


class PinnedBuffer:
    """Page-locked host memory from snrx_host_alloc, viewed as a numpy array."""

    def __init__(self, shape, dtype=np.complex64):
        self.lib = load()
        self.dtype = np.dtype(dtype)
        self.shape = tuple(shape) if not np.isscalar(shape) else (int(shape),)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = c_void_p()
        check(self.lib.snrx_host_alloc(byref(p), self.nbytes))
        self.ptr = p
        buf = (ctypes.c_char * self.nbytes).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            self.lib.snrx_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

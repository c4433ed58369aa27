"""TEST INFRASTRUCTURE ONLY -- CPU oracles of the receive path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this package.  Nothing under snout_b200/ does (tests/test_abi_layout.py enforces it).

Two kinds of oracle live here:

* "port"      -- plain-C restatements (ble_oracle.c, zb_oracle.c, pfb_oracle.c) built into
                 oracle/_build/liboracle.so; buildable anywhere gcc exists.
* "reference" -- the UNMODIFIED reference sources compiled from /root/reference into
                 oracle/_ref/*.so by `make -C oracle ref` (only where /root/reference exists;
                 the built files travel to the GPU box, the sources never enter this repo).
"""
from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint8, c_uint32, c_void_p

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE_ROOT = "/root/reference"

FRAME_DTYPE = np.dtype([
    ("sample_index", "<i8"), ("capture_id", "<u4"), ("window", "<u4"), ("channel", "<u2"),
    ("proto", "u1"), ("crc_ok", "u1"), ("lqi", "u1"), ("phase", "u1"), ("len", "<u2"),
    ("access_addr", "<u4"), ("bytes", "u1", (132,)),
], align=True)
assert FRAME_DTYPE.itemsize == 160

ZB_POST_HALO = 16448


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "vendor", "BTLE"))


_native_dir: str | None = None


def build(ref: bool | None = None, native: bool = False, quiet: bool = True) -> None:
    """Compile the port oracle, and the reference oracle when /root/reference is present.  native=True also builds
    liboracle_native.so (-O3 -march=native on THIS host): the library the CPU baseline legs of bench.py time.  It goes
    to a temporary directory, removed at exit, so that the benchmark can run from a read-only tree."""
    global _native_dir
    args = ["make", "-C", HERE]
    out = subprocess.run(args + ["all"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + out.stdout + out.stderr)
    if native:
        if _native_dir is None:
            _native_dir = tempfile.mkdtemp(prefix="snrx_oracle_native_")
            atexit.register(shutil.rmtree, _native_dir, True)
        out = subprocess.run(args + ["native", f"BUILD={_native_dir}"], capture_output=True, text=True)
        if out.returncode != 0:
            raise RuntimeError("native oracle build failed:\n" + out.stdout + out.stderr)
    if ref is None:
        ref = reference_available()
    if ref:
        out = subprocess.run(["make", "-C", HERE, "ref"], capture_output=True, text=True)
        if out.returncode != 0:
            raise RuntimeError("reference oracle build failed:\n" + out.stdout + out.stderr)
    _libs.clear()


_libs: dict[str, ctypes.CDLL] = {}


def _lib(name: str) -> ctypes.CDLL:
    if name in _libs:
        return _libs[name]
    if name == "native" and _native_dir is None:
        build(ref=False, native=True)
    path = {"port": os.path.join(HERE, "_build", "liboracle.so"),
            "native": os.path.join(_native_dir or "", "liboracle_native.so"),
            "btle_ref": os.path.join(HERE, "_ref", "libbtle_ref.so"),
            "zb_ref": os.path.join(HERE, "_ref", "libzbsink_ref.so")}[name]
    if not os.path.exists(path):
        if name == "port":
            build(ref=False)
        else:
            raise FileNotFoundError(f"{path} missing: run `make -C oracle ref` where /root/reference exists")
    lib = ctypes.CDLL(path)
    _libs[name] = lib
    return lib


def have_ref(name: str = "btle_ref") -> bool:
    return os.path.exists(os.path.join(HERE, "_ref", {"btle_ref": "libbtle_ref.so", "zb_ref": "libzbsink_ref.so"}[name]))


def _frames(n: int) -> np.ndarray:
    return np.zeros(max(n, 1), dtype=FRAME_DTYPE)


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(c_void_p)


# ------------------------------------------------------------------------ BLE

def as_int8_iq(iq) -> np.ndarray:
    """[n,2] int8 view of a capture given as int8 pairs."""
    a = np.ascontiguousarray(iq, dtype=np.int8).reshape(-1, 2)
    return a


def ble_quantize(iq_cf32: np.ndarray, scale: float) -> np.ndarray:
    """cf32 -> int8 grid, q = clamp(rint(x*scale), -128, 127)."""
    x = np.ascontiguousarray(iq_cf32).view(np.float32).reshape(-1)
    q = np.empty(x.shape[0], dtype=np.int8)
    lib = _lib("port")
    lib.ble_oracle_quantize(_ptr(x), c_int64(x.shape[0]), c_float(scale), _ptr(q))
    return q.reshape(-1, 2)


def ble_decode(iq_int8, channel: int, aa: int = 0x8E89BED6, crc_init: int = 0x555555,
               impl: str = "port", cap: int = 1 << 16, aa_mask: int = 0xFFFFFFFF,
               first_window: int = 0, n_windows: int = 0) -> np.ndarray:
    """Frames of one 4 Msps int8 channel stream, windowed exactly like btle_rx's main loop."""
    q = as_int8_iq(iq_int8)
    out = _frames(cap)
    if impl == "port":
        lib = _lib("port")
        n = lib.ble_oracle_windows_range(_ptr(q), c_int64(q.shape[0]), c_int(channel), c_uint32(aa),
                                         c_uint32(aa_mask), c_uint32(crc_init), c_int64(first_window),
                                         c_int64(n_windows), _ptr(out), c_int(cap))
    elif impl == "reference":
        lib = _lib("btle_ref")
        lib.btle_ref_set_mask(c_uint32(aa_mask))
        n = lib.btle_ref_windows(_ptr(q), c_int64(q.shape[0]), c_int(channel), c_uint32(aa),
                                 c_uint32(crc_init), _ptr(out), c_int(cap))
    else:
        raise ValueError(impl)
    if n < 0 or n > cap:
        raise RuntimeError(f"ble oracle returned {n}")
    return out[:n].copy()


def ble_reference_stdout(iq_int8, channel: int, aa: int = 0x8E89BED6, crc_init: int = 0x555555) -> str:
    """Text the reference receiver() prints for this capture (run in a child process)."""
    import sys
    import tempfile
    q = as_int8_iq(iq_int8)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "iq.i8")
        q.tofile(path)
        code = (
            "import ctypes, numpy as np\n"
            f"lib = ctypes.CDLL({os.path.join(HERE, '_ref', 'libbtle_ref.so')!r})\n"
            f"q = np.fromfile({path!r}, dtype=np.int8)\n"
            f"lib.btle_ref_receiver_print(q.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(len(q)//2), {channel}, ctypes.c_uint32({aa}), ctypes.c_uint32({crc_init}))\n"
        )
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True)
        return r.stdout


def ble_time(iq_int8, channel: int, reps: int = 1, impl: str = "port") -> tuple[float, int]:
    q = as_int8_iq(iq_int8)
    nf = c_int(0)
    if impl == "reference":
        lib = _lib("btle_ref")
        lib.btle_ref_time.restype = c_double
        t = lib.btle_ref_time(_ptr(q), c_int64(q.shape[0]), c_int(channel), c_uint32(0x8E89BED6),
                              c_uint32(0x555555), c_int(reps), ctypes.byref(nf))
    else:
        lib = _lib("port")
        lib.ble_oracle_time.restype = c_double
        t = lib.ble_oracle_time(_ptr(q), c_int64(q.shape[0]), c_int(channel), c_uint32(0x8E89BED6),
                                c_uint32(0x555555), c_int(reps), ctypes.byref(nf))
    return float(t), int(nf.value)


def ble_tables(impl: str = "port"):
    """(whitening [40,42] u8, crc table [256] u32, crc_init_internal(0x555555))."""
    if impl == "port":
        lib = _lib("port")
        lib.ble_oracle_whiten_row.restype = POINTER(c_uint8)
        w = np.array([[lib.ble_oracle_whiten_row(ch)[i] for i in range(42)] for ch in range(40)], dtype=np.uint8)
        lib.ble_oracle_crc_table.restype = c_uint32
        t = np.array([lib.ble_oracle_crc_table(i) for i in range(256)], dtype=np.uint32)
        lib.ble_oracle_crc_init_internal.restype = c_uint32
        return w, t, int(lib.ble_oracle_crc_init_internal(c_uint32(0x555555)))
    lib = _lib("btle_ref")
    lib.btle_ref_scramble_row.restype = POINTER(c_uint8)
    w = np.array([[lib.btle_ref_scramble_row(ch)[i] for i in range(42)] for ch in range(40)], dtype=np.uint8)
    lib.btle_ref_crc_table.restype = c_uint32
    t = np.array([lib.btle_ref_crc_table(i) for i in range(256)], dtype=np.uint32)
    lib.btle_ref_crc_init_reorder.restype = c_uint32
    return w, t, int(lib.btle_ref_crc_init_reorder(c_uint32(0x555555)))


def ble_crc24(data: bytes, init_internal: int = 0xAAAAAA, impl: str = "port") -> int:
    buf = (c_uint8 * len(data))(*data)
    if impl == "port":
        lib = _lib("port")
        lib.ble_oracle_crc24.restype = c_uint32
        return int(lib.ble_oracle_crc24(buf, c_int(len(data)), c_uint32(init_internal)))
    lib = _lib("btle_ref")
    lib.btle_ref_crc24.restype = c_uint32
    return int(lib.btle_ref_crc24(buf, c_int(len(data)), c_uint32(init_internal)))


# --------------------------------------------------------------------- Zigbee

def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def zb_quad_demod(iq_cf32: np.ndarray) -> np.ndarray:
    x = np.ascontiguousarray(iq_cf32, dtype=np.complex64)
    f = np.empty(x.shape[0], dtype=np.float32)
    _lib("port").zb_oracle_quad_demod(_ptr(x), c_int64(x.shape[0]), _ptr(f))
    return f


def zb_dc_remove(f: np.ndarray) -> np.ndarray:
    f = _f32(f)
    z = np.empty_like(f)
    _lib("port").zb_oracle_dc_remove(_ptr(f), c_int64(f.shape[0]), _ptr(z))
    return z


def zb_chain(z: np.ndarray, begin: int, end: int, body_lo: int, body_hi: int, channel: int = 11,
             threshold: int = 10, segment: int = 0, cap: int = 4096, want_chips: bool = False, hold: int = 0,
             want_stop: bool = False):
    """One clock-recovery + sink chain (sink held in its initial state until position `hold`).
    Returns (frames, soft chips, chip positions[, stop position])."""
    z = _f32(z)
    out = _frames(cap)
    nf = c_int(0)
    stop = c_int64(0)
    lib = _lib("port")
    lib.zb_oracle_chain_hold.restype = c_int64
    maxchips = (end - begin) // 2 + 64 if want_chips else 0
    chips = np.zeros(max(maxchips, 1), dtype=np.float32)
    pos = np.zeros(max(maxchips, 1), dtype=np.int64)
    n = lib.zb_oracle_chain_hold(_ptr(z), c_int64(begin), c_int64(end), c_int64(body_lo), c_int64(body_hi), c_int64(hold),
                                 c_int(threshold), c_int(channel), c_uint32(segment), _ptr(out), c_int(cap),
                                 ctypes.byref(nf), _ptr(chips) if want_chips else None,
                                 _ptr(pos) if want_chips else None, c_int64(maxchips), ctypes.byref(stop))
    n = int(n)
    res = (out[:nf.value].copy(), chips[:min(n, maxchips)], pos[:min(n, maxchips)])
    return res + (int(stop.value),) if want_stop else res


ZB_SEGMENT_DEFAULT, ZB_PREHALO_DEFAULT = 4096, 2048      # include/snoutrx.h


def zb_dc_remove_serial(f: np.ndarray) -> np.ndarray:
    """The published single-pole IIR + subtract, one serial recurrence (SURVEY App. H.2)."""
    f = _f32(f)
    z = np.empty_like(f)
    _lib("port").zb_oracle_dc_remove_serial(_ptr(f), c_int64(f.shape[0]), _ptr(z))
    return z


def zb_receive_serial(iq_cf32: np.ndarray, channel: int = 11, threshold: int = 10, cap: int = 1 << 16) -> np.ndarray:
    """The reference flowgraph as it is: serial DC tracker and ONE unsegmented clock-recovery + sink chain."""
    x = np.ascontiguousarray(iq_cf32, dtype=np.complex64)
    out = _frames(cap)
    n = _lib("port").zb_oracle_receive_serial(_ptr(x), c_int64(x.shape[0]), c_int(channel), c_int(threshold), _ptr(out), c_int(cap))
    if n < 0 or n > cap:
        raise RuntimeError(f"zb oracle returned {n}")
    return out[:n].copy()


def zb_receive(iq_cf32: np.ndarray, channel: int = 11, threshold: int = 10, segment: int = ZB_SEGMENT_DEFAULT,
               prehalo: int = ZB_PREHALO_DEFAULT, cap: int = 1 << 16) -> np.ndarray:
    x = np.ascontiguousarray(iq_cf32, dtype=np.complex64)
    out = _frames(cap)
    n = _lib("port").zb_oracle_receive(_ptr(x), c_int64(x.shape[0]), c_int(channel), c_int(threshold),
                                        c_int64(segment), c_int64(prehalo), _ptr(out), c_int(cap))
    if n < 0 or n > cap:
        raise RuntimeError(f"zb oracle returned {n}")
    return out[:n].copy()


def zb_receive_z(z: np.ndarray, channel: int = 11, threshold: int = 10, segment: int = ZB_SEGMENT_DEFAULT,
                 prehalo: int = ZB_PREHALO_DEFAULT, cap: int = 1 << 16) -> np.ndarray:
    z = _f32(z)
    out = _frames(cap)
    n = _lib("port").zb_oracle_receive_z(_ptr(z), c_int64(z.shape[0]), c_int(channel), c_int(threshold),
                                          c_int64(segment), c_int64(prehalo), _ptr(out), c_int(cap))
    return out[:n].copy()


def zb_time(iq_cf32: np.ndarray, channel: int = 11, segment: int = ZB_SEGMENT_DEFAULT, prehalo: int = ZB_PREHALO_DEFAULT, reps: int = 1):
    x = np.ascontiguousarray(iq_cf32, dtype=np.complex64)
    nf = c_int(0)
    lib = _lib("port")
    lib.zb_oracle_time.restype = c_double
    t = lib.zb_oracle_time(_ptr(x), c_int64(x.shape[0]), c_int(channel), c_int64(segment), c_int64(prehalo),
                           c_int(reps), ctypes.byref(nf))
    return float(t), int(nf.value)


def zb_fcs16(data: bytes) -> int:
    lib = _lib("port")
    lib.zb_oracle_fcs16.restype = ctypes.c_uint16
    buf = (c_uint8 * max(len(data), 1))(*data)
    return int(lib.zb_oracle_fcs16(buf, c_int(len(data))))


def zb_chip_words(impl: str = "port") -> np.ndarray:
    if impl == "port":
        lib = _lib("port")
        lib.zb_oracle_chip_word.restype = c_uint32
        return np.array([lib.zb_oracle_chip_word(i) for i in range(16)], dtype=np.uint32)
    lib = _lib("zb_ref")
    lib.zb_ref_chip_mapping.restype = c_uint32
    return np.array([lib.zb_ref_chip_mapping(i) for i in range(16)], dtype=np.uint32)


def zb_sink_reference(chips: np.ndarray, threshold: int = 10, cap: int = 4096):
    """Feed soft chips to the UNMODIFIED reference sink.  Returns [(end_chip, psdu bytes)]."""
    chips = _f32(chips)
    lib = _lib("zb_ref")
    lib.zb_ref_new.restype = c_void_p
    h = c_void_p(lib.zb_ref_new(c_int(threshold)))
    end = np.zeros(cap, dtype=np.int64)
    ln = np.zeros(cap, dtype=np.int32)
    by = np.zeros((cap, 128), dtype=np.uint8)
    k = lib.zb_ref_feed(h, _ptr(chips), c_int64(chips.shape[0]), c_int64(0), _ptr(end), _ptr(ln), _ptr(by), c_int(cap))
    lib.zb_ref_delete(h)
    k = min(int(k), cap)
    return [(int(end[i]), bytes(by[i, :ln[i]])) for i in range(k)]


# ------------------------------------------------------------------------ PFB

def set_threads(n: int) -> None:
    """OpenMP threads of the native library (torchrun exports OMP_NUM_THREADS=1 to its workers)."""
    _lib("native").pfb_oracle_set_threads(c_int(n))


def pfb(iq_cf32: np.ndarray, taps: np.ndarray, bins, m0: int = 0, m1: int | None = None, fast: bool = False,
        native: bool = False) -> np.ndarray:
    """Channel streams [len(bins), m1-m0] complex64 of a 96 Msps capture.  native=True: the -march=native build."""
    x = np.ascontiguousarray(iq_cf32, dtype=np.complex64)
    if m1 is None:
        m1 = x.shape[0] // 24
    b = np.ascontiguousarray(bins, dtype=np.int32)
    out = np.zeros((b.shape[0], m1 - m0), dtype=np.complex64)
    lib = _lib("native" if native else "port")
    if fast:
        h = np.ascontiguousarray(taps, dtype=np.float32)
        lib.pfb_oracle_fast(_ptr(x), c_int64(x.shape[0]), _ptr(h), c_int(h.shape[0]), _ptr(b), c_int(b.shape[0]),
                            c_int64(m0), c_int64(m1), _ptr(out))
    else:
        h = np.ascontiguousarray(taps, dtype=np.float64)
        lib.pfb_oracle_direct(_ptr(x), c_int64(x.shape[0]), _ptr(h), c_int(h.shape[0]), _ptr(b), c_int(b.shape[0]),
                              c_int64(m0), c_int64(m1), _ptr(out))
    return out


def threads() -> int:
    return int(_lib("port").pfb_oracle_threads())

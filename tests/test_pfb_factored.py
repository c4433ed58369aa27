"""The BLE channelizer's prime-factor 48-point transform and integer slicer without a GPU: the cores k_pfb_ble runs
(snout_b200/csrc/fft.cuh Pfa48, snout_b200/csrc/pfb.cuh), stepped on the CPU through tests/emu/emu_pfa.cu, against their
definitions."""
import ctypes
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_frames_equal
from quant_rule import check_q8
from snout_b200 import chanplan, synth
from test_emu_kernels import _back, _slice_nb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def emu_pfa(tmp_path_factory):
    """tests/emu/emu_pfa.cu built with the flags of tests/emu/Makefile into a temporary directory, at -O3 and with OpenMP
    for the exhaustive slicer check (2^32 cases)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    out = str(tmp_path_factory.mktemp("emu_pfa") / "libemu_pfa.so")
    r = subprocess.run([nvcc, "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "--expt-relaxed-constexpr",
                        "-Xcompiler", "-fPIC,-ffp-contract=off,-fopenmp", "-lgomp", "-shared", "-o", out,
                        os.path.join(ROOT, "tests", "emu", "emu_pfa.cu")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lib = ctypes.CDLL(out)
    lib.emu_quant_bits.restype = ctypes.c_uint32
    lib.emu_quant_bits.argtypes = [ctypes.c_float, ctypes.c_float]
    lib.emu_q8_of_biased.argtypes = [ctypes.c_uint32]
    lib.emu_slicer_words.argtypes = [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p]
    lib.emu_slicer_exhaustive.restype = ctypes.c_uint64
    return lib


def test_prime_factor_transform(emu_pfa):
    # the rotated passes and the twiddle-free combination along the kernel's route (V tile, column load) for the 32 lanes of a
    # tile, and Pfa48::run, against the float64 inverse DFT at the bound of test_fft_codelets
    rng = np.random.default_rng(48)
    x = (rng.standard_normal((32, 48)) + 1j * rng.standard_normal((32, 48))).astype(np.complex64)
    ref = np.fft.ifft(x.astype(np.complex128), axis=1) * 48
    y = np.zeros_like(x)
    emu_pfa.emu_pfa48_tile(P(x), P(y))
    assert np.abs(y - ref).max() / np.abs(ref).max() < 1e-6
    for lane in (0, 17):
        y1 = np.zeros(48, dtype=np.complex64)
        emu_pfa.emu_pfa48_run(P(np.ascontiguousarray(x[lane])), P(y1))
        assert np.abs(y1 - ref[lane]).max() / np.abs(ref[lane]).max() < 1e-6
    # one branch at a time: the map must route every input to every bin with the right phase, not just on average
    for r in range(48):
        e = np.zeros((32, 48), dtype=np.complex64)
        e[:, r] = 1.0 + 0.5j
        emu_pfa.emu_pfa48_tile(P(e), P(y))
        want = (1.0 + 0.5j) * np.exp(2j * np.pi * np.arange(48) * r / 48)
        assert np.abs(y - want).max() < 1e-5, r


@pytest.mark.parametrize("scale", [128.0, 100.0])
def test_biased_quantiser_bytes(emu_pfa, scale):
    # every q in [-128, 127]: t = 1.5 * 2^23 + q, byte 0 = q (int8), byte 3 = 0x4B, and the slicer words carry (I, ~Q, 0, 1) and
    # (Q, I, I, I) -- the DEBUG q8 is read back from the latter
    out = np.zeros(4, dtype=np.uint32)
    for q in range(-128, 128):
        t = emu_pfa.emu_quant_bits(q / scale, scale)
        assert t == (0x4B400000 + q) & 0xFFFFFFFF, (q, hex(t))
        assert t & 0xFF == q & 0xFF and t >> 24 == 0x4B
        assert emu_pfa.emu_q8_of_biased(t) == q
        tq = emu_pfa.emu_quant_bits(-q / scale, scale) if q > -128 else emu_pfa.emu_quant_bits(127 / scale, scale)
        qq = -q if q > -128 else 127
        emu_pfa.emu_slicer_words(t, tq, P(out))
        w, a = int(out[0]), int(out[1])
        assert [w & 0xFF, (w >> 8) & 0xFF, (w >> 16) & 0xFF, w >> 24] == [q & 0xFF, ~qq & 0xFF, 0, 1], (q, hex(w))
        assert [a & 0xFF, (a >> 8) & 0xFF, a >> 24] == [qq & 0xFF, q & 0xFF, q & 0xFF], (q, hex(a))
        assert np.int32(out[2]) == q and np.int32(out[3]) == qq
    # beyond full scale the quantiser saturates at exactly -128 / 127
    assert emu_pfa.emu_q8_of_biased(emu_pfa.emu_quant_bits(-1e3, scale)) == -128
    assert emu_pfa.emu_q8_of_biased(emu_pfa.emu_quant_bits(1e3, scale)) == 127


def test_integer_slicer_exhaustive(emu_pfa):
    # sign bit of dp4a(slicer_a(I0, Q0), slicer_w(I1, Q1)) against I0 Q1 - I1 Q0 > 0 for all 2^32 int8 (I0, Q0, I1, Q1)
    assert emu_pfa.emu_slicer_exhaustive() == 0


@pytest.mark.parametrize("nt,name", [(16, "BLE_384"), (32, "BLE_768")])
def test_pfb_tile_factored(emu, emu_pfa, oracle_mod, nt, name):
    # whole tiles along the kernel's path (prime-factor passes, twiddle-free combination, biased quantiser, integer slicer),
    # checked as test_pfb_tile_kernel checks the Cooley-Tukey statement, and against that statement tile by tile
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from gen_tables import PFB_DESIGNS, kaiser_lowpass
    h = kaiser_lowpass(*PFB_DESIGNS[name])
    hf = h.astype(np.float32)
    rho = np.array([hf[r + 24 * d] for r in range(24) for d in range(nt)], dtype=np.float32)
    cap = synth.wideband_capture(seconds=0.0025, kind="ble", seed=4000, gap=(200, 2000))
    x = np.ascontiguousarray(cap.iq)[: 24 * 8192 - 24 * 40]          # ragged: n_out = 8152, last tile partial
    n_in = len(x)
    n_out = n_in // 24
    T, stride = 32, emu.emu_pfb_ble_stride()
    tiles = (n_out + stride - 1) // stride
    wpp, lead = emu.emu_bits_words_for(n_out), emu.emu_bits_lead_words()
    bits = np.zeros((40, wpp), dtype=np.uint64)
    q8 = np.zeros((40, tiles * stride + 1, 2), dtype=np.int8)
    raw = np.zeros((40, tiles * stride + 1), dtype=np.complex64)
    xf = x.view(np.float32)
    n_moved = 0
    for t in range(tiles):
        w = np.zeros(40, dtype=np.uint32)
        q = np.zeros((40, T, 2), dtype=np.int8)
        r = np.zeros((40, T), dtype=np.complex64)
        emu_pfa.emu_pfa_ble_tile(nt, P(xf), ctypes.c_int64(n_in), n_out, t, P(rho), ctypes.c_float(100.0), P(w), P(q), P(r))
        w0, q0, r0 = np.zeros_like(w), np.zeros_like(q), np.zeros_like(r)
        emu.emu_pfb_ble_tile(nt, P(xf), ctypes.c_int64(n_in), n_out, t, P(rho), ctypes.c_float(100.0), P(w0), P(q0), P(r0))
        # the two transforms differ in the last bits only; a quantised value may move only off a rounding boundary
        assert np.abs(r - r0).max() <= 1e-5 * max(np.abs(r0).max(), 1e-30), t
        moved = q != q0
        if moved.any():
            y = np.stack([r.real, r.imag], axis=-1)[moved] * 100.0
            assert np.all(np.abs(q.astype(int) - q0)[moved] == 1) and np.all(np.abs(np.abs(y) % 1.0 - 0.5) < 1e-3), t
            n_moved += int(moved.sum())
        else:
            assert np.array_equal(w, w0), t
        g0 = t * stride
        wi, off = lead + (g0 >> 5), g0 & 31
        sh = w.astype(np.uint64) << np.uint64(off)
        bits[:, wi] |= sh & np.uint64(0xFFFFFFFF)
        bits[:, wi + 1] |= sh >> np.uint64(32)
        if t:
            assert np.array_equal(q8[:, g0], q[:, 0])
        q8[:, g0:g0 + T] = q
        raw[:, g0:g0 + T] = r
    assert n_moved <= 4
    bits = bits.astype(np.uint32)
    assert not q8[:, n_out:].any()
    q8, raw = q8[:, :n_out], raw[:, :n_out]
    yd = oracle_mod.pfb(x, h, [chanplan.ble_channel_bin(c) for c in range(40)])
    rms = np.sqrt(np.mean(np.abs(yd) ** 2))
    assert np.abs(raw - yd).max() / rms < 1e-4
    check_q8(q8, raw, yd, 100.0, what=f"{name} factored tile harness")
    n_frames = 0
    for c in range(40):
        b2, _, _ = _slice_nb(emu, q8[c].astype(np.float32) / 128.0, 128.0)
        assert np.array_equal(b2, bits[c]), f"slicer words of channel {c}"
        got = _back(emu, oracle_mod, np.ascontiguousarray(bits[c]), wpp, n_out, c)
        assert_frames_equal(got, oracle_mod.ble_decode(q8[c], c), what=f"channel {c}")
        n_frames += len(got)
    assert n_frames > 100

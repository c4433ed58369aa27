"""The BLE oracle is pinned against the reference's own code and golden vectors (SURVEY 8c, App. E).

`port`      = oracle/ble_oracle.c (plain-C restatement, travels everywhere)
`reference` = oracle/_ref/libbtle_ref.so (unmodified btle_rx.c, built where /root/reference exists)
Fixtures in tests/golden/ hold outputs of `reference`, so the port stays pinned on any machine.
"""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, assert_frames_equal
from snout_b200 import synth

GOLD_BYTES = [
    "40250289674523011e096861636b72662d736f6c6f2d62746c652d7478203200000000000000006d88c3",
    "40250389674523011e096861636b72662d736f6c6f2d62746c652d74782033000000000000000058c4cb",
    "40250089674523011e096861636b72662d736f6c6f2d62746c652d7478203000000000000000000710d3",
]


def test_golden_capture_port(oracle_mod, golden):
    g = golden("btle_sample_iq_4msps.npz")
    fr = oracle_mod.ble_decode(g["iq"], 37)
    assert list(fr["sample_index"]) == [97892, 501906, 905891]          # SURVEY Appendix E
    assert [bytes(f["bytes"][:f["len"]]).hex() for f in fr] == GOLD_BYTES
    assert fr["crc_ok"].all() and list(fr["window"]) == [11, 61, 110]
    assert_frames_equal(fr, g["frames"], what="port vs reference output fixture")


def test_welcome_vector_port(oracle_mod, golden):
    g = golden("btle_welcome.npz")
    fr = oracle_mod.ble_decode(g["iq"], 37)
    assert_frames_equal(fr, g["frames"], what="welcome message")
    pdu = bytes(fr[0]["bytes"][:fr[0]["len"]])
    assert pdu[0] & 0xF == 2 and pdu[1] == 37                          # ADV_NONCONN_IND, PloadL37
    assert pdu[2:8][::-1].hex() == "010203040506"                      # AdvA printed MSB first
    assert b"imecUGent SDRgroup welcome u!" in pdu


@pytest.mark.parametrize("seed", [1001, 1002, 1003, 1004])
def test_synthetic_port_matches_reference_fixture(oracle_mod, golden, seed):
    g = golden("btle_synth_ref.npz")
    s, esn0, ch, n = g[f"params_{seed}"]
    cap = synth.ble_capture(n=int(n), channel=int(ch), seed=int(s), esn0_db=float(esn0))
    fr = oracle_mod.ble_decode(oracle_mod.ble_quantize(cap.iq, 128.0), int(ch))
    assert len(fr) > 0
    assert_frames_equal(fr, g[f"frames_{seed}"], what=f"seed {seed}")


def test_window_boundary_rule(oracle_mod, golden):
    """SURVEY App. A.4: an AA starting in the last 6 samples of a window is reported twice."""
    g = golden("btle_sample_iq_4msps.npz")["iq"]
    b = golden("btle_boundary_ref.npz")
    counts = {}
    for d in range(403, 414):
        gd = np.concatenate([np.zeros((d, 2), np.int8), g[:200_000]])
        fr = oracle_mod.ble_decode(gd, 37)
        assert_frames_equal(fr, b[f"frames_{d}"], what=f"delay {d}")
        counts[d] = len(fr)
    assert [counts[d] for d in range(403, 414)] == [1, 1, 1, 2, 2, 2, 2, 2, 2, 1, 1]


def test_tables_and_kats(oracle_mod, golden):
    t = golden("btle_tables_ref.npz")
    w, crc, ci = oracle_mod.ble_tables("port")
    assert np.array_equal(w, t["scramble_table"]) and np.array_equal(crc, t["crc_table"])
    assert ci == int(t["crc_init_internal"]) == 0xAAAAAA and crc[128] == 0xDA6000
    for ch in range(40):
        assert np.array_equal(synth.ble_whitening(ch, 42), t["scramble_table"][ch])
    k = json.load(open(os.path.join(GOLDEN, "kats.json")))["ble_crc24"]
    pdu = bytes.fromhex(k["pdu_hex"])
    assert oracle_mod.ble_crc24(pdu).to_bytes(3, "little").hex() == k["crc_tx_hex"]
    assert synth.ble_crc24(pdu).hex() == k["crc_tx_hex"]
    assert [oracle_mod._lib("port").ble_oracle_channel_mhz(c) for c in (37, 38, 39, 0, 10, 11, 36)] == \
        [2402, 2426, 2480, 2404, 2424, 2428, 2478]


def test_edge_cases(oracle_mod):
    assert len(oracle_mod.ble_decode(np.zeros((1, 2), np.int8), 37)) == 0          # 1-sample capture
    assert len(oracle_mod.ble_decode(np.zeros((8192 * 3 + 5, 2), np.int8), 12)) == 0   # ragged, silent
    rng = np.random.default_rng(7)
    noise = rng.integers(-128, 128, (300_000, 2), dtype=np.int8)                        # full-scale noise incl. -128
    fr = oracle_mod.ble_decode(noise, 37)
    assert fr["crc_ok"].sum() == 0


def test_data_channel_no_length_gate(oracle_mod):
    cap = synth.ble_capture(n=300_000, channel=9, seed=55, esn0_db=30)
    fr = oracle_mod.ble_decode(oracle_mod.ble_quantize(cap.iq, 128.0), 9)
    truth = {bytes(t.data) for t in cap.truth}
    got = {bytes(f["bytes"][:f["len"]]) for f in fr if f["crc_ok"]}
    assert len(truth & got) >= 0.8 * len(truth)
    assert (fr["len"] - 5 <= 31).all()


# ---------------------------------------------------------------- needs the reference-compiled oracle
ref = pytest.mark.skipif(not os.path.exists(os.path.join(os.path.dirname(GOLDEN), "..", "oracle", "_ref", "libbtle_ref.so")),
                         reason="oracle/_ref not built (needs /root/reference)")


@ref
def test_port_equals_reference_live(oracle_mod):
    for seed, ch, esn0 in ((77, 37, 12.0), (78, 20, 18.0), (79, 39, 30.0)):
        cap = synth.ble_capture(n=500_000, channel=ch, seed=seed, esn0_db=esn0, gap=(100, 3000))
        q = oracle_mod.ble_quantize(cap.iq, 128.0)
        assert_frames_equal(oracle_mod.ble_decode(q, ch), oracle_mod.ble_decode(q, ch, impl="reference"), what=f"seed {seed}")


def test_restated_loop_equals_real_receiver_stdout(oracle_mod, golden):
    """The harness obtains records by walking receiver()'s steps with the reference's functions;
    the text the real receiver() prints must describe the same frames."""
    g = golden("btle_synth_ref.npz")
    for seed in (1001, 1002):
        lines = [l for l in str(g[f"stdout_{seed}"]).splitlines() if " Pkt" in l]
        fr = g[f"frames_{seed}"]
        assert len(lines) == len(fr)
        for line, f in zip(lines, fr):
            pdu = bytes(f["bytes"][:f["len"]])
            assert line.endswith(f"CRC{0 if f['crc_ok'] else 1}")
            assert f" Ch{f['channel']} " in line and f"PloadL{pdu[1] & 0x3F} " in line


def test_access_mask_port_matches_reference_fixture(oracle_mod, golden):
    """-m / access_bit_mask (btle_rx.c:1395-1401, 2301): masked-out bits do not take part in the match."""
    g = golden("btle_mask_ref.npz")
    s, esn0, ch, n = g["params"]
    cap = synth.ble_capture(n=int(n), channel=int(ch), seed=int(s), esn0_db=float(esn0), gap=(100, 1500))
    q = oracle_mod.ble_quantize(cap.iq, 128.0)
    sizes = []
    for mask in (0xFFFFFF00, 0x00FFFFFF, 0xFFFF0000, 0xFFFFFFFE):
        fr = oracle_mod.ble_decode(q, int(ch), aa_mask=mask)
        assert_frames_equal(fr, g[f"frames_{mask:08x}"], what=f"mask {mask:08x}")
        sizes.append(len(fr))
    assert min(sizes) > 10

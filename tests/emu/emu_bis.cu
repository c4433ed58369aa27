// TEST INFRASTRUCTURE ONLY.  Host-side stepping of the BLE broadcast-isochronous cores of snout_b200/csrc/ble_bis.cuh (the
// BIGInfo parse, the BIS access address and CRC init, the subevent channels, the payload number, the subevent window and the
// listed k range that the schedule kernels call with BigSched), built by nvcc into a temporary shared library by
// tests/test_ble_bis.py and run on the CPU (no GPU needed).  Never part of libsnoutrx.so.  A BIGInfo is passed as its bytes.
#include <cstdint>
#include "../../snout_b200/csrc/ble_bis.cuh"

using namespace snrx;

static BigInfo emu_bi(const uint8_t* b, int n) {
    BigInfo bi{};
    big_info_decode(b, n, bi);
    return bi;
}

extern "C" {

// f = offset, units_us, iso_interval, num_bis, nse, bn, sub_interval, pto, bis_spacing, irc, max_pdu, sdu_interval, max_sdu,
// phy, framing, encrypted, saa, base_crc, valid; -1 if the PDU carries no BIGInfo
int emu_big_info_find(const uint8_t* pdu, int n_payload, int64_t* f /*[19]*/, uint64_t* chm, uint64_t* payload_count) {
    BigInfo bi{};
    if (!big_info_find(pdu, n_payload, bi)) return -1;
    const int64_t v[19] = {bi.offset, bi.units_us, bi.iso_interval, bi.num_bis, bi.nse, bi.bn, bi.sub_interval, bi.pto, bi.bis_spacing,
                           bi.irc, bi.max_pdu, bi.sdu_interval, bi.max_sdu, bi.phy, bi.framing, bi.encrypted, bi.saa, bi.base_crc,
                           big_info_valid(bi) ? 1 : 0};
    for (int i = 0; i < 19; i++) f[i] = v[i];
    *chm = bi.chm;
    *payload_count = bi.payload_count;
    return 0;
}
uint32_t emu_bis_access_address(uint32_t saa, int n) { return bis_access_address(saa, n); }
uint32_t emu_bis_crc_init(uint32_t base, int n) { return bis_crc_init(base, n); }
int emu_bis_channel(uint32_t counter, uint32_t aa, uint64_t chm, int se) { return bis_channel(counter, aa, chm, se); }
uint64_t emu_bis_payload_number(const uint8_t* b, int n, int64_t k, int se) { return bis_payload_number(emu_bi(b, n), k, se); }
int64_t emu_big_s_min(const uint8_t* b, int n) { return big_s_min(emu_bi(b, n)); }
void emu_bis_window(const uint8_t* b, int n, int ppm, int64_t k, int bis, int se, int64_t* lo, int64_t* hi) {
    bis_window(emu_bi(b, n), ppm, k, bis, se, *lo, *hi);
}
void emu_big_k_range(const uint8_t* b, int n, int ppm, int64_t s, int sps, int64_t base, int64_t n_out, int64_t* k_lo, int64_t* k_hi) {
    big_k_range(emu_bi(b, n), ppm, s, sps, base, n_out, *k_lo, *k_hi);
}

}  // extern "C"

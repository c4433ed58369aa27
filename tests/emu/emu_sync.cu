// TEST INFRASTRUCTURE ONLY.  Host-side stepping of the BLE periodic-advertising cores of snout_b200/csrc/ble_sync.cuh (the
// SyncInfo parse, CSA#2, the event window and the listed k range that k_ble_sync_count / k_ble_sync_events call), built by
// nvcc into a temporary shared library by tests/test_ble_periodic.py and run on the CPU (no GPU needed).  Never part of
// libsnoutrx.so.
#include <cstdint>
#include "../../snout_b200/csrc/ble_sync.cuh"

using namespace snrx;

static SyncInfo emu_si(int offset, int units_us, int adjust, int interval, int sca) {
    SyncInfo si{};
    si.offset = offset; si.units_us = units_us; si.adjust = adjust; si.interval = interval; si.sca = sca; si.chm = 3;
    return si;
}

extern "C" {

// f = offset, units_us, adjust, interval, sca, aa, crc_init, pa_counter, valid; -1 if the PDU carries no SyncInfo
int emu_sync_info_parse(const uint8_t* pdu, int n_payload, int32_t* f /*[9]*/, uint64_t* chm) {
    SyncInfo si{};
    if (!sync_info_parse(pdu, n_payload, si)) return -1;
    f[0] = si.offset; f[1] = si.units_us; f[2] = si.adjust; f[3] = si.interval; f[4] = si.sca;
    f[5] = (int32_t)si.aa; f[6] = (int32_t)si.crc_init; f[7] = (int32_t)si.pa_counter; f[8] = sync_info_valid(si) ? 1 : 0;
    *chm = si.chm;
    return 0;
}
int emu_csa2_channel(uint32_t counter, uint32_t aa, uint64_t chm) { return csa2_channel(counter, aa, chm); }
void emu_sync_window(int offset, int units_us, int adjust, int interval, int sca, int64_t k, int64_t* lo, int64_t* hi) {
    sync_window(emu_si(offset, units_us, adjust, interval, sca), k, *lo, *hi);
}
void emu_sync_k_range(int offset, int units_us, int adjust, int interval, int sca, int64_t s, int sps, int64_t base, int64_t n_out,
                      int64_t* k_lo, int64_t* k_hi) {
    sync_k_range(emu_si(offset, units_us, adjust, interval, sca), s, sps, base, n_out, *k_lo, *k_hi);
}
uint32_t emu_crc_seed_of(uint32_t crc_init) { return crc_seed_of(crc_init); }

}  // extern "C"

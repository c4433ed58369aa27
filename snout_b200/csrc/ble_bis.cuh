// ble_bis.cuh -- BLE broadcast isochronous streams: follow the BIGInfo in every AUX_SYNC_IND that snrx_ble_periodic decoded
// to the BIS subevents it describes, on the 1M and 2M PHYs, in the slicer bit streams the batch left in HBM.  The contract
// (carriers, BIGInfo fields, BIS access addresses and CRC inits, subevent channels, payload numbers, windows, listed events,
// search, decode, statuses, order) is stated in include/snoutrx.h above snrx_ble_bis_t; oracle/bis_oracle.py restates it.
//
// Launched by snrx_ble_bis after the periodic list is built, no atomics and no sort: the schedule kernels of ble_sync.cuh
// with BigSched,
//   k_ble_sched_flag / exclusive_scan / k_ble_sched_fill   the BIGs, in source order (one warp per periodic entry: the
//                                                          earliest carrier of its (capture, SAA) by a ballot over the others)
//   k_ble_sched_count / exclusive_scan / k_ble_sched_entries  the listed events of every BIG, Num_BIS x NSE entries each,
//                                                          with their AAs, CRC inits, counters, channels, payload numbers,
//                                                          windows and OUTSIDE
//   k_ble_sync_search<snrx_ble_bis_t>                      one warp per entry: windowed search with AA_n, then the decode
//                                                          with crc_init_n
#pragma once
#include "ble_sync.cuh"

namespace snrx {

static_assert(sizeof(snrx_ble_bis_t) == 336 && sizeof(snrx_ble_bis_t) % 16 == 0, "snrx_ble_bis_t layout (include/snoutrx.h, _abi.BIS_DTYPE)");

constexpr int kAdBigInfo = 0x2C;

struct BigInfo {
    int offset, units_us, iso_interval, num_bis, nse, bn, sub_interval, pto, bis_spacing, irc, max_pdu;
    int sdu_interval, max_sdu, phy, framing, encrypted;
    uint32_t saa, base_crc;
    uint64_t chm;                 // bits 0..36
    uint64_t payload_count;       // 39 bits
};

// the fields of a BIGInfo of n = 33 or 57 bytes (the layout of include/snoutrx.h)
SNRX_HD void big_info_decode(const uint8_t* b, int n, BigInfo& bi) {
    auto le = [&](int at, int nb) { uint64_t v = 0; for (int i = nb - 1; i >= 0; i--) v = (v << 8) | b[at + i]; return v; };
    const uint64_t w0 = le(0, 4), w1 = le(4, 4), w2 = le(8, 4), w5 = le(17, 4), w7 = le(23, 5), w8 = le(28, 5);
    bi.offset = (int)(w0 & 0x3FFFu);
    bi.units_us = ((w0 >> 14) & 1u) ? 300 : 30;
    bi.iso_interval = (int)((w0 >> 15) & 0xFFFu);
    bi.num_bis = (int)((w0 >> 27) & 0x1Fu);
    bi.nse = (int)(w1 & 0x1Fu);
    bi.bn = (int)((w1 >> 5) & 7u);
    bi.sub_interval = (int)((w1 >> 8) & 0xFFFFFu);
    bi.pto = (int)((w1 >> 28) & 0xFu);
    bi.bis_spacing = (int)(w2 & 0xFFFFFu);
    bi.irc = (int)((w2 >> 20) & 0xFu);
    bi.max_pdu = (int)((w2 >> 24) & 0xFFu);
    bi.saa = (uint32_t)le(13, 4);
    bi.sdu_interval = (int)(w5 & 0xFFFFFu);
    bi.max_sdu = (int)((w5 >> 20) & 0xFFFu);
    bi.base_crc = (uint32_t)le(21, 2);
    bi.chm = w7 & ((1ull << 37) - 1ull);
    bi.phy = (int)((w7 >> 37) & 7u);
    bi.payload_count = w8 & ((1ull << 39) - 1ull);
    bi.framing = (int)((w8 >> 39) & 1u);
    bi.encrypted = n == 57;
}

// pdu = header(2) | payload; n_payload = payload bytes.  True if this is a PDU of type 7 whose extended header holds its
// flagged fields and an ACAD whose first AD structure of type 0x2C is a BIGInfo of 33 or 57 bytes (the walk stops at a
// length-0 structure or one that overruns the ACAD).
SNRX_HD bool big_info_find(const uint8_t* pdu, int n_payload, BigInfo& bi) {
    int off, end;                                                 // the ACAD is p[off, end)
    if (!ext_header_field(pdu, n_payload, kExtAcad, off, end)) return false;
    const uint8_t* p = pdu + 2;
    for (int at = off; at < end && p[at] != 0 && at + 1 + p[at] <= end; at += 1 + p[at]) {
        if (p[at + 1] != kAdBigInfo) continue;
        if (p[at] != 34 && p[at] != 58) return false;
        big_info_decode(p + at + 2, p[at] - 1, bi);
        return true;
    }
    return false;
}

// the least spacing of two packets of one BIS (us): within an event Sub_Interval, across events the rest of the interval
SNRX_HD int64_t big_s_min(const BigInfo& bi) {
    const int64_t I = 1250 * (int64_t)bi.iso_interval;
    if (bi.nse == 1) return I;
    const int64_t a = bi.sub_interval, b = I - (int64_t)(bi.nse - 1) * bi.sub_interval;
    return a < b ? a : b;
}

// a BIGInfo that describes a BIG this receiver follows
SNRX_HD bool big_info_valid(const BigInfo& bi) {
    const int64_t I = 1250 * (int64_t)bi.iso_interval;
    return bi.num_bis >= 1 && bi.bn >= 1 && bi.nse >= 1 && bi.nse % bi.bn == 0 && bi.irc >= 1 && bi.irc <= bi.nse / bi.bn &&
           bi.iso_interval >= 4 && bi.phy <= 1 && popcount64(bi.chm) >= 2 &&
           (int64_t)(bi.num_bis - 1) * bi.bis_spacing + (int64_t)(bi.nse - 1) * bi.sub_interval < I && big_s_min(bi) > 0;
}

// AA_n = SAA ^ DW_n, D = (35 n + 42) mod 128, DW_n bits 31..16 = D0 D0 D0 D0 D0 D0 D1 D6 D1 0 D5 D4 0 D3 D2 0
SNRX_HD uint32_t bis_access_address(uint32_t saa, int n) {
    const uint32_t d = (uint32_t)(35 * n + 42) & 0x7Fu;
    auto bit = [&](int i) { return (d >> i) & 1u; };
    const uint32_t dw = (bit(0) ? 0xFC000000u : 0u) | bit(1) << 25 | bit(6) << 24 | bit(1) << 23 | bit(5) << 21 | bit(4) << 20 |
                        bit(3) << 18 | bit(2) << 17;
    return saa ^ dw;
}

// crc_init_n as c0 << 16 | c1 << 8 | c2: the CRCInit BaseCRCInit << 8 | n sent least significant byte first
SNRX_HD uint32_t bis_crc_init(uint32_t base_crc, int n) {
    return ((uint32_t)n << 16) | ((base_crc & 0xFFu) << 8) | ((base_crc >> 8) & 0xFFu);
}

// The channel of subevent se of the event with counter `counter`, for access address aa and the used channels chm (at least
// 2): subevent 0 is csa2_channel, each later one steps prnSubEvent_lu from the event's prn_s and moves at least d used
// channels on from the previous one (Core Vol 6 Part B 4.5.8.3 as read in include/snoutrx.h).
SNRX_HD int bis_channel(uint32_t counter, uint32_t aa, uint64_t chm, int se) {
    const int ch0 = csa2_channel(counter, aa, chm);
    if (se == 0) return ch0;
    const uint32_t cid = ((aa >> 16) ^ aa) & 0xFFFFu;
    uint32_t u = csa2_prn_s(counter, cid);
    const int n = popcount64(chm);
    const int d3 = n - 5 < 3 ? n - 5 : 3, d11 = (n - 10) / 2 < 11 ? (n - 10) / 2 : 11;
    const int d = d3 > d11 ? (d3 > 1 ? d3 : 1) : (d11 > 1 ? d11 : 1);
    int idx = popcount64(chm & ((1ull << ch0) - 1ull));           // the used-channel number of subevent 0
    for (int j = 1; j <= se; j++) {
        u = csa2_perm_mam(u, cid);
        const uint32_t prn_se = u ^ cid;
        idx = (int)(((uint32_t)idx + (uint32_t)d + ((prn_se * (uint32_t)(n - 2 * d + 1)) >> 16)) % (uint32_t)n);
    }
    return csa2_used_channel(chm, idx);
}

// the payload number subevent se of event k carries: group g = se / BN (g >= IRC: pretransmissions PTO (g - IRC + 1) events
// ahead), i = se mod BN
SNRX_HD uint64_t bis_payload_number(const BigInfo& bi, int64_t k, int se) {
    const int g = se / bi.bn, i = se % bi.bn;
    const int64_t M = 1ll << 39;
    int64_t e = (int64_t)(bi.payload_count / (uint64_t)bi.bn) + k + (g < bi.irc ? 0 : (int64_t)bi.pto * (g - bi.irc + 1));
    e %= M;
    if (e < 0) e += M;
    return (uint64_t)e * (uint64_t)bi.bn + (uint64_t)i;
}

// D_lo of subevent (n, se) of event k, us after the source's AA bit 0
SNRX_HD int64_t bis_d_lo(const BigInfo& bi, int64_t k, int n, int se) {
    return (int64_t)bi.offset * bi.units_us + 1250 * (int64_t)bi.iso_interval * k + (int64_t)(n - 1) * bi.bis_spacing +
           (int64_t)se * bi.sub_interval;
}

// [lo, hi] of AA bit 0 positions of subevent (n, se) of event k, relative to the source's AA bit 0; p = the train's ppm
SNRX_HD void bis_window(const BigInfo& bi, int p, int64_t k, int n, int se, int64_t& lo, int64_t& hi) {
    const int64_t d = bis_d_lo(bi, k, n, se);
    drift_window(d, d + bi.units_us, p, lo, hi);
}

// rule (a) for one window: at most 2 S_min samples, half the same-address spacing
SNRX_HD bool bis_window_ok(const BigInfo& bi, int p, int64_t k, int n, int se) {
    int64_t lo, hi;
    bis_window(bi, p, k, n, se, lo, hi);
    return hi - lo + 1 <= 2 * big_s_min(bi);
}

SNRX_HD bool big_event_ok(const BigInfo& bi, int p, int64_t k) {
    for (int n = 1; n <= bi.num_bis; n++)
        for (int se = 0; se < bi.nse; se++)
            if (!bis_window_ok(bi, p, k, n, se)) return false;
    return true;
}

// The listed k of a BIG whose source's AA bit 0 is at capture index s, in a buffer of local decisions [0, n_out - 2] whose
// sample 0 is capture index base: [k_lo, k_hi], empty when k_lo > k_hi.
//   Rule (a).  A window's width late(D + U) - early(D) + 17 does not shrink as D grows from 0 (late gains at least 4 per us,
//   early at most 4), nor as D falls while D + U < 0 (the mirror image).  For k >= k_c every D is >= 0, so the widest window
//   of an event is its last subevent's and the widths grow with k: one monotone test.  For k <= k_c - 3 every D + U is below
//   0 (D_lo(1, 0) < 1250 ISO_Interval at k_c, and every subevent starts inside the interval), so the widest window is the
//   first subevent's and the widths grow as k falls: another monotone test.  Events k_c - 1 and k_c - 2 can hold windows
//   with D < 0 <= D + U, so every window of theirs is tested.  A window whose |D| exceeds 2 S_min 10^6 / (8 p) us is wider
//   than 2 S_min (the width is at least 8 |D| p / 10^6), so every D met is below 2 * 5 118 750 * 10^6 / (8 * 20) us plus two
//   intervals: 4 |D| 10^6 stays inside int64.
//   Disjointness.  Two packets of one BIS are at least S_min us apart; early() of the later one is at least
//   4 S (10^6 - p) / 10^6 - 1 samples past early() of the earlier one, whose window (at most 2 S_min samples, which rule (a)
//   needs to be at least 4 U + 17 >= 137) then ends more than 2 S_min - 0.002 S_min - 1 > 31 * 4 samples before the later
//   window starts.
//   Rule (b).  rule_b_range with the first window's start, win_lo(1, 0), and the last window's end, win_hi(Num_BIS, NSE - 1).
SNRX_HD void big_k_range(const BigInfo& bi, int p, int64_t s, int sps, int64_t base, int64_t n_out, int64_t& k_lo, int64_t& k_hi) {
    const int64_t I = 1250 * (int64_t)bi.iso_interval, O = (int64_t)bi.offset * bi.units_us, smin = big_s_min(bi);
    const int nb = bi.num_bis, se_last = bi.nse - 1;
    const int64_t kc = ceil_div(-O, I);                           // the first k with D_lo(1, 0) >= 0
    k_lo = kc; k_hi = kc - 1;
    if (!bis_window_ok(bi, p, kc, nb, se_last)) return;           // every window of event k_c (all D >= 0)
    const int64_t de = (2 * smin * 1000000 / (8 * (int64_t)p)) / I; // (de + 1) I > 2 S_min 10^6 / (8 p): no window that far passes
    int64_t a_hi = kc + de + 1;                                   // fails: its last subevent's D >= (de + 1) I
    while (a_hi > kc && !bis_window_ok(bi, p, a_hi, nb, se_last)) a_hi--;
    while (bis_window_ok(bi, p, a_hi + 1, nb, se_last)) a_hi++;
    int64_t a_lo;
    if (!big_event_ok(bi, p, kc - 1)) a_lo = kc;
    else if (!big_event_ok(bi, p, kc - 2)) a_lo = kc - 1;
    else {                                                        // k <= k_c - 3: the first subevent's test, true on [a_lo, k_c - 3]
        a_lo = kc - 3 - de;
        if (bis_window_ok(bi, p, a_lo, 1, 0)) { while (bis_window_ok(bi, p, a_lo - 1, 1, 0)) a_lo--; }
        else { while (a_lo < kc - 2 && !bis_window_ok(bi, p, a_lo, 1, 0)) a_lo++; }
    }
    rule_b_range(a_lo, a_hi, O, I, [&](int64_t k) { int64_t lo, hi; bis_window(bi, p, k, 1, 0, lo, hi); return lo; },
                 [&](int64_t k) { int64_t lo, hi; bis_window(bi, p, k, nb, se_last, lo, hi); return hi; }, s, sps, base, n_out, k_lo, k_hi);
}

struct BigGroup {
    BigInfo bi;
    int64_t s;                    // the source's sample_index
    int64_t k_lo;                 // first listed event (k_ble_sched_count)
    uint32_t capture_id, source;
    int ppm;                      // of the source's train's SCA
};

#if defined(__CUDACC__)
// snrx_ble_bis: periodic entry -> BigGroup -> Num_BIS x NSE entries per listed event (the schedule kernels of ble_sync.cuh)
struct BigSched {
    using Src = snrx_ble_sync_t;
    using Group = BigGroup;
    using Entry = snrx_ble_bis_t;
    // a carrier (status OK, crc_ok, a valid BIGInfo); grouped by its SAA
    static __device__ __forceinline__ bool candidate(const Src& r, uint32_t, uint32_t& key) {
        BigInfo bi;
        if (!(r.status == SNRX_AUX_OK && r.crc_ok && r.len >= 5 && big_info_find(r.bytes, (int)r.len - 5, bi) && big_info_valid(bi))) return false;
        key = bi.saa;
        return true;
    }
    static __device__ __forceinline__ Group group(const Src& r, uint32_t i) {
        BigGroup b{};
        big_info_find(r.bytes, (int)r.len - 5, b.bi);
        b.s = r.sample_index; b.capture_id = r.capture_id; b.source = i; b.ppm = sca_ppm(r.sca);
        return b;
    }
    static __device__ __forceinline__ void k_range(const Group& b, const AuxGeom& g, int64_t& k_lo, int64_t& k_hi) {
        big_k_range(b.bi, b.ppm, b.s, b.bi.phy == SNRX_AUX_PHY_2M ? 2 : 4, g.base, g.n_out, k_lo, k_hi);
    }
    static __device__ __forceinline__ uint32_t per_event(const Group& b) { return (uint32_t)(b.bi.num_bis * b.bi.nse); }
    // entry j = (n - 1) NSE + se: BIS n, subevent se.  A BIS whose AA is 0 is not searched.
    static __device__ __forceinline__ uint8_t entry(const Group& b, int64_t k, uint32_t j, Entry& r) {
        const BigInfo& bi = b.bi;
        const int n = (int)(j / (uint32_t)bi.nse) + 1, se = (int)(j % (uint32_t)bi.nse);
        int64_t lo, hi;
        bis_window(bi, b.ppm, k, n, se, lo, hi);
        const uint32_t counter = ((uint32_t)(bi.payload_count / (uint64_t)bi.bn) + (uint32_t)k) & 0xFFFFu;
        const uint32_t aa = bis_access_address(bi.saa, n);
        r.win_lo = b.s + lo; r.win_hi = b.s + hi;
        r.payload_number = bis_payload_number(bi, k, se);
        r.access_addr = aa;
        r.crc_init = bis_crc_init(bi.base_crc, n);
        r.event_counter = (uint16_t)counter;
        r.bis = (uint8_t)n;
        r.subevent = (uint8_t)se;
        r.channel = (uint8_t)bis_channel(counter, aa, bi.chm, se);
        r.phy = (uint8_t)bi.phy;
        r.flags = (uint8_t)((bi.encrypted ? SNRX_BIS_ENCRYPTED : 0) | (bi.framing ? SNRX_BIS_FRAMED : 0));
        return aa == 0u ? SNRX_AUX_NOT_FOUND : kAuxPending;
    }
};
#endif  // __CUDACC__

}  // namespace snrx

// ble_sync.cuh -- BLE periodic advertising: follow the SyncInfo of every AUX_ADV_IND that snrx_ble_aux decoded to the
// AUX_SYNC_IND train it describes, on the 1M and 2M PHYs, in the slicer bit streams the batch left in HBM.  The contract
// (train sources, SyncInfo fields, CSA#2, windows, listed events, search, decode, statuses, order) is stated in
// include/snoutrx.h above snrx_ble_sync_t; oracle/periodic_oracle.py restates it.
//
// Launched by snrx_ble_periodic after the pointer rounds of snrx_ble_aux, no atomics and no sort; the schedule kernels are
// shared with snrx_ble_bis (ble_bis.cuh), SyncSched is this list's instance:
//   k_ble_sched_flag / exclusive_scan / k_ble_sched_fill   the trains, in source order (one warp per aux entry: the earliest
//                                                         source of its (capture, AA) by a ballot over the other candidates)
//   k_ble_sched_count / exclusive_scan / k_ble_sched_entries  the listed events of every train, in ascending k, with their
//                                                         counters, CSA#2 channels, windows and OUTSIDE
//   k_ble_sync_search                                    one warp per event: windowed search with the train's AA, then the
//                                                         decode that k_ble_aux_search uses, with the train's CRC init
#pragma once
#include "ble_aux.cuh"

namespace snrx {

static_assert(sizeof(snrx_ble_sync_t) == 320 && sizeof(snrx_ble_sync_t) % 16 == 0, "snrx_ble_sync_t layout (include/snoutrx.h, _abi.SYNC_DTYPE)");

constexpr int64_t kSyncOffsetAdjustUs = 2457600;

struct SyncInfo {
    int offset, units_us, adjust, interval, sca;
    uint64_t chm;                 // bits 0..36
    uint32_t aa, crc_init;        // crc_init = c0 << 16 | c1 << 8 | c2
    uint32_t pa_counter;
};

// pdu = header(2) | payload; n_payload = payload bytes.  True if pdu carries a SyncInfo inside its extended header
// (ext_header_field).
SNRX_HD bool sync_info_parse(const uint8_t* pdu, int n_payload, SyncInfo& si) {
    int off, end;
    if (!ext_header_field(pdu, n_payload, kExtSyncInfo, off, end) || off + 18 > end) return false;
    const uint8_t* b = pdu + 2 + off;
    const int o = b[0] | (b[1] << 8);
    si.offset = o & 0x1FFF;
    si.units_us = (o & 0x2000) ? 300 : 30;
    si.adjust = (o >> 14) & 1;
    si.interval = b[2] | (b[3] << 8);
    uint64_t v = 0;
    for (int i = 4; i >= 0; i--) v = (v << 8) | b[4 + i];
    si.chm = v & ((1ull << 37) - 1ull);
    si.sca = (int)((v >> 37) & 7u);
    si.aa = (uint32_t)b[9] | ((uint32_t)b[10] << 8) | ((uint32_t)b[11] << 16) | ((uint32_t)b[12] << 24);
    si.crc_init = ((uint32_t)b[13] << 16) | ((uint32_t)b[14] << 8) | (uint32_t)b[15];
    si.pa_counter = (uint32_t)b[16] | ((uint32_t)b[17] << 8);
    return true;
}

SNRX_HD int popcount64(uint64_t x) {
    int n = 0;
    for (; x; x &= x - 1) n++;
    return n;
}

// a SyncInfo that describes a train
SNRX_HD bool sync_info_valid(const SyncInfo& si) {
    return si.offset != 0 && si.interval >= SNRX_SYNC_MIN_INTERVAL && popcount64(si.chm) >= 2;
}

SNRX_HD int sca_ppm(int sca) {
    constexpr int ppm[8] = {500, 250, 150, 100, 75, 50, 30, 20};
    return ppm[sca & 7];
}

// Channel Selection Algorithm #2 (Core Vol 6 Part B 4.5.8.3), shared by the periodic events and the BIS subevents.
SNRX_HD uint32_t csa2_perm_mam(uint32_t u, uint32_t cid) {
    uint32_t v = 0;                                               // PERM: the bits of each byte reversed
    for (int i = 0; i < 8; i++) v |= (((u >> i) & 0x0101u)) << (7 - i);
    return (17u * v + cid) & 0xFFFFu;                             // MAM
}

// prn_s of event counter `counter` for channel identifier cid
SNRX_HD uint32_t csa2_prn_s(uint32_t counter, uint32_t cid) {
    uint32_t u = (counter ^ cid) & 0xFFFFu;
    for (int r = 0; r < 3; r++) u = csa2_perm_mam(u, cid);
    return u;
}

// the idx-th used channel of chm (idx below the number of used channels)
SNRX_HD int csa2_used_channel(uint64_t chm, int idx) {
    for (int c = 0; c < 37; c++)
        if ((chm >> c) & 1u) { if (idx == 0) return c; idx--; }
    return -1;                                                    // not reached
}

// the channel of event counter `counter` for access address aa and the used channels chm (at least one)
SNRX_HD int csa2_channel(uint32_t counter, uint32_t aa, uint64_t chm) {
    const uint32_t cid = ((aa >> 16) ^ aa) & 0xFFFFu;
    const uint32_t prn_e = csa2_prn_s(counter, cid) ^ cid;
    const int unmapped = (int)(prn_e % 37u);
    if ((chm >> unmapped) & 1u) return unmapped;
    return csa2_used_channel(chm, (int)(((uint32_t)popcount64(chm) * prn_e) >> 16));
}

SNRX_HD int64_t floor_div(int64_t a, int64_t b) {                 // b > 0
    const int64_t q = a / b;
    return (a % b != 0 && a < 0) ? q - 1 : q;
}
SNRX_HD int64_t ceil_div(int64_t a, int64_t b) { return -floor_div(-a, b); }

// [early(d_lo) - 8, late(d_hi) + 8]: the AA bit 0 positions (4 Msps) of a packet due d_lo..d_hi us after a reference
// packet, by a clock of p ppm either way (mathematical floor and ceiling; shared by the periodic and the BIS windows)
SNRX_HD void drift_window(int64_t d_lo, int64_t d_hi, int64_t p, int64_t& lo, int64_t& hi) {
    lo = (d_lo >= 0 ? floor_div(4 * d_lo * (1000000 - p), 1000000) : floor_div(4 * d_lo * (1000000 + p), 1000000)) - kAuxGuard;
    hi = (d_hi >= 0 ? ceil_div(4 * d_hi * (1000000 + p), 1000000) : ceil_div(4 * d_hi * (1000000 - p), 1000000)) + kAuxGuard;
}

// [lo, hi] of AA bit 0 positions of event k, relative to the source's AA bit 0
SNRX_HD void sync_window(const SyncInfo& si, int64_t k, int64_t& lo, int64_t& hi) {
    const int64_t U = si.units_us, p = sca_ppm(si.sca);
    const int64_t O = (int64_t)si.offset * U + (si.adjust ? kSyncOffsetAdjustUs : 0);
    const int64_t d_lo = O + k * 1250 * (int64_t)si.interval;
    drift_window(d_lo, d_lo + U, p, lo, hi);
}

// rule (a): the window is at most half the interval long
SNRX_HD bool sync_rule_a(const SyncInfo& si, int64_t k) {
    int64_t lo, hi;
    sync_window(si, k, lo, hi);
    return hi - lo + 1 <= 2500 * (int64_t)si.interval;
}

// Rule (b) of a schedule list on the rule-(a) range [a_lo, a_hi]: the listed [k_lo, k_hi] (empty when k_lo > k_hi) of a
// schedule whose source's AA bit 0 is at capture index s, in a buffer of local decisions [0, n_out - 2] whose sample 0 is
// capture index base.  win_lo(k) is the start of event k's first window and win_hi(k) the end of its last one, relative to
// s.  Both grow with k, so s + win_hi(k) + 31 sps >= base is false, then true as k grows, and s + win_lo(k) <= base +
// n_out - 2 is true, then false: each bound is stepped from the estimate floor((floor((x - s) / 4) - O) / I), the event
// whose D_lo (O + k I us after the source) is due at capture index x.
template <class WinLo, class WinHi>
SNRX_HD void rule_b_range(int64_t a_lo, int64_t a_hi, int64_t O, int64_t I, WinLo win_lo, WinHi win_hi, int64_t s, int sps,
                          int64_t base, int64_t n_out, int64_t& k_lo, int64_t& k_hi) {
    const int64_t last = base + n_out - 2;
    auto meets_lo = [&](int64_t k) { return s + win_hi(k) + 31 * sps >= base; };
    auto meets_hi = [&](int64_t k) { return s + win_lo(k) <= last; };
    auto clamp = [](int64_t k, int64_t a, int64_t b) { return k < a ? a : (k > b ? b : k); };
    int64_t k = clamp(floor_div(floor_div(base - s, 4) - O, I), a_lo, a_hi);
    while (k > a_lo && meets_lo(k - 1)) k--;
    while (k <= a_hi && !meets_lo(k)) k++;
    k_lo = k;
    if (k_lo > a_hi) { k_hi = k_lo - 1; return; }
    k = clamp(floor_div(floor_div(last - s, 4) - O, I), k_lo, a_hi);
    while (k < a_hi && meets_hi(k + 1)) k++;
    while (k >= k_lo && !meets_hi(k)) k--;
    k_hi = k;
}

// The listed k of a train (rule_b_range's arguments): rule (a) holds on one contiguous range around the k where D changes
// sign (the width grows by at least 1.2 samples per event on either side, more than the two roundings can take back), found
// by stepping a monotone test from an estimate.  Every D met has |D| <= 2500 * 65535 * 10^6 / (8 * 20) us + one interval:
// 4 |D| 10^6 stays inside int64.
SNRX_HD void sync_k_range(const SyncInfo& si, int64_t s, int sps, int64_t base, int64_t n_out, int64_t& k_lo, int64_t& k_hi) {
    const int64_t I = 1250 * (int64_t)si.interval, U = si.units_us, p = sca_ppm(si.sca);
    const int64_t O = (int64_t)si.offset * U + (si.adjust ? kSyncOffsetAdjustUs : 0);
    const int64_t kc = ceil_div(-O, I);                           // the first k with D_lo >= 0; kc - 1 and kc satisfy (a)
    const int64_t dmax = (2500 * (int64_t)si.interval) * 1000000 / (8 * p);
    int64_t a_hi = kc + dmax / I, a_lo = kc - 1 - dmax / I;
    while (!sync_rule_a(si, a_hi)) a_hi--;
    while (sync_rule_a(si, a_hi + 1)) a_hi++;
    while (!sync_rule_a(si, a_lo)) a_lo++;
    while (sync_rule_a(si, a_lo - 1)) a_lo--;
    rule_b_range(a_lo, a_hi, O, I, [&](int64_t k) { int64_t lo, hi; sync_window(si, k, lo, hi); return lo; },
                 [&](int64_t k) { int64_t lo, hi; sync_window(si, k, lo, hi); return hi; }, s, sps, base, n_out, k_lo, k_hi);
}

// the CRC register seed of a crc_init given as c0 << 16 | c1 << 8 | c2 (btle_rx.c crc_init_reorder: byte swap, 24-bit
// bit reversal)
SNRX_HD uint32_t crc_seed_of(uint32_t crc_init) {
    const uint32_t sw = ((crc_init & 0xFFu) << 16) | (crc_init & 0xFF00u) | ((crc_init >> 16) & 0xFFu);
    uint32_t r = 0;
    for (int i = 0; i < 24; i++) r |= ((sw >> i) & 1u) << (23 - i);
    return r;
}

// A periodic-advertising train: the group SyncSched builds from its source
struct SyncTrain {
    SyncInfo si;
    int64_t s;                    // the source's sample_index
    int64_t k_lo;                 // first listed event (k_ble_sched_count)
    uint32_t capture_id, source;
    int phy;
};

#if defined(__CUDACC__)
// The schedule lists (snrx_ble_periodic, snrx_ble_bis) are built by the kernels below, templated on a schedule S that
// supplies, from its source entries S::Src:
//   candidate(r, i, key)   entry i is a candidate source, and its key: one group per (capture, key)
//   group(r, i)            the S::Group a source describes (s, capture_id, source and what its events need)
//   k_range(grp, g, ..)    the group's listed k; per_event(grp): the entries of one event
//   entry(grp, k, j, r)    entry j of event k: every field of r but those the kernel sets (zero bytes, sample_index -1,
//                          capture_id, source, event, OUTSIDE); returns its status inside the buffer

// One warp per source entry of [0, n): flags[i] = 1 when entry i is the source of its (capture, key) group -- no other
// candidate of the same (capture, key) has a smaller sample_index, or the same one and a lower index.
template <class S>
__global__ void __launch_bounds__(256) k_ble_sched_flag(const typename S::Src* __restrict__ src, uint32_t n, uint32_t* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
        const typename S::Src& r = src[i];
        uint32_t key, ko;
        bool first = S::candidate(r, i, key);                     // warp-uniform
        for (uint32_t b = 0; first && b < n; b += 32) {
            const uint32_t j = b + lane;
            bool earlier = false;
            if (j < n && j != i) {
                const typename S::Src& o = src[j];
                earlier = o.capture_id == r.capture_id && (o.sample_index < r.sample_index || (o.sample_index == r.sample_index && j < i)) &&
                          S::candidate(o, j, ko) && ko == key;
            }
            if (__ballot_sync(0xffffffffu, earlier)) first = false;
        }
        if (lane == 0) flags[i] = first ? 1u : 0u;
    }
}

template <class S>
__global__ void __launch_bounds__(256) k_ble_sched_fill(const typename S::Src* __restrict__ src, uint32_t n, const uint32_t* __restrict__ flags,
                                                        const uint32_t* __restrict__ offsets, typename S::Group* __restrict__ groups) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flags[i]) return;
    groups[offsets[i]] = S::group(src[i], i);
}

// one thread per group: its listed k range, counts[t] = its entries, capped at max_frames + 1 (the caller sums the counts
// in 64 bits and refuses more than max_frames before it scans them)
template <class S>
__global__ void __launch_bounds__(256) k_ble_sched_count(typename S::Group* __restrict__ groups, uint32_t n_groups, AuxGeom g, uint32_t cap,
                                                         uint32_t* __restrict__ counts) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_groups) return;
    typename S::Group& grp = groups[t];
    int64_t k_lo, k_hi;
    S::k_range(grp, g, k_lo, k_hi);
    grp.k_lo = k_lo;
    const int64_t m = k_hi >= k_lo ? (k_hi - k_lo + 1) * S::per_event(grp) : 0;
    counts[t] = (uint32_t)(m > (int64_t)cap ? (int64_t)cap + 1 : m);
}

// one thread per listed entry: S::entry's fields, then OUTSIDE or its status; offsets[0..n_groups] are the groups' first
// entries
template <class S>
__global__ void __launch_bounds__(256) k_ble_sched_entries(const typename S::Group* __restrict__ groups, uint32_t n_groups,
                                                           const uint32_t* __restrict__ offsets, uint32_t total, AuxGeom g,
                                                           typename S::Entry* __restrict__ list) {
    using E = typename S::Entry;
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    uint32_t a = 0, b = n_groups;                                 // the last t with offsets[t] <= e
    while (b - a > 1) { const uint32_t m = (a + b) >> 1; if (offsets[m] <= e) a = m; else b = m; }
    const typename S::Group& grp = groups[a];
    const uint32_t local = e - offsets[a], per_event = S::per_event(grp);
    const int64_t k = grp.k_lo + (int64_t)(local / per_event);
    E& r = list[e];
    uint4* d = reinterpret_cast<uint4*>(&r);
#pragma unroll
    for (int q = 0; q < (int)(sizeof(E) / 16); q++) d[q] = make_uint4(0u, 0u, 0u, 0u);
    const uint8_t st = S::entry(grp, k, local % per_event, r);
    r.sample_index = -1;
    r.capture_id = grp.capture_id;
    r.source = grp.source;
    r.event = (int32_t)k;
    const int sps = r.phy == SNRX_AUX_PHY_2M ? 2 : 4;
    const int64_t l = r.win_lo - g.base, x = r.win_hi - g.base + 31 * sps;      // local first / last decision of the search
    r.status = (l < 0 || x + 1 >= g.n_out) ? SNRX_AUX_OUTSIDE : st;
}

// snrx_ble_periodic: aux entry -> SyncTrain -> one event per listed k
struct SyncSched {
    using Src = snrx_ble_aux_t;
    using Group = SyncTrain;
    using Entry = snrx_ble_sync_t;
    // status OK, crc_ok, first == i, a valid SyncInfo; grouped by its AA
    static __device__ __forceinline__ bool candidate(const Src& r, uint32_t i, uint32_t& key) {
        SyncInfo si;
        if (!(r.status == SNRX_AUX_OK && r.crc_ok && r.first == i && r.len >= 5 && sync_info_parse(r.bytes, (int)r.len - 5, si) &&
              sync_info_valid(si)))
            return false;
        key = si.aa;
        return true;
    }
    static __device__ __forceinline__ Group group(const Src& r, uint32_t i) {
        SyncTrain t{};
        sync_info_parse(r.bytes, (int)r.len - 5, t.si);
        t.s = r.sample_index; t.capture_id = r.capture_id; t.source = i; t.phy = r.phy;
        return t;
    }
    static __device__ __forceinline__ void k_range(const Group& t, const AuxGeom& g, int64_t& k_lo, int64_t& k_hi) {
        sync_k_range(t.si, t.s, t.phy == SNRX_AUX_PHY_2M ? 2 : 4, g.base, g.n_out, k_lo, k_hi);
    }
    static __device__ __forceinline__ uint32_t per_event(const Group&) { return 1u; }
    static __device__ __forceinline__ uint8_t entry(const Group& t, int64_t k, uint32_t, Entry& r) {
        int64_t lo, hi;
        sync_window(t.si, k, lo, hi);
        const uint32_t counter = (t.si.pa_counter + (uint32_t)k) & 0xFFFFu;
        r.win_lo = t.s + lo; r.win_hi = t.s + hi;
        r.access_addr = t.si.aa;
        r.crc_init = t.si.crc_init;
        r.event_counter = (uint16_t)counter;
        r.interval = (uint16_t)t.si.interval;
        r.channel = (uint8_t)csa2_channel(counter, t.si.aa, t.si.chm);
        r.phy = (uint8_t)t.phy;
        r.sca = (uint8_t)t.si.sca;
        return kAuxPending;
    }
};

// One warp per pending entry of [0, n): the earliest full match of the entry's access address in its window, then the
// decode with its CRC init.  E is snrx_ble_sync_t (a periodic event) or snrx_ble_bis_t (a BIS subevent, ble_bis.cuh).
template <class E>
__global__ void __launch_bounds__(128) k_ble_sync_search(E* __restrict__ list, uint32_t n, AuxGeom g,
                                                         const uint32_t* __restrict__ crc_tab, const uint8_t* __restrict__ whiten /*[40][260]*/) {
    __shared__ uint32_t crc_s[256];
    __shared__ uint8_t buf_s[4][SNRX_AUX_MAX_BYTES];
    __shared__ AaTables tabs_s[4];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_s[i] = crc_tab[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    for (uint32_t k = blockIdx.x * (blockDim.x >> 5) + wib; k < n; k += warps) {
        E& r = list[k];
        if (r.status != kAuxPending) continue;                    // warp-uniform
        const uint32_t aa = r.access_addr;
        tabs_s[wib].want0[lane] = ((aa >> lane) & 1u) - 1u;
        tabs_s[wib].dont_care[lane] = 0u;
        __syncwarp();
        const int sps = r.phy == SNRX_AUX_PHY_2M ? 2 : 4;
        const int lo = (int)(r.win_lo - g.base), hi = (int)(r.win_hi - g.base);   // inside the buffer (k_ble_sched_entries)
        const uint32_t* pw = g.bits + g.lay.index(r.capture_id - g.first_capture, r.channel, 0);
        const int nf = aux_find(pw, g.lay.words_per_stream, lo, hi, sps, tabs_s[wib], lane);
        if (nf < 0) { if (lane == 0) r.status = SNRX_AUX_NOT_FOUND; __syncwarp(); continue; }
        aux_decode(r, pw, nf, sps, r.channel, g, crc_s, whiten, crc_seed_of(r.crc_init), buf_s[wib], lane);
    }
}
#endif  // __CUDACC__

}  // namespace snrx

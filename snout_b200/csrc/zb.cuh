// zb.cuh -- IEEE 802.15.4 (Zigbee) receive chain on the GPU.
//
// Reference chain (snout/modulations/Zigbee/hackrf/Zigbee_rx/top_block.py:52-89):
//   analog.quadrature_demod_cf(1) -> x - single_pole_iir_filter_ff(0.00016)(x)
//   -> digital.clock_recovery_mm_ff(2, 0.000225, 0.5, 0.03, 0.0002) -> ieee802_15_4.packet_sink(10)
// with the sink's in-tree statement scapy-radio/gnuradio/gr-zigbee/lib/packet_sink_scapy_impl.cc
// (enter_search 55-65, enter_have_sync 67-79, enter_have_header 81-92, decode_chips 95-125,
// general_work 158-374).  The three GNU Radio stream blocks are not vendored in the reference
// tree; their published algorithms are restated here (and, independently, in oracle/zb_oracle.c,
// which the kernels must match bit for bit: every float operation below is an explicitly rounded
// single operation in a fixed order).
//
// Parallel decomposition (DESIGN.md "Zigbee"):
//   k_zb_quad      one thread per sample: table atan2 of x[n] conj(x[n-1])
//   k_zb_iir_*     the single-pole DC tracker evaluated in blocks of 4096 samples (block-local
//                  recurrence + a carried state folded from the 8 preceding blocks), so blocks run
//                  in parallel and the result does not depend on where a time shard starts
//   k_zb_chain     one thread per (capture, channel, segment): Mueller-Mueller clock recovery feeding
//                  the packet-sink state machine; segments overlap by a warm-up pre-halo and a
//                  longest-frame post-halo, a frame belongs to the segment holding its SFD position
//   k_zb_gather    compaction of the per-chain frame slots into the batch frame list
#pragma once
#include <string>

#include "common.cuh"
#include "scan.cuh"
#define SNRX_TABLE_QUAL static const
#include "zb_tables.h"

namespace snrx {

constexpr int kZbPostHalo = 16448;          // PHR + 127 bytes = 256 symbols * 64 samples, + 64
constexpr int kZbMinSyncChips = 193;        // chips between the SFD-completing chips of two records of one chain, at least: PHR (64),
                                            // one byte (64; a PHR of 0 still waits for one), >= 1 chip to re-lock on the register that
                                            // enter_search() cleared, 7 (32) and 10 (32) -- packet_sink_scapy_impl.cc:55-65, 190-359.
                                            // Not 7 symbols: the cleared register lets the search lock after k < 32 fresh chips (k = 14
                                            // at threshold 10), and every chip advances the clock recovery by 1..3 samples
constexpr int kZbSinkLead = 1024;           // the sink starts this many samples before the body: SHR (640) + alignment
                                            // slack; the clock recovery starts `prehalo` samples early (warm-up only)
constexpr float kZbClamp = 16.0f;           // |z| <= pi + |DC| for any finite input; anything else (Inf / NaN samples in the
                                            // capture) is replaced by 0 so that the clock recovery state stays finite

// fast_atan2f as GNU Radio publishes it (256-entry arctan table of |min| / |max| with linear interpolation, octant fix-up;
// restated with branches in oracle/zb_oracle.c zb_tab_atan2).  Here WITHOUT a branch: sixteen of these run per output time of
// the wideband front end, and the branchy form cost that kernel ~200 BRA + 170 BSSY/BSYNC per tile and a "branch resolving"
// stall of 0.77 per issue (profiles/r02_zb_wb16_ncu.json).  Every arithmetic result is the one the branchy statement
// computes: the octant cases differ only by exact operations (negation, adding +0), e.g. base - pi == -(pi - base) and
// -hpi + base == -(hpi - base) under round-to-nearest, so  ang = +-( C + (+-base) )  with C in {0, pi, pi/2}.
SNRX_HD float f_flip(float v, bool neg) {          // exact: v or -v
#ifdef __CUDA_ARCH__
    return __uint_as_float(__float_as_uint(v) ^ (neg ? 0x80000000u : 0u));
#else
    return neg ? -v : v;
#endif
}
// the table as the kernels read it: entry idx and the step to entry idx + 1
struct AtanTab {                                   // the 257 values themselves
    const float* t;
    SNRX_HD void get(int idx, float& lo, float& d) const { lo = t[idx]; d = f_sub(t[idx + 1], lo); }
};
struct AtanTabPairs {                              // [256] {tab[i], tab[i+1] - tab[i]}: the same single-precision subtraction, done once on
    const float2* t;                               // the host (zb_create) -- one 8-byte load per lookup instead of two loads and an FADD
    SNRX_HD void get(int idx, float& lo, float& d) const {
#ifdef __CUDA_ARCH__
        const float2 e = __ldg(t + idx);
#else
        const float2 e = t[idx];
#endif
        lo = e.x; d = e.y;
    }
};
template <class Tab>
SNRX_HD float tab_atan2_g(float y, float x, Tab tab) {
    const float ya = fabsf(y), xa = fabsf(x);
    const bool x_major = xa > ya;                             // |x| > |y|: the angle is measured from the x axis
    const bool y_lt = ya < xa;
    const float z = f_div(y_lt ? ya : xa, y_lt ? xa : ya);    // (ya < xa) ? ya / xa : xa / ya
    const bool small = z < 0.003921569f;
    float alpha = f_mul(z, 255.0f);
    const int idx = small ? 0 : (((int)alpha) & 0xFF);        // the table is read either way; its value is dropped when small
    alpha = f_sub(alpha, (float)idx);
    float lo, d;
    tab.get(idx, lo, d);
    const float base = small ? z : f_add(lo, f_mul(d, alpha));
    const float pi = 3.14159265358979323846f, hpi = 1.57079632679489661923f;
    const bool xpos = x >= 0.0f, ypos = y >= 0.0f;
    const float c = x_major ? (xpos ? 0.0f : pi) : hpi;
    const float r = f_add(c, f_flip(base, x_major != xpos));  // x-major: base | pi - base;  y-major: hpi - base | hpi + base
    const float ang = f_flip(r, !ypos);
    return (ya > 0.0f || xa > 0.0f) ? ang : 0.0f;
}
SNRX_HD float tab_atan2(float y, float x, const float* tab /*[257]*/) { return tab_atan2_g(y, x, AtanTab{tab}); }

// f = arg(x * conj(p))
template <class Tab>
SNRX_HD float quad_demod_g(float xr, float xi, float pr, float pi, Tab tab) {
    const float re = f_add(f_mul(xr, pr), f_mul(xi, pi));
    const float im = f_sub(f_mul(xi, pr), f_mul(xr, pi));
    return tab_atan2_g(im, re, tab);
}
SNRX_HD float quad_demod(float xr, float xi, float pr, float pi, const float* tab) { return quad_demod_g(xr, xi, pr, pi, AtanTab{tab}); }

// discriminator-domain chip words of the 16 data symbols (derived from the 802.15.4 PN
// sequences; equal CHIP_MAPPING[] & 0x7FFFFFFE of packet_sink_scapy_impl.h:28-45)
struct ChipMap { uint32_t w[16]; };
inline ChipMap make_chip_map() {
    ChipMap m;
    const char* pn0 = "11011001110000110101001000101110";
    for (int s = 0; s < 16; s++) {
        int c[32];
        for (int k = 0; k < 32; k++) {
            c[k] = pn0[(k - 4 * (s & 7) + 64) % 32] - '0';
            if ((s & 8) && (k & 1)) c[k] ^= 1;
        }
        uint32_t v = 0;
        for (int k = 1; k < 32; k++) v |= (uint32_t)(c[k] ^ c[k - 1] ^ (k & 1)) << (31 - k);
        m.w[s] = v & 0x7FFFFFFEu;
    }
    return m;
}

SNRX_HD int popc32(uint32_t x) {
#ifdef __CUDA_ARCH__
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

SNRX_HD int zb_dist(uint32_t reg, uint32_t word) { return popc32((reg & 0x7FFFFFFEu) ^ word); }

SNRX_HD uint32_t zb_fcs16_byte(uint32_t crc, uint32_t c) {        // Dot15d4FCS.compute_fcs, dot15d4.py:151-164, one byte
    uint32_t q = (crc ^ c) & 15u;
    crc = ((crc >> 4) ^ (q * 4225u)) & 0xFFFFu;
    q = (crc ^ (c >> 4)) & 15u;
    return ((crc >> 4) ^ (q * 4225u)) & 0xFFFFu;
}
SNRX_HD uint16_t zb_fcs16(const uint8_t* d, int n) {
    uint32_t crc = 0;
    for (int i = 0; i < n; i++) crc = zb_fcs16_byte(crc, d[i]);
    return (uint16_t)crc;
}

// ---- DC tracker (a11: single_pole_iir_filter_ff(0.00016) and the subtraction, top_block.py:52,70,84-89) -----------------
// y[n] = a f[n] + (1-a) y[n-1] in double, z[n] = f[n] - (float) y[n], evaluated per block of SNRX_IIR_BLOCK samples on the
// absolute grid: a block starts from the carried state folded from the block-local end values of the
// SNRX_IIR_MEMORY_BLOCKS preceding blocks (oracle/zb_oracle.c zb_oracle_dc_remove states the same and bounds it against the
// serial recurrence).
SNRX_HD double zb_iir_step(double y, float f) { return d_add(d_mul(SNRX_IIR_ALPHA, (double)f), d_mul(SNRX_IIR_BETA, y)); }
SNRX_HD float zb_dc_out(float f, double y) {
    const float z = f_sub(f, (float)y);
    return (fabsf(z) <= kZbClamp) ? z : 0.0f;
}
// state carried into block b: fold of the (at most) SNRX_IIR_MEMORY_BLOCKS preceding block-local end values, oldest
// first; decay = (1-alpha)^SNRX_IIR_BLOCK
SNRX_HD double zb_iir_fold(const double* ends, int b, double decay) {
    double carry = 0.0;
    for (int j = (b > SNRX_IIR_MEMORY_BLOCKS ? b - SNRX_IIR_MEMORY_BLOCKS : 0); j < b; j++) carry = d_add(ends[j], d_mul(decay, carry));
    return carry;
}
inline double zb_iir_block_decay() {
    volatile double p = 1.0; const double b = SNRX_IIR_BETA;
    for (int i = 0; i < SNRX_IIR_BLOCK; i++) p = p * b;
    return p;
}

// ---- clock recovery (a12: clock_recovery_mm_ff(2, 0.000225, 0.5, 0.03, 0.0002), top_block.py:69) ---------------------------
struct ZbMm { float mu, omega, last; int32_t ii; };     // ii: position in the stream (n_out < 2^31)

// row of the MMSE interpolator table for the fractional delay mu: rint(mu * 128).  mu * 128 lies in [0, 128],
// so adding 1.5 * 2^23 rounds it to the nearest integer (ties to even, exactly rintf) in the low mantissa bits:
// one FADD instead of a conversion on the chain's critical path.
SNRX_HD int zb_mm_row(float mu) {
    const float t = f_add(f_mul(mu, (float)SNRX_MMSE_NSTEPS), 12582912.0f);
#ifdef __CUDA_ARCH__
    return __float_as_int(t) & 0x1FF;           // 0..128: mu stays in [0, 1) because every z is finite (kZbClamp)
#else
    uint32_t u; memcpy(&u, &t, 4); return (int)(u & 0x1FFu);
#endif
}

// one Mueller-Mueller step on the 8 samples in[0..8) = z[ii .. ii+8) with the interpolator row t = taps[zb_mm_row(mu)];
// returns the soft chip
SNRX_HD float zb_mm_step(ZbMm& st, const float (&in)[8], const float (&t)[8]) {
    const float omega_mid = 2.0f, gain_omega = 0.000225f, gain_mu = 0.03f;
    const float omega_lim = 2.0f * 0.0002f;
    const float p0 = f_mul(t[0], in[0]), p1 = f_mul(t[1], in[1]), p2 = f_mul(t[2], in[2]), p3 = f_mul(t[3], in[3]);
    const float p4 = f_mul(t[4], in[4]), p5 = f_mul(t[5], in[5]), p6 = f_mul(t[6], in[6]), p7 = f_mul(t[7], in[7]);
    const float s01 = f_add(p0, p1), s23 = f_add(p2, p3), s45 = f_add(p4, p5), s67 = f_add(p6, p7);
    const float out = f_add(f_add(s01, s23), f_add(s45, s67));
    const float sl = (st.last < 0.0f) ? -1.0f : 1.0f;
    const float so = (out < 0.0f) ? -1.0f : 1.0f;
    const float mm = f_sub(f_mul(sl, out), f_mul(so, st.last));
    st.last = out;
    const float om = f_add(st.omega, f_mul(gain_omega, mm));
    const float dv = f_sub(om, omega_mid);
    const float hi = fabsf(f_add(dv, omega_lim)), lo = fabsf(f_sub(dv, omega_lim));
    st.omega = f_add(omega_mid, f_mul(0.5f, f_sub(hi, lo)));
    const float g = f_mul(gain_mu, mm);
    const float m2 = f_add(f_add(st.mu, st.omega), g);
    const float fl = floorf(m2);
    // the advance is 1, 2 or 3 samples for every finite input (m2 lies in (1.6, 3.4)); the clamp only guards the loop
    const int adv = (int)fl;
    st.ii += adv < 1 ? 1 : adv > 3 ? 3 : adv;
    st.mu = f_sub(m2, fl);
    return out;
}

// ---- packet sink (a13-a15), one 32-chip window at a time ------------------------------------------------------------------
// packet_sink_scapy_impl.cc:158-374 pushes one chip at a time.  Here the clock recovery first produces 32 chips, then
// zb_sink_window replays the state machine over them: while the sink is locked (d_preamble_cnt > 0, or past the SFD) it
// only looks at its register every 32 chips, so a window holds exactly one such symbol boundary, always at the same offset
// jb; while it is unlocked it compares every chip position against symbol 0 (:190-201), which is one funnel shift + popcount
// per position with no dependence between positions.  A register cleared by enter_search() (:55-65) is modelled by zeroing
// the chips it no longer holds.  Every lane of a warp does its symbol boundary at the same point of the program, which a
// chip-by-chip state machine per lane cannot (each lane's boundary falls on a different chip).
struct ZbSinkW {
    int state;                 // 0 search (unlocked, or locked on the preamble / first SFD half), 1 have sync (PHR), 2 have header (PSDU)
    int locked;                // state 0: d_preamble_cnt > 0
    int jb;                    // offset of the next symbol boundary inside the coming window (valid while locked or state > 0)
    int byte, nibble_idx;      // d_packet_byte, d_packet_byte_index
    int frame_len, got;        // d_packetlen, d_payload_cnt
    unsigned lqi_sum, lqi_n;
    int32_t sync_pos;          // input position of the chip that completed the SFD
    uint32_t prev;             // the previous window's chips (first chip in bit 31), cleared chips read 0
    uint32_t crc, crc1, crc2;  // FCS-16 over the PSDU bytes so far / without the last / without the last two
    uint32_t last2;            // the last two PSDU bytes, little endian
};
SNRX_HD void zb_sinkw_init(ZbSinkW& s) {
    s.state = 0; s.locked = 0; s.jb = 0; s.byte = 0; s.nibble_idx = 0; s.frame_len = 0; s.got = 0; s.lqi_sum = 0; s.lqi_n = 0;
    s.sync_pos = 0; s.prev = 0; s.crc = s.crc1 = s.crc2 = 0; s.last2 = 0;
}

// Where a chain's frames go: the chain's slots in the batch's slot array, and what identifies the chain
struct ZbEmit {
    snrx_frame_t* slots; uint32_t cap, nf;
    int32_t lo, hi;            // body of the chain: only frames whose sync position lies in [lo, hi) are reported
    int64_t index_base;        // sample_index = sync_pos + index_base
    uint32_t capture_id, window; uint16_t channel;
    int64_t good_end;          // end (whole-capture index) of the last CRC-ok frame reported
};
SNRX_HD int64_t zb_frame_end(int64_t sample_index, int len) { return sample_index + (int64_t)(2 + 2 * len) * 64; }

// the register the reference sink holds right after the chip at offset j of the window C (previous window P)
SNRX_HD uint32_t zb_reg_at(uint32_t C, uint32_t P, int j) { return funnel_r(C, P, 31 - j); }

// One window.  C: its chips, first chip in bit 31 (absent chips 0); nvalid: chips it holds (< 32 only when the stream
// ended); jstop: chips whose position lies before the end of the chain's body; pos_evt: input position of the chip at
// offset s.jb; j_start: offset of the first chip the sink sees (> 0 only in the window in which the sink starts: the chips
// before it must be 0 in C).  Returns true when the chain ends inside this window, *consumed = the chips of it that
// count as processed.
SNRX_HD bool zb_sink_window(ZbSinkW& s, uint32_t C, int nvalid, int jstop, int32_t pos_evt, const uint32_t* map, int thr,
                            ZbEmit& em, int* consumed, int j_start = 0) {
    // a sink in the search state stops at the first chip past the body (zb_run_chain's loop condition), any sink stops
    // where the stream ends; 32 = not inside this window
    const int stop_x = nvalid;
    const int stop_0 = jstop < nvalid ? jstop : nvalid;
    uint32_t P = s.prev;
    int j0 = j_start;                                // the unlocked search resumes here
    int pushed = j_start;                            // chips dealt with so far
    if (s.locked || s.state != 0) {
        const int e = s.jb;
        const int limit = s.state == 0 ? stop_0 : stop_x;
        if (e >= limit) { *consumed = limit; return true; }
        const uint32_t reg = zb_reg_at(C, P, e);
        // decode_chips :95-125: distance to every symbol, first minimum wins (the symbol number sits below the distance)
        uint32_t best = 0xFFFFFFFFu;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const uint32_t v = ((uint32_t)zb_dist(reg, map[i]) << 4) | (uint32_t)i;
            best = v < best ? v : best;
        }
        const int best_d = (int)(best >> 4), best_i = (int)(best & 15u);
        bool reset = false;
        if (s.state == 0) {                                            // STATE_SYNC_SEARCH, locked :204-241
            if (s.byte == 0) {
                if (zb_dist(reg, map[0]) <= thr) { /* one more preamble symbol */ }
                else if (zb_dist(reg, map[7]) <= thr) s.byte = 7 << 4;
                else reset = true;
            } else if (zb_dist(reg, map[10]) <= thr) {                 // enter_have_sync :67-79
                s.state = 1; s.got = 0; s.byte = 0; s.nibble_idx = 0; s.lqi_sum = 0; s.lqi_n = 0;
                s.sync_pos = pos_evt; s.crc = s.crc1 = s.crc2 = 0; s.last2 = 0;
            } else reset = true;
        } else if (best_d >= thr) {
            reset = true;                                              // a symbol nobody recognises aborts the frame
        } else {
            if (s.lqi_n < 8) { s.lqi_sum += 32 - best_d; s.lqi_n++; }
            if (s.nibble_idx == 0) s.byte = best_i; else s.byte |= best_i << 4;
            s.nibble_idx++;
            if ((s.nibble_idx & 1) == 0) {
                if (s.state == 1) {                                    // STATE_HAVE_SYNC :247-291
                    if (s.byte <= 127) { s.state = 2; s.frame_len = s.byte; s.got = 0; s.byte = 0; s.nibble_idx = 0; }   // :81-92
                    else reset = true;
                } else {                                               // STATE_HAVE_HEADER :293-359
                    const uint32_t b = (uint32_t)s.byte;
                    if (em.nf < em.cap) em.slots[em.nf].bytes[s.got] = (uint8_t)b;
                    s.got++;
                    s.nibble_idx = 0;
                    s.crc2 = s.crc1; s.crc1 = s.crc; s.crc = zb_fcs16_byte(s.crc, b);
                    s.last2 = (s.last2 >> 8) | (b << 8);
                    if (s.got >= s.frame_len) {                        // publish :333-355
                        if (s.sync_pos >= em.lo && s.sync_pos < em.hi) {
                            if (em.nf < em.cap) {
                                snrx_frame_t& f = em.slots[em.nf];
                                f.sample_index = (int64_t)s.sync_pos + em.index_base;
                                f.capture_id = em.capture_id;
                                f.window = em.window;
                                f.channel = em.channel;
                                f.proto = SNRX_PROTO_ZIGBEE;
                                const unsigned scaled = (s.lqi_sum / 8) << 3;           // :334-335
                                f.lqi = (uint8_t)(scaled >= 256 ? 255 : scaled);
                                f.phase = 0;
                                f.len = (uint16_t)s.got;
                                f.access_addr = 0;
                                f.crc_ok = (uint8_t)(s.got >= 2 && s.crc2 == s.last2);
                                for (int i = s.got; i < 132; i++) f.bytes[i] = 0;
                                if (f.crc_ok) { const int64_t end = zb_frame_end(f.sample_index, s.got); if (end > em.good_end) em.good_end = end; }
                            }
                            em.nf++;
                        }
                        reset = true;
                    }
                }
            }
        }
        pushed = e + 1;
        if (reset) {                                                   // enter_search :55-65: the register is cleared
            s.state = 0; s.locked = 0; s.byte = 0;
            C &= (e < 31) ? ((1u << (31 - e)) - 1u) : 0u;
            P = 0;
            j0 = e + 1;
        }
    }
    if (s.state == 0 && !s.locked) {
        // unlocked search :190-201 over the offsets [j0, stop_0): first position whose register is within thr of symbol 0
        uint32_t hits = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) hits |= (uint32_t)(zb_dist(zb_reg_at(C, P, j), map[0]) < thr) << j;
        if (j0 > 0) hits &= j0 < 32 ? ~((1u << j0) - 1u) : 0u;
        if (stop_0 < 32) hits &= (1u << stop_0) - 1u;
        if (hits) {
#ifdef __CUDA_ARCH__
            s.jb = __ffs((int)hits) - 1;
#else
            s.jb = __builtin_ctz(hits);
#endif
            s.locked = 1;
        }
    }
    s.prev = C;
    const int limit = s.state == 0 ? stop_0 : stop_x;
    if (limit < 32) { *consumed = limit > pushed ? limit : pushed; return true; }
    *consumed = 32;
    return false;
}

struct ZbChainParams {
    int32_t n_out;            // channel-rate samples per capture in the buffer
    int32_t origin;           // local index where segment `first_segment` starts (pre halo length)
    int32_t body;             // body length (local samples from origin)
    int32_t segment, prehalo;
    int32_t n_segments;
    int32_t n_blocks;         // DC-tracker blocks per stream
    uint32_t first_segment, first_capture;
    uint32_t n_captures, n_channels;
    int32_t threshold;
    uint32_t slots_per_chain;
    size_t f_stride;          // floats between (capture, channel) streams
};

// One chain = (capture, channel, segment): clock recovery fresh at `begin` = lo - prehalo, the sink from the first chip at
// or after lo - kZbSinkLead.  The chain ends at the post halo, or as soon as it has passed its body with the sink in the
// search state: a sync found from there on completes at a position >= hi and belongs to the next segment, so nothing this
// chain could still report is lost (oracle/zb_oracle.c zb_oracle_chain_hold stops at the same chip).
struct ZbChain {
    ZbMm mm; ZbSinkW sink; ZbEmit em;
    int32_t begin, hi, end, sink_from;
    int32_t nchips;           // clock-recovery steps so far (= chips)
    int sink_on;
};
SNRX_HD void zb_chain_init(ZbChain& c, const ZbChainParams& p, int seg, int channel_number, uint32_t capture_id, snrx_frame_t* slots) {
    // all positions are < n_out + segment + post halo < 2^31 (zb_create bounds max_out)
    const int32_t lo = p.origin + seg * p.segment;
    int32_t hi = lo + p.segment;
    const int32_t body_end = p.origin + p.body;
    if (hi > body_end) hi = body_end;
    int32_t begin = lo - p.prehalo; if (begin < 0) begin = 0;
    int32_t end = hi + kZbPostHalo; if (end > p.n_out) end = p.n_out;
    c.begin = begin; c.hi = hi; c.end = end; c.sink_from = lo - kZbSinkLead;
    c.mm.mu = 0.5f; c.mm.omega = 2.0f; c.mm.last = 0.0f; c.mm.ii = begin;
    zb_sinkw_init(c.sink);
    c.em.slots = slots; c.em.cap = p.slots_per_chain; c.em.nf = 0; c.em.lo = lo; c.em.hi = hi;
    c.em.index_base = (int64_t)p.first_segment * p.segment - (int64_t)p.origin;
    c.em.capture_id = capture_id; c.em.window = p.first_segment + (uint32_t)seg; c.em.channel = (uint16_t)channel_number;
    c.em.good_end = 0;
    c.nchips = 0; c.sink_on = 0;
}

// what 32 clock-recovery steps leave behind for the sink
struct ZbWin {
    uint32_t C;               // hard chips, first chip in bit 31 (absent chips 0)
    int nvalid;               // chips produced (< 32 only when the stream ended)
    int below;                // chips whose position lies before the end of the body
    int before;               // chips whose position lies before the point where the sink starts
    int32_t pos_evt;          // position of the chip at the sink's boundary offset
};

// where a chain reads its samples from: straight from the DC-removed stream (host stepping harness) ...
struct ZbDirectSrc {
    const float* z;
    const float* taps;     // [129][8]
    template <int K, bool FAST> SNRX_HD void tick() {}
    SNRX_HD void get8(int32_t ii, float (&in)[8]) const {
#pragma unroll
        for (int k = 0; k < 8; k++) in[k] = z[ii + k];
    }
    SNRX_HD void row(float mu, float (&t)[8]) const {
        const int r = zb_mm_row(mu);
#pragma unroll
        for (int k = 0; k < 8; k++) t[k] = taps[r * SNRX_MMSE_NTAPS + k];
    }
};

template <int K, bool FAST, bool DEBUG, class Src>
SNRX_HD void zb_chain_step(ZbChain& c, Src& src, ZbWin& w, int j, int jb, float* chips_dbg, int64_t chips_cap) {
    if (FAST || c.mm.ii + 8 <= c.end) {
        const int32_t pos = c.mm.ii;
        float in[8], t[8];
        src.template tick<K, FAST>();
        src.row(c.mm.mu, t);
        src.get8(pos, in);
        const float soft = zb_mm_step(c.mm, in, t);
        if (DEBUG && chips_dbg && c.nchips + j < chips_cap) chips_dbg[c.nchips + j] = soft;
        w.C = (w.C << 1) | (soft > 0.0f ? 1u : 0u);
        w.below += pos < c.hi ? 1 : 0;
        w.before += pos < c.sink_from ? 1 : 0;
        w.pos_evt = (j == jb) ? pos : w.pos_evt;
        w.nvalid++;
    }
}

// 32 clock-recovery steps.  FAST: the caller guarantees that none of them can reach the end of the stream (every step
// advances by at most 3 samples), so the per-step end test is dropped.
template <bool FAST, bool DEBUG, class Src>
SNRX_HD void zb_chain_steps(ZbChain& c, Src& src, ZbWin& w, float* chips_dbg, int64_t chips_cap) {
    w.C = 0; w.nvalid = 0; w.below = 0; w.before = 0; w.pos_evt = 0;
    const int jb = c.sink.jb;
    for (int j8 = 0; j8 < 32; j8 += 8) {
        zb_chain_step<0, FAST, DEBUG>(c, src, w, j8 + 0, jb, chips_dbg, chips_cap);
        zb_chain_step<1, FAST, DEBUG>(c, src, w, j8 + 1, jb, chips_dbg, chips_cap);
        zb_chain_step<2, FAST, DEBUG>(c, src, w, j8 + 2, jb, chips_dbg, chips_cap);
        zb_chain_step<3, FAST, DEBUG>(c, src, w, j8 + 3, jb, chips_dbg, chips_cap);
        zb_chain_step<4, FAST, DEBUG>(c, src, w, j8 + 4, jb, chips_dbg, chips_cap);
        zb_chain_step<5, FAST, DEBUG>(c, src, w, j8 + 5, jb, chips_dbg, chips_cap);
        zb_chain_step<6, FAST, DEBUG>(c, src, w, j8 + 6, jb, chips_dbg, chips_cap);
        zb_chain_step<7, FAST, DEBUG>(c, src, w, j8 + 7, jb, chips_dbg, chips_cap);
    }
    if (w.nvalid < 32) w.C = w.nvalid ? w.C << (32 - w.nvalid) : 0u;
}

// the sink's part of a window; returns true when the chain has ended
SNRX_HD bool zb_chain_sink(ZbChain& c, const ZbWin& w, const uint32_t* map, int thr) {
    uint32_t C = w.C;
    int j_start = 0;
    if (!c.sink_on) {
        if (w.before >= w.nvalid) {                   // still warming up (or the stream ended before the sink started)
            c.nchips += w.nvalid;
            return w.nvalid < 32;
        }
        c.sink_on = 1;                                // the sink starts inside this window: it never saw the chips before
        j_start = w.before;
        if (j_start > 0) C &= (1u << (32 - j_start)) - 1u;
    }
    int consumed = 0;
    const bool done = zb_sink_window(c.sink, C, w.nvalid, w.below, w.pos_evt, map, thr, c.em, &consumed, j_start);
    c.nchips += consumed;
    return done;
}

// a whole chain on one thread (host stepping harness; the device kernel k_zb_rx drives the same functions)
template <bool DEBUG, class Src>
SNRX_HD uint32_t zb_run_chain(Src& src, const ZbChainParams& p, int seg, const uint32_t* map,
                              int channel_number, uint32_t capture_id, snrx_frame_t* slots, float* chips_dbg,
                              int64_t chips_cap, int64_t* nchips_out, int64_t* good_end_out) {
    ZbChain c;
    zb_chain_init(c, p, seg, channel_number, capture_id, slots);
    bool done = false;
    while (!done) {
        ZbWin w;
        if (c.mm.ii + 8 + 3 * 32 <= c.end) zb_chain_steps<true, DEBUG>(c, src, w, chips_dbg, chips_cap);
        else zb_chain_steps<false, DEBUG>(c, src, w, chips_dbg, chips_cap);
        done = zb_chain_sink(c, w, map, p.threshold);
    }
    if (nchips_out) *nchips_out = c.nchips;
    if (good_end_out) *good_end_out = c.em.good_end;
    return c.em.nf;
}

// Filter of one chain's records given the ends of the CRC-ok frames of the `lookback` preceding chains of its stream.
// Records are compacted in place; returns the number kept.
SNRX_HD uint32_t zb_filter_chain(snrx_frame_t* slots, uint32_t n, int64_t good_end) {
    uint32_t w = 0;
    for (uint32_t k = 0; k < n; k++) {
        const snrx_frame_t& f = slots[k];
        bool keep = true;
        if (f.crc_ok) { const int64_t e = zb_frame_end(f.sample_index, f.len); if (e > good_end) good_end = e; }
        else if (f.sample_index < good_end) keep = false;
        if (keep) { if (w != k) slots[w] = slots[k]; w++; }
    }
    return w;
}
SNRX_HD int zb_filter_lookback(int segment) { return (16384 + segment - 1) / segment + 1; }
// a body of `segment` samples holds at most this many syncs kZbMinSyncChips samples apart (22 at 4096); k_zb_rx still flags a
// chain that finds more (SNRX_EOVERFLOW)
SNRX_HD uint32_t zb_slots_per_chain(uint32_t segment) { return (segment - 1) / kZbMinSyncChips + 1; }

#if defined(__CUDACC__)
// ------------------------------------------------------------------------------------ kernels

struct ZbQuadArgs {
    const float2* x; uint64_t stride; int64_t n; uint32_t n_captures;
    float* f; size_t f_stride;            // [cap][1][f_stride]
    const float2* atan_pairs;             // [256] AtanTabPairs, global (L1 resident)
    uint32_t blocks_per_cap;              // the grid is n_captures * blocks_per_cap blocks
};

// Narrow-band discriminator, element-wise: a thread takes four consecutive samples (two 16-byte streaming loads + the
// sample before them, one 16-byte store); the table is read as {value, step} pairs through L1 like in k_pfb_zb_warp.
// Round 2's first version (one sample per thread, two 8-byte loads, the 257-entry table in shared memory at random
// indices) took 9.8 ms per 2.56 G samples with the GPU to itself, this one 6.1 ms (5.0 TB/s of reads + writes).
__global__ void __launch_bounds__(256) k_zb_quad(ZbQuadArgs a) {
    const AtanTabPairs tab{a.atan_pairs};
    // a block stays inside one capture: one 32-bit division per block, none per item (a 64-bit item index split per item cost
    // as much as the four discriminators it fed)
    const uint32_t cap = blockIdx.x / a.blocks_per_cap;
    const float2* xc = a.x + (size_t)cap * a.stride;
    float* fc = a.f + (size_t)cap * a.f_stride;
    const int64_t n4 = (a.n + 3) / 4;
    for (int64_t q = (int64_t)(blockIdx.x % a.blocks_per_cap) * blockDim.x + threadIdx.x; q < n4; q += (int64_t)a.blocks_per_cap * blockDim.x) {
        const int64_t n0 = q * 4;
        float2 prev = make_float2(0.f, 0.f);
        if (n0 > 0) prev = __ldg(xc + n0 - 1);
        if (n0 + 4 <= a.n && ((reinterpret_cast<uintptr_t>(xc + n0) | reinterpret_cast<uintptr_t>(fc + n0)) & 15) == 0) {
            const float4 u = __ldcs(reinterpret_cast<const float4*>(xc + n0));
            const float4 v = __ldcs(reinterpret_cast<const float4*>(xc + n0) + 1);
            float4 o;
            o.x = quad_demod_g(u.x, u.y, prev.x, prev.y, tab);
            o.y = quad_demod_g(u.z, u.w, u.x, u.y, tab);
            o.z = quad_demod_g(v.x, v.y, u.z, u.w, tab);
            o.w = quad_demod_g(v.z, v.w, v.x, v.y, tab);
            *reinterpret_cast<float4*>(fc + n0) = o;
        } else {
            for (int64_t n = n0; n < n0 + 4 && n < a.n; n++) {
                const float2 cur = __ldg(xc + n);
                fc[n] = quad_demod_g(cur.x, cur.y, prev.x, prev.y, tab);
                prev = cur;
            }
        }
    }
}

struct ZbIirArgs {
    const float* f; size_t stride;                // per (capture, channel) stream stride
    int32_t n; int32_t n_blocks; uint32_t n_streams;
    double* block_end;    // [stream][n_blocks]  block-local recurrence value at the block end
    double* carry_in;     // [stream][n_blocks]  carried state entering each block
    double decay;         // (1-alpha)^SNRX_IIR_BLOCK
    uint8_t* busy;        // [stream][n_blocks]  a frame seems to be on the air at the block's end (zb_chain_key), or null
};

// Scheduling hint only -- it never touches a result.  The discriminator output of an O-QPSK burst moves by +-pi/4 per sample
// (sum of f^2 over 64 samples: 37..51 at 25..9 dB Es/N0, p99 66), noise on an empty channel gives 172 (p1 125), a GFSK burst
// in a shared bin of a mixed capture about 10 (measured on the oracle's channel streams).
constexpr float kZbBusyLo = 24.0f, kZbBusyHi = 92.0f;
constexpr int kZbBusyWindow = 64;
constexpr int kZbKeys = 10;           // zb_chain_key() values 0 .. kZbKeys - 1

// A (stream, block) unit is one thread's SNRX_IIR_BLOCK-sample serial recurrence from 0.  Its samples are contiguous and
// 128-byte aligned, so the thread streams them as float4 with the next 32 samples (8 loads) already in
// flight while the current 32 go through the dependent double-precision chain.
constexpr int kIirPf = 8;             // float4 loads in flight per thread

__global__ void __launch_bounds__(64) k_zb_iir_sum(ZbIirArgs a) {
    const uint32_t total = a.n_streams * (uint32_t)a.n_blocks;
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    // consecutive threads take different streams (DRAM page spread, as in k_zb_rx)
    const uint32_t b = idx / a.n_streams, s = idx % a.n_streams;
    const float* f = a.f + (size_t)s * a.stride + (size_t)b * SNRX_IIR_BLOCK;
    const int len = min(SNRX_IIR_BLOCK, a.n - (int)b * SNRX_IIR_BLOCK);
    const int n4 = len >> 2;
    const float4* f4 = reinterpret_cast<const float4*>(f);
    double l = 0.0;
    float4 cur[kIirPf], nxt[kIirPf];
#pragma unroll
    for (int k = 0; k < kIirPf; k++) nxt[k] = (k < n4) ? __ldg(f4 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i4 = 0; i4 < n4; i4 += kIirPf) {
#pragma unroll
        for (int k = 0; k < kIirPf; k++) cur[k] = nxt[k];
#pragma unroll
        for (int k = 0; k < kIirPf; k++) nxt[k] = (i4 + kIirPf + k < n4) ? __ldg(f4 + i4 + kIirPf + k) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < kIirPf; k++) {
            if (i4 + k < n4) {
                l = zb_iir_step(l, cur[k].x);
                l = zb_iir_step(l, cur[k].y);
                l = zb_iir_step(l, cur[k].z);
                l = zb_iir_step(l, cur[k].w);
            }
        }
    }
    for (int i = n4 << 2; i < len; i++) l = zb_iir_step(l, f[i]);
    a.block_end[(size_t)s * a.n_blocks + b] = l;
    if (a.busy) {
        float e = 0.0f;
        if (len == SNRX_IIR_BLOCK) {
#pragma unroll
            for (int k = 0; k < kZbBusyWindow / 4; k++) {
                const float4 v = __ldg(f4 + (SNRX_IIR_BLOCK - kZbBusyWindow) / 4 + k);      // just read: L1
                e += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
            }
        }
        a.busy[(size_t)s * a.n_blocks + b] = (uint8_t)(e > kZbBusyLo && e < kZbBusyHi);
    }
}

// carried state entering block b: folded from the SNRX_IIR_MEMORY_BLOCKS preceding blocks (all full
// length), oldest first -- one thread per (stream, block), no serial pass over the stream
__global__ void __launch_bounds__(128) k_zb_iir_carry(ZbIirArgs a) {
    const uint32_t total = a.n_streams * (uint32_t)a.n_blocks;
    for (uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const uint32_t s = idx / (uint32_t)a.n_blocks;
        const int b = (int)(idx % (uint32_t)a.n_blocks);
        a.carry_in[idx] = zb_iir_fold(a.block_end + (size_t)s * a.n_blocks, b, a.decay);
    }
}

// ... or, on the device, from the raw discriminator stream f in HBM:
//   * every step the lane loads the raw pair it will need kZbQueue steps later (one 8-byte load into a register queue:
//     HBM / L2 latency is covered without shared-memory staging), runs its own DC tracker over the pair that has arrived
//     (zb_iir_step from the carried state of each SNRX_IIR_BLOCK block) and stores z = f - y into
//   * the z ring in shared memory: zr[r * 32 + lane], row r = sample mod 128, rows 0..7 mirrored at 128..135 so that the
//     8 interpolator taps never wrap; every access of a warp is bank-conflict free whatever the lanes' positions.
// The DC-removed stream never exists in HBM (only with SNRX_F_KEEP_STREAMS, for the parity tests).  The tracker is
// paced by the STEP COUNT -- two samples per clock-recovery step, the nominal advance -- not by each lane's position, so
// the loop body has no refill branches.  A lane's position wanders around 2 samples per step by about one sample per
// window (measured on the oracle: <= 1 per 32 steps, < 100 over 2 M steps); k_zb_rx re-centres the lead between
// windows, so correctness never depends on the pacing.
constexpr int kZbQueue = 8;           // raw pairs in flight per lane
constexpr int kZbZRows = 128;         // z samples per lane (power of two), + 8 mirrored rows
constexpr int kZbLead = 64;           // samples the tracker starts ahead of the clock recovery: two windows' worth, so that the
                                      // tracker's position stays a multiple of 64 at every window start and a block boundary
                                      // of the tracker (2048) can only fall on a window start
constexpr int kZbLeadMin = 44;        // a window may start with this much lead: 32 steps of 3 samples eat at most 32 of it, 8 are read
constexpr int kZbLeadMax = 84;        // beyond it the tracker pauses for a window (the ring holds 128 >= 84 + 32 + 8).  A paused
                                      // window converts nothing, so its reads must stay behind conv on their own: |mm| <=
                                      // max|out| <= 1.60 * 2 pi (largest sum of |taps| of a row, |z| <= 2 pi), so 31 steps advance
                                      // at most 1 + 31 * (2.0004 + 0.03 * 10.06) = 72.4 samples and the last read still has
                                      // 85 - 72.4 = 12.6 samples of lead against the 8 it reads: 4.6 to spare.  This is a
                                      // derived bound: no test input comes near it (windows under 3e-3 chip-rate drift pause
                                      // with a lead of 22 or more at every read)
constexpr int kZbTapsPlane = (SNRX_MMSE_NSTEPS + 1) * 16;   // bytes of one plane of the interpolator table in shared memory
constexpr int kZbRxWarps = 4;         // warps per CTA (they only share the interpolator table)
#ifndef SNRX_ZB_RX_MINCTAS
#define SNRX_ZB_RX_MINCTAS 4
#endif
#ifndef SNRX_ZB_RX_REFILL
#define SNRX_ZB_RX_REFILL 1             // 1 = lanes take their next chain inside the window loop; 0 = chain loop around a window loop
#endif
constexpr int kZbRxCtasPerSm = 3;          // what shared memory allows (74 KB per CTA)
constexpr int kZbRxMinCtas = SNRX_ZB_RX_MINCTAS;   // register budget of the kernel: 65536 / (128 * this)
constexpr int kZbRxSmem = (SNRX_MMSE_NSTEPS + 1) * SNRX_MMSE_NTAPS * 4 + kZbRxWarps * (kZbZRows + 8) * 32 * 4;

template <bool DEBUG>
struct ZbRegSrc {
    const float2* nxt;     // next raw pair to load
    const double* carry;   // carried tracker state of this stream's blocks
    float2 q[kZbQueue];    // raw pairs in flight / waiting for the tracker
    double y;              // tracker state
    uint32_t zr;           // shared-memory byte address of this lane's column of the z ring
    uint32_t zw;           // byte offset of the row the tracker writes next (row * 128)
    uint32_t taps_adj;     // shared-memory byte address of the interpolator table - 0xB4000000 (see row())
    int32_t begin;         // stream index of ring position 0 (a multiple of SNRX_IIR_BLOCK)
    int32_t conv;          // samples the tracker has converted, relative to begin
    bool enabled;          // slow windows only: the tracker runs
    float* z_dbg; int32_t z_lo, z_hi;    // debug: this chain stores z[z_lo, z_hi) of its stream

    // a block of the tracker starts here: its state is the carried one
    __device__ __forceinline__ void boundary() {
        const int32_t g = begin + conv;
        if ((g & (SNRX_IIR_BLOCK - 1)) == 0) y = __ldg(carry + (g >> 11));
    }
    // BOUNDARY = false: the caller knows that no block boundary falls on this pair (fast windows call boundary() once)
    template <int K, bool BOUNDARY>
    __device__ __forceinline__ void convert() {
        static_assert(SNRX_IIR_BLOCK == 2048, "boundary() shifts by 11");
        const float f0 = q[K].x, f1 = q[K].y;
        q[K] = __ldg(nxt);                                   // the pair kZbQueue steps ahead
        nxt++;
        if (BOUNDARY) boundary();
        y = zb_iir_step(y, f0);
        const float z0 = zb_dc_out(f0, y);
        y = zb_iir_step(y, f1);
        const float z1 = zb_dc_out(f1, y);
        const uint32_t dst = zr + zw;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst), "f"(z0) : "memory");
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst + 128u), "f"(z1) : "memory");
        if (zw < 8u * 128u) {
            asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst + 128u * kZbZRows), "f"(z0) : "memory");
            asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst + 128u * (kZbZRows + 1)), "f"(z1) : "memory");
        }
        if (DEBUG && z_dbg) {
            const int32_t g = begin + conv;
            if (g >= z_lo && g < z_hi) z_dbg[g] = z0;
            if (g + 1 >= z_lo && g + 1 < z_hi) z_dbg[g + 1] = z1;
        }
        zw = (zw + 256u) & (128u * kZbZRows - 1u);
        conv += 2;
    }
    __device__ __forceinline__ void burst() {                // 16 samples
        convert<0, true>(); convert<1, true>(); convert<2, true>(); convert<3, true>();
        convert<4, true>(); convert<5, true>(); convert<6, true>(); convert<7, true>();
    }
    __device__ __forceinline__ void start(const float* f, const double* carry_, int32_t begin_) {
        begin = begin_; conv = 0; zw = 0; y = 0.0; enabled = true;
        carry = carry_;
        nxt = reinterpret_cast<const float2*>(f + begin_);
#pragma unroll
        for (int k = 0; k < kZbQueue; k++) q[k] = __ldg(nxt + k);
        nxt += kZbQueue;
        while (conv < kZbLead) burst();
    }
    template <int K, bool FAST>
    __device__ __forceinline__ void tick() {
        if (FAST) convert<K, false>();
        else if (enabled) convert<K, true>();
    }
    // a fast window converts the 64 samples from conv on; conv is a multiple of 64 there
    __device__ __forceinline__ bool aligned() const { return ((begin + conv) & 63) == 0; }
    __device__ __forceinline__ void get8(int32_t ii, float (&in)[8]) {
        const uint32_t p = zr + ((uint32_t)((ii - begin) & (kZbZRows - 1)) << 7);
#pragma unroll
        for (int k = 0; k < 8; k++) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(in[k]) : "r"(p + 128u * k));
    }
    // interpolator row rint(mu * 128): mu * 128 is exact, so one FFMA with the magic number 1.5 * 2^23 gives the bits
    // 0x4B400000 + row; (bits << 4) = 0xB4000000 + 16 * row (mod 2^32), hence the adjusted base: one shift for the address.
    // The table lies in shared memory as TWO planes of 16-byte rows (taps 0..3 | taps 4..7, kZbTapsPlane bytes apart): the
    // lanes of a warp sit at unrelated rows, and 16-byte rows spread a 16-byte load over 8 bank groups where the natural
    // 32-byte rows allowed 4 (300 M bank conflicts per 10-s capture in round 2's first ncu capture of this kernel).
    __device__ __forceinline__ void row(float mu, float (&t)[8]) const {
        const uint32_t a = taps_adj + (__float_as_uint(__fmaf_rn(mu, (float)SNRX_MMSE_NSTEPS, 12582912.0f)) << 4);
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(t[0]), "=f"(t[1]), "=f"(t[2]), "=f"(t[3]) : "r"(a));
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(t[4]), "=f"(t[5]), "=f"(t[6]), "=f"(t[7]) : "r"(a + (uint32_t)kZbTapsPlane));
    }
};

struct ZbRxArgs {
    const float* f;              // [stream][f_stride] raw discriminator streams
    const double* carry;         // [stream][n_blocks]
    const float* taps;           // [129][8]
    const int32_t* channel_numbers;
    snrx_frame_t* slots; uint32_t* counts; int64_t* good_end;
    uint32_t* queue;             // next chain to hand out (zeroed before the launch)
    const uint32_t* order;       // [n_chains] queue position -> chain in natural order (k_zb_order), or null = natural order
    uint32_t* overflow;          // set to 1 when a chain found more frames than it has slots
    float* z_dbg;                // [stream][f_stride] or null
    float* chips_dbg; int64_t chips_cap; int64_t* nchips_dbg;
    ChipMap map;                 // kernel parameter: the chip words are constant-bank operands
    ZbChainParams p;
};

// DC tracker, clock recovery, packet sink and FCS of the chains (capture, channel, segment).  A lane runs one chain at a
// time and takes the next one from a queue when it is done: chains differ in length by a factor of four (a chain that
// holds a frame follows it through the post halo), and the warp is busy as long as any of its lanes is.
template <bool DEBUG>
__global__ void __launch_bounds__(kZbRxWarps * 32, kZbRxMinCtas) k_zb_rx(const __grid_constant__ ZbRxArgs a) {
    extern __shared__ __align__(16) unsigned char zb_smem[];
    float* taps = reinterpret_cast<float*>(zb_smem);
    float* zring = taps + (SNRX_MMSE_NSTEPS + 1) * SNRX_MMSE_NTAPS;
    for (int i = threadIdx.x; i < (SNRX_MMSE_NSTEPS + 1) * SNRX_MMSE_NTAPS; i += blockDim.x)            // [row][8] -> two planes of [row][4]
        taps[((i & 4) ? kZbTapsPlane / 4 : 0) + (i >> 3) * 4 + (i & 3)] = a.taps[i];
    __syncthreads();
    const ZbChainParams& p = a.p;
    const uint32_t n_streams = p.n_captures * p.n_channels;
    const uint32_t total = n_streams * (uint32_t)p.n_segments;
    ZbRegSrc<DEBUG> src;
    src.zr = (uint32_t)__cvta_generic_to_shared(zring + (threadIdx.x >> 5) * ((kZbZRows + 8) * 32) + (threadIdx.x & 31));
    src.taps_adj = (uint32_t)__cvta_generic_to_shared(taps) - 0xB4000000u;
    asm volatile("" : "+r"(src.zr), "+r"(src.taps_adj));               // opaque: stay in registers
#if SNRX_ZB_RX_REFILL
    // ONE loop over windows for the whole life of the warp: a lane whose chain has ended takes the next chain from the queue at
    // the top of the next iteration while the other lanes of its warp carry on with theirs.  (Round 2's first version nested
    // the window loop inside the chain loop; the warp reconverges behind the inner loop, so every lane waited for the longest
    // of the warp's 32 chains -- a chain that holds a frame follows it through the post halo and runs up to 3.7x as long as an
    // empty one: ncu counted 13.5 active lanes per instruction, profiles/r02_zb_wb16_ncu_v2.json.)  Which lane runs which chain
    // has no influence on any result: a chain's state is private and its records go to the chain's own slots.
    ZbChain c;
    uint32_t chain = 0;
    float* chips_dbg = nullptr;
    bool have = false, more = true;
    for (;;) {
        if (!have && more) {
            // consecutive chains belong to different streams, so that a warp touches many DRAM pages at once
            const uint32_t pos = atomicAdd(a.queue, 1u);
            if (pos >= total) {
                more = false;
            } else {
                const uint32_t idx = a.order ? __ldg(a.order + pos) : pos;
                const uint32_t seg = idx / n_streams, sc = idx % n_streams;
                const uint32_t cap = sc / p.n_channels, ch = sc % p.n_channels;
                chain = sc * (uint32_t)p.n_segments + seg;                 // output order
                zb_chain_init(c, p, (int)seg, a.channel_numbers[ch], p.first_capture + cap, a.slots + (size_t)chain * p.slots_per_chain);
                src.z_dbg = (DEBUG && a.z_dbg) ? a.z_dbg + (size_t)sc * p.f_stride : nullptr;
                src.z_lo = seg == 0 ? 0 : c.em.lo; src.z_hi = (int)seg == p.n_segments - 1 ? p.n_out : c.hi;
                src.start(a.f + (size_t)sc * p.f_stride, a.carry + (size_t)sc * p.n_blocks, c.begin);
                chips_dbg = (DEBUG && a.chips_dbg) ? a.chips_dbg + (size_t)chain * a.chips_cap : nullptr;
                have = true;
            }
        }
        if (!__any_sync(0xffffffffu, have)) break;                         // the queue is empty and every lane's chain has ended
        if (have) {
            // re-centre the tracker's lead (rare: a lane drifts by about one sample per window)
            int lead = src.conv - (c.mm.ii - src.begin);
            while (lead < kZbLeadMin) { src.burst(); src.burst(); src.burst(); src.burst(); lead += 8 * kZbQueue; }
            src.enabled = lead <= kZbLeadMax;
            ZbWin w;
            if (src.enabled && src.aligned() && c.mm.ii + 8 + 3 * 32 <= c.end) {
                src.boundary();
                zb_chain_steps<true, DEBUG>(c, src, w, chips_dbg, a.chips_cap);
            } else {
                zb_chain_steps<false, DEBUG>(c, src, w, chips_dbg, a.chips_cap);
            }
            if (zb_chain_sink(c, w, a.map.w, p.threshold)) {
                a.good_end[chain] = c.em.good_end;
                a.counts[chain] = c.em.nf < p.slots_per_chain ? c.em.nf : p.slots_per_chain;
                if (c.em.nf > p.slots_per_chain) *a.overflow = 1u;
                if (DEBUG && a.nchips_dbg) a.nchips_dbg[chain] = c.nchips;
                have = false;
            }
        }
    }
#else
    for (;;) {
        // consecutive chains belong to different streams, so that a warp touches many DRAM pages at once
        const uint32_t pos = atomicAdd(a.queue, 1u);
        if (pos >= total) break;
        const uint32_t idx = a.order ? __ldg(a.order + pos) : pos;
        const uint32_t seg = idx / n_streams, sc = idx % n_streams;
        const uint32_t cap = sc / p.n_channels, ch = sc % p.n_channels;
        const uint32_t chain = sc * (uint32_t)p.n_segments + seg;      // output order
        ZbChain c;
        zb_chain_init(c, p, (int)seg, a.channel_numbers[ch], p.first_capture + cap, a.slots + (size_t)chain * p.slots_per_chain);
        src.z_dbg = (DEBUG && a.z_dbg) ? a.z_dbg + (size_t)sc * p.f_stride : nullptr;
        src.z_lo = seg == 0 ? 0 : c.em.lo; src.z_hi = (int)seg == p.n_segments - 1 ? p.n_out : c.hi;
        src.start(a.f + (size_t)sc * p.f_stride, a.carry + (size_t)sc * p.n_blocks, c.begin);
        float* chips_dbg = (DEBUG && a.chips_dbg) ? a.chips_dbg + (size_t)chain * a.chips_cap : nullptr;
        bool done = false;
        while (!done) {
            // re-centre the tracker's lead (rare: a lane drifts by about one sample per window)
            int lead = src.conv - (c.mm.ii - src.begin);
            while (lead < kZbLeadMin) { src.burst(); src.burst(); src.burst(); src.burst(); lead += 8 * kZbQueue; }
            src.enabled = lead <= kZbLeadMax;
            ZbWin w;
            if (src.enabled && src.aligned() && c.mm.ii + 8 + 3 * 32 <= c.end) {
                src.boundary();
                zb_chain_steps<true, DEBUG>(c, src, w, chips_dbg, a.chips_cap);
            } else {
                zb_chain_steps<false, DEBUG>(c, src, w, chips_dbg, a.chips_cap);
            }
            done = zb_chain_sink(c, w, a.map.w, p.threshold);
        }
        a.good_end[chain] = c.em.good_end;
        a.counts[chain] = c.em.nf < p.slots_per_chain ? c.em.nf : p.slots_per_chain;
        if (c.em.nf > p.slots_per_chain) *a.overflow = 1u;
        if (DEBUG && a.nchips_dbg) a.nchips_dbg[chain] = c.nchips;
    }
#endif
}

// ---- the order in which k_zb_rx hands out its chains ------------------------------------------------------------------------
// A chain that finds a frame in its body follows it through the post halo and runs up to 3.6 times as long as an empty one
// (2048 + 4096 + 16448 samples against 6144); a lane that takes such a chain late keeps its warp -- and its CTA's 74 KB of
// shared memory -- alive long after the queue has run dry.  ncu of round 2's k_zb_rx: 15.9 of 32 lanes active per instruction on
// a 4.9-s capture; a model of the queue (a lane takes the next chain when it is done, a warp lives as long as its longest
// lane) gives the same factor 2.0 for the natural order and 1.05 when the long chains go first.  So the chains are handed out
// longest (expected) first.  The key of a chain: 0 when nothing seems to be on the air at the end of its body -- or when the
// air has been busy without a break since two blocks before the body (a frame that is not this chain's to decode) --, else the
// number of consecutive busy block ends from the end of its body onwards (1 .. 9: how far the chain will have to run on).
// A wrong guess costs time, never a result: which lane runs which chain has no influence on any record (tested with one CTA
// running 733 chains).
SNRX_HD int zb_chain_key(const uint8_t* busy /* this stream's blocks */, int n_blocks, const ZbChainParams& p, int seg) {
    const int32_t lo = p.origin + seg * p.segment;
    int32_t hi = lo + p.segment;
    if (hi > p.origin + p.body) hi = p.origin + p.body;
    if (hi <= lo || (hi & (SNRX_IIR_BLOCK - 1)) || (lo & (SNRX_IIR_BLOCK - 1))) return 0;
    const int kb = hi / SNRX_IIR_BLOCK - 1;                  // the block that ends where the body ends
    if (kb < 0 || kb >= n_blocks || !busy[kb]) return 0;
    const int kl = lo / SNRX_IIR_BLOCK - 1;                  // the block that ends where the body starts
    if (kl >= 1) {
        bool spans = true;
        for (int j = kl - 1; j < kb; j++) spans = spans && busy[j] != 0;
        if (spans) return 0;
    }
    int key = 0;
    for (int j = kb; j < n_blocks && busy[j] && key < kZbKeys - 1; j++) key++;
    return key;
}

struct ZbOrderArgs {
    const uint8_t* busy; ZbChainParams p;
    uint32_t* hist;       // [kZbKeys] chains per key | [kZbKeys] fill cursors (zeroed before the count pass)
    uint32_t* order;      // [n_chains] position in the queue -> index in natural order (idx = seg * n_streams + stream)
};
template <bool FILL>
__global__ void __launch_bounds__(256) k_zb_order(ZbOrderArgs a) {
    const uint32_t n_streams = a.p.n_captures * a.p.n_channels;
    const uint32_t total = n_streams * (uint32_t)a.p.n_segments;
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    int key = -1;
    if (idx < total) key = zb_chain_key(a.busy + (size_t)(idx % n_streams) * a.p.n_blocks, a.p.n_blocks, a.p, (int)(idx / n_streams));
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t peers = __match_any_sync(0xffffffffu, key);          // one atomic per key and warp
    const uint32_t leader = (uint32_t)__ffs((int)peers) - 1u;
    const uint32_t rank = (uint32_t)__popc(peers & ((1u << lane) - 1u));
    if (!FILL) {
        if (key >= 0 && lane == leader) atomicAdd(a.hist + key, (uint32_t)__popc(peers));
        return;
    }
    uint32_t start = 0;
    if (key >= 0 && lane == leader) start = atomicAdd(a.hist + kZbKeys + key, (uint32_t)__popc(peers));
    start = __shfl_sync(peers, start, (int)leader);
    if (key < 0) return;
    uint32_t base = 0;                                                   // longest first
    for (int k = kZbKeys - 1; k > key; k--) base += a.hist[k];
    a.order[base + start + rank] = idx;
}

// one thread per chain: drop the CRC-failed records that lie inside a CRC-ok frame of this or a preceding chain
__global__ void __launch_bounds__(128) k_zb_span_filter(snrx_frame_t* __restrict__ slots, uint32_t slots_per_chain,
                                                        uint32_t* __restrict__ counts, const int64_t* __restrict__ good_end,
                                                        uint32_t n_chains, uint32_t n_segments, int lookback) {
    const uint32_t chain = blockIdx.x * blockDim.x + threadIdx.x;
    if (chain >= n_chains) return;
    const uint32_t n = counts[chain];
    if (n == 0) return;
    const uint32_t seg = chain % n_segments;
    int64_t ge = 0;
    for (int j = 1; j <= lookback && (uint32_t)j <= seg; j++) { const int64_t e = good_end[chain - j]; if (e > ge) ge = e; }
    const uint32_t w = zb_filter_chain(slots + (size_t)chain * slots_per_chain, n, ge);
    if (w != n) counts[chain] = w;
}

__global__ void __launch_bounds__(128) k_zb_gather(const snrx_frame_t* __restrict__ slots, uint32_t slots_per_chain,
                                                   const uint32_t* __restrict__ counts, const uint32_t* __restrict__ offsets,
                                                   uint32_t n_chains, snrx_frame_t* __restrict__ frames, uint32_t frame_cap,
                                                   uint32_t* __restrict__ totals, int after_ble) {
    // one warp per chain, each frame copied as 10 x 16 bytes
    const int lane = threadIdx.x & 31;
    const uint32_t warps_per_block = blockDim.x >> 5;
    const uint32_t base = after_ble ? totals[0] : 0u;
    for (uint32_t c = blockIdx.x * warps_per_block + (threadIdx.x >> 5); c < n_chains; c += gridDim.x * warps_per_block) {
        const uint32_t n = counts[c], off = base + offsets[c];
        for (uint32_t k = 0; k < n; k++) {
            if (off + k >= frame_cap) break;
            const uint4* src = reinterpret_cast<const uint4*>(slots + (size_t)c * slots_per_chain + k);
            uint4* dst = reinterpret_cast<uint4*>(frames + off + k);
            if (lane < 10) dst[lane] = src[lane];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) totals[2] = offsets[n_chains];
}

// ------------------------------------------------------------------------------------ host side
struct ZbState {
    bool ready = false;
    uint32_t n_ch = 0, max_caps = 0, max_out = 0;
    size_t stride = 0;                 // floats per (capture, channel) stream
    float *d_f = nullptr, *d_z = nullptr;
    double *d_block_end = nullptr, *d_carry = nullptr;
    double decay = 0.0;
    float *d_atan = nullptr, *d_mmse = nullptr;
    float2* d_atan_pairs = nullptr;   // AtanTabPairs
    int32_t* d_channels = nullptr;
    snrx_frame_t* d_slots = nullptr; size_t slots_bytes = 0;
    uint32_t *d_counts = nullptr, *d_offsets = nullptr, *d_scratch = nullptr, *d_queue = nullptr;
    uint32_t *d_order = nullptr, *d_hist = nullptr; uint8_t* d_busy = nullptr;      // k_zb_order
    bool natural_order = false;   // SNRX_ZB_ORDER=0: chains handed out in natural order (A/B runs)
    int64_t* d_good_end = nullptr;
    uint32_t max_chains = 0, slots_per_chain = 0;
    float* d_chips = nullptr; int64_t* d_nchips = nullptr; int64_t chips_cap = 0;
    float *d_wb_taps_rho = nullptr, *d_wb_taps_flat = nullptr, *d_wb_taps_pass = nullptr; float2* d_wb_cf = nullptr; int wb_nt = 16;
    bool wb_cta_kernel = false;   // wideband front end
    uint32_t rx_cta_cap = 0;      // SNRX_ZB_RX_CTAS: upper bound of k_zb_rx's grid (tests: few lanes, many chains per lane); 0 = none
    ChipMap map;
    uint32_t last_chains = 0;
};

inline void zb_free(ZbState& s) {
    void* bufs[] = {s.d_f, s.d_z, s.d_block_end, s.d_carry, s.d_atan, s.d_mmse, s.d_channels, s.d_slots,
                    s.d_counts, s.d_offsets, s.d_scratch, s.d_queue, s.d_good_end, s.d_chips, s.d_nchips, s.d_atan_pairs, s.d_order, s.d_hist, s.d_busy, s.d_wb_taps_rho, s.d_wb_taps_flat, s.d_wb_taps_pass, s.d_wb_cf};
    for (void* b : bufs) if (b) cudaFree(b);
    s = ZbState();
}

#define ZCK(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            char b__[512];                                                                         \
            snprintf(b__, sizeof b__, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            err = b__;                                                                             \
            return e__ == cudaErrorMemoryAllocation ? SNRX_ENOMEM : SNRX_ECUDA;                    \
        }                                                                                          \
    } while (0)

inline int zb_create(ZbState& s, const snrx_config_t& cfg, bool wideband, uint32_t n_ch, uint32_t max_caps,
                     uint32_t max_out, int sm_count, std::string& err) {
    (void)sm_count;
    static_assert(SNRX_IIR_BLOCK == SNRX_ZB_IIR_BLOCK && SNRX_IIR_MEMORY_BLOCKS == SNRX_ZB_IIR_MEMORY_BLOCKS, "include/snoutrx.h and zb_tables.h disagree");
    s.n_ch = n_ch; s.max_caps = max_caps; s.max_out = max_out;
    { const char* e = getenv("SNRX_ZB_RX_CTAS"); const int v = e ? atoi(e) : 0; s.rx_cta_cap = v > 0 ? (uint32_t)v : 0u; }
    if (cfg.zb_segment % SNRX_IIR_BLOCK || cfg.zb_prehalo % SNRX_IIR_BLOCK) {
        err = "zigbee: zb_segment and zb_prehalo must be multiples of 2048 (the DC tracker's block grid)"; return SNRX_EINVAL;
    }
    if ((uint64_t)max_out + cfg.zb_segment + kZbPostHalo >= (1ull << 31)) { err = "zigbee: capture too long for 32-bit chain positions"; return SNRX_ERANGE; }
    s.stride = ((size_t)max_out + 8 + 31) & ~(size_t)31;
    const size_t streams = (size_t)max_caps * n_ch;
    const bool keep = (cfg.flags & SNRX_F_KEEP_STREAMS) != 0;
    // + slack: a chain's tracker runs up to kZbLeadMax + 32 + 2 * kZbQueue samples ahead of its clock recovery, i.e. past
    // the end of its stream (those values are computed and never used)
    ZCK(cudaMalloc((void**)&s.d_f, (streams * s.stride + 512) * sizeof(float)));
    ZCK(cudaMemset(s.d_f, 0, (streams * s.stride + 512) * sizeof(float)));
    if (keep) ZCK(cudaMalloc((void**)&s.d_z, streams * s.stride * sizeof(float)));
    const size_t nblk = (max_out + SNRX_IIR_BLOCK - 1) / SNRX_IIR_BLOCK;
    ZCK(cudaMalloc((void**)&s.d_block_end, streams * nblk * sizeof(double)));
    ZCK(cudaMalloc((void**)&s.d_carry, streams * nblk * sizeof(double)));
    ZCK(cudaMalloc((void**)&s.d_busy, streams * nblk));
    ZCK(cudaMalloc((void**)&s.d_hist, sizeof(uint32_t) * 2 * kZbKeys));
    { const char* e = getenv("SNRX_ZB_ORDER"); s.natural_order = e && atoi(e) == 0; }
    s.decay = zb_iir_block_decay();
    ZCK(cudaMalloc((void**)&s.d_atan, sizeof(SNRX_ATAN_TAB)));
    ZCK(cudaMemcpy(s.d_atan, SNRX_ATAN_TAB, sizeof(SNRX_ATAN_TAB), cudaMemcpyHostToDevice));
    {
        std::vector<float2> pairs(256);
        for (int i = 0; i < 256; i++) pairs[i] = make_float2(SNRX_ATAN_TAB[i], f_sub(SNRX_ATAN_TAB[i + 1], SNRX_ATAN_TAB[i]));
        ZCK(cudaMalloc((void**)&s.d_atan_pairs, sizeof(float2) * 256));
        ZCK(cudaMemcpy(s.d_atan_pairs, pairs.data(), sizeof(float2) * 256, cudaMemcpyHostToDevice));
    }
    ZCK(cudaMalloc((void**)&s.d_mmse, sizeof(SNRX_MMSE_TAPS)));
    ZCK(cudaMemcpy(s.d_mmse, SNRX_MMSE_TAPS, sizeof(SNRX_MMSE_TAPS), cudaMemcpyHostToDevice));
    int32_t chans[16];
    for (int i = 0; i < 16; i++) chans[i] = wideband ? 11 + i : cfg.channel;
    ZCK(cudaMalloc((void**)&s.d_channels, sizeof chans));
    ZCK(cudaMemcpy(s.d_channels, chans, sizeof chans, cudaMemcpyHostToDevice));
    const uint32_t max_segs = (max_out + cfg.zb_segment - 1) / cfg.zb_segment;
    s.max_chains = (uint32_t)(streams * max_segs);
    s.slots_per_chain = zb_slots_per_chain(cfg.zb_segment);
    s.slots_bytes = (size_t)s.max_chains * s.slots_per_chain * sizeof(snrx_frame_t);
    ZCK(cudaMalloc((void**)&s.d_slots, s.slots_bytes));
    ZCK(cudaMalloc((void**)&s.d_counts, sizeof(uint32_t) * ((size_t)s.max_chains + 1)));
    ZCK(cudaMalloc((void**)&s.d_offsets, sizeof(uint32_t) * ((size_t)s.max_chains + 1)));
    ZCK(cudaMalloc((void**)&s.d_scratch, sizeof(uint32_t) * scan_scratch_items(s.max_chains)));
    ZCK(cudaMalloc((void**)&s.d_good_end, sizeof(int64_t) * ((size_t)s.max_chains + 1)));
    ZCK(cudaMalloc((void**)&s.d_queue, sizeof(uint32_t)));
    ZCK(cudaMalloc((void**)&s.d_order, sizeof(uint32_t) * ((size_t)s.max_chains + 1)));
    ZCK(cudaFuncSetAttribute(k_zb_rx<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kZbRxSmem));
    ZCK(cudaFuncSetAttribute(k_zb_rx<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kZbRxSmem));
    if (keep) {
        s.chips_cap = ((int64_t)cfg.zb_segment + cfg.zb_prehalo + kZbPostHalo) / 2 + 64;
        ZCK(cudaMalloc((void**)&s.d_chips, sizeof(float) * (size_t)s.max_chains * (size_t)s.chips_cap));
        ZCK(cudaMalloc((void**)&s.d_nchips, sizeof(int64_t) * (size_t)s.max_chains));
    }
    s.map = make_chip_map();
    s.ready = true;
    return SNRX_OK;
}

// wideband front end (channelizer + discriminator): defined in pfb_zb.cuh
inline int zb_wideband_front(ZbState& s, const snrx_config_t& cfg, const float2* x, uint32_t n_captures, uint64_t n_samples,
                      uint64_t stride, uint32_t n_out, cudaStream_t st, int& launches, std::string& err);

// totals: [2] receives the Zigbee frame count, [3] is set when a chain ran out of frame slots
inline int zb_process(ZbState& s, const snrx_config_t& cfg, const float2* x, uint32_t n_captures, uint64_t n_samples,
                      uint64_t stride, uint32_t n_out, uint32_t pre_out, uint32_t body_out, uint32_t first_segment,
                      uint32_t first_capture, snrx_frame_t* frames, uint32_t frame_cap, uint32_t* totals, bool after_ble,
                      cudaStream_t st, int sm_count, int& launches, std::string& err, cudaEvent_t ev_front_done = nullptr) {
    const bool wideband = (cfg.mode != SNRX_MODE_ZB_NB);
    const bool keep = (cfg.flags & SNRX_F_KEEP_STREAMS) != 0;
    const uint32_t streams = n_captures * s.n_ch;
    if (wideband) {
        int r = zb_wideband_front(s, cfg, x, n_captures, n_samples, stride, n_out, st, launches, err);
        if (r != SNRX_OK) return r;
    } else {
        ZbQuadArgs q;
        q.x = x; q.stride = stride; q.n = (int64_t)n_samples; q.n_captures = n_captures;
        q.f = s.d_f; q.f_stride = s.stride; q.atan_pairs = s.d_atan_pairs;
        const uint64_t per_cap_max = ((n_samples + 3) / 4 + 255) / 256;
        q.blocks_per_cap = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(per_cap_max, ((uint64_t)sm_count * 8 + n_captures - 1) / n_captures));
        const unsigned grid = q.blocks_per_cap * n_captures;
        k_zb_quad<<<grid, 256, 0, st>>>(q);
        launches++;
    }
    if (ev_front_done) ZCK(cudaEventRecord(ev_front_done, st));      // front end = channelizer + discriminator (stats.gpu_ms_frontend)
    ZbIirArgs ia;
    ia.f = s.d_f; ia.stride = s.stride; ia.n = (int32_t)n_out;
    ia.n_blocks = (int32_t)((n_out + SNRX_IIR_BLOCK - 1) / SNRX_IIR_BLOCK); ia.n_streams = streams;
    ia.block_end = s.d_block_end; ia.carry_in = s.d_carry; ia.decay = s.decay; ia.busy = s.natural_order ? nullptr : s.d_busy;
    const uint32_t nb_total = streams * (uint32_t)ia.n_blocks;
    k_zb_iir_sum<<<(nb_total + 63) / 64, 64, 0, st>>>(ia);
    k_zb_iir_carry<<<std::min<uint32_t>((nb_total + 127) / 128, (uint32_t)sm_count * 8), 128, 0, st>>>(ia);
    launches += 2;

    ZbRxArgs a{};
    ZbChainParams& p = a.p;
    p.n_out = (int32_t)n_out; p.origin = (int32_t)pre_out; p.body = (int32_t)body_out;
    p.segment = (int32_t)cfg.zb_segment; p.prehalo = (int32_t)cfg.zb_prehalo;
    p.n_segments = (int32_t)((body_out + cfg.zb_segment - 1) / cfg.zb_segment);
    p.n_blocks = ia.n_blocks;
    p.first_segment = first_segment; p.first_capture = first_capture;
    p.n_captures = n_captures; p.n_channels = s.n_ch; p.threshold = cfg.zb_threshold;
    p.slots_per_chain = s.slots_per_chain; p.f_stride = s.stride;
    const uint32_t n_chains = streams * (uint32_t)p.n_segments;
    if (n_chains > s.max_chains) { err = "zigbee: more chains than capacity"; return SNRX_ERANGE; }
    a.f = s.d_f; a.carry = s.d_carry; a.taps = s.d_mmse; a.channel_numbers = s.d_channels;
    a.slots = s.d_slots; a.counts = s.d_counts; a.good_end = s.d_good_end; a.overflow = totals + 3;
    a.z_dbg = s.d_z; a.chips_dbg = s.d_chips; a.chips_cap = s.chips_cap; a.nchips_dbg = s.d_nchips; a.map = s.map;
    a.queue = s.d_queue;
    ZCK(cudaMemsetAsync(s.d_queue, 0, sizeof(uint32_t), st));
    a.order = nullptr;
    if (!s.natural_order && n_chains > 0) {                                 // longest chains first (zb_chain_key)
        ZbOrderArgs oa;
        oa.busy = s.d_busy; oa.p = p; oa.hist = s.d_hist; oa.order = s.d_order;
        ZCK(cudaMemsetAsync(s.d_hist, 0, sizeof(uint32_t) * 2 * kZbKeys, st));
        k_zb_order<false><<<(n_chains + 255) / 256, 256, 0, st>>>(oa);
        k_zb_order<true><<<(n_chains + 255) / 256, 256, 0, st>>>(oa);
        launches += 2;
        a.order = s.d_order;
    }
    const uint32_t per_cta = kZbRxWarps * 32;
    uint32_t grid = std::min<uint32_t>((n_chains + per_cta - 1) / per_cta, (uint32_t)sm_count * kZbRxCtasPerSm);
    if (s.rx_cta_cap) grid = std::min(grid, s.rx_cta_cap);
    if (keep) ZCK(cudaMemsetAsync(s.d_z, 0, (size_t)streams * s.stride * sizeof(float), st));
    if (keep) k_zb_rx<true><<<grid, per_cta, kZbRxSmem, st>>>(a);
    else k_zb_rx<false><<<grid, per_cta, kZbRxSmem, st>>>(a);
    k_zb_span_filter<<<(n_chains + 127) / 128, 128, 0, st>>>(s.d_slots, s.slots_per_chain, s.d_counts, s.d_good_end, n_chains,
                                                             (uint32_t)p.n_segments, zb_filter_lookback(p.segment));
    launches += 2 + exclusive_scan(s.d_counts, n_chains, s.d_offsets, s.d_scratch, st);
    k_zb_gather<<<std::max(1u, std::min<uint32_t>((n_chains + 3) / 4, (uint32_t)sm_count * 8)), 128, 0, st>>>(
        s.d_slots, s.slots_per_chain, s.d_counts, s.d_offsets, n_chains, frames, frame_cap, totals, after_ble ? 1 : 0);
    launches++;
    ZCK(cudaGetLastError());
    s.last_chains = n_chains;
    return SNRX_OK;
}

inline int zb_debug_stage(ZbState& s, int stage, uint32_t caps, uint32_t n_out, const void** src, uint64_t* bytes) {
    (void)n_out;
    if (!s.ready) return SNRX_ESTATE;
    if (stage == SNRX_STAGE_ZB_DISC) {
        if (!s.d_z) return SNRX_ESTATE;
        *src = s.d_z; *bytes = (uint64_t)caps * s.n_ch * s.stride * sizeof(float); return SNRX_OK;
    }
    if (stage == SNRX_STAGE_ZB_CHIPS) {
        if (!s.d_chips) return SNRX_ESTATE;
        *src = s.d_chips; *bytes = (uint64_t)s.last_chains * (uint64_t)s.chips_cap * sizeof(float); return SNRX_OK;
    }
    if (stage == SNRX_STAGE_ZB_NCHIPS) {
        if (!s.d_nchips) return SNRX_ESTATE;
        *src = s.d_nchips; *bytes = (uint64_t)s.last_chains * sizeof(int64_t); return SNRX_OK;
    }
    if (stage == SNRX_STAGE_ZB_F) { *src = s.d_f; *bytes = (uint64_t)caps * s.n_ch * s.stride * sizeof(float); return SNRX_OK; }
    if (stage == SNRX_STAGE_CHAN_CF32) {
        if (!s.d_wb_cf) return SNRX_ESTATE;
        *src = s.d_wb_cf; *bytes = (uint64_t)caps * s.n_ch * n_out * sizeof(float2); return SNRX_OK;
    }
    return SNRX_EINVAL;
}
#endif  // __CUDACC__

}  // namespace snrx

// TEST INFRASTRUCTURE ONLY.  Host-side stepping of the kernels' __host__ __device__ cores, built
// by nvcc into tests/emu/libemu.so and run on the CPU (no GPU needed).  It lets the CPU test
// suite check the kernels' index math and arithmetic against the oracle before GPU time is
// spent.  The glue between cores (shuffles, ballots, shared-memory hand-over) is restated here
// with plain loops; the cores themselves are the very functions the kernels call.
// Never part of libsnoutrx.so.
#include <cstring>
#include <vector>
#include "../../snout_b200/csrc/ble_back.cuh"
#include "../../snout_b200/csrc/ble_front.cuh"
#include "../../snout_b200/csrc/fft.cuh"
#include "../../snout_b200/csrc/pfb.cuh"
#include "../../snout_b200/csrc/ble_adv.cuh"
#include "../../snout_b200/csrc/ble_conn.cuh"
#include "../../snout_b200/csrc/zb.cuh"
#include "../../snout_b200/csrc/pfb_zb.cuh"
#include "../../snout_b200/csrc/zb_mac.cuh"

using namespace snrx;

template <int C>
static void zb_disc_tile_row(const cf* cur, const cf* nxt, float* f_out, int m) {
    f_out[C * kTileStride + m] = zb_disc<C>(cur[C], nxt[C], SNRX_ATAN_TAB);
    if constexpr (C + 1 < 16) zb_disc_tile_row<C + 1>(cur, nxt, f_out, m);
}

extern "C" {

void emu_idft48(const float* in, float* out) {
    cf a[48], b[48];
    for (int i = 0; i < 48; i++) { a[i].r = in[2 * i]; a[i].i = in[2 * i + 1]; }
    Idft3xQ<48>::run(a, b);
    for (int i = 0; i < 48; i++) { out[2 * i] = b[i].r; out[2 * i + 1] = b[i].i; }
}
void emu_idft96(const float* in, float* out) {
    cf a[96], b[96];
    for (int i = 0; i < 96; i++) { a[i].r = in[2 * i]; a[i].i = in[2 * i + 1]; }
    Idft3xQ<96>::run(a, b);
    for (int i = 0; i < 96; i++) { out[2 * i] = b[i].r; out[2 * i + 1] = b[i].i; }
}

int emu_ble_channel_of_q(int q) { return ble_channel_of_q(q); }

// k_zb_order's per-chain key (a scheduling hint: which chains k_zb_rx hands out first) and the busy flag k_zb_iir_sum derives
// from the last 64 discriminator samples of a block
int emu_zb_chain_key(const uint8_t* busy, int n_blocks, int origin, int body, int segment, int seg) {
    ZbChainParams p{};
    p.origin = origin; p.body = body; p.segment = segment; p.n_blocks = n_blocks;
    return zb_chain_key(busy, n_blocks, p, seg);
}
int emu_zb_block_busy(const float* f_last64) {
    float e = 0.0f;
    for (int i = 0; i < kZbBusyWindow; i++) e += f_last64[i] * f_last64[i];
    return (e > kZbBusyLo && e < kZbBusyHi) ? 1 : 0;
}
int emu_zb_keys() { return kZbKeys; }

}  // extern "C"

// ---- one tile of k_pfb_ble<NT, *>, phases 0..3 --------------------------------------------------
// x: capture cf32 (n_in samples).  Outputs: words[40] = the 31 decisions of samples g_first .. g_first+30
// (bit = time), q8[40][32][2] (int8), raw[40][32] cf32 for samples g_first .. g_first+31.
template <int NT>
static void pfb_tile(const float* x, int64_t n_in, int n_out, int tile, const float* taps_rho,
                     float scale, uint32_t* words, int8_t* q8, float* raw_out) {
    using B = PfbBleGeom<NT>;
    using G = typename B::G;
    constexpr int T = B::kT;
    std::vector<float2> xs(G::kXsLen, make_float2(0.f, 0.f));
    std::vector<float4> V(8 * 32, make_float4(0.f, 0.f, 0.f, 0.f));
    const int g_first = B::kStride * tile;
    const int64_t x0 = (int64_t)kPfbD * g_first - G::kHist;
    constexpr int kPer = 24 * kChunkT, kPairs = kPer / 2;
    for (int idx = 0; idx < G::kPieces * kPairs; idx++) {              // pfb_stage_tile
        const int p = idx / kPairs, t = idx - p * kPairs;
        const int ip = kPer * p - 12 + 2 * t;
        if (ip >= 0 && ip < G::kTileIn) {
            const int64_t i = x0 + ip;
            const bool ok = (i >= 0) && (i + 1 < n_in);
            for (int k = 0; k < 2; k++)
                xs[ip + 8 * p + k] = ok ? make_float2(x[2 * (i + k)], x[2 * (i + k) + 1]) : make_float2(0.f, 0.f);
        }
    }
    std::vector<cf> F(T * 3 * 16);                                     // f[gi][16] of every lane
    for (int gi = 0; gi < 3; gi++) {                                   // phase 1
        for (int lane = 0; lane < 32; lane++) {
            const int rl = lane & 7, c = lane >> 3;
            const int rho = gi + 3 * rl;
            float g[NT];
            for (int d = 0; d < NT; d++) g[d] = taps_rho[rho * NT + d];
            float2 acc[2][kChunkT];
            pfb_fir_thread<NT, 2, kChunkT>(xs.data() + fir_base<NT, kChunkT>(rho, c), rho <= 12 ? 8 : 0, g, acc);
            for (int e = 0; e < kChunkT; e++)
                V[v_pos(rl, 8 * c + e)] = make_float4(acc[0][e].x, acc[0][e].y, acc[1][e].x, acc[1][e].y);
        }
        for (int lane = 0; lane < 32; lane++) {
            cf v16[16], f16[16];
            pfb_load_col16(V.data(), lane, v16);
            IdftPow2<16, 1>::run(v16, f16);
            for (int k = 0; k < 16; k++) F[(lane * 3 + gi) * 16 + k] = f16[k];
        }
    }
    std::vector<cf> Y(T * 48);
    for (int m = 0; m < T; m++) {                                      // phase 2
        const int mg = g_first + m;
        const float s = (mg < n_out) ? scale : 0.0f;
        cf y[48], raw[48], f0[16], f1[16], f2[16];
        for (int k = 0; k < 16; k++) { f0[k] = F[(m * 3 + 0) * 16 + k]; f1[k] = F[(m * 3 + 1) * 16 + k]; f2[k] = F[(m * 3 + 2) * 16 + k]; }
        pfb_combine_quant(f0, f1, f2, y, s, (mg & 1) ? -s : s, raw, true);
        for (int qq = 0; qq < 48; qq++) {
            Y[m * 48 + qq] = y[qq];
            const int ch = ble_channel_of_q(qq);
            if (ch >= 0) {
                q8[(ch * T + m) * 2] = (int8_t)y[qq].r;
                q8[(ch * T + m) * 2 + 1] = (int8_t)y[qq].i;
                const float sg = ((qq & 1) && (mg & 1)) ? -1.0f : 1.0f;
                raw_out[(ch * T + m) * 2] = raw[qq].r * sg;
                raw_out[(ch * T + m) * 2 + 1] = raw[qq].i * sg;
            }
        }
    }
    // phase 3: per-lane slot words, then the shuffle transposes
    uint32_t wa[32], wb[32];
    for (int lane = 0; lane < 32; lane++) {
        const int nx = lane < 31 ? lane + 1 : lane;                    // __shfl_down: lane 31 reads itself
        uint32_t a = 0, b = 0;
        for (int L = 23; L >= 0; L--) {
            const int qq = ble_q_of_slot_a(L);
            a = shift_in_sign(a, slicer_sign(Y[lane * 48 + qq].r, Y[lane * 48 + qq].i, Y[nx * 48 + qq].r, Y[nx * 48 + qq].i));
        }
        for (int L = 15; L >= 0; L--) {
            const int qq = ble_q_of_slot_b(L);
            b = shift_in_sign(b, slicer_sign(Y[lane * 48 + qq].r, Y[lane * 48 + qq].i, Y[nx * 48 + qq].r, Y[nx * 48 + qq].i));
        }
        wa[lane] = a; wb[lane] = b;
    }
    auto xchg = [](uint32_t* w, int j, uint32_t m) {
        uint32_t o[32];
        for (int lane = 0; lane < 32; lane++) o[lane] = transpose_step(w[lane], w[lane ^ j], lane, j, m);
        memcpy(w, o, sizeof o);
    };
    { uint32_t o[32]; for (int lane = 0; lane < 32; lane++) o[lane] = (wb[lane] & 0xFFFFu) | (wb[lane ^ 16] << 16); memcpy(wb, o, sizeof o); }
    xchg(wa, 16, 0x0000FFFFu);
    for (int j = 8; j >= 1; j >>= 1) {
        const uint32_t m = j == 8 ? 0x00FF00FFu : j == 4 ? 0x0F0F0F0Fu : j == 2 ? 0x33333333u : 0x55555555u;
        xchg(wa, j, m); xchg(wb, j, m);
    }
    memset(words, 0, sizeof(uint32_t) * 40);
    for (int L = 0; L < 24; L++) words[ble_channel_of_q(ble_q_of_slot_a(L))] = wa[L] & 0x7FFFFFFFu;
    for (int L = 0; L < 16; L++) words[ble_channel_of_q(ble_q_of_slot_b(L))] = wb[L] & 0x7FFFFFFFu;
}

// ---- one tile of k_pfb_zb<NT, *>: f[g_first+1 .. g_first+127] for 16 channels, rotated streams for debug
template <int NT>
static void pfb_zb_tile(const float* x, int64_t n_in, int n_out, int tile, const float* taps_rho,
                        float* f_out /*[16][127]*/, float* y_out /*[16][128] cf32 rotated*/) {
    using G = PfbGeom<NT, kZbChunkT>;
    std::vector<float2> xs(G::kXsLen, make_float2(0.f, 0.f));
    std::vector<float2> V(96 * kZbVStride, make_float2(0.f, 0.f));
    const int g_first = kTileStride * tile;
    const int64_t x0 = (int64_t)kPfbD * g_first - G::kHist;
    constexpr int kPer = 24 * kZbChunkT;
    for (int tid = 0; tid < kPer / 2; tid++)
        for (int p = 0; p < G::kPieces; p++) {
            const int ip = kPer * p - 12 + 2 * tid;
            if (ip >= 0 && ip < G::kTileIn) {
                const int64_t i = x0 + ip;
                const bool ok = (i >= 0) && (i + 1 < n_in);
                for (int k = 0; k < 2; k++)
                    xs[ip + 8 * p + k] = ok ? make_float2(x[2 * (i + k)], x[2 * (i + k) + 1]) : make_float2(0.f, 0.f);
            }
        }
    for (int tid = 0; tid < kZbFirThreads; tid++) {
        const int lane = tid & 31, wid = tid >> 5;
        const int rho = 8 * (wid % 3) + (lane & 7), q = 4 * (wid / 3) + (lane >> 3);
        float g[NT];
        for (int d = 0; d < NT; d++) g[d] = taps_rho[rho * NT + d];
        float2 acc[4][kZbChunkT];
        pfb_fir_thread<NT, 4, kZbChunkT>(xs.data() + fir_base<NT, kZbChunkT>(rho, q), rho <= 12 ? 8 : 0, g, acc);
        for (int br = 0; br < 4; br++)
            for (int e = 0; e < kZbChunkT; e++) V[(rho + 24 * br) * kZbVStride + kZbChunkT * q + e] = acc[br][e];
    }
    std::vector<cf> Y(kTileT * 16);
    for (int m = 0; m < kTileT; m++) {
        cf y[16];
        pfb_dft96_zb(V.data() + m, y);
        const int mg = g_first + m;
        for (int c = 0; c < 16; c++) {
            Y[m * 16 + c] = y[c];
            const int rot = (zb_bin_of_slot(c) * (mg & 3)) & 3;
            const float rr = rot == 0 ? y[c].r : rot == 1 ? y[c].i : rot == 2 ? -y[c].r : -y[c].i;
            const float ii = rot == 0 ? y[c].i : rot == 1 ? -y[c].r : rot == 2 ? -y[c].i : y[c].r;
            y_out[(c * kTileT + m) * 2] = rr; y_out[(c * kTileT + m) * 2 + 1] = ii;
        }
    }
    for (int m = 0; m < kTileStride; m++) zb_disc_tile_row<0>(&Y[m * 16], &Y[(m + 1) * 16], f_out, m);
}

extern "C" {

void emu_pfb_zb_tile(int nt, const float* x, int64_t n_in, int n_out, int tile, const float* taps_rho, float* f_out, float* y_out) {
    if (nt == 16) pfb_zb_tile<16>(x, n_in, n_out, tile, taps_rho, f_out, y_out);
    else pfb_zb_tile<32>(x, n_in, n_out, tile, taps_rho, f_out, y_out);
}
int emu_zb_bin_of_slot(int c) { return zb_bin_of_slot(c); }

int emu_pfb_tile_stride(void) { return kTileStride; }          // Zigbee kernel

// BLE channelizer tile (one warp): 32 samples computed, 31 decisions emitted
int emu_pfb_ble_stride(void) { return PfbBleGeom<16>::kStride; }
void emu_pfb_ble_tile(int nt, const float* x, int64_t n_in, int n_out, int tile, const float* taps_rho,
                      float scale, uint32_t* words, int8_t* q8, float* raw) {
    if (nt == 16) pfb_tile<16>(x, n_in, n_out, tile, taps_rho, scale, words, q8, raw);
    else pfb_tile<32>(x, n_in, n_out, tile, taps_rho, scale, words, q8, raw);
}

int emu_bits_words_for(int n_out) { return (int)bits_words_for((uint32_t)n_out); }
int emu_bits_lead_words(void) { return kBitsLeadWords; }

// ---- narrow-band slicer: whole capture -> bit stream words (BitsLayout, 1 channel) --------------
void emu_ble_slice_nb(const float* x, int64_t n, float scale, uint32_t* bits, uint32_t nw, int8_t* q8) {
    memset(bits, 0, sizeof(uint32_t) * nw);
    auto qv = [&](int64_t k, int c) -> float { return k < n ? quant_exact(x[2 * k + c], scale) : quant_exact(0.f, scale); };
    for (int64_t k = 0; k < n; k++) {
        if (q8) { q8[2 * k] = (int8_t)qv(k, 0); q8[2 * k + 1] = (int8_t)qv(k, 1); }
        if (slicer_bit(qv(k, 0), qv(k, 1), qv(k + 1, 0), qv(k + 1, 1)))
            bits[(size_t)kBitsLeadWords + (size_t)(k >> 5)] |= 1u << (k & 31);
    }
}

// ---- BLE back end over one (capture, channel) bit stream: aa search, decode, resolve -----------
int emu_ble_back(const uint32_t* bits, uint32_t nw, int n_out, int m_origin, int n_windows, uint32_t first_window,
                 int channel, uint32_t aa, uint32_t aa_mask, uint32_t crc_init_internal, const uint32_t* crc_tab,
                 const uint32_t* whiten /*[40][11]*/, snrx_frame_t* out, int cap, int* n_cands_out) {
    BleParams p{};
    p.aa = aa; p.aa_mask = aa_mask; p.crc_init_internal = crc_init_internal; p.n_out = n_out; p.m_origin = m_origin;
    p.n_windows = n_windows; p.first_window = first_window; p.first_capture = 0; p.n_captures = 1; p.n_channels = 1;
    const int z = aa_virtual_bits(aa, aa_mask);
    const uint32_t mask_hi = aa_mask & ~((1u << z) - 1u);
    std::vector<Cand> cands;
    for (uint32_t w = 0; w < nw; w++) {                                // k_aa_search + k_aa_fill
        uint32_t ww[5];
        for (int d = 0; d < 5; d++) ww[d] = (w + d < nw) ? bits[w + d] : 0u;
        const AaTables tabs = make_aa_tables(aa, mask_hi);
        uint32_t h = aa_word_hits(ww, tabs, [](uint32_t m) { return m != 0u; });
        const int nvalid = n_out - 32 * ((int)w - kBitsLeadWords);
        if (nvalid <= 0) h = 0u; else if (nvalid < 32) h &= (1u << nvalid) - 1u;
        for (int i = 0; i < 32; i++)
            if ((h >> i) & 1u) {
                const int s = 32 * ((int)w - kBitsLeadWords) + i;
                const uint32_t d = (symbols32(bits, s) ^ aa) & aa_mask;
                Cand c; c.s = s; c.ch_idx = 0; c.vneed = (uint8_t)hi_bit_plus1(d); c.pad = 0; c.cap = 0;
                cands.push_back(c);
            }
    }
    std::vector<Dec> decs(cands.size());
    for (size_t k = 0; k < cands.size(); k++) {                        // k_ble_decode
        const Cand c = cands[k];
        uint32_t chunk[11];
        for (int q = 0; q < 11; q++) chunk[q] = symbols32(bits, c.s + 128 + 128 * q) ^ whiten[channel * 11 + q];
        Dec d; d.s = c.s; d.resume = 0; d.vneed = c.vneed;
        ble_finish(chunk, channel >= 37 && channel <= 39, crc_init_internal, crc_tab, d);
        decs[k] = d;
    }
    int n = 0;
    for (int w = 0; w < n_windows; w++) {
        const int W = m_origin + kWindow * w;
        ble_resolve_window(cands.data(), decs.data(), 0, (int)cands.size(), W, z, [&](int k) {
            if (n < cap) ble_fill_frame(out[n], cands[k], decs[k], p, w, channel);
            n++;
        });
    }
    if (n_cands_out) *n_cands_out = (int)cands.size();
    return n;
}

// ---- Zigbee cores -----------------------------------------------------------------------------
void emu_zb_quad(const float* x, int64_t n, float* f) {
    for (int64_t k = 0; k < n; k++) {
        const float pr = k ? x[2 * (k - 1)] : 0.f, pi = k ? x[2 * (k - 1) + 1] : 0.f;
        f[k] = quad_demod(x[2 * k], x[2 * k + 1], pr, pi, SNRX_ATAN_TAB);
    }
}
void emu_zb_dc(const float* f, int64_t n, float* z) {
    const double decay = zb_iir_block_decay();
    const int nb = (int)((n + SNRX_IIR_BLOCK - 1) / SNRX_IIR_BLOCK);
    std::vector<double> block_end(nb), carry_in(nb);
    for (int b = 0; b < nb; b++) {                      // k_zb_iir_sum
        const int len = (int)std::min<int64_t>(SNRX_IIR_BLOCK, n - (int64_t)b * SNRX_IIR_BLOCK);
        double l = 0.0;
        for (int i = 0; i < len; i++) l = zb_iir_step(l, f[(size_t)b * SNRX_IIR_BLOCK + i]);
        block_end[b] = l;
    }
    for (int b = 0; b < nb; b++) carry_in[b] = zb_iir_fold(block_end.data(), b, decay);   // k_zb_iir_carry
    for (int b = 0; b < nb; b++) {                      // the tracker inside k_zb_rx (ZbRingSrc::convert2)
        const int len = (int)std::min<int64_t>(SNRX_IIR_BLOCK, n - (int64_t)b * SNRX_IIR_BLOCK);
        double y = carry_in[b];
        for (int i = 0; i < len; i++) {
            const float fv = f[(size_t)b * SNRX_IIR_BLOCK + i];
            y = zb_iir_step(y, fv);
            z[(size_t)b * SNRX_IIR_BLOCK + i] = zb_dc_out(fv, y);
        }
    }
}
uint32_t emu_zb_slots_per_chain(uint32_t segment) { return zb_slots_per_chain(segment); }
void emu_zb_mmse_taps(float* out /*[129][8]*/) { memcpy(out, SNRX_MMSE_TAPS, sizeof(SNRX_MMSE_TAPS)); }
// k_zb_rx's tracker pacing: kZbLead, kZbLeadMin, kZbLeadMax
void emu_zb_lead_params(int* out) { out[0] = kZbLead; out[1] = kZbLeadMin; out[2] = kZbLeadMax; }

// chains over a DC-removed stream: zb_run_chain (the per-thread code of k_zb_rx) with the samples read straight from z.
// Returns the number of records, or -(seg + 1) when chain seg found more records than its slots hold (k_zb_rx sets the
// overflow flag there and the batch fails with SNRX_EOVERFLOW).
int emu_zb_chains(const float* z, int n_out, int origin, int body, int segment, int prehalo, uint32_t first_segment,
                  int threshold, int channel, snrx_frame_t* out, int cap, int64_t* nchips_out /* [n_segments] or null */) {
    ZbChainParams p{};
    p.n_out = n_out; p.origin = origin; p.body = body; p.segment = segment; p.prehalo = prehalo;
    p.n_segments = (body + segment - 1) / segment; p.first_segment = first_segment; p.first_capture = 0;
    p.n_captures = 1; p.n_channels = 1; p.threshold = threshold; p.slots_per_chain = zb_slots_per_chain(segment);
    p.f_stride = 0;
    ChipMap map = make_chip_map();
    // k_zb_rx: every chain into its own slots + the end of its CRC-ok frames
    std::vector<snrx_frame_t> slots((size_t)p.slots_per_chain * p.n_segments);
    std::vector<uint32_t> counts(p.n_segments);
    std::vector<int64_t> good_end(p.n_segments);
    for (int seg = 0; seg < p.n_segments; seg++) {
        ZbDirectSrc src{z, &SNRX_MMSE_TAPS[0][0]};
        int64_t nchips = 0;
        uint32_t nf = zb_run_chain<false>(src, p, seg, map.w, channel, 0, slots.data() + (size_t)seg * p.slots_per_chain, nullptr, 0,
                                          &nchips, &good_end[seg]);
        if (nchips_out) nchips_out[seg] = nchips;
        if (nf > p.slots_per_chain) return -(seg + 1);
        counts[seg] = nf;
    }
    // k_zb_span_filter (one thread per chain), then k_zb_gather
    const int lookback = zb_filter_lookback(segment);
    int n = 0;
    for (int seg = 0; seg < p.n_segments; seg++) {
        int64_t ge = 0;
        for (int j = 1; j <= lookback && j <= seg; j++) ge = std::max(ge, good_end[seg - j]);
        const uint32_t w = zb_filter_chain(slots.data() + (size_t)seg * p.slots_per_chain, counts[seg], ge);
        for (uint32_t k = 0; k < w; k++) { if (n < cap) out[n] = slots[(size_t)seg * p.slots_per_chain + k]; n++; }
    }
    return n;
}

// the windowed sink alone on given hard chips (one bit per chip), against which the reference sink is compared:
// returns the number of frames, lens[k] / bytes[k][128] / end_chip[k] (index of the chip that completed frame k)
int emu_zb_sink_chips(const uint8_t* chips, int64_t n, int threshold, int32_t* lens, uint8_t* bytes, int64_t* end_chip, int cap) {
    ChipMap map = make_chip_map();
    ZbSinkW s; zb_sinkw_init(s);
    snrx_frame_t slot;
    ZbEmit em{};
    em.slots = &slot; em.cap = 1; em.nf = 0; em.lo = 0; em.hi = 0x7FFFFFFF; em.index_base = 0; em.good_end = 0;
    int k = 0;
    for (int64_t w0 = 0; w0 < n; w0 += 32) {
        const int nvalid = (int)std::min<int64_t>(32, n - w0);
        uint32_t C = 0;
        for (int j = 0; j < nvalid; j++) C = (C << 1) | (chips[w0 + j] & 1u);
        if (nvalid < 32) C <<= (32 - nvalid);
        int consumed = 0;
        const int jb = s.jb;
        const bool done = zb_sink_window(s, C, nvalid, nvalid, (int32_t)(w0 + jb), map.w, threshold, em, &consumed);
        if (em.nf) {                                     // a frame completed at the boundary of this window
            if (k < cap) { lens[k] = slot.len; memcpy(bytes + (size_t)k * 128, slot.bytes, 128); end_chip[k] = w0 + jb; }
            k++; em.nf = 0;
        }
        if (done) break;
    }
    return k;
}

// one record through zb_mac_parse (k_zb_mac_summary's per-thread code)
void emu_zb_mac_parse(const uint8_t* psdu, int len, snrx_zbmac_t* out) { zb_mac_parse(psdu, len, *out); out->frame = 0; }

// one record through ble_adv_parse (k_ble_adv_summary's per-thread code)
void emu_ble_adv_parse(const uint8_t* pdu, int len, snrx_adv_t* out) { ble_adv_parse(pdu, len, *out); out->frame = 0; }

// one record through ble_conn_parse (k_ble_conn_fill's per-thread code); returns 1 for a CONNECT_REQ
int emu_ble_conn_parse(const uint8_t* pdu, int len, snrx_conn_t* out) { memset(out, 0, sizeof *out); return ble_conn_parse(pdu, len, *out) ? 1 : 0; }

}  // extern "C"

// TEST INFRASTRUCTURE ONLY.  Host-side stepping of the BLE channelizer's prime-factor 48-point transform and integer slicer
// (snout_b200/csrc/fft.cuh Pfa48, snout_b200/csrc/pfb.cuh), built by nvcc into a temporary shared library by
// tests/test_pfb_factored.py and run on the CPU (no GPU needed).  Never part of libsnoutrx.so.
#include <cstring>
#include <vector>
#include "../../snout_b200/csrc/pfb.cuh"

using namespace snrx;

// ---- one tile of k_pfb_ble<NT, *>, phases 0..3, along the kernel's path (prime-factor passes, integer slicer) -------------
// The glue between cores (shuffles, shared-memory hand-over) is restated with plain loops, as in tests/emu/emu.cu; the cores
// are the functions the kernel calls.  x: capture cf32 (n_in samples).  Outputs: words[40] = the 31 decisions of samples
// g_first .. g_first+30 (bit = time), q8[40][32][2] (int8), raw[40][32] cf32 for samples g_first .. g_first+31.
template <int NT>
static void pfa_tile(const float* x, int64_t n_in, int n_out, int tile, const float* taps_rho, float scale, uint32_t* words,
                     int8_t* q8, float* raw_out) {
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
            pfb_load_col16_pfa(V.data(), lane, gi, v16);
            IdftPow2<16, 1>::run(v16, f16);
            for (int k = 0; k < 16; k++) F[(lane * 3 + gi) * 16 + k] = f16[k];
        }
    }
    std::vector<uint32_t> SW(T * 48), SA(T * 48);                      // slicer words of every lane
    for (int m = 0; m < T; m++) {                                      // phase 2
        const int mg = g_first + m;
        const float s = (mg < n_out) ? scale : 0.0f;
        cf raw[48], f0[16], f1[16], f2[16];
        uint32_t sw[48], sa[48];
        for (int k = 0; k < 16; k++) { f0[k] = F[(m * 3 + 0) * 16 + k]; f1[k] = F[(m * 3 + 1) * 16 + k]; f2[k] = F[(m * 3 + 2) * 16 + k]; }
        pfb_combine_quant_pfa(f0, f1, f2, sw, sa, s, (mg & 1) ? -s : s, raw, true);
        for (int qq = 0; qq < 48; qq++) {
            SW[m * 48 + qq] = sw[qq]; SA[m * 48 + qq] = sa[qq];
            const int ch = ble_channel_of_q(qq);
            if (ch >= 0) {
                q8[(ch * T + m) * 2] = slicer_a_i(sa[qq]);
                q8[(ch * T + m) * 2 + 1] = slicer_a_q(sa[qq]);
                const float sg = ((qq & 1) && (mg & 1)) ? -1.0f : 1.0f;
                raw_out[(ch * T + m) * 2] = raw[qq].r * sg;
                raw_out[(ch * T + m) * 2 + 1] = raw[qq].i * sg;
            }
        }
    }
    uint32_t wa[32], wb[32];                                           // phase 3: per-lane slot words, then the transposes
    for (int lane = 0; lane < 32; lane++) {
        const int nx = lane < 31 ? lane + 1 : lane;                    // __shfl_down: lane 31 reads itself
        uint32_t a = 0, b = 0;
        for (int L = 23; L >= 0; L--) {
            const int qq = ble_q_of_slot_a(L);
            a = shift_in_sign(a, slicer_sign_dp4a(SA[lane * 48 + qq], SW[nx * 48 + qq]));
        }
        for (int L = 15; L >= 0; L--) {
            const int qq = ble_q_of_slot_b(L);
            b = shift_in_sign(b, slicer_sign_dp4a(SA[lane * 48 + qq], SW[nx * 48 + qq]));
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

extern "C" {

void emu_pfa_ble_tile(int nt, const float* x, int64_t n_in, int n_out, int tile, const float* taps_rho, float scale,
                      uint32_t* words, int8_t* q8, float* raw) {
    if (nt == 16) pfa_tile<16>(x, n_in, n_out, tile, taps_rho, scale, words, q8, raw);
    else pfa_tile<32>(x, n_in, n_out, tile, taps_rho, scale, words, q8, raw);
}

// 32 independent 48-point inverse DFTs, in[32][48] -> out[32][48] (cf32), along k_pfb_ble's route: branch r of vector `lane`
// goes to the V tile where the FIR lane of pass r mod 3 stores it, pfb_load_col16 reads the pass's column in the rotated order,
// IdftPow2<16, 1> transforms it, and the twiddle-free combination writes the 48 bins
void emu_pfa48_tile(const float* in, float* out) {
    float4 V[3][8 * 32];
    for (int gi = 0; gi < 3; gi++)
        for (int rl = 0; rl < 8; rl++)
            for (int col = 0; col < 32; col++) {
                const float* a = in + 2 * (48 * col + gi + 3 * rl);        // branch rho = gi + 3 rl
                const float* b = in + 2 * (48 * col + gi + 3 * rl + 24);   // and rho + 24
                V[gi][v_pos(rl, col)] = make_float4(a[0], a[1], b[0], b[1]);
            }
    for (int lane = 0; lane < 32; lane++) {
        cf f[3][16], y[48];
        for (int gi = 0; gi < 3; gi++) {
            cf v16[16];
            pfb_load_col16_pfa(V[gi], lane, gi, v16);
            IdftPow2<16, 1>::run(v16, f[gi]);
        }
        Pfa48::combine<0>(f[0], f[1], f[2], y);
        for (int k = 0; k < 48; k++) { out[2 * (48 * lane + k)] = y[k].r; out[2 * (48 * lane + k) + 1] = y[k].i; }
    }
}

void emu_pfa48_run(const float* in, float* out) {
    cf a[48], b[48];
    for (int i = 0; i < 48; i++) { a[i].r = in[2 * i]; a[i].i = in[2 * i + 1]; }
    Pfa48::run(a, b);
    for (int i = 0; i < 48; i++) { out[2 * i] = b[i].r; out[2 * i + 1] = b[i].i; }
}

// the wideband quantiser's biased result for one component y at quantiser scale `scale`, as k_pfb_ble forms it
uint32_t emu_quant_bits(float y, float scale) { return f_bits(quant_pair_biased(make_float2(y, y), f_mul(scale, 1.0f / 255.0f)).x); }
int emu_q8_of_biased(uint32_t t) { return q8_of_biased(t); }

// slicer words of one sample from the bits of its biased (I, Q): out = {slicer_w, slicer_a, slicer_a_i, slicer_a_q}
void emu_slicer_words(uint32_t t_i, uint32_t t_q, uint32_t* out) {
    const uint32_t a = slicer_a(t_i, t_q);
    out[0] = slicer_w(t_i, t_q); out[1] = a; out[2] = (uint32_t)(int)slicer_a_i(a); out[3] = (uint32_t)(int)slicer_a_q(a);
}

// decision bit of sample (I0, Q0) with successor (I1, Q1) through the slicer helpers, for every int8 (I0, Q0, I1, Q1): returns
// the number of the 2^32 cases whose bit differs from I0 Q1 - I1 Q0 > 0
uint64_t emu_slicer_exhaustive(void) {
    static uint32_t W[65536];
    for (int j = 0; j < 65536; j++) {                       // j = (I1 + 128) * 256 + (Q1 + 128)
        const int i1 = (j >> 8) - 128, q1 = (j & 255) - 128;
        W[j] = slicer_w(f_bits(kMagic + (float)i1), f_bits(kMagic + (float)q1));
    }
    uint64_t bad = 0;
#pragma omp parallel for reduction(+ : bad) schedule(static)
    for (int k = 0; k < 65536; k++) {
        const int i0 = (k >> 8) - 128, q0 = (k & 255) - 128;
        const uint32_t a = slicer_a(f_bits(kMagic + (float)i0), f_bits(kMagic + (float)q0));
        for (int j = 0; j < 65536; j++) {
            const int i1 = (j >> 8) - 128, q1 = (j & 255) - 128;
            const uint32_t got = slicer_sign_dp4a(a, W[j]) >> 31;
            bad += got != (uint32_t)(i0 * q1 - i1 * q0 > 0);
        }
    }
    return bad;
}

}  // extern "C"

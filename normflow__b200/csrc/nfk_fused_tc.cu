// nfk_fused_tc.cu -- kernel and launch of the tensor-core fused coupling step
// (design notes: nfk_fused_tc.cuh).  Persistent CTAs (two per SM) loop over samples; per
// sample the lattice is walked in strips of R rows.
//
// Per strip (rows = output rows, r0 = first lattice row), linear index = row * WS + slot,
// slot = column + 1:
//   x  strip : rows r0-3 .. r0+rows+2   fp32   [rows+6][WS]
//   h1 strip : rows r0-2 .. r0+rows+1   fp16 hi/lo planes of 16-byte records (8 channels)
//   h2 strip : rows r0-1 .. r0+rows     the same, split by the parity of the linear index
// A strip that continues a sample copies its first h2 rows (0, 1) and the h1 rows they need (2, 3)
// from the bottom of the previous strip instead of recomputing them (tc_carry).
//
//   compute warps                                   MMA warp
//   -------------                                   --------
//   load x strip                    |barC|
//   P1: h1 = tanh(conv1(x frozen))  -> arrive H1    sync H1: layer-2 tiles (9 MMAs each, N = 16),
//   E2: per tile wait m2[j]; TMEM -> bias, tanh,             commit m2[j] per tile
//       split -> h2                 -> arrive H2    sync H2: layer-3 tiles on ACTIVE sites
//   E3: per tile wait m3[k]; TMEM -> spline/affine           (9 MMAs, N = N3), commit m3[k]
//       -> y into the x strip       |barC|
//   copy the strip's rows to y      |barC|

#include <stdlib.h>

#include <type_traits>

#include "nfk_common.cuh"
#include "nfk_fused_tc.cuh"

using namespace nfk;

struct TcArgs {
    const float *x, *w1, *b1, *w2, *b2, *w3, *b3, *log_in;
    float *y, *log_out;
    long long B;
    TcGeom g;
    RqsCfg cfg;
    long long* trace;      // debug: per-phase clock64 stamps of CTA 0 (NULL in production)
    // training forward (SAVE): what the backward kernels need, channel-major fp32
    float *save_h1, *save_h2;   // [B][8][L0][L1] post-activation hidden layers
    float *save_out;            // [B][P][L0][L1] conditioner output (written at the active sites only)
};

// debug hook (not part of the C ABI): a device buffer of 2 x 4096 int64 that CTA 0 fills with
// clock64() stamps, [0, 4096) compute warps, [4096, 8192) MMA warp
static long long* g_trace = nullptr;
extern "C" void nfk_debug_tc_trace(long long* device_buffer) { g_trace = device_buffer; }

namespace {

// 8 broadcast weights as two 128-bit shared loads
__device__ __forceinline__ void load_w8(const float* p, float (&wv)[8]) {
    const float4 t0 = reinterpret_cast<const float4*>(p)[0], t1 = reinterpret_cast<const float4*>(p)[1];
    wv[0] = t0.x; wv[1] = t0.y; wv[2] = t0.z; wv[3] = t0.w; wv[4] = t1.x; wv[5] = t1.y; wv[6] = t1.z; wv[7] = t1.w;
}

__device__ __forceinline__ int wrap_idx(int v, int L) {
    v %= L;
    return v < 0 ? v + L : v;
}

// 8 channel values of one site -> the hi / lo fp16 records
__device__ __forceinline__ void make_records(const float (&v)[8], uint4& hi, uint4& lo) {
    float l[8], h[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) h[c] = tc_split(v[c], l[c]);
    hi = make_uint4(tc_pack(h[0], h[1]), tc_pack(h[2], h[3]), tc_pack(h[4], h[5]), tc_pack(h[6], h[7]));
    lo = make_uint4(tc_pack(l[0], l[1]), tc_pack(l[2], l[3]), tc_pack(l[4], l[5]), tc_pack(l[6], l[7]));
}

template <int KIND, int K, int INV, bool SAVE>
__global__ void __launch_bounds__(kTcThreads, 2) fused2d_tc_kernel(const TcArgs a) {
    constexpr int P = KIND == 0 ? 2 : 3 * K - 2;
    using Shape = TcShape<P>;
    constexpr int N3 = Shape::N3;
    extern __shared__ __align__(128) uint8_t smem[];
    const TcGeom& g = a.g;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int WS = g.WS, L0 = g.L0, L1 = g.L1;

    float* xs = reinterpret_cast<float*>(smem + g.off_xs);
    uint8_t* h1 = smem + g.off_h1 + kTcGuard * 16;            // record 0 of the hi plane
    uint8_t* h2 = smem + g.off_h2 + kTcGuard * 16;            // record 0 of parity 0, hi plane
    __half* B2 = reinterpret_cast<__half*>(smem + g.off_b2);  // [tap][kgroup][16][8]
    __half* B3 = reinterpret_cast<__half*>(smem + g.off_b3);  // [tap][kgroup][N3][8]
    float* w1s = reinterpret_cast<float*>(smem + g.off_w1);   // [tap][8] | b1[8] | b2[8] | b3[P]
    float* b1s = w1s + 72;                                    // layer-1 weights and b1, b2 are stored times
    float* b2s = b1s + 8;                                     // 2 log2(e): the tanh argument comes out scaled
    float* b3s = b2s + 8;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + g.off_bar);   // m2[16] | m3[8]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 24);
    float* red = reinterpret_cast<float*>(tmem_slot + 2);             // one float per compute warp (<= 12)

    // ---- one-time set-up: weights -> fp16 pair operands, barriers, TMEM -------------------
    for (int e = tid; e < 9 * 16 * 8; e += kTcThreads) {                 // layer 2: N = [8 hi | 8 lo]
        const int ci = e & 7, n = (e >> 3) & 15, t = e >> 7;
        const int co = n & 7;
        const float w = NFK_LDG(a.w2 + (co * 8 + ci) * 9 + t);
        const __half hi = __float2half_rn(w);
        const __half val = n < 8 ? hi : __float2half_rn((w - __half2float(hi)) * kLoScale);
        B2[((t * 2 + 0) * 16 + n) * 8 + ci] = val;
        B2[((t * 2 + 1) * 16 + n) * 8 + ci] = val;
    }
    for (int e = tid; e < 9 * N3 * 8; e += kTcThreads) {                 // layer 3: N = [8 hi | 8 lo] per group
        const int ci = e & 7, n = (e >> 3) % N3, t = (e >> 3) / N3;
        const int grp = n >> 4, w16 = n & 15;
        const int gs = P - 8 * grp < 8 ? P - 8 * grp : 8;                // channels of this group (<= 0: padding)
        const bool is_lo = w16 >= gs;
        const int p = 8 * grp + (is_lo ? w16 - gs : w16);
        __half val = __float2half_rn(0.f);
        if (w16 < 2 * gs) {
            const float w = NFK_LDG(a.w3 + (p * 8 + ci) * 9 + t);
            const __half hi = __float2half_rn(w);
            val = is_lo ? __float2half_rn((w - __half2float(hi)) * kLoScale) : hi;
        }
        B3[((t * 2 + 0) * N3 + n) * 8 + ci] = val;
        B3[((t * 2 + 1) * N3 + n) * 8 + ci] = val;
    }
    for (int e = tid; e < 72 + 8 + 8 + P; e += kTcThreads) {
        float v;
        if (e < 72) v = kTwoLog2e * NFK_LDG(a.w1 + (e & 7) * 9 + (e >> 3));          // w1s[tap][co]
        else if (e < 80) v = a.b1 ? kTwoLog2e * NFK_LDG(a.b1 + e - 72) : 0.f;
        else if (e < 88) v = a.b2 ? kTwoLog2e * NFK_LDG(a.b2 + e - 80) : 0.f;
        else v = (a.b3 && e - 88 < P) ? NFK_LDG(a.b3 + e - 88) : 0.f;
        w1s[e] = v;
    }
    if (tid == 0) {
        for (int i = 0; i < 24; ++i) tc::mbar_init(tc::smem_u32(bars + i), 1);
        tc::fence_mbar_init();
    }
    if (warp == kTcComputeWarps) tc::tmem_alloc(tc::smem_u32(tmem_slot), kTcTmemCols);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const int cbase = tc_cbase(WS);

    // The CTA's work is the flat sequence of (sample, strip) units; both roles walk it in step.
    struct Unit { long long b; int r0; };
    const int Rr = g.R;
    auto next_unit = [&](Unit u) {
        u.r0 += Rr;
        if (u.r0 >= L0) { u.r0 = 0; u.b += gridDim.x; }
        return u;
    };

    if (warp >= kTcComputeWarps) {
        // =============================== MMA warps ========================================
        const int iw = warp - kTcComputeWarps;                     // this issuer takes tiles iw, iw + kTcIssuers, ...
        const bool lead = tc::elect_one();
        const uint32_t idesc2 = tc::make_idesc(0, 128, 16), idesc3 = tc::make_idesc(0, 128, N3);
        const uint64_t a1_desc = tc::make_desc(tc::smem_u32(h1), g.h1_comp_bytes, 128);
        const uint64_t a2_desc0 = tc::make_desc(tc::smem_u32(h2), g.h2_comp_bytes, 128);
        const uint64_t a2_desc1 = tc::make_desc(tc::smem_u32(h2 + g.h2_par_bytes), g.h2_comp_bytes, 128);
        const uint64_t b2_desc = tc::make_desc(tc::smem_u32(B2), 16 * 16, 128);
        const uint64_t b3_desc = tc::make_desc(tc::smem_u32(B3), N3 * 16, 128);
        int tn = 0;
        auto stamp = [&](int) {
            if (a.trace && blockIdx.x == 0 && lead && iw == 0 && tn < 4000) a.trace[4096 + tn++] = clock64();
        };
        for (Unit u{blockIdx.x, 0}; u.b < a.B; u = next_unit(u)) {
            const int r0 = u.r0, rows = L0 - r0 < Rr ? L0 - r0 : Rr;
            const int c2 = tc_carry(r0);
            const int t2 = tc_tiles2(rows, WS, c2), t3 = tc_tiles3(rows, WS, L1);
            const int plin = (g.active_val - 1 + g.mask_parity - r0) & 1;
            // ---- layer 2: out record i2 = c2 WS + 128 j + m reads h1 records i2 + WS + dr WS + dc
            stamp(0);
            tc::bar_sync(kBarH1, kTcThreads);
            tc::fence_after_sync();
            stamp(1);
            if (lead) {
                for (int j = iw; j < t2; j += kTcIssuers) {
#pragma unroll
                    for (int t = 0; t < 9; ++t) {
                        const int delta = (t / 3 - 1) * WS + (t % 3 - 1);
                        tc::mma_f16(tmem + j * 16, tc::desc_advance(a1_desc, j * 128 + (c2 + 1) * WS + delta),
                                    tc::desc_advance(b2_desc, t * 2 * 16), idesc2, t > 0);
                    }
                    tc::mma_commit(tc::smem_u32(bars + j));
                }
            }
            __syncwarp();
            stamp(2);
            // ---- layer 3: active record c (site s = 2c + plin) reads s + dr WS + dc
            tc::bar_sync(kBarH2, kTcThreads);
            tc::fence_after_sync();
            stamp(3);
            if (lead) {
                for (int k = iw; k < t3; k += kTcIssuers) {
#pragma unroll
                    for (int t = 0; t < 9; ++t) {
                        const int sh = plin + (t / 3 - 1) * WS + (t % 3 - 1);   // parity and offset of the source
                        const uint64_t ad = (sh & 1) ? a2_desc1 : a2_desc0;
                        tc::mma_f16(tmem + k * N3, tc::desc_advance(ad, cbase + k * 128 + (sh >> 1)),
                                    tc::desc_advance(b3_desc, t * 2 * N3), idesc3, t > 0);
                    }
                    tc::mma_commit(tc::smem_u32(bars + 16 + k));
                }
            }
            __syncwarp();
            stamp(4);
        }
    } else {
        // ============================= compute warps ======================================
        const int q = warp & 3, set = warp >> 2;
        uint32_t ph2 = 0, ph3 = 0;                                 // phase parity per barrier (my tiles)
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        const bool has_b3 = a.b3 != nullptr;
        const int xs_stride = (Rr + 7) * WS;                       // floats per x-strip buffer

        // x strip of unit u: global loads into registers (issued early, consumed after the layer-2
        // epilogue has hidden their latency), then stored into the strip buffer.  Element e of the
        // strip is (row e / WS, slot e % WS); periodic wrap by index.
        constexpr int kXPerThread = 6;                             // (R + 6) WS <= 6 * 256 (checked on the host)
        float xr[kXPerThread];
        auto xload_issue = [&](const Unit& u) {
            const int rows = L0 - u.r0 < Rr ? L0 - u.r0 : Rr;
            const float* xb = a.x + u.b * (long long)L0 * L1;
            const int n = (rows + 6) * WS;
#pragma unroll
            for (int k = 0; k < kXPerThread; ++k) {
                const int e = tid + k * kTcComputeThreads;
                xr[k] = 0.f;
                if (e < n) {
                    const int j = tc_div(e, g.magic_ws), slot = e - j * WS;
                    int r = u.r0 - 3 + j;
                    r += r < 0 ? L0 : 0;                                  // twice: a 2-row lattice wraps twice
                    r += r < 0 ? L0 : 0;
                    r -= r >= L0 ? L0 : 0;
                    r -= r >= L0 ? L0 : 0;
                    int c = slot - 1;
                    c = c < 0 ? c + L1 : c;
                    c = c >= L1 ? c - L1 : c;
                    xr[k] = NFK_LDG(xb + r * L1 + c);
                }
            }
        };
        auto xload_store = [&](const Unit& u, float* xbuf) {
            const int rows = L0 - u.r0 < Rr ? L0 - u.r0 : Rr;
            const int n = (rows + 6) * WS;
#pragma unroll
            for (int k = 0; k < kXPerThread; ++k) {
                const int e = tid + k * kTcComputeThreads;
                if (e < n) xbuf[e] = xr[k];
            }
        };

        // ---- P1: h1 = tanh(conv1(x on the frozen sites)).  An item is a vertical pair of sites
        // (rows 2 jp, 2 jp + 1 of the h1 strip, column c): one of the two is an ACTIVE site -- its
        // 4 cross neighbours carry x, centre and diagonals are masked to zero -- and the other a
        // FROZEN one (centre + 4 diagonals).  The nine inputs are selected by the pair's
        // orientation, so only the 72 non-zero FMAs of the 144 are issued, and lanes walk
        // consecutive columns (conflict-free shared-memory traffic).
        // NI items (it0, it0 + 256, ...) per trip share every weight fetched from shared memory
        auto layer1_items = [&](auto ni_tag, int it0, long long b, int r0, int rows, const float* xbuf) {
            constexpr int NI = decltype(ni_tag)::value;
            float in[NI][9];                                              // by weight tap kh * 3 + kw
            bool up_active[NI];
            int jp[NI], cc[NI];
#pragma unroll
            for (int z = 0; z < NI; ++z) {
                const int it = it0 + z * kTcComputeThreads;
                jp[z] = tc_div(it, g.magic_l1);
                cc[z] = it - jp[z] * L1;
                const float* xw = xbuf + (2 * jp[z]) * WS + cc[z];        // window rows 0..3, slots c..c+2
                // mask bit of the upper site (lattice row r0 - 2 + 2 jp, column c)
                const bool ua = ((1 - g.mask_parity + r0 + cc[z]) & 1) == g.active_val;
                up_active[z] = ua;
                const float x00 = xw[0], x01 = xw[1], x02 = xw[2];
                const float x10 = xw[WS], x11 = xw[WS + 1], x12 = xw[WS + 2];
                const float x20 = xw[2 * WS], x21 = xw[2 * WS + 1], x22 = xw[2 * WS + 2];
                const float x30 = xw[3 * WS], x31 = xw[3 * WS + 1], x32 = xw[3 * WS + 2];
                in[z][1] = ua ? x01 : x11;    // active site: N, W, E, S
                in[z][3] = ua ? x10 : x20;
                in[z][5] = ua ? x12 : x22;
                in[z][7] = ua ? x21 : x31;
                in[z][4] = ua ? x21 : x11;    // frozen site: centre, NW, NE, SW, SE
                in[z][0] = ua ? x10 : x00;
                in[z][2] = ua ? x12 : x02;
                in[z][6] = ua ? x30 : x20;
                in[z][8] = ua ? x32 : x22;
            }
            float acc[NI][2][8];                                          // [item][0 active site / 1 frozen site][co]
            {
                float bv[8];
                load_w8(b1s, bv);
#pragma unroll
                for (int z = 0; z < NI; ++z)
#pragma unroll
                    for (int co = 0; co < 8; ++co) acc[z][0][co] = acc[z][1][co] = bv[co];
            }
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                float wv[8];
                load_w8(w1s + t * 8, wv);
                const int which = (t & 1) ? 0 : 1;                        // odd taps: cross -> active site
#pragma unroll
                for (int co = 0; co < 8; ++co)
#pragma unroll
                    for (int z = 0; z < NI; ++z) acc[z][which][co] = fmaf(in[z][t], wv[co], acc[z][which][co]);
            }
#pragma unroll
            for (int z = 0; z < NI; ++z) {
                uint4 rec[2][2];                                          // [site][hi / lo]
                float vv[2][8];
#pragma unroll
                for (int s = 0; s < 2; ++s) {
#pragma unroll
                    for (int co = 0; co < 8; ++co) vv[s][co] = tanh_from_scaled(acc[z][s][co]);
                    make_records(vv[s], rec[s][0], rec[s][1]);
                }
                const int c = cc[z], i1 = (2 * jp[z]) * WS + c + 1;
#pragma unroll
                for (int s = 0; s < 2; ++s) {                             // s = 0 upper row, 1 lower row
                    if (s == 1 && 2 * jp[z] + 1 >= rows + 4) break;
                    const bool take_active = (s == 0) == up_active[z];
                    uint4 hi, lo;
                    hi.x = take_active ? rec[0][0].x : rec[1][0].x; hi.y = take_active ? rec[0][0].y : rec[1][0].y;
                    hi.z = take_active ? rec[0][0].z : rec[1][0].z; hi.w = take_active ? rec[0][0].w : rec[1][0].w;
                    lo.x = take_active ? rec[0][1].x : rec[1][1].x; lo.y = take_active ? rec[0][1].y : rec[1][1].y;
                    lo.z = take_active ? rec[0][1].z : rec[1][1].z; lo.w = take_active ? rec[0][1].w : rec[1][1].w;
                    uint8_t* dst = h1 + (i1 + s * WS) * 16;
                    *reinterpret_cast<uint4*>(dst) = hi;
                    *reinterpret_cast<uint4*>(dst + g.h1_comp_bytes) = lo;
                    if (c == 0 || c == L1 - 1) {                          // periodic copies: slot L1+1 / slot 0
                        uint8_t* dw = c == 0 ? dst + L1 * 16 : dst - L1 * 16;
                        *reinterpret_cast<uint4*>(dw) = hi;
                        *reinterpret_cast<uint4*>(dw + g.h1_comp_bytes) = lo;
                    }
                    if (SAVE) {   // rows of the strip proper, and the two the next strip takes over (tc_carry)
                        const int j1 = 2 * jp[z] + s;
                        if (j1 >= 2 && r0 - 2 + j1 < L0) {
                            float* dsth = a.save_h1 + (b * 8 * L0 + (r0 - 2 + j1)) * (long long)L1 + c;
#pragma unroll
                            for (int co = 0; co < 8; ++co)
                                dsth[(long long)co * L0 * L1] = take_active ? vv[0][co] : vv[1][co];
                        }
                    }
                }
            }
        };
        auto layer1 = [&](const Unit& u, const float* xbuf) {
            const int r0 = u.r0, rows = L0 - r0 < Rr ? L0 - r0 : Rr;
            const int npair = (rows + 5) >> 1, items = npair * L1;
            int it0 = tid + tc_carry(r0) * L1;                        // first pair: h1 rows 2 carry, 2 carry + 1
            for (; it0 + kTcComputeThreads < items; it0 += 2 * kTcComputeThreads)
                layer1_items(std::integral_constant<int, 2>{}, it0, u.b, r0, rows, xbuf);
            if (it0 < items) layer1_items(std::integral_constant<int, 1>{}, it0, u.b, r0, rows, xbuf);
        };

        // one warp of each tile set polls the MMA barrier; the other three block in hardware
        auto tile_wait = [&](uint64_t* bar, uint32_t parity) {
            if (q == 0) tc::mbar_wait(tc::smem_u32(bar), parity);
            tc::bar_sync(kBarSet0 + set, 128);
            tc::fence_after_sync();
        };

        // ---- E2: accumulators of layer 2 -> h2 records
        auto epilogue2 = [&](const Unit& u) {
            const int rows = L0 - u.r0 < Rr ? L0 - u.r0 : Rr;
            const int c2 = tc_carry(u.r0);
            const int t2 = tc_tiles2(rows, WS, c2);
            float bv[8];
            load_w8(b2s, bv);
            for (int j = set; j < t2; j += kTcSets) {
                tile_wait(bars + j, (ph2 >> j) & 1u);
                ph2 ^= 1u << j;
                float acc[16];
                tc::tmem_ld16(lane_addr + j * 16, acc);
                tc::tmem_ld_wait();
                const int i2 = c2 * WS + j * 128 + q * 32 + lane;
                const int j2 = tc_div(i2, g.magic_ws), slot = i2 - j2 * WS;
                if (j2 < rows + 2 && slot >= 1 && slot <= L1) {
                    float v[8];
#pragma unroll
                    for (int c = 0; c < 8; ++c)
                        v[c] = tanh_from_scaled(fmaf(acc[8 + c], kTwoLog2e / kLoScale, fmaf(acc[c], kTwoLog2e, bv[c])));
                    uint4 hi, lo;
                    make_records(v, hi, lo);
                    uint8_t* dst = h2 + (i2 & 1) * g.h2_par_bytes + (i2 >> 1) * 16;
                    *reinterpret_cast<uint4*>(dst) = hi;
                    *reinterpret_cast<uint4*>(dst + g.h2_comp_bytes) = lo;
                    if (slot == 1 || slot == L1) {            // periodic copies: slot L1+1 / slot 0
                        const int iw = slot == 1 ? i2 + L1 : i2 - L1;
                        uint8_t* dw = h2 + (iw & 1) * g.h2_par_bytes + (iw >> 1) * 16;
                        *reinterpret_cast<uint4*>(dw) = hi;
                        *reinterpret_cast<uint4*>(dw + g.h2_comp_bytes) = lo;
                    }
                    if (SAVE && j2 >= 1 && u.r0 - 1 + j2 < L0) {     // row rows + 1: the next strip's row 1
                        float* dsth = a.save_h2 + (u.b * 8 * L0 + (u.r0 - 1 + j2)) * (long long)L1 + slot - 1;
#pragma unroll
                        for (int c = 0; c < 8; ++c) dsth[(long long)c * L0 * L1] = v[c];
                    }
                }
            }
        };

        // ---- E3: accumulators of layer 3 at the active sites -> transform, y into the x strip
        // `next_cols` = TMEM columns layer 2 of the NEXT unit will overwrite (0: there is none).  A
        // thread releases that unit's layer 2 (arrive on H1) as soon as it has drained every
        // accumulator tile of its own that lives in those columns: layer 2 of the next unit then
        // runs on the tensor core while the rest of this epilogue is still at work.
        auto epilogue3 = [&](const Unit& u, float* xbuf, int next_cols) -> float {
            const int r0 = u.r0, rows = L0 - r0 < Rr ? L0 - r0 : Rr;
            const int t3 = tc_tiles3(rows, WS, L1);
            const int plin = (g.active_val - 1 + g.mask_parity - r0) & 1;
            float lsum = 0.f;
            bool released = next_cols == 0;
            auto release_if_clear = [&](int k_next) {             // k_next: my next tile (or >= t3)
                if (!released && (k_next >= t3 || k_next * N3 >= next_cols)) {
                    tc::fence_before_sync();                      // my TMEM reads so far are done
                    tc::bar_arrive(kBarH1, kTcThreads);
                    released = true;
                }
            };
            release_if_clear(set);
            for (int k = set; k < t3; k += kTcSets) {
                tile_wait(bars + 16 + k, (ph3 >> k) & 1u);
                ph3 ^= 1u << k;
                float prm[P];
#pragma unroll
                for (int grp = 0; grp < Shape::kFull; ++grp) {
                    float v[16];                                  // [8 hi | 8 lo]
                    tc::tmem_ld16(lane_addr + k * N3 + grp * 16, v);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int c = 0; c < 8; ++c) prm[grp * 8 + c] = fmaf(v[8 + c], 1.f / kLoScale, v[c]);
                }
                if constexpr (Shape::kTail > 0) {                 // [kTail hi | kTail lo]
                    constexpr int kT = Shape::kTail;
                    float v[2 * kT <= 8 ? 8 : 16];
                    const uint32_t col = lane_addr + k * N3 + Shape::kFull * 16;
                    if constexpr (2 * kT <= 8) tc::tmem_ld8(col, v);
                    else tc::tmem_ld16(col, v);
                    tc::tmem_ld_wait();
#pragma unroll
                    for (int c = 0; c < kT; ++c) prm[Shape::kFull * 8 + c] = fmaf(v[kT + c], 1.f / kLoScale, v[c]);
                }
                if (has_b3) {
#pragma unroll
                    for (int c = 0; c < P; ++c) prm[c] += b3s[c];
                }
                const int s = 2 * (cbase + k * 128 + q * 32 + lane) + plin;
                const int j2 = tc_div(s, g.magic_ws), slot = s - j2 * WS;
                if (j2 >= 1 && j2 <= rows && slot >= 1 && slot <= L1) {
                    if (SAVE) {
                        float* dsto = a.save_out + (u.b * P * L0 + (r0 + j2 - 1)) * (long long)L1 + slot - 1;
#pragma unroll
                        for (int c = 0; c < P; ++c) dsto[(long long)c * L0 * L1] = prm[c];
                    }
                    float* px = xbuf + (j2 + 2) * WS + slot;
                    const float xv = *px;
                    float out, l;
                    if (KIND == 0) {
                        const float t = prm[0], sc = fabsf(prm[1]);
                        if (!INV) { out = fmaf(xv, fast_ex2(-sc * kInvLn2), t); l = -sc; }
                        else { out = (xv - t) * fast_ex2(sc * kInvLn2); l = sc; }
                    } else {
                        tc_rqs<K, INV, P>(prm, a.cfg, xv, out, l);
                    }
                    *px = out;
                    lsum += l;
                }
                release_if_clear(k + kTcSets);
            }
            return lsum;
        };

        // tc_carry: h1 rows rows + 2, rows + 3 (hi and lo planes) -> rows 2, 3 for the next strip
        auto carry_h1 = [&](int rows) {
            const int n = 2 * WS;
            for (int e = tid; e < 2 * n; e += kTcComputeThreads) {
                const int plane = e >= n, i = e - plane * n;
                uint8_t* dst = h1 + plane * g.h1_comp_bytes + (2 * WS + i) * 16;
                *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(dst + rows * WS * 16);
            }
        };
        // tc_carry: h2 rows rows, rows + 1 -> rows 0, 1 (the shift moves a record to the other parity
        // plane when rows is odd)
        auto carry_h2 = [&](int rows) {
            const int n = 2 * WS;
            for (int e = tid; e < 2 * n; e += kTcComputeThreads) {
                const int plane = e >= n, i = e - plane * n, is = rows * WS + i;
                uint8_t* h2c = h2 + plane * g.h2_comp_bytes;
                *reinterpret_cast<uint4*>(h2c + (i & 1) * g.h2_par_bytes + (i >> 1) * 16) =
                    *reinterpret_cast<const uint4*>(h2c + (is & 1) * g.h2_par_bytes + (is >> 1) * 16);
            }
        };

        // Software pipeline over units: while the tensor core runs layer 3 of unit i, the compute
        // warps already build h1 of unit i+1 (its x strip was prefetched during E2 of unit i).
        Unit cur{blockIdx.x, 0};
        int buf = 0;
        float lacc = 0.f;
        int tn = 0;
        auto stamp = [&](int) {
            if (a.trace && blockIdx.x == 0 && tid == 0 && tn < 4000) a.trace[tn++] = clock64();
        };
        if (cur.b < a.B) {
            xload_issue(cur);
            xload_store(cur, xs);
            tc::bar_sync(kBarCompute, kTcComputeThreads);
            layer1(cur, xs);
            tc::fence_before_sync();
            tc::fence_async_smem();
            tc::bar_arrive(kBarH1, kTcThreads);
        }
        while (cur.b < a.B) {
            const Unit nxt = next_unit(cur);
            const bool has_next = nxt.b < a.B;
            const bool carry = has_next && tc_carry(nxt.r0) > 0;
            const int rows = L0 - cur.r0 < Rr ? L0 - cur.r0 : Rr;
            float* xcur = xs + buf * xs_stride;
            float* xnext = xs + (buf ^ 1) * xs_stride;
            stamp(0);
            if (has_next) xload_issue(nxt);                           // in flight while E2 runs
            epilogue2(cur);
            stamp(1);
            tc::fence_before_sync();
            tc::fence_async_smem();
            tc::bar_arrive(kBarH2, kTcThreads);                       // layer 3 of `cur` may start
            if (has_next) xload_store(nxt, xnext);
            tc::bar_sync(kBarCompute, kTcComputeThreads);             // x of `nxt` visible; every layer-2 tile of `cur` consumed
            stamp(2);
            int next_cols = 0;
            if (carry) {
                carry_h1(rows);
                tc::bar_sync(kBarCompute, kTcComputeThreads);         // before layer 1 of `nxt` overwrites the source rows
            }
            if (has_next) {
                layer1(nxt, xnext);                                   // overlaps layer 3 of `cur` on the tensor core
                tc::fence_async_smem();                               // h1 of `nxt` visible to the tensor core
                const int nrows = L0 - nxt.r0 < Rr ? L0 - nxt.r0 : Rr;
                next_cols = 16 * tc_tiles2(nrows, WS, tc_carry(nxt.r0));
            }
            stamp(3);
            lacc += epilogue3(cur, xcur, next_cols);                  // releases layer 2 of `nxt` on the way
            stamp(4);
            tc::bar_sync(kBarCompute, kTcComputeThreads);             // y of the strip complete in xcur
            if (carry) carry_h2(rows);                               // every layer-3 MMA of `cur` has completed
            {   // the strip's rows (active: transformed, frozen: copied) -> y, one warp per row
                float* yb = a.y + cur.b * (long long)L0 * L1;
                for (int j = warp; j < rows; j += kTcComputeWarps) {
                    const float* src = xcur + (j + 3) * WS + 1;
                    float* dst = yb + (cur.r0 + j) * L1;
                    for (int col = lane; col < L1; col += 32) dst[col] = src[col];
                }
            }
            if (cur.r0 + Rr >= L0) {      // last strip of the sample: log|det J| (fixed reduction tree)
                lacc = warp_sum(lacc);
                if (lane == 0) red[warp] = lacc;
                tc::bar_sync(kBarCompute, kTcComputeThreads);
                if (tid == 0 && a.log_out) {
                    float tot = 0.f;
#pragma unroll
                    for (int w = 0; w < kTcComputeWarps; ++w) tot += red[w];
                    a.log_out[cur.b] = (a.log_in ? a.log_in[cur.b] : 0.f) + tot;
                }
                lacc = 0.f;
            }
            tc::bar_sync(kBarCompute, kTcComputeThreads);             // xcur (and `red`) free for reuse
            stamp(5);
            cur = nxt;
            buf ^= 1;
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == kTcComputeWarps) tc::tmem_dealloc(tmem, kTcTmemCols);
}

template <int KIND, int K, int INV, bool SAVE>
int tc_launch(TcArgs a, cudaStream_t st) {
    constexpr int P = KIND == 0 ? 2 : 3 * K - 2;
    // every GPU of a B200 box is the same part: queried once (thread-safe static initialisation)
    struct Props { int sm_count, max_smem; };
    static const Props props = [] {
        Props p{0, 0};
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&p.sm_count, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&p.max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (p.sm_count <= 0) p.sm_count = 148;
        return p;
    }();
    const int sm_count = props.sm_count, max_smem = props.max_smem;
    // two CTAs per SM: each may use half of the SM's shared memory (minus the 1 KB system slice)
    const uint32_t budget = (uint32_t)((max_smem > 0 ? max_smem : 227 * 1024) + 1024) / 2 - 1024;
    int best = 0;
    float best_cost = 1e30f;
    TcGeom g = a.g;
    for (int R = 2; R <= a.g.L0; ++R) {
        if (!tc_plan<P>(g, R, budget)) continue;
        const float c = tc_cost_per_row<P>(g.L0, g.L1, g.WS, R);
        if (c < best_cost) { best_cost = c; best = R; }
    }
    if (const char* e = getenv("NFK_TC_R")) {             // tuning override of the strip height
        const int r = atoi(e);
        TcGeom t = a.g;
        if (r >= 2 && r <= a.g.L0 && tc_plan<P>(t, r, budget)) best = r;
    }
    if (best == 0) return NFK_EUNSUPPORTED;
    tc_plan<P>(a.g, best, budget);
    a.g.magic_ws = (uint32_t)((0x100000000ULL + a.g.WS - 1) / a.g.WS);
    a.g.magic_l1 = (uint32_t)((0x100000000ULL + a.g.L1 - 1) / a.g.L1);
    if (ensure_dynamic_smem<fused2d_tc_kernel<KIND, K, INV, SAVE>>((int)budget) != NFK_OK) return NFK_ECUDA;
    long long grid = 2LL * sm_count;
    if (grid > a.B) grid = a.B;
    fused2d_tc_kernel<KIND, K, INV, SAVE><<<(unsigned)grid, kTcThreads, a.g.smem_bytes, st>>>(a);
    return check_launch();
}

template <int KIND, int K>
int tc_launch_dir(const TcArgs& a, int inverse, cudaStream_t st) {
    if (a.save_out) return inverse ? NFK_EINVAL : tc_launch<KIND, K, 0, true>(a, st);
    return inverse ? tc_launch<KIND, K, 1, false>(a, st) : tc_launch<KIND, K, 0, false>(a, st);
}

}  // namespace

namespace nfk {

// Tensor-core fused step; NFK_EUNSUPPORTED when the geometry / knot count is outside what
// this kernel covers (the caller then runs the CUDA-core kernel of nfk_fused.cu).
int fused2d_tc_step(const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                    const float* w3, const float* b3, int kind, const nfk_rqs_params& prm, int mask_parity,
                    int parity, int inverse, const float* log_in, float* y, float* log_out, int L0, int L1,
                    int64_t B, cudaStream_t st, float* save_h1, float* save_h2, float* save_out) {
    if ((L0 & 1) || (L1 & 1) || L1 < 2 || L0 < 2) return NFK_EUNSUPPORTED;   // checkerboard must wrap consistently
    if ((save_h1 || save_h2 || save_out) && !(save_h1 && save_h2 && save_out)) return NFK_EINVAL;
    TcArgs a;
    a.x = x; a.w1 = w1; a.b1 = b1; a.w2 = w2; a.b2 = b2; a.w3 = w3; a.b3 = b3;
    a.log_in = log_in; a.y = y; a.log_out = log_out; a.B = B;
    a.trace = g_trace;
    a.save_h1 = save_h1; a.save_h2 = save_h2; a.save_out = save_out;
    a.g = TcGeom{};
    a.g.L0 = L0; a.g.L1 = L1; a.g.WS = L1 + 3;
    a.g.mask_parity = mask_parity; a.g.active_val = parity == 0 ? 1 : 0;
    a.cfg = RqsCfg{0.f, 1.f, 0.f, 1.f, 0, 0};
    if (kind == 0) return tc_launch_dir<0, 2>(a, inverse, st);
    a.cfg = RqsCfg{prm.xlim0, prm.xlim1 - prm.xlim0, prm.ylim0, prm.ylim1 - prm.ylim0, prm.extrap_left,
                   prm.extrap_right};
    switch (prm.n_knots) {
        case 4: return tc_launch_dir<1, 4>(a, inverse, st);
        case 5: return tc_launch_dir<1, 5>(a, inverse, st);
        case 6: return tc_launch_dir<1, 6>(a, inverse, st);
        case 8: return tc_launch_dir<1, 8>(a, inverse, st);
        case 10: return tc_launch_dir<1, 10>(a, inverse, st);
        default: return NFK_EUNSUPPORTED;
    }
}

}  // namespace nfk

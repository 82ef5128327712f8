// nfk_fused_tc.cuh -- the fused 2-D coupling step with its conditioner on the tensor cores.
//
// Same operator as nfk_fused.cuh (Coupling_.forward step k, couplings_.py:56-64, with the
// ConvAct(1 -> 8 -> 8 -> P) conditioner of modules.py:131-145 and the affine / RQ-spline
// transform of couplings_.py:123-139, 178-262), but layers 2 and 3 of the conditioner run as
// implicit GEMMs on tcgen05:
//
//   * operands are fp16 PAIRS: every activation / weight v is carried as v = hi + lo with
//     hi = fp16(v), lo = fp16(v - hi) (weights: lo scaled by 2^11 to stay normal).  One
//     kind::f16 MMA has K = 16 = [8 channels of hi | 8 channels of lo] of the activations
//     against [w_hi ; w_hi] in accumulator columns [0, N) and [w_lo ; w_lo] in columns
//     [N, 2N) (layer 3 interleaves the two per group of 8 channels, TcShape):
//     acc = (a_hi + a_lo) w_hi + 2^-11 (a_hi + a_lo) w_lo' -- 22 significant bits
//     per factor, fp32 accumulation in TMEM.  The 1e-5 parity contract rules out plain
//     fp16 / bf16 / tf32 (SURVEY 7, hard part 1); this split costs ONE MMA per tap.
//   * a strip of the lattice lives in shared memory as 16-byte records (one site = 8 fp16
//     channels) in LINEAR order with an odd row stride WS = L1 + 3 (slot 0 / L1+1 hold the
//     periodic wrap copies), so (i) an M = 128 tile of consecutive records is a valid
//     K-major no-swizzle UMMA operand and a conv tap is a shifted start address, and (ii) the
//     checkerboard parity of a site is the parity of its linear index: layer 3 runs on the
//     ACTIVE sites only, from parity-split copies of h2 (index >> 1 within a parity plane).
//   * one MMA warp issues; eight compute warps run layer 1 (CUDA cores), the TMEM epilogues
//     (bias, tanh, fp16 split; spline) and the field I/O.  MMAs of a strip overlap with the
//     epilogue of earlier tiles, and two CTAs per SM overlap each other's phases.
//
// Measured basis (scratch/tc_probe.cu on a B200): an M=128 kind::f16/tf32 MMA costs ~41
// cycles for any N <= 32 (A-operand read bound), 50 at N = 64; the shifted-start layout and
// the split reproduce fp64 to 4e-7 of sum|terms|.
#pragma once

#include <cuda_fp16.h>

#include "nfk_fused.cuh"
#include "nfk_tc.cuh"

namespace nfk {

#ifndef NFK_TC_COMPUTE_WARPS
#define NFK_TC_COMPUTE_WARPS 8
#endif
constexpr int kTcComputeWarps = NFK_TC_COMPUTE_WARPS;          // multiple of 4 (one warp per TMEM lane quarter)
constexpr int kTcSets = kTcComputeWarps / 4;                   // tile sets working in parallel
constexpr int kTcComputeThreads = 32 * kTcComputeWarps;
#ifndef NFK_TC_ISSUERS
#define NFK_TC_ISSUERS 1
#endif
// MMA-issuing warps (the last ones; one elected thread each, M tiles dealt round robin).  Measured at the BASELINE
// geometry (B = 16384, 64 x 64, K = 10): 1 issuer 2.834 ms, 2 issuers 2.884 ms, 3 issuers 3.64 ms (register cap):
// this kernel is bound by the shared-memory data pipe (MMA operand reads + TMEM / LDS / STS traffic, 79 % busy),
// not by the issuing thread -- unlike the N-D kernels (nfk_convnd_tc.cu), whose single issuer was the bottleneck.
constexpr int kTcIssuers = NFK_TC_ISSUERS;
constexpr int kTcThreads = kTcComputeThreads + 32 * kTcIssuers;
constexpr int kTcTmemCols = 256;            // per CTA: two CTAs share the SM's 512 columns
constexpr int kTcGuard = 8;                 // 16-byte records of slack in front of every plane
constexpr float kLoScale = 2048.f;          // weights' lo part is stored times 2^11

enum { kBarCompute = 1, kBarH1 = 2, kBarH2 = 3, kBarSet0 = 4 };   // kBarSet0 + {0, 1}: the two tile sets

// launch geometry (host-computed, passed by value)
struct TcGeom {
    int L0, L1, WS;              // lattice rows, columns, WS = L1 + 3 (odd)
    int R;                       // output rows per strip
    int mask_parity, active_val;
    // shared-memory map (byte offsets from the dynamic shared-memory base; 16-byte alignment suffices)
    uint32_t off_xs, off_h1, off_h2, off_b2, off_b3, off_w1, off_bar;
    uint32_t h1_comp_bytes;      // hi plane -> lo plane of h1
    uint32_t h2_comp_bytes;      // hi plane -> lo plane of h2 (within a parity)
    uint32_t h2_par_bytes;       // parity 0 -> parity 1
    uint32_t smem_bytes;
    uint32_t magic_ws, magic_l1; // ceil(2^32 / WS), ceil(2^32 / L1): exact n / d for n d < 2^32
};

__device__ __forceinline__ int tc_div(int n, uint32_t magic) { return (int)__umulhi((uint32_t)n, magic); }

NFK_HD int tc_div_up(int a, int b) { return (a + b - 1) / b; }
// A strip that continues a sample (r0 > 0) takes over from the previous strip of that sample the
// rows both need: h2 rows 0, 1 and h1 rows 2, 3 (h1 rows 0, 1 are then read by no output).  Its
// layer 2 starts at h2 row `carry` and its layer 1 at h1 row 2 `carry`.
NFK_HD int tc_carry(int r0) { return r0 > 0 ? 2 : 0; }
// tiles of layer 2 / layer 3 for a strip with `rows` output rows
NFK_HD int tc_tiles2(int rows, int WS, int carry) { return tc_div_up((rows + 2 - carry) * WS, 128); }
NFK_HD int tc_cbase(int WS) { return (WS + 1) >> 1; }
NFK_HD int tc_tiles3(int rows, int WS, int L1) {
    // linear indices of the output sites in the h2 strip: rows 1..rows, slots 1..L1
    const int s_max = rows * WS + L1;
    return tc_div_up((s_max >> 1) - tc_cbase(WS) + 1, 128);
}

// Layer-3 accumulator columns, packed by groups of 8 output channels: group g holds
// [hi of its gs channels | lo of the same], gs = min(8, P - 8 g), at columns 16 g ... 16 g + 2 gs.
// One 16-column TMEM load (8 for a tail of <= 4 channels) then carries both halves of its
// channels: the epilogue loads 2P columns rounded up to 8, not 2 x (P rounded up to 16).
template <int P>
struct TcShape {
    static constexpr int kFull = P / 8, kTail = P % 8;      // full groups, channels of the last group
    static constexpr int kCols = 16 * kFull + 2 * kTail;    // accumulator columns in use
    static constexpr int N3 = (kCols + 15) / 16 * 16;       // the MMA's N (multiple of 16 at M = 128)
};

// Fills the geometry for a given R; returns false when it does not fit one CTA's budget.
template <int P>
inline bool tc_plan(TcGeom& g, int R, uint32_t smem_budget) {
    const int WS = g.WS;
    g.R = R;
    const int t2 = tc_tiles2(R, WS, 0), t3 = tc_tiles3(R, WS, g.L1);
    if (t2 > 16 || t2 * 16 > kTcTmemCols || t3 > 8 || t3 * TcShape<P>::N3 > kTcTmemCols) return false;
    if ((R + 6) * WS > 6 * kTcComputeThreads) return false;                 // x strip staged in 6 registers per thread
    auto align = [](uint32_t v) { return (v + 127u) & ~127u; };
    uint32_t off = 0;
    g.off_xs = off; off = align(off + 2u * (uint32_t)(R + 7) * WS * 4); // two strips (+ 1 row: P1 pairs may peek past the end)
    const int e2 = t2 * 128 > 2 * WS + tc_tiles2(R, WS, 2) * 128 ? t2 * 128 : 2 * WS + tc_tiles2(R, WS, 2) * 128;
    const int n1 = e2 + 2 * WS + 2;                                         // records an M2 tile may touch
    g.h1_comp_bytes = align((uint32_t)(kTcGuard + n1) * 16);
    g.off_h1 = off; off += 2 * g.h1_comp_bytes;
    int n2 = tc_cbase(WS) + t3 * 128 + (WS + 1) / 2 + 2;                    // per parity plane
    const int n2_min = ((R + 2) * WS + 1) / 2 + 1;
    if (n2 < n2_min) n2 = n2_min;
    g.h2_comp_bytes = align((uint32_t)(kTcGuard + n2) * 16);
    g.h2_par_bytes = 2 * g.h2_comp_bytes + 64;          // odd multiple of 64: the two parities hit different banks
    g.off_h2 = off; off += 2 * g.h2_par_bytes;
    g.off_b2 = off; off = align(off + 9 * 2 * 16 * 16);
    g.off_b3 = off; off = align(off + 9 * 2 * TcShape<P>::N3 * 16);
    g.off_w1 = off; off = align(off + (72 + 8 + 8 + P) * 4);
    g.off_bar = off; off = align(off + 24 * 8 + 64);
    g.smem_bytes = off;
    return g.smem_bytes <= smem_budget;
}

// MMA + epilogue cost model of a strip height (cycles per lattice row, measured MMA costs):
// used on the host to pick R
template <int P>
inline float tc_cost_per_row(int L0, int L1, int WS, int R) {
    const float c2 = 9 * 41.f, c3 = 9 * (TcShape<P>::N3 <= 32 ? 42.f : TcShape<P>::N3 <= 64 ? 50.f : 66.f);
    float total = 0.f;
    for (int r0 = 0; r0 < L0; r0 += R) {
        const int rows = L0 - r0 < R ? L0 - r0 : R;
        total += tc_tiles2(rows, WS, tc_carry(r0)) * c2 + tc_tiles3(rows, WS, L1) * c3 + 600.f;   // + per-strip sync overhead
    }
    return total / L0;
}

// fp16 pair of a float: hi = v truncated to 11 significant bits (exact in fp16 for normal fp16
// magnitudes), lo = v - hi (13 bits, of which fp16 keeps 11: 22 bits in all).
__device__ __forceinline__ float tc_split(float v, float& lo) {
    const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    lo = v - hi;
    return hi;
}
__device__ __forceinline__ uint32_t tc_pack(float a, float b) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));      // low half = a
    return r;
}

// ---- fast scalar maths (MUFU based, 1-2 ulp): what the epilogues run per site
__device__ __forceinline__ float fast_ex2(float v) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float fast_lg2(float v) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float fast_rcp(float v) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
constexpr float kTwoLog2e = 2.88539008177792681f;      // 2 log2(e)
// tanh(u) from a = 2 log2(e) u:  1 - 2 / (2^a + 1)   (abs error ~1e-7; saturates cleanly)
__device__ __forceinline__ float tanh_from_scaled(float a) {
    return fmaf(-2.f, fast_rcp(fast_ex2(a) + 1.f), 1.f);
}
// log2(1 + 2^z), the softplus with beta = ln 2 (couplings_.py:173-176; identity above z ln2 > 20)
__device__ __forceinline__ float fast_softplus_ln2(float z) {
    const float e = fast_ex2(z);
    const float r = e < 2.44140625e-4f ? e * (kInvLn2 - 0.5f * kInvLn2 * e) : fast_lg2(1.f + e);   // log1p series below 2^-12
    return z * kLn2 > 20.f ? z : r;
}

// Rational-quadratic coupling spline at one site from the raw conditioner channels p[0..3K-2)
// held in registers (same maths as rqs_site_forward / rqs_site_inverse in nfk_math.cuh --
// couplings_.py:211-262, spline.py:154-287 -- arranged for registers: the bin is found by
// comparing UNNORMALISED prefix sums, and every run-time index becomes a select chain).
template <int K, int INV, int NPR>
__device__ __forceinline__ void tc_rqs(const float (&p)[NPR], const RqsCfg& cfg, float v, float& out, float& l) {
    constexpr float kL2e = 1.44269504088896341f;
    float mx = p[0], my = p[K - 1];
#pragma unroll
    for (int c = 1; c < K - 1; ++c) {
        mx = fmaxf(mx, p[c]);
        my = fmaxf(my, p[K - 1 + c]);
    }
    mx *= -kL2e;
    my *= -kL2e;
    float rx[K - 1], ry[K - 1];          // running sums of the unnormalised softmax terms
    float sx = 0.f, sy = 0.f;
#pragma unroll
    for (int c = 0; c < K - 1; ++c) {
        sx += fast_ex2(fmaf(p[c], kL2e, mx));
        sy += fast_ex2(fmaf(p[K - 1 + c], kL2e, my));
        rx[c] = sx;
        ry[c] = sy;
    }
    const float lo = INV ? cfg.ylim0 : cfg.xlim0, wd = INV ? cfg.yw : cfg.xw;
    if (cfg.left == kExtrapLinear && v <= lo) {                 // spline.py:466-470
        const float D = fast_softplus_ln2(p[2 * K - 2]);
        if (!INV) { out = cfg.ylim0 + D * (v - cfg.xlim0); l = logf(D); }
        else { out = cfg.xlim0 + __fdividef(v - cfg.ylim0, D); l = -logf(D); }
        return;
    }
    if (cfg.right == kExtrapLinear && v > lo + wd) {            // spline.py:476-478
        const float D = fast_softplus_ln2(p[3 * K - 3]);
        if (!INV) { out = (cfg.ylim0 + cfg.yw) + D * (v - (cfg.xlim0 + cfg.xw)); l = logf(D); }
        else { out = (cfg.xlim0 + cfg.xw) + __fdividef(v - (cfg.ylim0 + cfg.yw), D); l = -logf(D); }
        return;
    }
    // segment j = number of interior knots strictly below v (searchsorted right=False + clamp):
    // knot c+1 = lo + r[c] wd / s  <  v   <=>   r[c] < (v - lo) s / wd
    const float ss = INV ? sy : sx;
    const float t = (v - lo) * ss * fast_rcp(wd);
    float cx = 0.f, cy = 0.f;                                   // prefix sums below the segment
    float pw = p[0], ph = p[K - 1];                             // raw width / height channel of the segment
    float d0 = p[2 * K - 2], d1 = p[2 * K - 1];
#pragma unroll
    for (int c = 0; c < K - 2; ++c) {
        const bool below = (INV ? ry[c] : rx[c]) < t;
        cx = below ? rx[c] : cx;
        cy = below ? ry[c] : cy;
        pw = below ? p[c + 1] : pw;
        ph = below ? p[K + c] : ph;
        d0 = below ? p[2 * K - 1 + c] : d0;
        d1 = below ? p[2 * K + c] : d1;
    }
    // the segment's own softmax terms, re-evaluated (a difference of prefix sums would lose
    // the low bits of a narrow bin)
    const float qx = cfg.xw * fast_rcp(sx), qy = cfg.yw * fast_rcp(sy);
    const float X0 = fmaf(cx, qx, cfg.xlim0), w = fast_ex2(fmaf(pw, kL2e, mx)) * qx;
    const float Y0 = fmaf(cy, qy, cfg.ylim0), h = fast_ex2(fmaf(ph, kL2e, my)) * qy;
    const float D0 = fast_softplus_ln2(d0), D1 = fast_softplus_ln2(d1);
    const float rw = fast_rcp(w);
    const float m = h * rw;
    const float sig = D0 + D1 - 2.f * m;
    float th;
    if (!INV) {
        th = (v - X0) * rw;
    } else {                                                    // stable root, cf. rq_theta_from_eta
        const float eta = __fdividef(v - Y0, h);
        const float a2 = fmaf(-sig, eta, D0 - m);
        const float a1 = -a2 - m;
        const float a0 = m * eta;
        const float disc = fmaxf(fmaf(a1, a1, -4.f * a0 * a2), 0.f);
        th = __fdividef(2.f * a0, sqrtf(disc) - a1);
    }
    const float om = 1.f - th, tom = th * om;
    const float den = fmaf(sig, tom, m);
    const float rden = fast_rcp(den);
    const float Q = fmaf(D1 * th, th, fmaf(2.f * m, tom, D0 * om * om));
    // logf, not lg2.approx: log g is close to 0 at most sites and the approximation's ABSOLUTE error
    // was measured to double the error of the per-sample log|det J| sum
    const float lg = logf(m * m * Q * rden * rden);
    if (!INV) {
        out = fmaf(h * fmaf(m * th, th, D0 * tom), rden, Y0);
        l = lg;
    } else {
        out = fmaf(w, th, X0);
        l = -lg;
    }
}

}  // namespace nfk

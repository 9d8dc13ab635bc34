// Device kernels of libame (sm_100a).  See DESIGN.md for the data layout and the per-kernel rooflines.
//
// Time parallelism: every 30 s chunk of the reference restarts all filter state from zero
// (audio_mastering_engine.py:185-199), and inside a chunk the filters are stable LTI systems, so a
// tile of T frames is computed by ONE lane pair (L lane, R lane) that first runs `warm` frames of the
// preceding audio from zero state.  `warm` is chosen on the host so that the state error has decayed
// below 1e-13 of the signal level (FP64 rounding level) when the tile proper starts; the first tile
// of a chunk needs no warm-up and is exact by construction.
//
// All 32 lanes of a warp run the SAME number of 4-frame groups (the warp maximum), so every shuffle is a
// plain full-mask SHFL; lanes past their own range keep computing on stale input and simply do not store.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "ame_layout.h"

namespace ame {

constexpr unsigned kFull = 0xffffffffu;

__constant__ double c_hist_bounds[1001];
__constant__ double c_hist_energy[1000];

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg16(const uint4 *p) { return __ldg(p); }

__device__ __forceinline__ double bq_step(const ame_biquad &c, double &z0, double &z1, double x) {
    // DF-II transposed, the form scipy evaluates (lfilter / sosfilt) - FMA-contracted.
    double y = fma(c.b0, x, z0);
    z0 = fma(-c.a1, y, fma(c.b1, x, z1));
    z1 = fma(-c.a2, y, c.b2 * x);
    return y;
}

// exact int16 -> double without the conversion pipe: 2^52 + 2^31 + x as raw bits, minus the bias
__device__ __forceinline__ double i16_to_f64(int x) {
    return __hiloint2double(0x43300000, (int)(0x80000000u ^ (unsigned)x)) - 4503601774854144.0;
}

// np.clip(x,-1,1) * 32767 -> astype(int16)  (truncate toward zero), float64 flavour
// (clip first or clamp the truncated product: same integer - the product is monotone in v, +-32767 are exact, and
// cvt.rzi saturates; the integer clamp avoids two DSETP-based double min/max)
__device__ __forceinline__ int to_pcm_f64(double v) {
    return min(max(__double2int_rz(__dmul_rn(v, 32767.0)), -32767), 32767);
}
__device__ __forceinline__ int to_pcm_f32(float v) {
    v = fminf(fmaxf(v, -1.0f), 1.0f);
    return __float2int_rz(__fmul_rn(v, 32767.0f));
}
__device__ __forceinline__ int sat16(int v) { return v > 32767 ? 32767 : (v < -32768 ? -32768 : v); }
__device__ __forceinline__ uint32_t pack16(int lo, int hi) { return (uint32_t)(uint16_t)lo | ((uint32_t)(uint16_t)hi << 16); }

// Butterworth second-order section, numerator b0 * (1 + 2S z^-1 + z^-2) with S = +1 (zeros at z = -1:
// low-pass type) or S = -1 (zeros at z = +1: high-pass type), a0 = 1.  Every section scipy.signal.butter
// returns for the reference's shelves / band-passes / crossovers has this shape (validated on the host),
// which saves two coefficient registers per section.  DF-II transposed as scipy evaluates it:
//   y = b0 x + z0 ; z0 = (z1 + b1 x) - a1 y ; z1 = b2 x - a2 y        with b1 x = 2S (b0 x) exactly.
template <int S, typename F>
__device__ __forceinline__ F bw_step(F b0, F a1, F a2, F &z0, F &z1, F x) {
    const F y = fma(b0, x, z0);
    const F t = b0 * x;
    z0 = fma(-a1, y, fma((F)(2.0 * S), t, z1));
    z1 = fma(-a2, y, t);
    return y;
}
template <int S, typename F>   // b0 == 1
__device__ __forceinline__ F bw_step1(F a1, F a2, F &z0, F &z1, F x) {
    const F y = x + z0;
    z0 = fma(-a1, y, fma((F)(2.0 * S), x, z1));
    z1 = fma(-a2, y, x);
    return y;
}

// apply_shelf_filter with a negative gain (:289): samples * g + (y - samples * g), i.e. y up to one rounding.  When the
// stage is the first active one its input is still the float32 channel, and numpy evaluates samples * g in float32
// (a Python float does not widen a float32 array); later stages see float64.  No FMA contraction.
template <bool FIRST>
__device__ __forceinline__ double shelf_cut(double v, double f, double g) {
    const double t = FIRST ? (double)__fmul_rn((float)v, (float)g) : __dmul_rn(v, g);
    return __dadd_rn(t, __dsub_rn(f, t));
}
template <bool FIRST>
__device__ __forceinline__ float shelf_cut(float v, float f, float g) {          // the FP32 experiment (precision = 1)
    const float t = __fmul_rn(v, g);
    return __fadd_rn(t, __fsub_rn(f, t));
}

template <typename F>
struct PeakCoef { F b0, a1[4], a2[4]; };          // butter(4, bandpass, sos): signs (+,+,-,-), sections 1..3 unit gain
template <typename F>
__device__ __forceinline__ void load_peak(PeakCoef<F> &c, const ame_eq_stage &st) {
    c.b0 = (F)st.s[0].b0;
#pragma unroll
    for (int i = 0; i < 4; ++i) { c.a1[i] = (F)st.s[i].a1; c.a2[i] = (F)st.s[i].a2; }
}
template <typename F>
__device__ __forceinline__ F peak_step(const PeakCoef<F> &c, F *z, F x) {
    F t = bw_step<1, F>(c.b0, c.a1[0], c.a2[0], z[0], z[1], x);
    t = bw_step1<1, F>(c.a1[1], c.a2[1], z[2], z[3], t);
    t = bw_step1<-1, F>(c.a1[2], c.a2[2], z[4], z[5], t);
    return bw_step1<-1, F>(c.a1[3], c.a2[3], z[6], z[7], t);
}

// exact int16 -> x / 32768 as double in ONE add: bits of 2^37 + (x + 2^31) * 2^-15, minus 2^37 + 2^16
__device__ __forceinline__ double i16_to_unit(int x) {
    return __hiloint2double(0x42400000, (int)(0x80000000u ^ (unsigned)x)) - 137439019008.0;
}

// ------------------------------------------------------------------------------------------------
// k_eq: int16 in -> [warmth -> int16] -> float32 -> 4-stage EQ in FP64 -> float32 -> [width] -> int16
// ONE THREAD per tile, both channels: the L and R cascades are two independent dependency chains in one
// instruction stream (the kernel is bound by FP64 latency, not by registers), and the cross-channel
// stages (warmth, width, packing) need no shuffles.  MASK = active EQ stages, WARM = warmth on.
// F = double is the product (what scipy computes, :272-298); F = float is the precision experiment of DESIGN.md
// (ame_plan_options.precision = 1): the same cascade with float32 coefficients and state.
// ------------------------------------------------------------------------------------------------
// SKEW (experiment, not instantiated in the product): the four stages work on four consecutive frames at once - stage
// s on frame i - s, handing its output to stage s + 1 through a register - so that one iteration holds 8 independent
// dependency chains instead of 2.  Same bytes out; measured 11.00 ms against 11.07 ms for the plain order on the
// 128-track launch (profiles/r02/summary.md): the compiler's schedule of the plain loop already overlaps the stages.
template <int MASK, bool WARM, typename F, bool SKEW>
__device__ __forceinline__ void eq_tile(const TileJob &job, const ame_track_params *__restrict__ tp,
                                        const double *__restrict__ luts, const int16_t *__restrict__ in,
                                        int16_t *__restrict__ pre) {
    const bool widen = (tp->flags & AME_F_WIDTH) != 0;
    const float wfac = tp->width;
    const double *lut = WARM ? luts + (size_t)tp->warm_lut * 65536 + 32768 : nullptr;
    double wl_b0 = 0, wl_b1 = 0, wl_a1 = 0, wl_gm1 = 0, wh_b0 = 0, wh_b1 = 0, wh_a1 = 0, wh_gm1 = 0;
    if (WARM) {
        wl_b0 = tp->wl_b0; wl_b1 = tp->wl_b1; wl_a1 = tp->wl_a1; wl_gm1 = tp->wl_gm1;
        wh_b0 = tp->wh_b0; wh_b1 = tp->wh_b1; wh_a1 = tp->wh_a1; wh_gm1 = tp->wh_gm1;
    }
    F s0_b0 = 0, s0_a1 = 0, s0_a2 = 0, g0 = 0, gm0 = 0, s3_b0 = 0, s3_a1 = 0, s3_a2 = 0, g3 = 0, gm3 = 0, gm1 = 0, gm2 = 0;
    bool boost0 = false, boost3 = false;
    PeakCoef<F> p1, p2;
    if (MASK & 1) {
        s0_b0 = (F)tp->eq[0].s[0].b0; s0_a1 = (F)tp->eq[0].s[0].a1; s0_a2 = (F)tp->eq[0].s[0].a2;
        g0 = (F)tp->eq[0].g; gm0 = (F)tp->eq[0].gm1; boost0 = tp->eq[0].kind == AME_EQ_SHELF_BOOST;
    }
    if (MASK & 2) { load_peak(p1, tp->eq[1]); gm1 = (F)tp->eq[1].gm1; }
    if (MASK & 4) { load_peak(p2, tp->eq[2]); gm2 = (F)tp->eq[2].gm1; }
    if (MASK & 8) {
        s3_b0 = (F)tp->eq[3].s[0].b0; s3_a1 = (F)tp->eq[3].s[0].a1; s3_a2 = (F)tp->eq[3].s[0].a2;
        g3 = (F)tp->eq[3].g; gm3 = (F)tp->eq[3].gm1; boost3 = tp->eq[3].kind == AME_EQ_SHELF_BOOST;
    }
    F zl[20], zr[20];
#pragma unroll
    for (int i = 0; i < 20; ++i) { zl[i] = 0; zr[i] = 0; }

    const int64_t warm = (MASK != 0) ? (int64_t)tp->warm_eq : 0;
    int64_t f_lo = job.tile_begin - warm;
    if (f_lo < job.chunk_begin) f_lo = job.chunk_begin;
    const int64_t f_hi = job.tile_end;
    if (f_hi <= f_lo) return;
    const int64_t g0f = f_lo & ~(int64_t)3;               // first 4-aligned group
    const int n_it = (int)((f_hi - g0f + 3) >> 2);

    auto st0 = [&](F v, F *z) -> F {   // apply_shelf_filter 250 Hz low (:283-289)
        if (MASK & 1) {
            const F f = bw_step<1, F>(s0_b0, s0_a1, s0_a2, z[0], z[1], v);
            v = boost0 ? v + (f - v) * gm0 : shelf_cut<true>(v, f, g0);
        }
        return v;
    };
    auto st1 = [&](F v, F *z) -> F { return (MASK & 2) ? v + peak_step(p1, z + 2, v) * gm1 : v; };    // apply_peak_filter 1 kHz (:290-298)
    auto st2 = [&](F v, F *z) -> F { return (MASK & 4) ? v + peak_step(p2, z + 10, v) * gm2 : v; };   // apply_peak_filter 4 kHz
    auto st3 = [&](F v, F *z) -> F {   // apply_shelf_filter 8 kHz high
        if (MASK & 8) {
            const F f = bw_step<-1, F>(s3_b0, s3_a1, s3_a2, z[18], z[19], v);
            v = boost3 ? v + (f - v) * gm3 : shelf_cut<(MASK & 7) == 0>(v, f, g3);
        }
        return v;
    };
    auto cascade = [&](F v, F *z) -> float {               // one channel through the 4 EQ stages
        return (float)st3(st2(st1(st0(v, z), z), z), z);   // samples[:, i] = ... into the float32 array (:274), round to nearest
    };
    F q0l = 0, q0r = 0, q1l = 0, q1r = 0, q2l = 0, q2r = 0, q3l = 0, q3r = 0;     // SKEW: stage outputs of the last four frames

    // one frame -> packed (L | R << 16) int16 output.  lutL / lutR = tanh table values (fetched a group ahead).
    auto frame = [&](uint32_t w, double lutL, double lutR) -> uint32_t {
        int xl = (int)(int16_t)(w & 0xffffu), xr = (int)(int16_t)(w >> 16);
        if (WARM) {
            // apply_analog_character (:258-266): tanh in float32 (table = the host's own np.tanh, widened
            // exactly to double), then two order-2 "shelves" that lfilter(axis=-1) runs ACROSS the channels:
            //   y0 = b0*L ; y1 = (b1*L - a1*y0) + b0*R ; blend x + (y - x)*(g - 1)       (no FMA contraction)
            double L = lutL, R = lutR;
            double y0 = __dmul_rn(wl_b0, L);
            double y1 = __dadd_rn(__dsub_rn(__dmul_rn(wl_b1, L), __dmul_rn(wl_a1, y0)), __dmul_rn(wl_b0, R));
            const double L1 = __dadd_rn(L, __dmul_rn(__dsub_rn(y0, L), wl_gm1));
            const double R1 = __dadd_rn(R, __dmul_rn(__dsub_rn(y1, R), wl_gm1));
            y0 = __dmul_rn(wh_b0, L1);
            y1 = __dadd_rn(__dsub_rn(__dmul_rn(wh_b1, L1), __dmul_rn(wh_a1, y0)), __dmul_rn(wh_b0, R1));
            L = __dadd_rn(L1, __dmul_rn(__dsub_rn(y0, L1), wh_gm1));
            R = __dadd_rn(R1, __dmul_rn(__dsub_rn(y1, R1), wh_gm1));
            xl = to_pcm_f64(L);                            // float_array_to_audio_segment (:254-257)
            xr = to_pcm_f64(R);
        }
        // audio_segment_to_float_array (:250-253): x / 32768 is exact in float32 and in float64
        float yl, yr;
        if (SKEW && MASK != 0) {
            yl = (float)q3l; yr = (float)q3r;              // the frame that entered four iterations ago leaves
            const F o3l = st3(q2l, zl), o3r = st3(q2r, zr);
            const F o2l = st2(q1l, zl), o2r = st2(q1r, zr);
            const F o1l = st1(q0l, zl), o1r = st1(q0r, zr);
            q0l = st0((F)i16_to_unit(xl), zl); q0r = st0((F)i16_to_unit(xr), zr);
            q3l = o3l; q3r = o3r; q2l = o2l; q2r = o2r; q1l = o1l; q1r = o1r;
        } else if (MASK != 0) {
            yl = cascade((F)i16_to_unit(xl), zl);
            yr = cascade((F)i16_to_unit(xr), zr);
        } else {
            yl = __fmul_rn((float)xl, 1.0f / 32768.0f);
            yr = __fmul_rn((float)xr, 1.0f / 32768.0f);
        }
        if (widen) {          // apply_stereo_width (:267-271), float32 arithmetic
            const float mid = __fmul_rn(__fadd_rn(yl, yr), 0.5f);
            const float side = __fmul_rn(__fmul_rn(__fsub_rn(yl, yr), 0.5f), wfac);
            yl = __fadd_rn(mid, side);
            yr = __fsub_rn(mid, side);
        }
        return pack16(to_pcm_f32(yl), to_pcm_f32(yr));     // clip inside to_pcm == np.clip of (:270) then (:255)
    };

    const uint4 *src = reinterpret_cast<const uint4 *>(in) + (g0f >> 2);
    uint4 *dst = reinterpret_cast<uint4 *>(pre) + (g0f >> 2);
    // software pipeline: input words two groups ahead, tanh-table values one group ahead
    uint4 cur = ldg16(src), nxt = make_uint4(0, 0, 0, 0);
    if (g0f + 0 < job.chunk_begin) cur.x = 0;              // frames before the chunk start keep the zero state
    if (g0f + 1 < job.chunk_begin) cur.y = 0;
    if (g0f + 2 < job.chunk_begin) cur.z = 0;
    if (n_it > 1) nxt = ldg16(src + 1);
    double lutL[4] = {0, 0, 0, 0}, lutR[4] = {0, 0, 0, 0};
    auto fetch_lut = [&](const uint4 &q, double *l, double *r) {
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            l[k] = __ldg(lut + (int)(int16_t)(w[k] & 0xffffu));
            r[k] = __ldg(lut + (int)(int16_t)(w[k] >> 16));
        }
    };
    if (WARM) fetch_lut(cur, lutL, lutR);
    constexpr int LAG = (SKEW && MASK != 0) ? 1 : 0;       // groups between a frame entering and leaving
    for (int it = 0; it < n_it + LAG; ++it) {              // the extra iteration drains the pipeline (its input is not used)
        uint4 nn = nxt;
        if (it + 2 < n_it) nn = ldg16(src + it + 2);
        double nL[4] = {0, 0, 0, 0}, nR[4] = {0, 0, 0, 0};
        if (WARM) fetch_lut(nxt, nL, nR);
        const int64_t g = g0f + 4 * (int64_t)(it - LAG);   // first frame of the group that leaves in this iteration
        const uint32_t w[4] = {cur.x, cur.y, cur.z, cur.w};
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] = frame(w[k], lutL[k], lutR[k]);
        if (it < LAG) {
        } else if (g >= job.tile_begin && g + 4 <= f_hi) {
            dst[it - LAG] = make_uint4(o[0], o[1], o[2], o[3]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (g + k >= job.tile_begin && g + k < f_hi) reinterpret_cast<uint32_t *>(dst + it - LAG)[k] = o[k];
        }
        cur = nxt; nxt = nn;
#pragma unroll
        for (int k = 0; k < 4; ++k) { lutL[k] = nL[k]; lutR[k] = nR[k]; }
    }
}

#define AME_EQ_KERNEL(NAME, F, SK)                                                                                  \
__global__ void __launch_bounds__(256, 1)                                                                          \
NAME(const TileJob *__restrict__ jobs, int n_jobs, const ame_track_params *__restrict__ tracks,                    \
     const double *__restrict__ luts, const int16_t *__restrict__ in, int16_t *__restrict__ pre) {                 \
    const int j = blockIdx.x * blockDim.x + threadIdx.x;                                                           \
    if (j >= n_jobs) return;                                                                                       \
    const TileJob job = jobs[j];                                                                                   \
    if (job.tile_end <= job.tile_begin) return;           /* padding job (tracks get whole warps) */               \
    const ame_track_params *tp = tracks + job.track;                                                               \
    switch (job.variant) {      /* bits 0-3: EQ stages, bit 4: warmth */                                           \
        AME_EQ_CASE(0, F, SK) AME_EQ_CASE(1, F, SK) AME_EQ_CASE(2, F, SK) AME_EQ_CASE(3, F, SK) AME_EQ_CASE(4, F, SK)    \
        AME_EQ_CASE(5, F, SK) AME_EQ_CASE(6, F, SK) AME_EQ_CASE(7, F, SK) AME_EQ_CASE(8, F, SK) AME_EQ_CASE(9, F, SK)    \
        AME_EQ_CASE(10, F, SK) AME_EQ_CASE(11, F, SK) AME_EQ_CASE(12, F, SK) AME_EQ_CASE(13, F, SK) AME_EQ_CASE(14, F, SK) \
        AME_EQ_CASE(15, F, SK)                                                                                     \
    }                                                                                                              \
}
#define AME_EQ_CASE(M, F, SK) case M: eq_tile<M, false, F, SK>(job, tp, luts, in, pre); break; \
                              case M + 16: eq_tile<M, true, F, SK>(job, tp, luts, in, pre); break;
AME_EQ_KERNEL(k_eq, double, false)
AME_EQ_KERNEL(k_eq_f32, float, false)      // precision experiment only (ame_plan_options.precision = 1)
#undef AME_EQ_CASE
#undef AME_EQ_KERNEL

// ------------------------------------------------------------------------------------------------
// k_band_split: int16 pre -> Butterworth-4 LP 250 / HP 4k in FP64, mid = x - low - high, each band
// truncated to int16 (apply_multiband_compressor :300-305).  One thread per tile, both channels, same
// warm-up scheme.  bands = 3 planes of mb_frames frames each.
// ------------------------------------------------------------------------------------------------
// UNI: every multiband track of the launch has the same crossover (same sample rate) - the usual case; the
// coefficients then come from the kernel parameter and live in uniform registers.
template <bool UNI>
__global__ void __launch_bounds__(128, 3)
k_band_split(const __grid_constant__ XoverCfg xc, const TileJob *__restrict__ jobs, int n_jobs, const ame_track_params *__restrict__ tracks,
             const int64_t *__restrict__ mb_delta,   // per track: mb_offset - offset_frames
             const int16_t *__restrict__ pre, int16_t *__restrict__ bands, int64_t mb_frames) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_jobs) return;
    const TileJob job = jobs[j];
    const ame_track_params *tp = tracks + job.track;
    const double lb0 = UNI ? xc.lb0 : tp->xlp[0].b0, la10 = UNI ? xc.la10 : tp->xlp[0].a1, la20 = UNI ? xc.la20 : tp->xlp[0].a2,
                 la11 = UNI ? xc.la11 : tp->xlp[1].a1, la21 = UNI ? xc.la21 : tp->xlp[1].a2;
    const double hb0 = UNI ? xc.hb0 : tp->xhp[0].b0, ha10 = UNI ? xc.ha10 : tp->xhp[0].a1, ha20 = UNI ? xc.ha20 : tp->xhp[0].a2,
                 ha11 = UNI ? xc.ha11 : tp->xhp[1].a1, ha21 = UNI ? xc.ha21 : tp->xhp[1].a2;
    const int64_t delta = mb_delta[job.track];
    double zl[8], zr[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { zl[i] = 0.0; zr[i] = 0.0; }
    int64_t f_lo = job.tile_begin - (int64_t)tp->warm_xover;
    if (f_lo < job.chunk_begin) f_lo = job.chunk_begin;
    const int64_t f_hi = job.tile_end;
    if (f_hi <= f_lo) return;
    const int64_t g0f = f_lo & ~(int64_t)7;                // 8 frames = one 32-byte sector per iteration
    const int n_it = (int)((f_hi - g0f + 7) >> 3);
    uint32_t *b0 = reinterpret_cast<uint32_t *>(bands) + delta;
    uint32_t *b1 = b0 + mb_frames;
    uint32_t *b2 = b1 + mb_frames;

    auto split = [&](int xm, double *z, int &p0, int &p1, int &p2) {
        const double x = i16_to_unit(xm);
        const double lo = bw_step1<1, double>(la11, la21, z[2], z[3], bw_step<1, double>(lb0, la10, la20, z[0], z[1], x));
        const double hi = bw_step1<-1, double>(ha11, ha21, z[6], z[7], bw_step<-1, double>(hb0, ha10, ha20, z[4], z[5], x));
        const double mid = __dsub_rn(__dsub_rn(x, lo), hi);
        p0 = to_pcm_f64(lo); p1 = to_pcm_f64(mid); p2 = to_pcm_f64(hi);
    };

    const uint4 *src = reinterpret_cast<const uint4 *>(pre) + (g0f >> 2);
    uint4 c0 = ldg16(src), c1 = ldg16(src + 1), n0 = make_uint4(0, 0, 0, 0), n1 = n0;
    {   // keep the zero state until the chunk starts
        uint32_t *cw0 = reinterpret_cast<uint32_t *>(&c0), *cw1 = reinterpret_cast<uint32_t *>(&c1);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (g0f + k < job.chunk_begin) cw0[k] = 0;
            if (g0f + 4 + k < job.chunk_begin) cw1[k] = 0;
        }
    }
    if (n_it > 1) { n0 = ldg16(src + 2); n1 = ldg16(src + 3); }
    for (int it = 0; it < n_it; ++it) {
        uint4 m0 = n0, m1 = n1;
        if (it + 2 < n_it) { m0 = ldg16(src + 2 * it + 4); m1 = ldg16(src + 2 * it + 5); }
        const int64_t g = g0f + 8 * (int64_t)it;
        const uint32_t w[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
        uint32_t o0[8], o1[8], o2[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            int l0, l1, l2, r0, r1, r2;
            split((int)(int16_t)(w[k] & 0xffffu), zl, l0, l1, l2);
            split((int)(int16_t)(w[k] >> 16), zr, r0, r1, r2);
            o0[k] = pack16(l0, r0); o1[k] = pack16(l1, r1); o2[k] = pack16(l2, r2);
        }
        if (g >= job.tile_begin && g + 8 <= f_hi) {
            uint4 *q0 = reinterpret_cast<uint4 *>(b0 + g), *q1 = reinterpret_cast<uint4 *>(b1 + g), *q2 = reinterpret_cast<uint4 *>(b2 + g);
            q0[0] = make_uint4(o0[0], o0[1], o0[2], o0[3]); q0[1] = make_uint4(o0[4], o0[5], o0[6], o0[7]);
            q1[0] = make_uint4(o1[0], o1[1], o1[2], o1[3]); q1[1] = make_uint4(o1[4], o1[5], o1[6], o1[7]);
            q2[0] = make_uint4(o2[0], o2[1], o2[2], o2[3]); q2[1] = make_uint4(o2[4], o2[5], o2[6], o2[7]);
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (g + k >= job.tile_begin && g + k < f_hi) { b0[g + k] = o0[k]; b1[g + k] = o1[k]; b2[g + k] = o2[k]; }
        }
        c0 = n0; c1 = n1; n0 = m0; n1 = m1;
    }
}

// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// Multiband compressor = pydub compress_dynamic_range per band (:306-308), split by what is sequential:
//   k_window_flag    (time-parallel)  window rms of the previous look_frames frames; emits the integer rms
//                                     for frames ABOVE threshold and 0 otherwise (2 B per band frame)
//   k_compact        (time-parallel)  one CTA per tile of a chain: COMPACTS the flagged frames into the chain's dense
//                                     list of rms values (rank = flagged frames of the chain's earlier tiles + a
//                                     scan inside the tile) and leaves per 32-frame group a record {bit mask of
//                                     flagged frames, number of flagged frames before the group}.  Below threshold
//                                     the reference never releases (max_attenuation = 0 => dec = 0), so unflagged
//                                     frames are no-ops of the recurrence.
//   k_att_chain      (one CTA per (chunk, band))  the attenuation recurrence over the dense list, cut into S segments
//                                     of EQUAL step count that are walked in parallel from a guessed start and
//                                     repaired until every segment starts from its predecessor's true end (exact);
//                                     emits the attenuation after every flagged frame as a dense list.
//   k_compress_apply (time-parallel)  attenuation in force at frame i = list[base + popc(mask up to i) - 1] (0 before
//                                     the first flagged frame of the chunk); gain = 10^(-att/20), audioop.mul,
//                                     low.overlay(mid).overlay(high) (:309).
// pydub: rms_at(i) = audioop.rms(frames [max(i-look,0), i)) = (unsigned)sqrt(S / n) with S the exact integer
// sum of squares and n = 2 * frames.  rms > thresh  <=>  rms >= thr_i  <=>  S >= thr_i^2 * n (integers), so
// only flagged frames take the square root (S/n is never within a relative 2^-43 of a perfect square unless equal,
// hence the double-precision expression of audioop truncates to the exact integer root).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned energy_of(uint32_t w) {          // l^2 + r^2 <= 2^31
    const int l = (int16_t)(w & 0xffffu), r = (int16_t)(w >> 16);
    return (unsigned)(l * l) + (unsigned)(r * r);
}

__device__ __forceinline__ void load8(const uint32_t *__restrict__ p, int64_t idx, int64_t lo, int64_t hi, uint32_t *w) {
    // 8 consecutive frames p[idx .. idx+8) with frames outside [lo, hi) read as zero
    if (idx >= lo && idx + 8 <= hi && ((reinterpret_cast<uintptr_t>(p + idx) & 15) == 0)) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(p + idx));
        const uint4 b = __ldg(reinterpret_cast<const uint4 *>(p + idx) + 1);
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) w[k] = (idx + k >= lo && idx + k < hi) ? __ldg(p + idx + k) : 0u;
    }
}

// floor(sqrt(s / n)) in exact integers, for s / n <= 2^30 (rms <= 32768) and n = 2 * window frames <= 8192 (look_frames
// <= 4096 is validated; 384 kHz needs 3840): audioop.rms is (unsigned)sqrt(S / n) in double, which truncates to exactly
// this (header comment above: S / n below a square k^2 stays below it by >= 1 / n, a relative 2^-43, far more than the
// double division and root can lose).  The float estimate (float(s), __fdividef within 2 ulp, a rounded root) is within
// 2^-20 relative, < 0.04 absolute, of the root, so truncation leaves it within 1; two integer tests settle it without
// overflow ((2^15 + 1)^2 * 2^13 < 2^44), and the double division + square root (~55 FP64 instructions per flagged frame)
// go away.
__device__ __forceinline__ unsigned isqrt_ratio(unsigned long long s, unsigned n) {
    unsigned r = (unsigned)__fsqrt_rn(__fdividef((float)s, (float)n));
    if ((unsigned long long)r * r * n > s) --r;
    else if ((unsigned long long)(r + 1) * (r + 1) * n <= s) ++r;
    return r;
}

__global__ void __launch_bounds__(kWfThreads)
k_window_flag(const WfJob *__restrict__ jobs, const int16_t *__restrict__ bands, uint16_t *__restrict__ rms,
              int *__restrict__ tile_cnt, GrpRec *__restrict__ grp) {
    __shared__ long long s_scan[kWfThreads / 32];
    __shared__ unsigned long long s_head[kWfThreads / 32];
    __shared__ int s_flag[kWfThreads / 32];
    const WfJob job = jobs[blockIdx.x];
    const uint32_t *bp = reinterpret_cast<const uint32_t *>(bands) + job.plane_off;
    uint16_t *rp = rms + job.plane_off;
    const int64_t n = job.n, t0 = job.tile_begin;
    const int look = job.look;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t i0 = t0 + (int64_t)threadIdx.x * 8;
    // all loads first (the kernel is bound by memory latency): this thread's 8 frames, the 8 frames `look` earlier,
    // and its share of the window entering the tile
    uint32_t w[8], wo[8];
    load8(bp, i0, 0, n, w);
    load8(bp, i0 - look, 0, n, wo);
    // window sum entering the tile: frames [t0 - look, t0)
    unsigned long long head = 0;
    for (int64_t j = t0 - look + threadIdx.x; j < t0; j += kWfThreads)
        if (j >= 0) head += energy_of(__ldg(bp + j));
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) head += __shfl_xor_sync(kFull, head, d);
    if (lane == 0) s_head[wid] = head;
    // D_j = e_j - e_{j-look}; S_i = head + sum_{t0 <= j < i} D_j
    long long pre[8];          // exclusive prefix of D inside the thread
    long long run = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        pre[k] = run;
        run += (long long)energy_of(w[k]) - (long long)energy_of(wo[k]);
    }
    long long incl = run;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long v = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_scan[wid] = incl;
    __syncthreads();
    long long base = incl - run;
    unsigned long long h = 0;
#pragma unroll
    for (int q = 0; q < kWfThreads / 32; ++q) {
        if (q < wid) base += s_scan[q];
        h += s_head[q];
    }
    base += (long long)h;
    const unsigned long long thr2 = (unsigned long long)job.thr_i * job.thr_i;
    const bool never = job.thr_i > 32768u;         // rms <= 32768 can never exceed it
    uint32_t o[4] = {0, 0, 0, 0};
    unsigned m8 = 0;                               // flagged frames of this thread (thr_i >= 1, so a flagged frame has rms >= 1)
    if (t0 >= look && i0 + 8 <= n) {          // the window is full (all but the first look_frames of a chunk): one constant bound
        const unsigned long long bound = thr2 * (unsigned long long)(2 * look);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const unsigned long long s = (unsigned long long)(base + pre[k]);
            unsigned r = 0;
            if (!never && s >= bound) r = isqrt_ratio(s, (unsigned)(2 * look));
            m8 |= (r != 0 ? 1u : 0u) << k;
            o[k >> 1] |= (r & 0xffffu) << ((k & 1) * 16);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int64_t i = i0 + k;
            const long long s = base + pre[k];
            const int64_t nfr = i < look ? i : look;
            unsigned r = 0;
            if (!never && i < n && nfr > 0 && (unsigned long long)s >= thr2 * (unsigned long long)(2 * nfr))
                r = isqrt_ratio((unsigned long long)s, (unsigned)(2 * nfr));
            m8 |= (r != 0 ? 1u : 0u) << k;
            o[k >> 1] |= (r & 0xffffu) << ((k & 1) * 16);
        }
    }
    // rank of every flagged frame inside the tile: exclusive scan of the per-thread counts over the CTA
    const int cnt = __popc(m8);
    int fincl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(kFull, fincl, d);
        if (lane >= d) fincl += v;
    }
    if (lane == 31) s_flag[wid] = fincl;
    // the four threads of a 32-frame group sit in one warp (threadIdx.x & 3 == 0 leads)
    const unsigned m1 = __shfl_down_sync(kFull, m8, 1), m2 = __shfl_down_sync(kFull, m8, 2), m3 = __shfl_down_sync(kFull, m8, 3);
    __syncthreads();
    int fbase = 0, total = 0;
#pragma unroll
    for (int q = 0; q < kWfThreads / 32; ++q) {
        if (q < wid) fbase += s_flag[q];
        total += s_flag[q];
    }
    const int rank = fbase + fincl - cnt;
    if ((threadIdx.x & 3) == 0 && i0 < n)
        grp[job.grp_begin + (i0 >> 5)] = GrpRec{m8 | (m1 << 8) | (m2 << 16) | (m3 << 24), (uint32_t)rank};   // k_compact adds the tile's rank
    if (m8) {                  // the tile's flagged rms values, dense from the tile's first slot of the rms plane
        uint16_t *dp = rp + t0 + rank;
        int slot = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (m8 & (1u << k)) dp[slot++] = (uint16_t)((o[k >> 1] >> ((k & 1) * 16)) & 0xffffu);
    }
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
}

// att' = (att <= M) ? min(att + inc, M) : max(att - dec, 0), evaluated as
//   att > M ? att - dec : (att < tau ? att + inc : M)
// * max(., 0) never binds: att - dec > M - M/release_frames >= 0.
// * tau is precomputed per table entry (host), so BOTH predicates are functions of the old attenuation and
//   evaluate in parallel with the two DADDs; the loop-carried path is max(DADD, compare) + select, ~18 cycles
//   on B200 against ~36 for DADD -> fmin (DSETP + FSEL) -> select (profiles/micro/att_chain_latency.cu).
// * all operands are non-negative doubles, for which integer order of the bit patterns == numeric order.
__device__ __forceinline__ double att_update(double att, double m, double inc, double dec, double tau) {
    const long long ia = __double_as_longlong(att);
    const bool above = ia > __double_as_longlong(m);
    const bool rising = ia < __double_as_longlong(tau);
    const double s = att + inc;
    const double d = att - dec;
    const double r = above ? d : m;
    return (rising && !above) ? s : r;
}

// ------------------------------------------------------------------------------------------------
// k_att_chain: the attenuation recurrence of one (chunk, band), exact, parallel in time.
//
// k_compact has turned the chain's rms plane into a dense list of the n_f flagged frames (below threshold the reference
// never releases - max_attenuation = 0 => dec = 0 - so unflagged frames are no-ops of the recurrence).
// Speculation and repair over the dense list of n_f steps.  S lanes take S contiguous segments of equal
//   step count (a multiple of 8).  Pass 1 starts every segment from a guess - the max_attenuation of the step just
//   before it, which is exactly right whenever the compressor was clamped there; lane 0 from 0, as the reference
//   resets the attenuation per chunk.  In a repair pass lane t takes the end value lane t-1 produced in the previous
//   pass; if that differs (bitwise) from the start it used, it walks its segment again carrying BOTH attenuations
//   (old start, new start - two independent chains in one thread) and stops at the first 8-step block after which
//   they are bit-equal: from there on what it stored before is right, and so is its old end value.  When no lane's
//   start changed, every lane has been walked from the true end of its predecessor, i.e. the stored values are
//   those of the sequential loop.  Trajectories meet whenever both clamp to the same max_attenuation
//   (att in [tau, M] -> M), which a tracking compressor does constantly.  Where they cannot meet - an attenuation
//   parked above M for a long stretch releases by M / release_frames per step, hardly at all - each pass settles one
//   more segment and the lanes of a warp run in lockstep, so the chain degrades to the cost of the sequential loop
//   (~30 cycles per step), never below it: no fallback kernel is needed.
// The walk is a software pipeline: rms values two 8-step blocks ahead, table entries (one 32-byte gather per step)
// one block ahead, 25 cycles per dependent step (profiles/micro/att_chain_latency3.cu).
// ------------------------------------------------------------------------------------------------
struct RmsBlk { uint32_t w[4]; };         // 8 consecutive entries of the dense rms list

// entries [i, i+8) of the list, entries at or past `lim` read as 0 (= the no-op table entry)
__device__ __forceinline__ RmsBlk list_load(const uint16_t *__restrict__ lp, int64_t i, int64_t lim, bool vec) {
    RmsBlk q;
    q.w[0] = q.w[1] = q.w[2] = q.w[3] = 0;
    if (vec && i + 8 <= lim) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(lp + i));
        q.w[0] = v.x; q.w[1] = v.y; q.w[2] = v.z; q.w[3] = v.w;
    } else if (i < lim) {
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (i + k < lim) q.w[k >> 1] |= (uint32_t)__ldg(lp + i + k) << ((k & 1) * 16);
    }
    return q;
}

// k_tile_prefix: one CTA per chain.  tile_base[j] = flagged frames of the chain in front of its tile j (exclusive scan of
// the k_window_flag counts, a few hundred ints); n_flagged = the chain's total.
__global__ void __launch_bounds__(kWfThreads)
k_tile_prefix(const ChainJob *__restrict__ jobs, const int *__restrict__ tile_cnt, int *__restrict__ tile_base,
              int *__restrict__ n_flagged) {
    __shared__ int s_warp[kWfThreads / 32];
    const ChainJob job = jobs[blockIdx.x];
    const int n_tiles = (int)((job.n + kWfTile - 1) / kWfTile);
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    int carry = 0;
    for (int j0 = 0; j0 < n_tiles; j0 += kWfThreads) {
        const int j = j0 + t;
        const int c = j < n_tiles ? tile_cnt[job.tile0 + j] : 0;
        int incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(kFull, incl, d);
            if (lane >= d) incl += v;
        }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        int base = carry, total = 0;
#pragma unroll
        for (int q = 0; q < kWfThreads / 32; ++q) {
            if (q < wid) base += s_warp[q];
            total += s_warp[q];
        }
        if (j < n_tiles) tile_base[job.tile0 + j] = base + incl - c;
        carry += total;
        __syncthreads();
    }
    if (t == 0) n_flagged[blockIdx.x] = carry;
}

// k_compact: one WARP per k_window_flag tile.  Moves the tile's dense run of flagged rms values (the tile's first
// tile_cnt slots of the rms plane) to its place in the chain's dense list and adds the tile's rank to the tile's group
// records (64 of them).
__global__ void __launch_bounds__(kWfThreads)
k_compact(const WfJob *__restrict__ jobs, int n_tiles, const uint16_t *__restrict__ rms, const int *__restrict__ tile_cnt,
          const int *__restrict__ tile_base, uint16_t *__restrict__ list, GrpRec *__restrict__ grp) {
    const int lane = threadIdx.x & 31;
    const int tile = blockIdx.x * (kWfThreads / 32) + (threadIdx.x >> 5);
    if (tile >= n_tiles) return;
    const WfJob job = jobs[tile];
    const int cnt = tile_cnt[tile], base = tile_base[tile];
    if (base) {                                            // the first tiles of a chain (rank 0) keep their records
        const int64_t frames = min((int64_t)kWfTile, job.n - job.tile_begin);
        const int ng = (int)((frames + 31) >> 5);
        GrpRec *gr = grp + job.grp_begin + (job.tile_begin >> 5);
        for (int g = lane; g < ng; g += 32) gr[g].base += (uint32_t)base;
    }
    const uint16_t *rp = rms + job.plane_off + job.tile_begin;
    uint16_t *lp = list + job.plane_off + base;
    for (int j = lane; j < cnt; j += 32) lp[j] = rp[j];
}


// table entries of the 8 steps of a block: one 32-byte gather each (entry 0 is all zeros = no-op).  Plain asm, not
// volatile: the table is constant and tbl + r is always a valid aligned entry, so the compiler may schedule the loads
// as it likes.
__device__ __forceinline__ void list_entries(AttEntry *e, const AttEntry *tbl, const RmsBlk &q) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const unsigned r = (q.w[k >> 1] >> ((k & 1) * 16)) & 0xffffu;
        asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(e[k].m), "=d"(e[k].inc), "=d"(e[k].dec), "=d"(e[k].tau) : "l"(tbl + r));
    }
}

// What a repair walk learns about the trajectory it stores (the one from the NEW start), so that the next change of
// the start can usually be applied without walking again:
//   the first p steps all took the release branch (attenuation parked above max_attenuation: att' = att - dec).
//   Inside one binade a double is (exponent, integer mantissa n), and fl(n u - dec) = (n - q) u with q = the nearest
//   integer to dec / u - the SAME q for every n of the binade unless dec / u is exactly half-way (a tie, decided by
//   the parity of n).  So on that prefix a start moved by d ulps moves every value by d ulps, exactly, as long as
//   (a) no step is a tie, (b) the moved values stay in the binade, (c) they stay above every max_attenuation
//   (margin = min over the prefix of bits(att) - bits(M) stays positive).
//   At step p the stored trajectory left the release branch.  If it was CLAMPED there (tau <= att <= M -> M) and the
//   moved value still lies in [tau, M], both trajectories are M from step p on: the end value does not move.
//   If the whole segment is parked (p = its length) the end value moves by d as well.
// A chain parked for seconds (pydub releases by M / release_frames per frame, hardly at all) therefore costs one
// walk per segment plus an integer add per stored value, instead of one walk per segment PER PASS.
struct SegSum {
    long long margin;      // min over the parked prefix of bits(att before the step) - bits(M of the step)
    long long at_p;        // bits(att before step p)
    long long lo, hi;      // bits(tau), bits(M) of step p
    int64_t p;             // steps in the parked prefix
    int exp0;              // exponent field of the start
    bool open;             // still inside the prefix (while walking); afterwards: the whole segment is parked
    bool ok;               // no tie, one binade
};

__device__ __forceinline__ void segsum_begin(SegSum &u, double start) {
    u.margin = 0x7fffffffffffffffLL; u.at_p = 0; u.lo = 0; u.hi = -1; u.p = 0;
    u.exp0 = (int)(__double_as_longlong(start) >> 52);
    u.open = true; u.ok = u.exp0 > 0;
}

// 8 steps of the recurrence (steps [i, i+8) of the list) from attenuation b - with DUAL also from a - storing the
// b trajectory.  True when DUAL and a == b afterwards.
template <bool DUAL>
__device__ __forceinline__ bool list_step8(const AttEntry *e, double *al, int64_t i, int64_t lim, bool avec, double &a, double &b,
                                           SegSum &u, double &max_m, double &sum_dec) {
    double o[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (!DUAL) { max_m = fmax(max_m, e[k].m); sum_dec += e[k].dec; }   // the first walk also sizes the segment (forecast below)
        if (DUAL && u.open && i + k < lim) {
            const long long ib = __double_as_longlong(b), im = __double_as_longlong(e[k].m);
            if (ib > im) {
                u.margin = min(u.margin, ib - im);
                const long long id = __double_as_longlong(e[k].dec);
                if (id != 0) {
                    const int ed = (int)(id >> 52);
                    const long long mant = (id & 0xfffffffffffffLL) | (ed ? (1LL << 52) : 0LL);
                    if ((ed ? ed : 1) + (__ffsll(mant) - 1) == u.exp0 - 1) u.ok = false;      // half an ulp exactly: a tie
                }
                ++u.p;
            } else {
                u.open = false;
                u.at_p = ib; u.lo = __double_as_longlong(e[k].tau); u.hi = im;
                if ((int)(ib >> 52) != u.exp0) u.ok = false;
            }
        }
        b = att_update(b, e[k].m, e[k].inc, e[k].dec, e[k].tau);
        if (DUAL) a = att_update(a, e[k].m, e[k].inc, e[k].dec, e[k].tau);
        o[k] = b;
    }
    if (avec && i + 8 <= lim) {
        double2 *d = reinterpret_cast<double2 *>(al + i);
        d[0] = make_double2(o[0], o[1]); d[1] = make_double2(o[2], o[3]);
        d[2] = make_double2(o[4], o[5]); d[3] = make_double2(o[6], o[7]);
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (i + k < lim) al[i + k] = o[k];
    }
    return DUAL && __double_as_longlong(a) == __double_as_longlong(b);
}

// steps [b0, b1) of the list (b0 a multiple of 8) from attenuation b; with DUAL also from a, returning true after the
// first block that leaves the two bit-equal.  b holds the attenuation reached.
template <bool DUAL>
__device__ __forceinline__ bool list_walk(const uint16_t *lp, const AttEntry *tbl, double *al, int64_t b0, int64_t b1, bool vec,
                                          bool avec, double a, double &b, SegSum &u, double &max_m, double &sum_dec) {
    if (b0 >= b1) return false;
    RmsBlk r0 = list_load(lp, b0, b1, vec), r1 = list_load(lp, b0 + 8, b1, vec);
    AttEntry ea[8], eb[8];
    list_entries(ea, tbl, r0);
    for (int64_t i = b0; i < b1; i += 16) {
        r0 = list_load(lp, i + 16, b1, vec);
        list_entries(eb, tbl, r1);
        if (list_step8<DUAL>(ea, al, i, b1, avec, a, b, u, max_m, sum_dec)) return true;
        if (i + 8 >= b1) break;
        r1 = list_load(lp, i + 24, b1, vec);
        list_entries(ea, tbl, r0);
        if (list_step8<DUAL>(eb, al, i + 8, b1, avec, a, b, u, max_m, sum_dec)) return true;
    }
    return false;
}

__global__ void __launch_bounds__(kChainMaxThreads)
k_att_chain(const ChainJob *__restrict__ jobs, const uint16_t *__restrict__ list, const int *__restrict__ n_flagged,
            const AttEntry *__restrict__ tables, double *att, int64_t mb_frames, int n_lanes,
            int *__restrict__ stats) {   // stats[chain] = {flagged steps, passes}
    __shared__ double s_end[kChainMaxThreads], s_maxm[kChainMaxThreads], s_dec[kChainMaxThreads], s_guess[kChainMaxThreads];
    const ChainJob job = jobs[blockIdx.x];
    const int t = threadIdx.x;
    const uint16_t *lp = list + (int64_t)job.band * mb_frames + job.mb_begin;
    double *al = att + (int64_t)job.band * mb_frames + job.mb_begin;
    const AttEntry *tbl = tables + (size_t)job.table * 32769;
    const bool vec = (reinterpret_cast<uintptr_t>(lp) & 15) == 0;
    const bool avec = (reinterpret_cast<uintptr_t>(al) & 15) == 0;
    const int64_t n_f = n_flagged[blockIdx.x];        // k_compact counted the chain's flagged frames

    // ---- phase 1: the recurrence over n_f steps in S segments, speculation and repair ---------------------------
    int S = n_lanes < 1 ? 1 : (n_lanes > (int)blockDim.x ? (int)blockDim.x : n_lanes);
    int64_t seg = (((n_f + S - 1) / S) + 7) & ~(int64_t)7;
    if (seg < 64) seg = 64;                                   // a lane is not worth less than a few blocks
    const int S_used = (int)((n_f + seg - 1) / seg);
    const int64_t b0 = min(n_f, (int64_t)t * seg), b1 = min(n_f, b0 + seg);
    double start = 0.0;
    if (t > 0 && b0 < b1) start = tbl[__ldg(lp + b0 - 1)].m;
    double end = start;
    SegSum u;
    segsum_begin(u, start);
    u.ok = false;                                             // nothing is known after the plain first walk
    double max_m = 0.0, sum_dec = 0.0;
    list_walk<false>(lp, tbl, al, b0, b1, vec, avec, 0.0, end, u, max_m, sum_dec);
    // Forecast (decides only which guesses are tried next, never what is stored).  Follow the attenuation from lane 0's
    // end - which is final - through the segments: where it enters a segment above everything that segment can ask for,
    // even after all the release it could get there, the true trajectory is parked throughout.  Such a lane walks
    // again from the forecast value: a start in the right binade and within a few thousand ulps of the true one, so
    // that when the true start arrives (one lane per pass) it is applied as an integer shift (SegSum) instead of
    // another walk - a chain parked for its whole length costs two walks per lane instead of one walk per lane per pass.
    s_end[t] = end; s_maxm[t] = max_m; s_dec[t] = sum_dec; s_guess[t] = -1.0;
    __syncthreads();
    if (t == 0) {
        double lb = s_end[0];
        for (int v = 1; v < S_used; ++v) {
            const double lo = lb - 1.000001 * s_dec[v];
            if (lb > 0.0 && lo > s_maxm[v]) { s_guess[v] = lb; lb = lo; }
            else lb = s_end[v];
        }
    }
    __syncthreads();
    long long pending = 0;                                    // ulps still to be added to the stored prefix [b0, b0 + u.p)
    auto flush = [&]() {
        if (pending) {
            for (int64_t i = b0; i < b0 + u.p; ++i) al[i] = __longlong_as_double(__double_as_longlong(al[i]) + pending);
            pending = 0;
        }
    };
    int passes = 1;
    for (;;) {
        s_end[t] = end;
        __syncthreads();
        double from = (t > 0 && t < S_used) ? s_end[t - 1] : 0.0;
        if (passes == 1 && t < S_used && s_guess[t] >= 0.0) from = s_guess[t];
        const bool redo = t < S_used && __double_as_longlong(from) != __double_as_longlong(start);
        const int n_redo = __syncthreads_count(redo);     // also orders the reads of s_end before the next round's writes
        if (!n_redo) break;
        ++passes;
        if (redo) {
            const long long fb = __double_as_longlong(from), d = fb - __double_as_longlong(start);
            const bool parked = u.open;                   // the whole segment is a parked prefix
            bool quick = u.ok && (int)(fb >> 52) == u.exp0 && (d >= 0 || u.p == 0 || u.margin > -d);
            if (quick && parked) quick = (int)((__double_as_longlong(end) + d) >> 52) == u.exp0;
            // step p must clamp (tau <= att <= M -> M) on the stored trajectory and on the moved one
            if (quick && !parked) quick = u.at_p >= u.lo && u.at_p <= u.hi && u.at_p + d >= u.lo && u.at_p + d <= u.hi &&
                                          (int)((u.at_p + d) >> 52) == u.exp0;
            if (quick) {                                  // every stored value of the prefix moves by d ulps, nothing else does
                pending += d;
                if (u.p) u.margin += d;
                if (parked) end = __longlong_as_double(__double_as_longlong(end) + d);
                else u.at_p += d;
                start = from;
            } else {
                flush();                                  // the stored values must be the trajectory from `start` again
                double b = from;
                segsum_begin(u, from);
                const bool met = list_walk<true>(lp, tbl, al, b0, b1, vec, avec, start, b, u, max_m, sum_dec);
                if (!met) end = b;
                // still "open" means every step walked was parked: that describes the segment only if the walk covered it
                if (u.open && (met || (int)(__double_as_longlong(end) >> 52) != u.exp0)) u.ok = false;
                start = from;
            }
        }
    }
    flush();
    if (stats && t == 0) { stats[2 * blockIdx.x] = (int)min(n_f, (int64_t)0x7fffffff); stats[2 * blockIdx.x + 1] = passes; }
}

// audioop.mul: fbound(x * f) = floor(clamp(x * f)).  Here 0 < f <= 1 (f = 10^(-att/20), att > 0) and |x| <= 32768, so
// |x * f| <= 32768: the upper clamp never binds and the lower one only replaces a value in (-32768, -32767) by -32768,
// which floor() yields anyway.  (The max() is a guard against an exp10 one ulp above 1.0, not a case that occurs.)
__device__ __forceinline__ int mul_floor(int x, double f) {
    return max(__double2int_rd(__dmul_rn((double)x, f)), -32768);
}

// pydub db_to_float(-att) = 10 ** (-att / 20); out of line so the call sites of k_compress_apply share one copy
// (the fully inlined kernel thrashed the instruction cache: stall_no_instruction 1.7 per issue).  CUDA exp10 is within
// 1 ulp of the correctly rounded value, CPython's is glibc pow: a different last bit of the gain moves x * gain by
// < 4e-12 LSB, so floor() flips only when the product is that close to an integer (DESIGN.md, parity decisions).
__device__ __noinline__ double gain_of_att(double att) { return exp10(-att / 20.0); }

// k_compress_apply: one warp per 256-frame segment, all three bands.  The attenuation in force at a frame is the
// list value of the last flagged frame at or before it: rank = group base + popc(mask up to the lane); 0 before the
// first flagged frame of the chunk.  gain = 10^(-att/20) (pydub db_to_float), audioop.mul = floor(clip(x * gain)),
// skipped when att == 0 exactly as pydub does, then low.overlay(mid).overlay(high) = saturating adds (:309).
__global__ void __launch_bounds__(128, 5)
k_compress_apply(const MbChunk *__restrict__ chunks, int n_chunks, int64_t seg_lo, int64_t seg_hi,
                 const int16_t *__restrict__ bands, const GrpRec *__restrict__ grp, const double *__restrict__ att,
                 int16_t *__restrict__ pre, int64_t mb_frames) {
    const int64_t seg = seg_lo + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (seg >= seg_hi) return;
    const int lane = threadIdx.x & 31;
    int lo = 0, hi = n_chunks - 1;                 // last chunk (of this launch's slice) with seg_prefix <= seg
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (chunks[mid].seg_prefix <= seg) lo = mid; else hi = mid - 1;
    }
    const MbChunk ck = chunks[lo];
    const int64_t lseg = seg - ck.seg_prefix;
    const int64_t f0 = lseg * kSeg;
    const int64_t n = ck.n;
    // issue every load of the segment first (24 groups x {record, band word}), then the attenuations
    uint32_t wv[3][8];
    GrpRec rec[3][8];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        const uint32_t *bp = reinterpret_cast<const uint32_t *>(bands) + (int64_t)b * mb_frames + ck.mb_begin;
        const GrpRec *gp = grp + ck.grp_begin[b] + lseg * 8;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const int64_t i = f0 + g * 32 + lane;
            wv[b][g] = (i < n) ? __ldg(bp + i) : 0u;
            const uint2 r = (f0 + g * 32 < n) ? __ldg(reinterpret_cast<const uint2 *>(gp + g)) : make_uint2(0u, 0u);
            rec[b][g] = GrpRec{r.x, r.y};
        }
    }
    // the attenuation in force at every (band, frame): all 24 gathers in flight before the first one is used
    double av[3][8];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        const double *ap = att + (int64_t)b * mb_frames + ck.mb_begin;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const unsigned rank = rec[b][g].base + __popc(rec[b][g].mask & (0xffffffffu >> (31 - lane)));
            av[b][g] = rank ? __ldg(ap + (rank - 1)) : 0.0;
        }
    }
    int accl[8], accr[8];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        double c_att = 0.0, c_fac = 1.0;           // per-lane cache of the last gain computed
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const uint32_t w = wv[b][g];
            int l = (int16_t)(w & 0xffffu), r = (int16_t)(w >> 16);
            const double mine = av[b][g];
            if (mine != 0.0) {
                if (mine != c_att) { c_att = mine; c_fac = gain_of_att(mine); }
                l = mul_floor(l, c_fac);
                r = mul_floor(r, c_fac);
            }
            accl[g] = b ? sat16(accl[g] + l) : l;
            accr[g] = b ? sat16(accr[g] + r) : r;
        }
    }
    uint32_t *out = reinterpret_cast<uint32_t *>(pre) + ck.abs_begin;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        const int64_t i = f0 + g * 32 + lane;
        if (i < n) out[i] = pack16(accl[g], accr[g]);
    }
}

// ------------------------------------------------------------------------------------------------
// k_kweight_energy: s16 -> x/32768 -> BS.1770 pre-filter + RLB (2 biquads, FP64) -> sum of squares
// per 100 ms sub-block (ebur128.c filter + gating-block sums).  K-filter state runs through the
// whole track (the reference measures the concatenated file), so warm-up may cross chunk joins.
// One thread per tile of sub-blocks, both channels (two independent chains).
// ------------------------------------------------------------------------------------------------
// UNI: every track of the launch has the same K filter (same sample rate): coefficients from the kernel parameter.
template <bool UNI>
__global__ void __launch_bounds__(128, 5)
k_kweight_energy(const __grid_constant__ KwCfg kc, const KwJob *__restrict__ jobs, int n_jobs, const ame_track_params *__restrict__ tracks,
                 const TrackDev *__restrict__ tdev, const int16_t *__restrict__ pre,
                 double *__restrict__ energy, int *__restrict__ peak) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_jobs) return;
    const KwJob job = jobs[j];
    const ame_track_params *tp = tracks + job.track;
    const TrackDev td = tdev[job.track];
    const ame_biquad k0 = UNI ? ame_biquad{kc.b0, kc.b1, kc.b2, kc.a1, kc.a2} : tp->kw[0];
    const ame_biquad k1 = UNI ? ame_biquad{1.0, -2.0, 1.0, kc.ra1, kc.ra2} : tp->kw[1];
    const int64_t s100 = td.s100;
    const int64_t base = tp->offset_frames;                      // multiple of 8
    const int64_t t_begin = (int64_t)job.sb_begin * s100;        // relative to the track
    const int64_t t_end = (int64_t)job.sb_end * s100;
    int64_t f_lo = t_begin - (int64_t)tp->warm_kw;
    if (f_lo < 0) f_lo = 0;
    f_lo &= ~(int64_t)7;                                         // extra warm-up frames are harmless
    double zl[4] = {0, 0, 0, 0}, zr[4] = {0, 0, 0, 0}, accl = 0, accr = 0;
    int pk = 0;
    int64_t next_end = t_begin + s100;
    int sb = job.sb_begin;
    const uint4 *src = reinterpret_cast<const uint4 *>(reinterpret_cast<const uint32_t *>(pre) + base + f_lo);
    const int n_it = (int)((t_end - f_lo + 7) >> 3);             // 8 frames = one 32-byte sector per iteration
    uint4 c0 = ldg16(src), c1 = ldg16(src + 1), n0 = c0, n1 = c1;
    if (n_it > 1) { n0 = ldg16(src + 2); n1 = ldg16(src + 3); }
    // Three kinds of 8-frame groups: in front of the tile (warm-up: filter only), inside one sub-block of the tile
    // (accumulate, no per-frame test - all of them at 48 / 96 / 192 kHz, where a sub-block is a whole number of groups),
    // and the ones a tile or sub-block boundary cuts (per-frame tests; 44.1 kHz: one group in 551).
    for (int it = 0; it < n_it; ++it) {
        uint4 m0 = n0, m1 = n1;
        if (it + 2 < n_it) { m0 = ldg16(src + 2 * it + 4); m1 = ldg16(src + 2 * it + 5); }
        const int64_t g = f_lo + 8 * (int64_t)it;
        const uint32_t w[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
        if (g + 8 <= t_begin) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int xl = (int)(int16_t)(w[k] & 0xffffu), xr = (int)(int16_t)(w[k] >> 16);
                bq_step(k1, zl[2], zl[3], bq_step(k0, zl[0], zl[1], i16_to_unit(xl)));
                bq_step(k1, zr[2], zr[3], bq_step(k0, zr[0], zr[1], i16_to_unit(xr)));
            }
        } else if (g >= t_begin && g + 8 <= next_end) {          // next_end <= t_end
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int xl = (int)(int16_t)(w[k] & 0xffffu), xr = (int)(int16_t)(w[k] >> 16);
                const double yl = bq_step(k1, zl[2], zl[3], bq_step(k0, zl[0], zl[1], i16_to_unit(xl)));
                const double yr = bq_step(k1, zr[2], zr[3], bq_step(k0, zr[0], zr[1], i16_to_unit(xr)));
                accl = fma(yl, yl, accl);
                accr = fma(yr, yr, accr);
                pk = max(pk, max(abs(xl), abs(xr)));
            }
            if (g + 8 == next_end) {
                energy[td.sb_offset + sb] = accl + accr;         // ebur128: per-channel sums, then added
                accl = 0; accr = 0; ++sb; next_end += s100;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int64_t f = g + k;
                const int xl = (int)(int16_t)(w[k] & 0xffffu), xr = (int)(int16_t)(w[k] >> 16);
                const double yl = bq_step(k1, zl[2], zl[3], bq_step(k0, zl[0], zl[1], i16_to_unit(xl)));
                const double yr = bq_step(k1, zr[2], zr[3], bq_step(k0, zr[0], zr[1], i16_to_unit(xr)));
                if (f >= t_begin && f < t_end) {
                    accl = fma(yl, yl, accl);
                    accr = fma(yr, yr, accr);
                    pk = max(pk, max(abs(xl), abs(xr)));
                    if (f + 1 == next_end) {
                        energy[td.sb_offset + sb] = accl + accr;
                        accl = 0; accr = 0; ++sb; next_end += s100;
                    }
                }
            }
        }
        c0 = n0; c1 = n1; n0 = m0; n1 = m1;
    }
    atomicMax(peak + job.track, pk);
}

// tail frames beyond the last complete sub-block still count for the sample peak
__global__ void k_tail_peak(const ame_track_params *__restrict__ tracks, const TrackDev *__restrict__ tdev,
                            int track_lo, int track_hi, const int16_t *__restrict__ pre, int *__restrict__ peak) {
    const int t = track_lo + blockIdx.x;
    if (t >= track_hi) return;
    const int64_t begin = (int64_t)tdev[t].n_sb * tdev[t].s100;
    const int16_t *p = pre + 2 * tracks[t].offset_frames;
    int pk = 0;
    for (int64_t i = 2 * begin + threadIdx.x; i < 2 * tdev[t].n_total; i += blockDim.x) pk = max(pk, abs((int)p[i]));
    atomicMax(peak + t, pk);
}

__device__ __forceinline__ int hist_index(double e) {   // ebur128.c find_histogram_index
    int lo = 0, hi = 1000;
    do {
        int mid = (lo + hi) >> 1;
        if (e >= c_hist_bounds[mid]) lo = mid; else hi = mid;
    } while (hi - lo != 1);
    return lo;
}

// k_block_hist: 400 ms blocks every 100 ms -> 1000-bin histogram (absolute gate = bin floor, -70 LUFS), and the
// short-term histogram behind loudness range: 3 s windows, the first ending at 3 s, then one per second
// (ebur128.c: short_term_frame_counter reaches 30 sub-blocks, is reset to 20).
__global__ void __launch_bounds__(256)
k_block_hist(const TrackDev *__restrict__ tdev, int track_lo, const double *__restrict__ energy, long long *__restrict__ hist,
             int *__restrict__ hist_st) {
    __shared__ unsigned s_hist[1000];
    __shared__ unsigned s_st[1000];
    const int t = track_lo + blockIdx.x;
    for (int i = threadIdx.x; i < 1000; i += blockDim.x) { s_hist[i] = 0; s_st[i] = 0; }
    __syncthreads();
    const TrackDev td = tdev[t];
    const double *e = energy + td.sb_offset;
    const double denom = (double)(4 * (int64_t)td.s100);
    for (int j = td.first_block + threadIdx.x; j + 3 < td.n_sb; j += blockDim.x) {
        const double s = (((e[j] + e[j + 1]) + e[j + 2]) + e[j + 3]) / denom;
        if (s >= c_hist_bounds[0]) atomicAdd(&s_hist[hist_index(s)], 1u);
    }
    const double denom_st = (double)(30 * (int64_t)td.s100);
    for (int k = threadIdx.x; 10 * k + 29 < td.n_sb; k += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < 30; ++j) s += e[10 * k + j];
        s /= denom_st;
        if (s >= c_hist_bounds[0]) atomicAdd(&s_st[hist_index(s)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 1000; i += blockDim.x) {
        hist[(int64_t)t * 1000 + i] = (long long)s_hist[i];
        hist_st[(int64_t)t * 1000 + i] = (int)s_st[i];
    }
}

// ebur128_gated_loudness over a 400 ms block histogram, in ebur128.c's order (the sums are order-sensitive in the last
// bit, and that bit can decide the '%.2f' the gain is made of; products and sums rounded separately, as the C library
// computes them - an FMA there moved the relative gate by one ulp): blocks above the absolute gate, the relative gate (as
// energy and in LUFS; -70 when no block passes) and the gated loudness (-inf when no block passes the relative gate).
// k_finalize and k_meter_finalize both walk with it.
struct GateWalk { long long count, above; double rel, thresh, integrated; };
template <class H>
__device__ __forceinline__ GateWalk gate_walk(const H *h) {
    GateWalk g{0, 0, 0.0, -70.0, -INFINITY};
    double rel = 0.0; long long count = 0;
    for (int j = 0; j < 1000; ++j) { rel = __dadd_rn(rel, __dmul_rn((double)h[j], c_hist_energy[j])); count += h[j]; }
    g.count = count;
    if (count > 0) {
        rel /= (double)count;
        rel *= 0.1;                                  // RELATIVE_GATE_FACTOR = 10^(-10/10)
        g.rel = rel;
        g.thresh = 10.0 * log10(rel) - 0.691;        // ff_ebur128_relative_threshold
        int start;
        if (rel < c_hist_bounds[0]) start = 0;
        else { start = hist_index(rel); if (rel > c_hist_energy[start]) ++start; }
        double gated = 0.0; long long above = 0;
        for (int j = start; j < 1000; ++j) { gated = __dadd_rn(gated, __dmul_rn((double)h[j], c_hist_energy[j])); above += h[j]; }
        g.above = above;
        if (above > 0) {
            gated /= (double)above;
            g.integrated = 10.0 * log10(gated) - 0.691;
        }
    }
    return g;
}

// ff_ebur128_loudness_range over a short-term histogram: blocks above (mean power - 20 dB), 10th .. 95th percentile; 0
// when there is none
template <class HS>
__device__ __forceinline__ double lra_walk(const HS *hs) {
    long long n = 0; double power = 0.0;
    for (int j = 0; j < 1000; ++j) { n += hs[j]; power = __dadd_rn(power, __dmul_rn((double)hs[j], c_hist_energy[j])); }
    if (n > 0) {
        power /= (double)n;
        const double integ = 0.01 * power;           // MINUS_20DB
        int idx;
        if (integ < c_hist_bounds[0]) idx = 0;
        else { idx = hist_index(integ); if (integ > c_hist_energy[idx]) ++idx; }
        long long m = 0;
        for (int j = idx; j < 1000; ++j) m += hs[j];
        if (m > 0) {
            const long long p_lo = (long long)((double)(m - 1) * 0.1 + 0.5), p_hi = (long long)((double)(m - 1) * 0.95 + 0.5);
            long long acc = 0; int j = idx;
            while (acc <= p_lo) acc += hs[j++];
            const double l_en = c_hist_energy[j - 1];
            while (acc <= p_hi) acc += hs[j++];
            const double h_en = c_hist_energy[j - 1];
            return (10.0 * log10(h_en) - 0.691) - (10.0 * log10(l_en) - 0.691);
        }
    }
    return 0.0;
}

// k_finalize: ebur128_gated_loudness + loudness range + the linear-mode gain of af_loudnorm.  One CTA per track: the
// two 1000-bin histograms are staged in shared memory by all threads, then ONE thread walks them.
__global__ void __launch_bounds__(128)
k_finalize(const ame_track_params *__restrict__ tracks, int track_lo, int track_hi,
           const long long *__restrict__ hist, const int *__restrict__ hist_st, const int *__restrict__ peak,
           const unsigned *__restrict__ tp_bits, ame_track_result *__restrict__ res) {
    __shared__ long long s_h[1000];
    __shared__ int s_hs[1000];
    const int t = track_lo + blockIdx.x;
    if (t >= track_hi) return;
    for (int i = threadIdx.x; i < 1000; i += blockDim.x) {
        s_h[i] = hist[(int64_t)t * 1000 + i];
        s_hs[i] = hist_st[(int64_t)t * 1000 + i];
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    ame_track_result r;
    r.input_i = -INFINITY; r.measured_i_2dp = -INFINITY; r.gain = 1.0; r.rel_threshold = 0.0;
    r.n_blocks = 0; r.normalized = 0; r.sample_peak = peak[t];
    r.input_lra = 0.0; r.input_thresh = -70.0;
    r.true_peak = ((tracks[t].flags & AME_F_TRUE_PEAK) && tracks[t].sample_rate < 192000) ? (double)__uint_as_float(tp_bits[t])
                                                                                           : (double)peak[t] * (1.0 / 32768.0);
    const GateWalk g = gate_walk(s_h);
    r.n_blocks = g.count;
    if (g.count > 0) {
        r.rel_threshold = g.rel;
        r.input_thresh = g.thresh;
        if (g.above > 0) {
            r.input_i = g.integrated;
            if (tracks[t].flags & AME_F_NORMALIZE) {
                r.measured_i_2dp = rint(r.input_i * 100.0) / 100.0;   // the '%.2f' string of pass 1
                r.gain = pow(10.0, (tracks[t].target_lufs - r.measured_i_2dp) / 20.0);
                r.normalized = 1;
            }
        }
    }
    r.input_lra = lra_walk(s_hs);
    res[t] = r;
}

// k_apply_gain: loudnorm linear mode: s16 -> x/32768 -> * gain -> lrint(x * 32768) clipped to s16.
// Tracks with the limiter stage write the normalised signal to the slot's `norm` buffer instead of `out` (k_limiter
// reads it) and record, per limiter tile, the last frame whose peak exceeds the limiter's limit (lim_last, preset to -1).
__global__ void __launch_bounds__(256)
k_apply_gain(const GainJob *__restrict__ jobs, const ame_track_result *__restrict__ res, const ame_track_params *__restrict__ tracks,
             const TrackDev *__restrict__ tdev, const int16_t *__restrict__ pre, int16_t *__restrict__ out,
             int16_t *__restrict__ norm, long long *__restrict__ lim_last) {
    const GainJob job = jobs[blockIdx.x];
    const ame_track_result r = res[job.track];
    const ame_track_params *tp = tracks + job.track;
    const bool lim = (tp->flags & AME_F_LIMITER) != 0;
    const int thr_i = tp->lim_thr_i;
    const int64_t t_begin = tp->offset_frames + tp->halo_frames;
    const int lim_tile0 = tdev[job.track].lim_tile0, lim_shift = tdev[job.track].lim_shift;
    const uint4 *src = reinterpret_cast<const uint4 *>(pre);
    uint4 *dst = reinterpret_cast<uint4 *>(lim ? norm : out);
    const int64_t v0 = job.begin >> 2, v1 = (job.end + 3) >> 2;   // 4 frames per uint4; tiles are 4-aligned
    long long last = -1;                                           // last over-limit frame seen in limiter tile `last_tile`
    int last_tile = -1;
    const double g = r.gain;
    for (int64_t v = v0 + threadIdx.x; v < v1; v += blockDim.x) {
        const uint4 q = __ldg(src + v);
        uint32_t w[4] = {q.x, q.y, q.z, q.w};
        if (r.normalized) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int l = (int16_t)(w[k] & 0xffffu), rr = (int16_t)(w[k] >> 16);
                int ol = __double2int_rn(__dmul_rn(__dmul_rn((double)l * (1.0 / 32768.0), g), 32768.0));
                int orr = __double2int_rn(__dmul_rn(__dmul_rn((double)rr * (1.0 / 32768.0), g), 32768.0));
                w[k] = (uint32_t)(uint16_t)sat16(ol) | ((uint32_t)(uint16_t)sat16(orr) << 16);
            }
        }
        if (lim) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int l = (int16_t)(w[k] & 0xffffu), rr = (int16_t)(w[k] >> 16);
                const int64_t f = 4 * v + k;
                if (max(abs(l), abs(rr)) >= thr_i && f >= job.begin && f < job.end) {
                    const int tile = lim_tile0 + (int)((f - t_begin) >> lim_shift);
                    if (tile != last_tile) {
                        if (last_tile >= 0) atomicMax(lim_last + last_tile, last);
                        last_tile = tile;
                    }
                    last = f;                                      // a thread's frames only grow
                }
            }
        }
        dst[v] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    if (lim && last_tile >= 0) atomicMax(lim_last + last_tile, last);
}

// ------------------------------------------------------------------------------------------------
// ffmpeg alimiter (audio_mastering_engine.py:223; af_alimiter.c with level_in = level_out = 1, auto level on, asc off,
// latency off) on the normalised signal.  The filter is one sequential state machine per track: a look-ahead ring of B
// frames (output = input delayed by B - 1 frames), an attenuation `att` that moves by `delta` per frame, and a queue of
// the over-limit peaks inside the ring with the slope each will hand over when it leaves.
// What makes it parallel in time:
//   (1) after G = B + release_frames + 8 frames without an over-limit frame the state is the initial one again (att 1,
//       delta 0, empty queue: the last queued peak has left the ring and its linear release has reached 1), and in that
//       state the filter is elementwise, out[n] = clip(x[n - B + 1]) / limit.  k_apply_gain leaves per 32768-frame tile
//       the last frame over the limit, so every tile knows whether it STARTS in the initial state and whether it is
//       elementwise throughout (all 256 threads, copy speed - the common case for mastered material);
//   (2) a tile that does not start in the initial state (a track that is over the limit all the time - a hot loudness
//       target clips) takes a GUESS of its start state: the machine run from the initial state over the 2 G frames in
//       front of the tile.  The machine forgets: when a queued peak leaves the ring the attenuation is SET to
//       limit / peak, and everything else in the state (slope, queue) is made of peaks inside the ring.  Every tile
//       records the state it started from and the state it ended in; k_lim_verify compares each tile's start with its
//       predecessor's end, field by field and bit by bit; a tile whose guess was wrong runs again from its
//       predecessor's end (two rounds), and what is still open after that is walked sequentially by k_lim_fallback
//       until the live state equals a recorded start.  When every start equals its predecessor's end, the tiles are
//       the sequential run: exact.
// One warp per non-elementwise tile: lane 0 walks the state 32 frames at a time, all lanes load the frames before and
// scale / round / store them after.
// ------------------------------------------------------------------------------------------------
// The machine between two frames, as recorded per tile.  The queue (one entry per over-limit frame still inside the
// look-ahead ring: up to B of them while the signal clips) lives in two side arrays of `keep` = B_max + 2 entries per tile.
struct LimState {
    double att, delta;
    int qlen;
    int exact;                      // as a tile's START state: known to be the true one (initial state / track start)
};
struct LimStore {                   // where the recorded states of a launch live
    LimState *st;                   // [tiles]
    int *qframe;                    // [tiles][keep] frame (relative to the track) of every queued peak, in queue order
    double *qdelta;                 // [tiles][keep]
    int keep;
};

struct LimSmem {                    // views into the CTA's dynamic shared memory (lim_smem)
    double *qdelta;                 // [cap]
    double *qratio;                 // [cap]  limit / peak of the queued frame (af_alimiter.c recomputes it from the ring at every search)
    double *att;                    // [32]
    int *qframe;                    // [cap]  -1 = none (the sentinel af_alimiter.c keeps behind the last entry)
    int *pin, *pout;                // [32] peak (max |s16|) of the frame entering / leaving the ring at each of 32 steps
    int mask;                       // cap - 1, cap = a power of two >= look-ahead frames + 4
};
__host__ __device__ inline size_t lim_smem_bytes(int cap) { return (size_t)cap * 20 + 32 * 16; }
__device__ __forceinline__ LimSmem lim_smem(unsigned char *raw, int cap) {
    LimSmem sm;
    sm.qdelta = reinterpret_cast<double *>(raw);
    sm.qratio = sm.qdelta + cap;
    sm.att = sm.qratio + cap;
    sm.qframe = reinterpret_cast<int *>(sm.att + 32);
    sm.pin = sm.qframe + cap;
    sm.pout = sm.pin + 32;
    sm.mask = cap - 1;
    return sm;
}

struct LimCtx {
    const uint32_t *x;              // normalised signal (packed buffer)
    uint32_t *y;                    // output
    int64_t t_begin, t_end;         // the track
    int B, thr_i;
    double limit, level, fsrel;
};

struct LimRegs { double att, delta; int qiter, qlen; };      // the scalar part of the machine, the same in every lane

__device__ __forceinline__ int lim_out_sample(int x, double att, double limit, double level) {
    double v = __dmul_rn((double)x * (1.0 / 32768.0), att);          // buf[c] * att
    v = fmin(fmax(v, -limit), limit);                                 // av_clipd(dst, -limit, limit)
    v = __dmul_rn(v, level);                                          // * level (* level_out = 1)
    return sat16(__double2int_rn(__dmul_rn(v, 32768.0)));             // swresample dbl -> s16
}

__device__ __forceinline__ void lim_emit(const LimCtx &c, int64_t n, double att) {   // output frame n = input frame n - (B - 1)
    const int64_t m = n - (c.B - 1);
    const uint32_t w = m >= c.t_begin ? __ldg(c.x + m) : 0u;
    c.y[n] = pack16(lim_out_sample((int16_t)(w & 0xffffu), att, c.limit, c.level), lim_out_sample((int16_t)(w >> 16), att, c.limit, c.level));
}

__device__ __forceinline__ void lim_reset(LimRegs &r, LimSmem &sm, int lane) {
    for (int i = lane; i <= sm.mask; i += 32) { sm.qframe[i] = -1; sm.qdelta[i] = 0.0; }
    r.att = 1.0; r.delta = 0.0; r.qiter = 0; r.qlen = 0;
    __syncwarp();
}

__device__ __forceinline__ void lim_save(const LimRegs &r, const LimSmem &sm, const LimStore &S, int tile, int exact, int lane) {
    if (lane == 0) S.st[tile] = LimState{r.att, r.delta, r.qlen, exact};
    for (int k = lane; k < r.qlen; k += 32) {
        S.qframe[(size_t)tile * S.keep + k] = sm.qframe[(r.qiter + k) & sm.mask];
        S.qdelta[(size_t)tile * S.keep + k] = sm.qdelta[(r.qiter + k) & sm.mask];
    }
}

__device__ __forceinline__ void lim_load(LimRegs &r, LimSmem &sm, const LimStore &S, int tile, int lane) {
    lim_reset(r, sm, lane);
    const LimState st = S.st[tile];
    r.att = st.att; r.delta = st.delta; r.qiter = 0; r.qlen = st.qlen;
    for (int k = lane; k < st.qlen; k += 32) {
        sm.qframe[k] = S.qframe[(size_t)tile * S.keep + k];
        sm.qdelta[k] = S.qdelta[(size_t)tile * S.keep + k];
    }
    __syncwarp();
}

// limit / peak of every queued frame, from the signal (after a load; the machine keeps them current itself)
__device__ __forceinline__ void lim_ratios(const LimCtx &c, const LimRegs &r, LimSmem &sm, int lane) {
    for (int k = lane; k < r.qlen; k += 32) {
        const int j = (r.qiter + k) & sm.mask;
        const uint32_t w = __ldg(c.x + c.t_begin + sm.qframe[j]);
        sm.qratio[j] = c.limit / ((double)max(abs((int)(int16_t)(w & 0xffffu)), abs((int)(int16_t)(w >> 16))) * (1.0 / 32768.0));
    }
    __syncwarp();
}

// recorded state (A, tile a) == recorded state (B, tile b), field by field and bit by bit (whole warp; same result in every lane)
__device__ __forceinline__ bool lim_equal(const LimStore &A, int a, const LimStore &Bs, int b, int lane) {
    const LimState x = A.st[a], y = Bs.st[b];
    bool eq = x.qlen == y.qlen && __double_as_longlong(x.att) == __double_as_longlong(y.att) &&
              __double_as_longlong(x.delta) == __double_as_longlong(y.delta);
    if (eq)
        for (int k = lane; k < x.qlen; k += 32)
            eq = eq && A.qframe[(size_t)a * A.keep + k] == Bs.qframe[(size_t)b * Bs.keep + k] &&
                 __double_as_longlong(A.qdelta[(size_t)a * A.keep + k]) == __double_as_longlong(Bs.qdelta[(size_t)b * Bs.keep + k]);
    return __all_sync(kFull, eq);
}

// the live machine == recorded state (S, tile)
__device__ __forceinline__ bool lim_equal_live(const LimRegs &r, const LimSmem &sm, const LimStore &S, int tile, int lane) {
    const LimState y = S.st[tile];
    bool eq = r.qlen == y.qlen && __double_as_longlong(r.att) == __double_as_longlong(y.att) &&
              __double_as_longlong(r.delta) == __double_as_longlong(y.delta);
    if (eq)
        for (int k = lane; k < r.qlen; k += 32)
            eq = eq && sm.qframe[(r.qiter + k) & sm.mask] == S.qframe[(size_t)tile * S.keep + k] &&
                 __double_as_longlong(sm.qdelta[(r.qiter + k) & sm.mask]) == __double_as_longlong(S.qdelta[(size_t)tile * S.keep + k]);
    return __all_sync(kFull, eq);
}

// The machine over frames [n_lo, n_hi) of the packed buffer; output is stored when `emit`.  The whole warp runs the
// frame loop in lockstep with the scalar state replicated in every lane (same inputs, same arithmetic); only the search
// through the queue when an over-limit frame arrives (af_alimiter.c walks it entry by entry - up to B entries while the
// signal clips) is spread over the lanes, 32 entries per step.
__device__ __forceinline__ void lim_run(const LimCtx &c, LimRegs &r, LimSmem &sm, int64_t n_lo, int64_t n_hi, bool emit, int lane) {
    const int bufsize = 2 * c.B;
    double att = r.att, delta = r.delta;
    int qiter = r.qiter, qlen = r.qlen;
    for (int64_t n0 = n_lo; n0 < n_hi; n0 += 32) {
        const int64_t n = n0 + lane, m = n - (c.B - 1);
        const uint32_t win = n < n_hi ? __ldg(c.x + n) : 0u;
        const uint32_t wout = (n < n_hi && m >= c.t_begin) ? __ldg(c.x + m) : 0u;
        sm.pin[lane] = max(abs((int)(int16_t)(win & 0xffffu)), abs((int)(int16_t)(win >> 16)));
        sm.pout[lane] = max(abs((int)(int16_t)(wout & 0xffffu)), abs((int)(int16_t)(wout >> 16)));
        const unsigned over = __ballot_sync(kFull, n < n_hi && sm.pin[lane] >= c.thr_i);
        __syncwarp();
        const int n_valid = (int)min((int64_t)32, n_hi - n0);
        if (over == 0 && qlen == 0 && delta == 0.0) {                 // nothing can happen in these 32 frames
            if (lane < n_valid) sm.att[lane] = att;
        } else {
            for (int k = 0; k < n_valid; ++k) {
                const int rel = (int)(n0 + k - c.t_begin);
                if (over & (1u << k)) {                               // the entering frame is over the limit
                    const double peak = (double)sm.pin[k] * (1.0 / 32768.0);
                    const double patt = fmin(c.limit / peak, 1.0);
                    const double rdelta = (1.0 - patt) / c.fsrel;
                    const double ratio = c.limit / peak;
                    const double d = (ratio - att) / bufsize * 2;
                    if (d < delta) {
                        delta = d;
                        if (lane == 0) { sm.qframe[0] = rel; sm.qframe[1] = -1; sm.qdelta[0] = rdelta; sm.qratio[0] = ratio; }
                        qlen = 1; qiter = 0;
                    } else {
                        int found = -1;                               // first queue position whose slope the new peak undercuts
                        for (int i0 = 0; i0 < qlen && found < 0; i0 += 32) {
                            const int i = i0 + lane;
                            bool hit = false;
                            double pdelta = 0.0;
                            if (i < qlen) {
                                const int j = (qiter + i) & sm.mask;
                                pdelta = (ratio - sm.qratio[j]) / (double)(rel - sm.qframe[j]);     // (limit/peak - limit/ppeak) / distance
                                hit = pdelta < sm.qdelta[j];
                            }
                            const unsigned hits = __ballot_sync(kFull, hit);
                            if (hits) {
                                const int first = __ffs(hits) - 1;
                                found = i0 + first;
                                const double pd = __shfl_sync(kFull, pdelta, first);
                                if (lane == 0) sm.qdelta[(qiter + found) & sm.mask] = pd;
                            }
                        }
                        if (found >= 0) {
                            qlen = found + 1;
                            if (lane == 0) {
                                sm.qframe[(qiter + qlen) & sm.mask] = rel;
                                sm.qdelta[(qiter + qlen) & sm.mask] = rdelta;
                                sm.qratio[(qiter + qlen) & sm.mask] = ratio;
                                sm.qframe[(qiter + qlen + 1) & sm.mask] = -1;
                            }
                            ++qlen;
                        }
                    }
                    __syncwarp();
                }
                att += delta;
                if (lane == 0) sm.att[k] = att;                       // the leaving frame is scaled by this
                if (rel >= c.B - 1 && rel - (c.B - 1) == sm.qframe[qiter]) {   // a queued peak leaves the ring
                    delta = sm.qdelta[qiter];
                    att = c.limit / ((double)sm.pout[k] * (1.0 / 32768.0));
                    --qlen;
                    __syncwarp();
                    if (lane == 0) sm.qframe[qiter] = -1;
                    qiter = (qiter + 1) & sm.mask;
                    __syncwarp();
                }
                if (att > 1.0) { att = 1.0; delta = 0.0; qiter = 0; qlen = 0; __syncwarp(); if (lane == 0) sm.qframe[0] = -1; __syncwarp(); }
                if (att <= 0.0) { att = 0.0000000000001; delta = (1.0 - att) / c.fsrel; }
                if (att != 1.0 && (1.0 - att) < 0.0000000000001) att = 1.0;
                if (delta != 0.0 && fabs(delta) < 0.00000000000001) delta = 0.0;
            }
        }
        __syncwarp();
        if (emit && lane < n_valid) lim_emit(c, n, sm.att[lane]);
        __syncwarp();
    }
    r.att = att; r.delta = delta; r.qiter = qiter; r.qlen = qlen;
}

struct LimTile { bool limiter, first, quiet_start, simple; int64_t G; };

__device__ __forceinline__ LimTile lim_classify(const GainJob *jobs, int tile, const long long *lim_last, const ame_track_params *tp) {
    LimTile t;
    const GainJob job = jobs[tile];
    t.limiter = (tp->flags & AME_F_LIMITER) != 0;
    t.G = (int64_t)tp->lim_frames + tp->lim_release_frames + 8;
    t.first = tile == 0 || jobs[tile - 1].track != job.track;
    const long long prev_last = t.first ? -1 : lim_last[tile - 1];
    t.quiet_start = t.first || prev_last < 0 || (job.begin - 1 - prev_last >= t.G);
    t.simple = t.quiet_start && lim_last[tile] < 0;
    return t;
}

__device__ __forceinline__ LimCtx lim_ctx(const ame_track_params *tp, const int16_t *norm, int16_t *out) {
    LimCtx c;
    c.x = reinterpret_cast<const uint32_t *>(norm);
    c.y = reinterpret_cast<uint32_t *>(out);
    c.t_begin = tp->offset_frames + tp->halo_frames;
    c.t_end = c.t_begin + tp->n_frames;
    c.B = tp->lim_frames; c.thr_i = tp->lim_thr_i;
    c.limit = tp->lim_limit; c.level = tp->lim_level; c.fsrel = tp->lim_fs_release;
    return c;
}

// round 0: every tile (elementwise tiles by all threads, the others by warp 0 from the initial state or from a guess);
// round >= 1: the tiles k_lim_verify left open, from their predecessor's recorded end state.
// guess: frames the round-0 guess runs over in front of its tile; -1 = 2 G (ame_plan_set_limiter_guess)
__global__ void __launch_bounds__(256)
k_limiter(const GainJob *__restrict__ jobs, int n_jobs, const long long *__restrict__ lim_last,
          const ame_track_params *__restrict__ tracks, const int16_t *__restrict__ norm, int16_t *__restrict__ out,
          LimStore IN, LimStore OUT, int *__restrict__ need, int round, int cap, int guess) {
    // round 0 is launched twice: 256 threads per tile for the elementwise tiles (the others leave at once) and ONE warp
    // per tile for the sequential ones (so that a few thousand of them are resident at a time)
    extern __shared__ __align__(16) unsigned char lim_raw[];
    LimSmem sm = lim_smem(lim_raw, cap);
    const int tile = blockIdx.x;
    const GainJob job = jobs[tile];
    const ame_track_params *tp = tracks + job.track;
    const LimTile t = lim_classify(jobs, tile, lim_last, tp);
    if (!t.limiter) { if (round == 0 && threadIdx.x == 0) need[tile] = 0; return; }
    if (round == 0 && t.simple != (blockDim.x > 32)) return;
    const LimCtx c = lim_ctx(tp, norm, out);
    const int lane = threadIdx.x & 31;
    LimRegs r;
    if (round == 0) {
        if (t.simple) {                                               // initial state throughout: elementwise
            for (int64_t n = job.begin + threadIdx.x; n < job.end; n += blockDim.x) lim_emit(c, n, 1.0);
            if (threadIdx.x == 0) {
                IN.st[tile] = LimState{1.0, 0.0, 0, 1};
                OUT.st[tile] = LimState{1.0, 0.0, 0, 0};
                need[tile] = 0;
            }
            return;
        }
        lim_reset(r, sm, lane);
        int exact = 1;
        if (!t.quiet_start) {                                         // guess: the machine over the 2 G frames in front
            const int64_t ws = max(c.t_begin, job.begin - (guess < 0 ? 2 * t.G : (int64_t)guess));
            exact = ws == c.t_begin;                                  // from the track start it is no guess
            lim_run(c, r, sm, ws, job.begin, false, lane);
        }
        lim_save(r, sm, IN, tile, exact, lane);
    } else {
        // open, and the predecessor is settled (it does not run in this round, so its recorded end is stable)
        if (!need[tile] || need[tile - 1]) return;
        lim_load(r, sm, OUT, tile - 1, lane);
        lim_ratios(c, r, sm, lane);
        lim_save(r, sm, IN, tile, 0, lane);
    }
    lim_run(c, r, sm, job.begin, job.end, true, lane);
    lim_save(r, sm, OUT, tile, 0, lane);
}

// does every tile start where its predecessor ended?  One warp per tile; counts the open tiles of this pass.
__global__ void __launch_bounds__(128)
k_lim_verify(const GainJob *__restrict__ jobs, int n_jobs, const ame_track_params *__restrict__ tracks,
             LimStore IN, LimStore OUT, int *__restrict__ need, int *__restrict__ open_count) {
    const int tile = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (tile >= n_jobs) return;
    const GainJob job = jobs[tile];
    int open = 0;
    if ((tracks[job.track].flags & AME_F_LIMITER) && tile > 0 && jobs[tile - 1].track == job.track && !IN.st[tile].exact)
        open = !lim_equal(IN, tile, OUT, tile - 1, lane);
    if (lane == 0) {
        need[tile] = open;
        if (open) atomicAdd(open_count, 1);
    }
}

// what the repair rounds left open: ONE warp per track walks its tiles in order; at an open tile it resumes from the
// predecessor's end and keeps walking until its live state equals the recorded start of a tile that is not open -
// from there on the recorded tiles are the sequential run again
__global__ void __launch_bounds__(32)
k_lim_fallback(const GainJob *__restrict__ jobs, int n_jobs, const ame_track_params *__restrict__ tracks,
               const int16_t *__restrict__ norm, int16_t *__restrict__ out, LimStore IN, LimStore OUT,
               const int *__restrict__ need, int cap) {
    extern __shared__ __align__(16) unsigned char lim_raw[];
    LimSmem sm = lim_smem(lim_raw, cap);
    const int first_tile = blockIdx.x;
    const int track = jobs[first_tile].track;
    if (first_tile > 0 && jobs[first_tile - 1].track == track) return;       // not the first tile of its track
    const ame_track_params *tp = tracks + track;
    if (!(tp->flags & AME_F_LIMITER)) return;
    const LimCtx c = lim_ctx(tp, norm, out);
    const int lane = threadIdx.x;
    LimRegs r;
    bool walking = false;
    for (int tile = first_tile; tile < n_jobs && jobs[tile].track == track; ++tile) {
        if (!walking) {
            if (!need[tile]) continue;
            lim_load(r, sm, OUT, tile - 1, lane);                             // an open tile has a predecessor in its track
            lim_ratios(c, r, sm, lane);
            walking = true;
        }
        lim_run(c, r, sm, jobs[tile].begin, jobs[tile].end, true, lane);
        lim_save(r, sm, OUT, tile, 0, lane);
        __syncwarp();
        const int next = tile + 1;
        if (next < n_jobs && jobs[next].track == track && !need[next] && (IN.st[next].exact || lim_equal_live(r, sm, IN, next, lane)))
            walking = false;
    }
}

// ------------------------------------------------------------------------------------------------
// k_true_peak: ITU-R BS.1770-4 Annex 2 true-peak estimate of the pre-normalisation signal (what loudnorm's
// measured_TP / the linear-mode test TP=-1.5 at :229,240 stand on): the signal oversampled 4x (fs < 96 kHz), 2x
// (fs < 192 kHz) or taken as is, by the 4-phase x 12-tap interpolator of the recommendation, maximum |y| over both
// channels.  One CTA per k_apply_gain tile; float32 arithmetic (a level meter, not on the audio path).
// ------------------------------------------------------------------------------------------------
__constant__ float c_tp_fir[4][12] = {
    {0.0017089843750f, 0.0109863281250f, -0.0196533203125f, 0.0332031250000f, -0.0594482421875f, 0.1373291015625f,
     0.9721679687500f, -0.1022949218750f, 0.0476074218750f, -0.0266113281250f, 0.0148925781250f, -0.0083007812500f},
    {-0.0291748046875f, 0.0292968750000f, -0.0517578125000f, 0.0891113281250f, -0.1665039062500f, 0.4650878906250f,
     0.7797851562500f, -0.2003173828125f, 0.1015625000000f, -0.0582275390625f, 0.0330810546875f, -0.0189208984375f},
    {-0.0189208984375f, 0.0330810546875f, -0.0582275390625f, 0.1015625000000f, -0.2003173828125f, 0.7797851562500f,
     0.4650878906250f, -0.1665039062500f, 0.0891113281250f, -0.0517578125000f, 0.0292968750000f, -0.0291748046875f},
    {-0.0083007812500f, 0.0148925781250f, -0.0266113281250f, 0.0476074218750f, -0.1022949218750f, 0.9721679687500f,
     0.1373291015625f, -0.0594482421875f, 0.0332031250000f, -0.0196533203125f, 0.0109863281250f, 0.0017089843750f}};

// The interpolator over one tile (GainJob) of the track that starts at frame t_begin (the frames before the tile are its
// history), maximum |y| over both channels into the track's float bits.  k_true_peak and k_meter_peak both run it.
__device__ __forceinline__ void true_peak_tile(const GainJob &job, const ame_track_params *tp, const uint32_t *x,
                                               unsigned *__restrict__ tp_bits) {
    const int fs = tp->sample_rate;
    const int step = fs < 96000 ? 1 : 2;                               // phases 0,1,2,3 (4x) or 0,2 (2x)
    const int64_t t_begin = tp->offset_frames + tp->halo_frames;
    float best = 0.0f;
    // 8 frames per thread and iteration, 11 frames of history in front
    for (int64_t n0 = job.begin + (int64_t)threadIdx.x * 8; n0 < job.end; n0 += (int64_t)blockDim.x * 8) {
        float l[19], r[19];
#pragma unroll
        for (int k = 0; k < 19; ++k) {
            const int64_t m = n0 - 11 + k;
            const uint32_t w = (m >= t_begin && m < job.end) ? __ldg(x + m) : 0u;
            l[k] = (float)(int16_t)(w & 0xffffu) * (1.0f / 32768.0f);
            r[k] = (float)(int16_t)(w >> 16) * (1.0f / 32768.0f);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (n0 + i >= job.end) break;
            for (int p = 0; p < 4; p += step) {
                float yl = 0.0f, yr = 0.0f;
#pragma unroll
                for (int k = 0; k < 12; ++k) {                        // y[4n + p] = sum_k h_p[k] x[n - k]
                    yl = fmaf(c_tp_fir[p][k], l[11 + i - k], yl);
                    yr = fmaf(c_tp_fir[p][k], r[11 + i - k], yr);
                }
                best = fmaxf(best, fmaxf(fabsf(yl), fabsf(yr)));
            }
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) best = fmaxf(best, __shfl_xor_sync(kFull, best, d));
    if ((threadIdx.x & 31) == 0 && best > 0.0f) atomicMax(tp_bits + job.track, __float_as_uint(best));
}

__global__ void __launch_bounds__(256)
k_true_peak(const GainJob *__restrict__ jobs, const ame_track_params *__restrict__ tracks, const int16_t *__restrict__ pre,
            unsigned *__restrict__ tp_bits) {
    const GainJob job = jobs[blockIdx.x];
    const ame_track_params *tp = tracks + job.track;
    if (!(tp->flags & AME_F_TRUE_PEAK)) return;
    if (tp->sample_rate >= 192000) return;                             // no oversampling: k_finalize reports the sample peak
    true_peak_tile(job, tp, reinterpret_cast<const uint32_t *>(pre), tp_bits);
}

// ------------------------------------------------------------------------------------------------
// The output meter (AME_F_MEASURE_OUTPUT): EBU R128 over any buffer in the packed layout, for the flagged tracks of a
// wave.  k_kweight_energy fills the meter's own sub-block energies (and the sample peak of the complete sub-blocks),
// k_meter_peak the true peak and the sample peak of every frame, k_meter_finalize the histograms, the maxima and the
// walk.  Every array is indexed by track, so the waves of different slots never share an entry.
// ------------------------------------------------------------------------------------------------
// One CTA per meter peak tile (the k_apply_gain tiles): the BS.1770 interpolator below 192 kHz (whatever the track's
// AME_F_TRUE_PEAK), and max |s16| of every frame of the tile.
__global__ void __launch_bounds__(256)
k_meter_peak(const GainJob *__restrict__ jobs, const ame_track_params *__restrict__ tracks, const int16_t *__restrict__ buf,
             unsigned *__restrict__ tp_bits, int *__restrict__ peak) {
    const GainJob job = jobs[blockIdx.x];
    const ame_track_params *tp = tracks + job.track;
    const uint32_t *x = reinterpret_cast<const uint32_t *>(buf);
    if (tp->sample_rate < 192000) true_peak_tile(job, tp, x, tp_bits);
    int pk = 0;
    for (int64_t f = job.begin + threadIdx.x; f < job.end; f += blockDim.x) {
        const uint32_t w = __ldg(x + f);
        pk = max(pk, max(abs((int)(int16_t)(w & 0xffffu)), abs((int)(int16_t)(w >> 16))));
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) pk = max(pk, __shfl_xor_sync(kFull, pk, d));
    if ((threadIdx.x & 31) == 0 && pk > 0) atomicMax(peak + job.track, pk);
}

__device__ __forceinline__ double block_max(double v, double *s_warp) {   // over the CTA; every thread gets the result
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, d));
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
    __syncthreads();
    v = s_warp[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) v = fmax(v, s_warp[i]);
    __syncthreads();
    return v;
}

__device__ __forceinline__ double lufs_or_inf(double e) { return e >= 0.0 ? 10.0 * log10(e) - 0.691 : -INFINITY; }

// One CTA of 256 threads per flagged track of the wave: both histograms in shared memory exactly as k_block_hist builds
// them, the ungated maxima of the momentary (400 ms) and short-term (3 s) energies at every 100 ms sub-block, then ONE
// thread walks the histograms as k_finalize does and writes the track's ame_loudness.
__global__ void __launch_bounds__(256)
k_meter_finalize(const int32_t *__restrict__ mtracks, const ame_track_params *__restrict__ tracks, const TrackDev *__restrict__ mtdev,
                 const double *__restrict__ energy, const int *__restrict__ peak, const unsigned *__restrict__ tp_bits,
                 ame_loudness *__restrict__ res) {
    __shared__ unsigned s_hist[1000];
    __shared__ unsigned s_st[1000];
    __shared__ double s_warp[8];
    const int t = mtracks[blockIdx.x];
    for (int i = threadIdx.x; i < 1000; i += blockDim.x) { s_hist[i] = 0; s_st[i] = 0; }
    __syncthreads();
    const TrackDev td = mtdev[t];
    const double *e = energy + td.sb_offset;
    const double denom = (double)(4 * (int64_t)td.s100);
    double mom = -1.0, st = -1.0;                    // energies are >= 0: -1 = no complete window
    for (int j = threadIdx.x; j + 3 < td.n_sb; j += blockDim.x) {
        const double s = (((e[j] + e[j + 1]) + e[j + 2]) + e[j + 3]) / denom;
        mom = fmax(mom, s);
        if (s >= c_hist_bounds[0]) atomicAdd(&s_hist[hist_index(s)], 1u);
    }
    // 3 s windows at every sub-block; the ones starting at a whole second are the loudness-range histogram's
    const double denom_st = (double)(30 * (int64_t)td.s100);
    for (int k = threadIdx.x; k + 29 < td.n_sb; k += blockDim.x) {
        double s = 0.0;
        for (int j = 0; j < 30; ++j) s += e[k + j];
        s /= denom_st;
        st = fmax(st, s);
        if (k % 10 == 0 && s >= c_hist_bounds[0]) atomicAdd(&s_st[hist_index(s)], 1u);
    }
    __syncthreads();
    mom = block_max(mom, s_warp);
    st = block_max(st, s_warp);
    if (threadIdx.x != 0) return;
    ame_loudness r;
    const GateWalk g = gate_walk(s_hist);
    r.integrated = g.integrated; r.thresh = g.thresh; r.n_blocks = g.count;
    r.lra = lra_walk(s_st);
    r.sample_peak = peak[t];
    r.true_peak = tracks[t].sample_rate < 192000 ? (double)__uint_as_float(tp_bits[t]) : (double)peak[t] * (1.0 / 32768.0);
    r.max_momentary = lufs_or_inf(mom);
    r.max_short_term = lufs_or_inf(st);
    r.measured = 1;
    res[t] = r;
}

}  // namespace ame

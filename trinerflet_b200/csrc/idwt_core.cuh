// Core of the IDWT level kernels: per-thread phase functions, written so that the SAME code compiles
// for the device (idwt.cu) and for a host-side lock-step emulator used only by the CPU test-suite
// (tests/emu/idwt_emu.cpp) to check the index arithmetic without a GPU.  The product path is the
// CUDA kernel; the emulator is never linked into libtrinerflet_b200.so.
//
// Behavioural contract: one iteration of the level loop of TriPlaneVolume.build_planes
// (/root/reference/reconstruction/triplaneencoder/triplane_encoder.py:379-394):
//     yl = 2*x ; pad yl, yh by 4 ; x' = DWTInverse('bior6.8', mode='zero')((yl, [yh]))
// per axis   y[i] = sum_m lo[m]*g0[i+8-2m] + hi[m]*g1[i+8-2m]   (0 <= i+8-2m < 18, zero outside),
// H axis first on (2*LL, yh0) and (yh1, yh2), then W axis (pytorch_wavelets SFB2D order).
// The other wavelets of the reference's pad table (haar, bior2.2, bior2.6, bior4.4: length L, pad (L-2)/4) use the same
// closed form: their taps sit in the 18-tap frame at G[k + 9 - L/2] = g[k], and padding by 4 with G gives exactly what
// padding by their own pad with g gives.  Every tap is a compile-time constant, so the zero taps of the shorter banks cost
// no instruction.
#pragma once
#include <math.h>
#include <stddef.h>

#include "../../include/trinerflet_b200.h"   // TNL_WAVELET_*

#ifdef __CUDACC__
#define TNL_HD __host__ __device__ __forceinline__
#else
#define TNL_HD inline
#endif

namespace tnl {

// synthesis taps g0 = rec_lo, g1 = rec_hi of wavelet W (TNL_WAVELET_*) in the 18-tap frame
template <int W>
TNL_HD constexpr float rec_lo(int k);
template <int W>
TNL_HD constexpr float rec_hi(int k);

// PyWavelets bior6.8 synthesis taps (rec_lo = g0 has 11 non-zero taps, rec_hi = g1 has 17).
template <>
TNL_HD constexpr float rec_lo<TNL_WAVELET_BIOR6_8>(int k) {
    switch (k) {
        case 3: return 0.014426282505624435f;
        case 4: return 0.014467504896790148f;
        case 5: return -0.07872200106262882f;
        case 6: return -0.04036797903033992f;
        case 7: return 0.41784910915027457f;
        case 8: return 0.7589077294536541f;
        case 9: return 0.41784910915027457f;
        case 10: return -0.04036797903033992f;
        case 11: return -0.07872200106262882f;
        case 12: return 0.014467504896790148f;
        case 13: return 0.014426282505624435f;
        default: return 0.0f;
    }
}
template <>
TNL_HD constexpr float rec_hi<TNL_WAVELET_BIOR6_8>(int k) {
    switch (k) {
        case 1: return -0.0019088317364812906f;
        case 2: return -0.0019142861290887667f;
        case 3: return 0.016990639867602342f;
        case 4: return 0.01193456527972926f;
        case 5: return -0.04973290349094079f;
        case 6: return -0.07726317316720414f;
        case 7: return 0.09405920349573646f;
        case 8: return 0.4207962846098268f;
        case 9: return -0.8259229974584023f;
        case 10: return 0.4207962846098268f;
        case 11: return 0.09405920349573646f;
        case 12: return -0.07726317316720414f;
        case 13: return -0.04973290349094079f;
        case 14: return 0.01193456527972926f;
        case 15: return 0.016990639867602342f;
        case 16: return -0.0019142861290887667f;
        case 17: return -0.0019088317364812906f;
        default: return 0.0f;
    }
}

// PyWavelets haar, bior2.2, bior2.6, bior4.4 (tests/wavelet_oracle.py), placed in the frame
template <>
TNL_HD constexpr float rec_lo<TNL_WAVELET_HAAR>(int k) {
    switch (k) {
        case 8: return 0.7071067811865476f;
        case 9: return 0.7071067811865476f;
        default: return 0.0f;
    }
}
template <>
TNL_HD constexpr float rec_hi<TNL_WAVELET_HAAR>(int k) {
    switch (k) {
        case 8: return 0.7071067811865476f;
        case 9: return -0.7071067811865476f;
        default: return 0.0f;
    }
}
template <>
TNL_HD constexpr float rec_lo<TNL_WAVELET_BIOR2_2>(int k) {
    switch (k) {
        case 7: return 0.3535533905932738f;
        case 8: return 0.7071067811865476f;
        case 9: return 0.3535533905932738f;
        default: return 0.0f;
    }
}
template <>
TNL_HD constexpr float rec_hi<TNL_WAVELET_BIOR2_2>(int k) {
    switch (k) {
        case 7: return 0.1767766952966369f;
        case 8: return 0.3535533905932738f;
        case 9: return -1.0606601717798214f;
        case 10: return 0.3535533905932738f;
        case 11: return 0.1767766952966369f;
        default: return 0.0f;
    }
}
template <>
TNL_HD constexpr float rec_lo<TNL_WAVELET_BIOR2_6>(int k) {
    switch (k) {
        case 7: return 0.3535533905932738f;
        case 8: return 0.7071067811865476f;
        case 9: return 0.3535533905932738f;
        default: return 0.0f;
    }
}
template <>
TNL_HD constexpr float rec_hi<TNL_WAVELET_BIOR2_6>(int k) {
    switch (k) {
        case 3: return 0.006905339660024878f;
        case 4: return 0.013810679320049757f;
        case 5: return -0.046956309688169176f;
        case 6: return -0.10772329869638811f;
        case 7: return 0.16987135563661201f;
        case 8: return 0.4474660099696121f;
        case 9: return -0.966747552403483f;
        case 10: return 0.4474660099696121f;
        case 11: return 0.16987135563661201f;
        case 12: return -0.10772329869638811f;
        case 13: return -0.046956309688169176f;
        case 14: return 0.013810679320049757f;
        case 15: return 0.006905339660024878f;
        default: return 0.0f;
    }
}
template <>
TNL_HD constexpr float rec_lo<TNL_WAVELET_BIOR4_4>(int k) {
    switch (k) {
        case 5: return -0.06453888262869706f;
        case 6: return -0.04068941760916406f;
        case 7: return 0.41809227322161724f;
        case 8: return 0.7884856164055829f;
        case 9: return 0.41809227322161724f;
        case 10: return -0.04068941760916406f;
        case 11: return -0.06453888262869706f;
        default: return 0.0f;
    }
}
template <>
TNL_HD constexpr float rec_hi<TNL_WAVELET_BIOR4_4>(int k) {
    switch (k) {
        case 5: return -0.03782845550726404f;
        case 6: return -0.023849465019556843f;
        case 7: return 0.11062440441843718f;
        case 8: return 0.37740285561283066f;
        case 9: return -0.8526986790088938f;
        case 10: return 0.37740285561283066f;
        case 11: return 0.11062440441843718f;
        case 12: return -0.023849465019556843f;
        case 13: return -0.03782845550726404f;
        default: return 0.0f;
    }
}

// W-axis synthesis (fwd_phase_b): does window element i reach a non-zero tap of g1 (HI) or g0 for one of its two output
// pairs e (tap index d = i - e)?  Elements that reach none are not loaded.
template <int W, bool HI>
TNL_HD constexpr bool wsyn_reaches(int i) {
    for (int e = 0; e < 2; ++e) {
        const int d = i - e;
        if (d < 0 || d > 8) continue;
        const float ge = HI ? rec_hi<W>(16 - 2 * d) : rec_lo<W>(16 - 2 * d);
        const float go = HI ? rec_hi<W>(17 - 2 * d) : rec_lo<W>(17 - 2 * d);
        if (ge != 0.f || go != 0.f) return true;
    }
    return false;
}

// async 4-byte global->shared copy with zero fill; the host emulator provides a synchronous version
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int sz = valid ? 4 : 0;  // src-size 0 => destination zero-filled (this IS the zero padding)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }
#else
inline void cp_async4(float* smem_dst, const float* gsrc, bool valid) { *smem_dst = valid ? *gsrc : 0.0f; }
inline void cp_async_commit() {}
template <int N>
inline void cp_async_wait() {}
#endif

// packed pair of floats; on the device an FFMA2 (sm_100 packed fp32 FMA, one issue slot for two FMAs) with the tap as
// a broadcast immediate, on the host (emulator) two fmaf() -- identical round-to-nearest results.
#if defined(__CUDA_ARCH__)
typedef float2 f2;
__device__ __forceinline__ f2 mk2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ f2 fma2(float g, f2 w, f2 acc) { return __ffma2_rn(make_float2(g, g), w, acc); }
#else
struct f2 { float x, y; };
inline f2 mk2(float a, float b) { f2 r; r.x = a; r.y = b; return r; }
inline f2 fma2(float g, f2 w, f2 acc) { f2 r; r.x = fmaf(g, w.x, acc.x); r.y = fmaf(g, w.y, acc.y); return r; }
#endif

template <int CG_, int TW_>
struct IdwtCfg {
    static constexpr int CG = CG_;      // channels per CTA (even)
    static constexpr int TW = TW_;      // fine-resolution columns per strip (32)
    static constexpr int TM = TW / 2;   // coarse-resolution columns per strip (16)
    static constexpr int RA = 3;        // coarse rows per step
    static constexpr int RB = 2 * RA;   // fine rows per step
    static constexpr int WIN = TM + 8;  // coarse columns incl. halo (24) == fine columns incl. halo / 2
    static constexpr int NT = WIN * CG; // threads per CTA
    static constexpr int pad_to(int len) { return len + (((CG - len) % 32) + 32) % 32; }  // stride == CG (mod 32)
    static constexpr int RS_F = pad_to(WIN * CG);      // forward mid row stride (floats)
    static constexpr int RS_B = 2 * WIN * CG;          // backward mid row stride (pairs (a,b); 48 fine columns)
    static constexpr int MID_F = 2 * RB * RS_F;        // floats per forward mid buffer  (2 bands x 6 rows)
    static constexpr int MID_B = 2 * RA * RS_B;        // floats per backward mid buffer (3 rows x 48 cols x CG x (a,b))
    static constexpr int STAGE = 4 * RA * NT;          // floats per input stage (12 per thread)
    static constexpr int NSTAGE = 3;                   // cp.async ring depth: inputs are staged two steps ahead
    static constexpr size_t SMEM_F = sizeof(float) * (2 * MID_F + NSTAGE * STAGE);
    static constexpr size_t SMEM_B = sizeof(float) * (2 * MID_B + NSTAGE * STAGE);
    static_assert(CG % 2 == 0, "channel pairs");
    static_assert(RB * (TW / 4) * (CG / 2) == NT, "forward phase-B item count must equal the thread count");
    static_assert(RA * (TM / 2) * CG == NT, "backward phase-B item count must equal the thread count");
};

struct IdwtBlock {
    int bx, by, bz;
};

// per-thread geometry shared by both directions
struct IdwtGeom {
    int n, C, plane, c0, m0, row_lo, row_hi, col, chan;
    int begin, end, nsteps;  // streamed coarse rows (fwd) / fine row pairs (bwd): [begin, end)
};

template <typename Cfg>
TNL_HD IdwtGeom idwt_geom(int tid, IdwtBlock b, int n, int C, int rows_per_cta) {
    IdwtGeom g;
    g.n = n;
    g.C = C;
    // channel chunks of the same strip are adjacent in launch order (bx fastest): they read the two halves of the same
    // 128-byte lines, so the second one hits L2 (ncu: with the chunk in bz every input line came from DRAM twice)
    const int chunks = C / Cfg::CG;
    g.plane = b.bz;
    g.c0 = (b.bx % chunks) * Cfg::CG;
    g.m0 = (b.bx / chunks) * Cfg::TM;
    g.row_lo = b.by * rows_per_cta;
    g.row_hi = g.row_lo + rows_per_cta < n ? g.row_lo + rows_per_cta : n;
    g.col = tid / Cfg::CG;
    g.chan = g.c0 + tid % Cfg::CG;
    // centre row m needs streamed rows m-4 .. m+4 (bwd: fine row pairs m-4 .. m+4); m is emitted when m+4 arrives
    g.begin = g.row_lo - 4;
    g.end = g.row_hi + 4;
    g.nsteps = (g.end - g.begin + Cfg::RA - 1) / Cfg::RA;
    return g;
}

// work-list mode: the CTA's block comes from an item {plane, first coarse column, row_lo, row_hi} instead of the grid
struct IdwtItem {
    int plane, m0, row_lo, row_hi;
};

template <typename Cfg>
TNL_HD IdwtGeom idwt_geom_item(int tid, int chunk, IdwtItem it, int n, int C) {
    IdwtGeom g;
    g.n = n;
    g.C = C;
    g.plane = it.plane;
    g.c0 = chunk * Cfg::CG;
    g.m0 = it.m0;
    g.row_lo = it.row_lo;
    g.row_hi = it.row_hi < n ? it.row_hi : n;
    g.col = tid / Cfg::CG;
    g.chan = g.c0 + tid % Cfg::CG;
    g.begin = g.row_lo - 4;
    g.end = g.row_hi + 4;
    g.nsteps = (g.end - g.begin + Cfg::RA - 1) / Cfg::RA;
    return g;
}

// ================================================================================================
// forward
// ================================================================================================
struct FwdState {
    f2 wL[9];       // (2*LL, HL): both enter the H-axis low-pass taps
    f2 wH[9];       // (LH, HH):   both enter the H-axis high-pass taps
    float abs_acc;  // sum |yh| over the detail coefficients this thread owns (wavelet L1 regulariser by-product)
    const float *pLL, *pH0, *pH1, *pH2;  // running pointers: this thread's column at the next row to stage
    int next_j;                          // that row index (may be negative / past the end: staged as zeros)
    unsigned j_lim;                      // rows [0, j_lim) are real data for this CTA
    bool col_ok;
    // phase-B item (constant over the steps): mid-buffer offsets, output offset
    int b_lo, b_hi, b_r, b_sb;
    size_t b_out;
};

template <typename Cfg>
TNL_HD void fwd_state_init(FwdState& st, const IdwtGeom& g, const float* x, const float* yh, int tid) {
    for (int i = 0; i < 9; ++i) st.wL[i] = st.wH[i] = mk2(0.f, 0.f);
    st.abs_acc = 0.f;
    const int mcol = g.m0 - 4 + g.col;
    st.col_ok = mcol >= 0 && mcol < g.n;
    const long long plane_px = (long long)g.n * g.n;
    const long long row_stride = (long long)g.n * g.C;
    st.next_j = g.begin;
    st.j_lim = (unsigned)(g.end < g.n ? g.end : g.n);
    const long long off = (long long)(st.col_ok ? mcol : 0) * g.C + g.chan + (long long)g.begin * row_stride;
    st.pLL = x + (long long)g.plane * plane_px * g.C + off;
    st.pH0 = yh + (long long)(g.plane * 3 + 0) * plane_px * g.C + off;
    st.pH1 = yh + (long long)(g.plane * 3 + 1) * plane_px * g.C + off;
    st.pH2 = yh + (long long)(g.plane * 3 + 2) * plane_px * g.C + off;
    const int cp = tid % (Cfg::CG / 2), rs = tid / (Cfg::CG / 2);
    st.b_r = rs % Cfg::RB;
    st.b_sb = rs / Cfg::RB;
    st.b_lo = (0 * Cfg::RB + st.b_r) * Cfg::RS_F + (2 * st.b_sb) * Cfg::CG + 2 * cp;
    st.b_hi = (1 * Cfg::RB + st.b_r) * Cfg::RS_F + (2 * st.b_sb) * Cfg::CG + 2 * cp;
    const int n2 = 2 * g.n;
    st.b_out = ((size_t)g.plane * n2 * n2 + (size_t)2 * (g.m0 + 2 * st.b_sb)) * g.C + g.c0 + 2 * cp;
}

// stage the next RA coarse rows for this thread's column: stage[(rr*NT + tid)*4 + {LL, HL, LH, HH}]
// (that order makes one 128-bit shared load deliver the register pairs (LL,HL) and (LH,HH) without moves).
// Rows outside the tensor / the chunk are zero-filled (src-size 0: the address is not dereferenced).
template <typename Cfg>
TNL_HD void fwd_issue_stage(const IdwtGeom& g, FwdState& st, float* stage, int tid) {
    const long long row_stride = (long long)g.n * g.C;
    float* d = stage + (size_t)tid * 4;
#pragma unroll
    for (int rr = 0; rr < Cfg::RA; ++rr) {
        const bool ok = st.col_ok && (unsigned)(st.next_j + rr) < st.j_lim;
        cp_async4(d + rr * Cfg::NT * 4 + 0, st.pLL + rr * row_stride, ok);
        cp_async4(d + rr * Cfg::NT * 4 + 1, st.pH1 + rr * row_stride, ok);
        cp_async4(d + rr * Cfg::NT * 4 + 2, st.pH0 + rr * row_stride, ok);
        cp_async4(d + rr * Cfg::NT * 4 + 3, st.pH2 + rr * row_stride, ok);
    }
    cp_async_commit();
    st.next_j += Cfg::RA;
    st.pLL += Cfg::RA * row_stride;
    st.pH0 += Cfg::RA * row_stride;
    st.pH1 += Cfg::RA * row_stride;
    st.pH2 += Cfg::RA * row_stride;
}

// The phase functions take the wavelet as their last template argument; it defaults to bior6.8 for the lock-step emulator
// (tests/emu/idwt_emu.cpp).
// H-axis synthesis; newest sample at ring slot SLOT:  W[d] = w[(SLOT + 1 + d) % 9], d = 0 (row m-4) .. 8 (row m+4)
//   even = sum_d W[d] g[16-2d],  odd = sum_d W[d] g[17-2d];  .x = low band pair (2LL, LH), .y = high band pair (HL, HH)
template <int SLOT, int W = TNL_WAVELET_BIOR6_8>
TNL_HD void synth_rows(const f2 (&wL)[9], const f2 (&wH)[9], f2& even, f2& odd) {
    f2 e = mk2(0.f, 0.f), o = mk2(0.f, 0.f);
#pragma unroll
    for (int d = 0; d < 9; ++d) {
        const f2 l = wL[(SLOT + 1 + d) % 9], h = wH[(SLOT + 1 + d) % 9];
        const float ge0 = rec_lo<W>(16 - 2 * d), go0 = rec_lo<W>(17 - 2 * d);
        const float ge1 = rec_hi<W>(16 - 2 * d), go1 = rec_hi<W>(17 - 2 * d);
        if (ge0 != 0.f) e = fma2(ge0, l, e);
        if (go0 != 0.f) o = fma2(go0, l, o);
        if (ge1 != 0.f) e = fma2(ge1, h, e);
        if (go1 != 0.f) o = fma2(go1, h, o);
    }
    even = e;
    odd = o;
}

template <int SLOT, int W = TNL_WAVELET_BIOR6_8>
TNL_HD void fwd_row(FwdState& st, const float* stage, float* mid, int tid, int rr, int NT, int RB, int RS, bool own) {
    const f2* s = reinterpret_cast<const f2*>(stage + ((size_t)rr * NT + tid) * 4);
    f2 l = s[0];                     // (LL, HL)
    const f2 h = s[1];               // (LH, HH)
    if (own) st.abs_acc += fabsf(l.y) + fabsf(h.x) + fabsf(h.y);
    l.x = l.x + l.x;                 // yl = 2*x (exact)
    st.wL[SLOT] = l;
    st.wH[SLOT] = h;
    f2 e, o;
    synth_rows<SLOT, W>(st.wL, st.wH, e, o);
    mid[(0 * RB + 2 * rr) * RS + tid] = e.x;
    mid[(0 * RB + 2 * rr + 1) * RS + tid] = o.x;
    mid[(1 * RB + 2 * rr) * RS + tid] = e.y;
    mid[(1 * RB + 2 * rr + 1) * RS + tid] = o.y;
}

// phase A of step phase PH (= step index mod 3): RA rows enter the windows at ring slots 3*PH .. 3*PH+2
template <typename Cfg, int PH, int W = TNL_WAVELET_BIOR6_8>
TNL_HD void fwd_phase_a(const IdwtGeom& g, FwdState& st, const float* stage, float* mid, int tid, int ss) {
    // a coefficient is "owned" by exactly one CTA: its column lies in the strip proper (not the halo) and its row in the chunk
    const bool col_own = g.col >= 4 && g.col < 4 + Cfg::TM;
    const int j0 = g.begin + ss * Cfg::RA;
    fwd_row<(PH * 3 + 0) % 9, W>(st, stage, mid, tid, 0, Cfg::NT, Cfg::RB, Cfg::RS_F, col_own && j0 + 0 >= g.row_lo && j0 + 0 < g.row_hi);
    fwd_row<(PH * 3 + 1) % 9, W>(st, stage, mid, tid, 1, Cfg::NT, Cfg::RB, Cfg::RS_F, col_own && j0 + 1 >= g.row_lo && j0 + 1 < g.row_hi);
    fwd_row<(PH * 3 + 2) % 9, W>(st, stage, mid, tid, 2, Cfg::NT, Cfg::RB, Cfg::RS_F, col_own && j0 + 2 >= g.row_lo && j0 + 2 < g.row_hi);
}

// phase B: W-axis synthesis. item = (mid row r, strip sb of 4 output columns, channel pair cp)
template <typename Cfg, int W = TNL_WAVELET_BIOR6_8>
TNL_HD void fwd_phase_b(const IdwtGeom& g, const FwdState& st, const float* mid, float* out, int ss) {
    const int r = st.b_r;
    const int m = g.begin + ss * Cfg::RA + (r >> 1) - 4;  // coarse row whose synthesis produced mid row r
    if (m < g.row_lo || m >= g.row_hi) return;
    const f2* mlo = reinterpret_cast<const f2*>(mid + st.b_lo);
    const f2* mhi = reinterpret_cast<const f2*>(mid + st.b_hi);
    // stream the window: element i feeds output pair e with tap index d = i - e; nothing is kept but the accumulators
    f2 ev[2] = {mk2(0.f, 0.f), mk2(0.f, 0.f)}, od[2] = {mk2(0.f, 0.f), mk2(0.f, 0.f)};
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        f2 h = mk2(0.f, 0.f), l = mk2(0.f, 0.f);
        if (wsyn_reaches<W, true>(i)) h = mhi[i * (Cfg::CG / 2)];
        if (wsyn_reaches<W, false>(i)) l = mlo[i * (Cfg::CG / 2)];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int d = i - e;
            if (d < 0 || d > 8) continue;
            const float ge0 = rec_lo<W>(16 - 2 * d), go0 = rec_lo<W>(17 - 2 * d);
            const float ge1 = rec_hi<W>(16 - 2 * d), go1 = rec_hi<W>(17 - 2 * d);
            if (ge0 != 0.f) ev[e] = fma2(ge0, l, ev[e]);
            if (go0 != 0.f) od[e] = fma2(go0, l, od[e]);
            if (ge1 != 0.f) ev[e] = fma2(ge1, h, ev[e]);
            if (go1 != 0.f) od[e] = fma2(go1, h, od[e]);
        }
    }
    const int Y = 2 * m + (r & 1);
    const int n2 = 2 * g.n;
    f2* orow = reinterpret_cast<f2*>(out + st.b_out + (size_t)Y * n2 * g.C);
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int X = 2 * (g.m0 + 2 * st.b_sb + e);
        if (X < n2) {
            orow[(size_t)(2 * e) * (g.C / 2)] = ev[e];
            orow[(size_t)(2 * e + 1) * (g.C / 2)] = od[e];
        }
    }
}

// ================================================================================================
// backward (adjoint).  g_out [3][2n][2n][C] -> g_x [3][n][n][C] (includes the factor 2), g_yh [3][3][n][n][C]
//   a[m][X] = sum_k g0[k] G[2m-8+k][X]         b[m][X] = sum_k g1[k] G[2m-8+k][X]        (H-axis adjoint)
//   gLL[m][w] = 2 sum_k g0[k] a[m][2w-8+k]      gHL[m][w] = sum_k g1[k] a[m][2w-8+k]      (W-axis adjoint)
//   gLH[m][w] =   sum_k g0[k] b[m][2w-8+k]      gHH[m][w] = sum_k g1[k] b[m][2w-8+k]
// thread <-> two fine columns (Xa = 2*m0-8+col, Xb = Xa + WIN) x channel, 18-deep register windows of pairs (G[.][Xa], G[.][Xb]).
// ================================================================================================
struct BwdState {
    f2 w[18];
    const float *pa, *pb;  // running pointers: columns Xa / Xb at the next fine row to stage
    int next_y;
    unsigned y_lim;
    bool oka, okb;
};

template <typename Cfg>
TNL_HD void bwd_state_init(BwdState& st, const IdwtGeom& g, const float* gout) {
    for (int i = 0; i < 18; ++i) st.w[i] = mk2(0.f, 0.f);
    const int n2 = 2 * g.n;
    const int Xa = 2 * g.m0 - 8 + g.col, Xb = Xa + Cfg::WIN;
    st.oka = Xa >= 0 && Xa < n2;
    st.okb = Xb >= 0 && Xb < n2;
    st.next_y = 2 * g.begin;
    st.y_lim = (unsigned)(2 * g.end < n2 ? 2 * g.end : n2);
    const long long row_stride = (long long)n2 * g.C;
    const long long base = (long long)g.plane * n2 * row_stride + g.chan + (long long)st.next_y * row_stride;
    st.pa = gout + base + (long long)(st.oka ? Xa : 0) * g.C;
    st.pb = gout + base + (long long)(st.okb ? Xb : 0) * g.C;
}

// stage[(rr2*NT + tid)*2 + {a, b}], rr2 = 0 .. 2*RA-1 fine rows of the step
template <typename Cfg>
TNL_HD void bwd_issue_stage(const IdwtGeom& g, BwdState& st, float* stage, int tid) {
    const long long row_stride = (long long)(2 * g.n) * g.C;
    float* d = stage + (size_t)tid * 2;
#pragma unroll
    for (int rr = 0; rr < 2 * Cfg::RA; ++rr) {
        const bool rok = (unsigned)(st.next_y + rr) < st.y_lim;
        cp_async4(d + rr * Cfg::NT * 2 + 0, st.pa + rr * row_stride, rok && st.oka);
        cp_async4(d + rr * Cfg::NT * 2 + 1, st.pb + rr * row_stride, rok && st.okb);
    }
    cp_async_commit();
    st.next_y += 2 * Cfg::RA;
    st.pa += 2 * Cfg::RA * row_stride;
    st.pb += 2 * Cfg::RA * row_stride;
}

// newest sample (k = 17) at ring slot SLOT;  U[k] = w[(SLOT + 1 + k) % 18];  .x = column Xa, .y = column Xb
template <int SLOT, int W = TNL_WAVELET_BIOR6_8>
TNL_HD void analyse(const f2 (&w)[18], f2& a, f2& b) {
    f2 ra = mk2(0.f, 0.f), rb = mk2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 18; ++k) {
        const f2 u = w[(SLOT + 1 + k) % 18];
        const float g0 = rec_lo<W>(k), g1 = rec_hi<W>(k);
        if (g0 != 0.f) ra = fma2(g0, u, ra);
        if (g1 != 0.f) rb = fma2(g1, u, rb);
    }
    a = ra;
    b = rb;
}

template <int SLOT, int W = TNL_WAVELET_BIOR6_8>  // SLOT = ring slot of the second (newest) row of the pair; odd
TNL_HD void bwd_row(BwdState& st, const float* stage, float* mid, int tid, int rr, int NT, int RS) {
    const f2* s = reinterpret_cast<const f2*>(stage);
    st.w[(SLOT + 17) % 18] = s[(size_t)(2 * rr) * NT + tid];
    st.w[SLOT] = s[(size_t)(2 * rr + 1) * NT + tid];
    f2 a, b;
    analyse<SLOT, W>(st.w, a, b);
    // mid layout [row rr][fine column 0..2*WIN)[CG] of pairs (a, b); this thread owns columns col and col + WIN
    f2* m2 = reinterpret_cast<f2*>(mid);
    m2[(size_t)rr * RS + tid] = mk2(a.x, b.x);
    m2[(size_t)rr * RS + NT + tid] = mk2(a.y, b.y);
}

template <typename Cfg, int PH, int W = TNL_WAVELET_BIOR6_8>
TNL_HD void bwd_phase_a(BwdState& st, const float* stage, float* mid, int tid) {
    bwd_row<(2 * (PH * 3 + 0) + 1) % 18, W>(st, stage, mid, tid, 0, Cfg::NT, Cfg::RS_B);
    bwd_row<(2 * (PH * 3 + 1) + 1) % 18, W>(st, stage, mid, tid, 1, Cfg::NT, Cfg::RS_B);
    bwd_row<(2 * (PH * 3 + 2) + 1) % 18, W>(st, stage, mid, tid, 2, Cfg::NT, Cfg::RS_B);
}

TNL_HD float signf_(float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); }  // torch.sign

// phase B: W-axis adjoint. item = (row r, pair of coarse columns sb, channel cb).
// yh / reg: optional fused gradient of the wavelet L1 regulariser, g_yh += reg * sign(yh)  (nerf/utils.py:640-655)
template <typename Cfg, int W = TNL_WAVELET_BIOR6_8>
TNL_HD void bwd_phase_b(const IdwtGeom& g, const float* mid, float* g_x, float* g_yh, int tid, int ss, const float* yh,
                        float reg) {
    const int cb = tid % Cfg::CG;
    const int rs = tid / Cfg::CG;  // 0 .. 23 = 3 rows x 8 column pairs
    const int r = rs % Cfg::RA;
    const int sb = rs / Cfg::RA;   // coarse columns m0 + 2*sb, m0 + 2*sb + 1
    const int m = g.begin + ss * Cfg::RA + r - 4;
    if (m < g.row_lo || m >= g.row_hi) return;
    const size_t plane_px = (size_t)g.n * g.n;
    const int w0 = g.m0 + 2 * sb;
    // issue the regulariser's coefficient loads first so that their latency hides behind the FMA work
    float y[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
    if (yh != nullptr) {
#pragma unroll
        for (int e = 0; e < 2; ++e)
            if (w0 + e < g.n) {
                const size_t px = (size_t)m * g.n + w0 + e;
#pragma unroll
                for (int b = 0; b < 3; ++b) y[e][b] = yh[((size_t)(g.plane * 3 + b) * plane_px + px) * g.C + g.c0 + cb];
            }
    }
    // fine column X = 2w - 8 + k ; buffer column = X - (2*m0 - 8) = 2*(w - m0) + k.  Streamed: window element i feeds
    // coarse column e with tap k = i - 2e.
    const f2* mab = reinterpret_cast<const f2*>(mid) + (size_t)r * Cfg::RS_B + (4 * sb) * Cfg::CG + cb;
    f2 lo[2] = {mk2(0.f, 0.f), mk2(0.f, 0.f)}, hi[2] = {mk2(0.f, 0.f), mk2(0.f, 0.f)};  // lo = (gLL/2, gLH), hi = (gHL, gHH)
#pragma unroll
    for (int i = 0; i < 20; ++i) {
        const f2 v = mab[i * Cfg::CG];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int k = i - 2 * e;
            if (k < 0 || k > 17) continue;
            const float g0 = rec_lo<W>(k), g1 = rec_hi<W>(k);
            if (g0 != 0.f) lo[e] = fma2(g0, v, lo[e]);
            if (g1 != 0.f) hi[e] = fma2(g1, v, hi[e]);
        }
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int w = w0 + e;
        if (w < g.n) {
            const size_t px = (size_t)m * g.n + w;
            float lh = lo[e].y, hl = hi[e].x, hh = hi[e].y;
            if (yh != nullptr) {
                lh = fmaf(reg, signf_(y[e][0]), lh);
                hl = fmaf(reg, signf_(y[e][1]), hl);
                hh = fmaf(reg, signf_(y[e][2]), hh);
            }
            g_x[((size_t)g.plane * plane_px + px) * g.C + g.c0 + cb] = 2.0f * lo[e].x;
            g_yh[((size_t)(g.plane * 3 + 0) * plane_px + px) * g.C + g.c0 + cb] = lh;
            g_yh[((size_t)(g.plane * 3 + 1) * plane_px + px) * g.C + g.c0 + cb] = hl;
            g_yh[((size_t)(g.plane * 3 + 2) * plane_px + px) * g.C + g.c0 + cb] = hh;
        }
    }
}

// launch geometry shared by the kernel launcher and the emulator
template <typename Cfg>
inline void idwt_grid(unsigned n, unsigned C, unsigned num_sm, unsigned& gx, unsigned& gy, unsigned& gz, unsigned& rows) {
    gx = ((n + Cfg::TM - 1) / Cfg::TM) * (C / Cfg::CG);
    gz = 3;
    rows = 96;  // halo overhead 8/rows; shrink the chunk until the grid covers the machine a few times
    while (rows > 24 && gx * ((n + rows - 1) / rows) * gz < 4 * num_sm) rows /= 2;
    if (rows > n) rows = n;
    gy = (n + rows - 1) / rows;
}

}  // namespace tnl

// ts_common.cuh -- index remapping, weight split and interpolation arithmetic shared by every
// kernel of the B200 shift operator (host+device so the CPU-side tests can pin the formulas).
//
// Semantics follow the reference (paths relative to torchshifts/csrc/ops/):
//   remap_literal          kernels/shifts_kernels.h:10-29   infer_index
//   axis_index             kernels/shifts_kernels.h:40-50   size-1 axes ignore their shift
//   split_forward/backward cpu/shifts_cpu.cpp:223-224, :242-244
//   lerp / interp          kernels/interpolation.h:3-38     (three separately rounded ops, no FMA)
//   weight partials        kernels/interpolation.h:9-61, shifts_kernels.h:132-154
// but none of the code is taken from there: the device form below is division-free (shifts are
// reduced once per channel to a bounded congruent value, then wraps are done by compare/add).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/torchshifts_b200.h"

#define TS_HD __host__ __device__ __forceinline__
#define TS_D __device__ __forceinline__

namespace ts {

// ------------------------------------------------------------------------------------------
// Geometry handed to kernels by value.
struct Geo {
    int dim, pad;
    int wf32;            // weights are fp32 whatever the element type (TS_WEIGHTS_F32 with fp16 / bf16 x)
    long long N, C;
    int S[3];            // input sizes
    int OS[3];           // output sizes (rb - lb)
    int lb[3];
    long long xs[5];     // x strides in elements
    long long in_plane;  // S0*S1*S2
    long long out_plane; // OS0*OS1*OS2
};

// Tensor axis of a LEVEL (0 slab, 1 row, 2 column) of a `dim`-dimensional geometry; negative: the level is absent.
TS_HD int level_axis(int level, int dim) { return level - (3 - dim); }

// Exact division by a launch-invariant (n < 2^31), set up on the host; the device side is fdiv (ts_ptx.cuh).
struct FastDiv { unsigned m, l, d; };
inline FastDiv make_fastdiv(unsigned d) {
    FastDiv f;
    f.d = d ? d : 1;
    unsigned l = 0;
    while ((1ull << l) < f.d) ++l;
    f.l = l;
    f.m = (unsigned)(((((unsigned long long)1 << l) - f.d) << 32) / f.d + 1);
    return f;
}

// ------------------------------------------------------------------------------------------
// Index remap.
TS_HD int pmod(int a, int b) { return (b + (a % b)) % b; }

// Literal formula (divisions).  Negative result = "outside, use the pad value".
TS_HD int remap_literal(int idx, int len, int pad) {
    switch (pad) {
    case TS_PAD_BORDER: return idx < 0 ? 0 : (idx > len - 1 ? len - 1 : idx);
    case TS_PAD_PERIODIC: return pmod(idx, len);
    case TS_PAD_REFLECT: {
        int neg = idx < 0 ? 1 : 0, a = idx < 0 ? -idx : idx;
        int odd = (neg + (a - neg) / (len - 1)) & 1;
        int m = pmod(idx, len - 1);
        return odd ? (len - 1 - m) : m;
    }
    case TS_PAD_SYMMETRIC: {
        int neg = idx < 0 ? 1 : 0, a = idx < 0 ? -idx : idx;
        int odd = (neg + (a - neg) / len) & 1;
        int m = pmod(idx, len);
        return odd ? (len - 1 - m) : m;
    }
    default: return idx > len - 1 ? -1 : idx;
    }
}

// Period of the remap as a function of the index (0 = not periodic: zeros / border).
TS_HD int remap_period(int len, int pad) {
    return pad == TS_PAD_PERIODIC ? len : pad == TS_PAD_REFLECT ? 2 * (len - 1) : pad == TS_PAD_SYMMETRIC ? 2 * len : 0;
}

// Replace an arbitrary 64-bit shift by a bounded one that gives the same remapped index for
// every position in [0,len) and its +1 neighbour.  |result| <= len+1 (zeros/border) or < period.
TS_HD int reduce_shift(long long s, int len, int pad) {
    if (len <= 1) return 0;                     // size-1 axis: the shift is ignored altogether
    const int period = remap_period(len, pad);
    if (period == 0) {
        const long long lim = (long long)len + 1;
        return (int)(s < -lim ? -lim : (s > lim ? lim : s));
    }
    return (int)(s % (long long)period);
}

// Division-free remap, valid for idx in [-(P-1), len+P-1] (P = period), i.e. for
// idx = pos - reduce_shift(..) (+1) with pos in [0,len).  Template so PAD folds at compile time
// in the staged kernels; the generic kernels pass it at run time.
TS_HD int remap_bounded(int idx, int len, int pad) {
    switch (pad) {
    case TS_PAD_BORDER: return idx < 0 ? 0 : (idx > len - 1 ? len - 1 : idx);
    case TS_PAD_PERIODIC:
        if (idx < 0) idx += len;
        if (idx >= len) idx -= len;
        return idx;
    case TS_PAD_REFLECT: {
        const int P = 2 * (len - 1);
        if (idx < 0) idx += P;
        if (idx >= P) idx -= P;
        return idx <= len - 1 ? idx : P - idx;
    }
    case TS_PAD_SYMMETRIC: {
        const int P = 2 * len;
        if (idx < 0) idx += P;
        if (idx >= P) idx -= P;
        return idx < len ? idx : P - 1 - idx;
    }
    default: return idx > len - 1 ? -1 : idx;
    }
}

// One axis of get_shifted_value: a size-1 axis always maps to 0.
TS_HD int axis_index(int idx, int len, int pad) { return len == 1 ? 0 : remap_bounded(idx, len, pad); }
// same with the literal (division) formula: valid for ANY index, not only idx = pos - reduce_shift(..) (+1)
TS_HD int axis_index_literal(int idx, int len, int pad) { return len == 1 ? 0 : remap_literal(idx, len, pad); }

// ------------------------------------------------------------------------------------------
// Unfused arithmetic (the oracle is compiled without FMA; active forward / grad_input must be
// bit-exact, so every product and sum is rounded separately).
template <typename T> struct Arith;
template <> struct Arith<float> {
    static TS_HD float add(float a, float b) {
#ifdef __CUDA_ARCH__
        return __fadd_rn(a, b);
#else
        volatile float r = a + b; return r;
#endif
    }
    static TS_HD float sub(float a, float b) {
#ifdef __CUDA_ARCH__
        return __fsub_rn(a, b);
#else
        volatile float r = a - b; return r;
#endif
    }
    static TS_HD float mul(float a, float b) {
#ifdef __CUDA_ARCH__
        return __fmul_rn(a, b);
#else
        volatile float r = a * b; return r;
#endif
    }
    static TS_HD float floor_(float a) { return floorf(a); }
    static TS_HD float ceil_(float a) { return ceilf(a); }
    static TS_HD float rint_(float a) { return rintf(a); }
};
template <> struct Arith<double> {
    static TS_HD double add(double a, double b) {
#ifdef __CUDA_ARCH__
        return __dadd_rn(a, b);
#else
        volatile double r = a + b; return r;
#endif
    }
    static TS_HD double sub(double a, double b) {
#ifdef __CUDA_ARCH__
        return __dsub_rn(a, b);
#else
        volatile double r = a - b; return r;
#endif
    }
    static TS_HD double mul(double a, double b) {
#ifdef __CUDA_ARCH__
        return __dmul_rn(a, b);
#else
        volatile double r = a * b; return r;
#endif
    }
    static TS_HD double floor_(double a) { return floor(a); }
    static TS_HD double ceil_(double a) { return ceil(a); }
    static TS_HD double rint_(double a) { return rint(a); }
};

template <typename T> TS_HD T lerp(T a, T b, T x) {
    using A = Arith<T>;
    return A::add(A::mul(a, A::sub((T)1, x)), A::mul(b, x));
}
// v: neighbours in reference order (bit0 = +1 on axis 0, bit1 = +1 on axis 1, bit2 = +1 on axis 2)
template <typename T> TS_HD T interp2(const T* v, T x, T y) { return lerp(lerp(v[0], v[1], x), lerp(v[2], v[3], x), y); }
template <typename T, int DIM> TS_HD T interpolate(const T* v, const T* d) {
    if (DIM == 1) return lerp(v[0], v[1], d[0]);
    if (DIM == 2) return interp2(v, d[0], d[1]);
    return lerp(interp2(v, d[0], d[1]), interp2(v + 4, d[0], d[1]), d[2]);
}
template <typename T> TS_HD T dx2(const T* v, T y) { using A = Arith<T>; return lerp(A::sub(v[2], v[0]), A::sub(v[3], v[1]), y); }
template <typename T> TS_HD T dy2(const T* v, T x) { using A = Arith<T>; return A::sub(lerp(v[2], v[3], x), lerp(v[0], v[1], x)); }
// The reference's per-element "gradient w.r.t. shift" factors (quirks included: in 2D/3D g[0],
// which goes to the axis-0 weight, is a difference along axis 1).
template <typename T, int DIM> TS_HD void weight_partials(const T* v, const T* d, T* g) {
    using A = Arith<T>;
    if (DIM == 1) { g[0] = A::sub(v[1], v[0]); return; }
    if (DIM == 2) { g[0] = dx2(v, d[1]); g[1] = dy2(v, d[0]); return; }
    g[0] = lerp(dx2(v, d[1]), dx2(v + 4, d[1]), d[2]);
    g[1] = lerp(dy2(v, d[0]), dy2(v + 4, d[0]), d[2]);
    g[2] = A::sub(interp2(v + 4, d[0], d[1]), interp2(v, d[0], d[1]));
}

// ------------------------------------------------------------------------------------------
// Weight split.  CT = compute type (float or double).
template <typename CT> TS_HD long long to_ll_trunc(CT v) {
    // saturating, NaN -> 0 (the reference's cast is undefined there)
    if (!(v == v)) return 0;
    if (v >= (CT)9.2e18) return (long long)9200000000000000000LL;
    if (v <= (CT)-9.2e18) return (long long)-9200000000000000000LL;
    return (long long)v;
}
template <typename CT> TS_HD void split_forward(CT w, bool active, long long& iw, CT& dw) {
    using A = Arith<CT>;
    if (active) { iw = to_ll_trunc(A::floor_(w)); dw = A::sub(w, (CT)iw); }
    else { iw = to_ll_trunc(A::rint_(w)); dw = (CT)0; }
}
template <typename CT> TS_HD void split_backward(CT w, bool active, long long& iw, CT& dw) {
    using A = Arith<CT>;
    if (active) { dw = A::sub(w, A::floor_(w)); iw = to_ll_trunc(A::sub(w, dw)); }
    else { dw = w > (CT)0 ? A::sub(w, A::floor_(w)) : A::sub(A::ceil_(w), w); iw = to_ll_trunc(A::rint_(w)); }
}

// ------------------------------------------------------------------------------------------
// Element types.  ST = storage type, CT = compute type.
template <typename ST> struct Elem;
template <> struct Elem<float> { using CT = float; static TS_D float ld(float v) { return v; } static TS_D float st(float v) { return v; } };
template <> struct Elem<double> { using CT = double; static TS_D double ld(double v) { return v; } static TS_D double st(double v) { return v; } };
template <> struct Elem<__half> { using CT = float; static TS_D float ld(__half v) { return __half2float(v); } static TS_D __half st(float v) { return __float2half_rn(v); } };
template <> struct Elem<__nv_bfloat16> { using CT = float; static TS_D float ld(__nv_bfloat16 v) { return __bfloat162float(v); } static TS_D __nv_bfloat16 st(float v) { return __float2bfloat16_rn(v); } };

// Per-channel shift parameters, computed in every thread's registers (a handful of operations
// once per (n,c) plane or work unit; replaces the reference's weights_init kernels and the
// half-dozen ATen launches around them, cuda/shifts_cuda.cu:168-199, :219-229).
template <typename CT, int DIM> struct ShiftParams {
    int sx[DIM];   // shift reduced against the input sizes  (fetches from x)
    int sg[DIM];   // shift reduced against the output sizes (fetches from grad, backward only)
    CT d[3];       // fractional parts (0 for the sparse forward)
};

// Weight `idx` of a layer with `ST` elements, in the compute type: a 16-bit layer may carry fp32 weights (g.wf32), which are
// split as they are -- never rounded to 16 bits first.
template <typename ST>
TS_D typename Elem<ST>::CT load_weight(const ST* __restrict__ w, long long idx, const Geo& g) {
    if constexpr (sizeof(ST) == 2) {
        if (g.wf32) return reinterpret_cast<const float*>(w)[idx];
    }
    return Elem<ST>::ld(w[idx]);
}

template <typename ST, int DIM>
TS_D ShiftParams<typename Elem<ST>::CT, DIM> load_params(const ST* __restrict__ w, long long c, const Geo& g,
                                                         bool active, bool backward) {
    using CT = typename Elem<ST>::CT;
    ShiftParams<CT, DIM> p;
    p.d[0] = p.d[1] = p.d[2] = (CT)0;
#pragma unroll
    for (int a = 0; a < DIM; ++a) {
        const CT wv = load_weight<ST>(w, c * DIM + a, g);
        long long iw; CT dw;
        if (backward) split_backward<CT>(wv, active, iw, dw); else split_forward<CT>(wv, active, iw, dw);
        p.sx[a] = reduce_shift(iw, g.S[a], g.pad);
        p.sg[a] = reduce_shift(iw, g.OS[a], g.pad);
        p.d[a] = dw;
    }
    return p;
}

// Integer shifts of the quantized path: raw integer weight minus its zero point
// (quantized/shifts_quantized.cpp:113-114, kernels/shifts_kernels.h:553-555).
template <int DIM>
TS_HD void load_qshifts(const void* __restrict__ qw, int kind, long long wzp, long long c, const Geo& g, int* sx) {
#pragma unroll
    for (int a = 0; a < DIM; ++a) {
        long long raw;
        if (kind == TS_QW_U8) raw = ((const uint8_t*)qw)[c * DIM + a];
        else if (kind == TS_QW_I8) raw = ((const int8_t*)qw)[c * DIM + a];
        else raw = ((const int32_t*)qw)[c * DIM + a];
        sx[a] = reduce_shift(raw - wzp, g.S[a], g.pad);
    }
}

// ------------------------------------------------------------------------------------------
// How the integer shifts are obtained in the sparse/quantized gather kernels.
enum { WK_F32 = 0, WK_F64 = 1, WK_F16 = 2, WK_BF16 = 3, WK_QUANT = 4 };

// Integer shift of weight `idx` = c * dim + axis for the sparse forward (rounded float weight) or the quantized forward
// (raw weight minus its zero point).  The arguments are references into the kernel's parameters, so that each is read only
// on the path that uses it.
TS_D long long sparse_shift(const void* const& w, const int& wk, const int& qkind, const long long& wzp, long long idx) {
    long long iw = 0;
    switch (wk) {
    case WK_F32: { float d; split_forward<float>(((const float*)w)[idx], false, iw, d); break; }
    case WK_F64: { double d; split_forward<double>(((const double*)w)[idx], false, iw, d); break; }
    case WK_F16: { float d; split_forward<float>(__half2float(((const __half*)w)[idx]), false, iw, d); break; }
    case WK_BF16: { float d; split_forward<float>(__bfloat162float(((const __nv_bfloat16*)w)[idx]), false, iw, d); break; }
    default:
        if (qkind == TS_QW_U8) iw = (long long)((const uint8_t*)w)[idx] - wzp;
        else if (qkind == TS_QW_I8) iw = (long long)((const int8_t*)w)[idx] - wzp;
        else iw = (long long)((const int32_t*)w)[idx] - wzp;
    }
    return iw;
}

// ------------------------------------------------------------------------------------------
// Shared-memory vector loads as opaque instructions.  Written as plain C++ (`*(const uint4*)p`) the
// compiler narrows a 128-bit load to the words a misaligned window actually uses (LDS.32 + LDS.64 ...),
// and those narrower loads are 16-byte strided across a warp: 4-way bank conflicts (measured with ncu:
// half of all shared-memory wavefronts of the first TMA kernels).  LDS.128 of consecutive lanes is
// conflict-free, so the loads are pinned with inline PTX.  Addresses are 32-bit shared-window addresses.
#ifdef __CUDACC__
TS_D unsigned shared_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
TS_D uint4 lds128(unsigned addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
TS_D uint2 lds64(unsigned addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
TS_D unsigned lds32(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// ------------------------------------------------------------------------------------------
// 16-byte windows of staged boxes, shared by the staged and TMA families.  16-bit element types keep fp32 arithmetic: a
// window is resolved with a compile-time word select plus a half-word shift, and the store rounds once (Pack::pack).
// NW 32-bit words starting WS words into the aligned 16-byte group at byte offset `off` of `base`
// (off is a multiple of 16).  Loads the second group only when the window needs it.
template <int WS, int NW>
TS_D void load_words(unsigned base, int off, unsigned* w) {
    const uint4 A = lds128(base + off);
    unsigned W[8] = {A.x, A.y, A.z, A.w, 0u, 0u, 0u, 0u};
    if (WS + NW > 4) {
        const uint4 B = lds128(base + off + 16);
        W[4] = B.x; W[5] = B.y; W[6] = B.z; W[7] = B.w;
    }
#pragma unroll
    for (int t = 0; t < NW; ++t) w[t] = W[(t + WS) & 7];
}

// Element-type traits of the arithmetic kernels: V elements per 16-byte item; a window of NV
// elements spans words(NV) 32-bit words (one more than NV/2 for 16-bit types: half-word shift).
template <typename ST> struct Pack;
template <> struct Pack<float> {
    static constexpr int V = 4;
    static __host__ __device__ constexpr int words(int nv) { return nv; }
    template <int NV> static TS_D void unpack(const unsigned* w, int, float* out) {
#pragma unroll
        for (int t = 0; t < NV; ++t) out[t] = __uint_as_float(w[t]);
    }
    template <int NV, int HS> static TS_D void unpack_c(const unsigned* w, float* out) {
#pragma unroll
        for (int t = 0; t < NV; ++t) out[t] = __uint_as_float(w[t]);
    }
    static TS_D uint4 pack(const float* o) {
        return make_uint4(__float_as_uint(o[0]), __float_as_uint(o[1]), __float_as_uint(o[2]), __float_as_uint(o[3]));
    }
};
template <> struct Pack<__nv_bfloat16> {
    static constexpr int V = 8;
    static __host__ __device__ constexpr int words(int nv) { return nv / 2 + 1; }
    template <int NV> static TS_D void unpack(const unsigned* w, int hs, float* out) {
#pragma unroll
        for (int k = 0; k < (NV + 1) / 2; ++k) {
            const unsigned v = __funnelshift_r(w[k], w[k + 1], hs);
            out[2 * k] = __uint_as_float(v << 16);
            if (2 * k + 1 < NV) out[2 * k + 1] = __uint_as_float(v & 0xffff0000u);
        }
    }
    // compile-time half-word phase HS (0 / 16 bits): no funnel shift, one conversion per element
    template <int NV, int HS> static TS_D void unpack_c(const unsigned* w, float* out) {
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            const int h = t + (HS ? 1 : 0);
            out[t] = __uint_as_float((h & 1) ? (w[h >> 1] & 0xffff0000u) : (w[h >> 1] << 16));
        }
    }
    static TS_D uint4 pack(const float* o) {
        unsigned r[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const __nv_bfloat162 v = __floats2bfloat162_rn(o[2 * k], o[2 * k + 1]);
            r[k] = *(const unsigned*)&v;
        }
        return make_uint4(r[0], r[1], r[2], r[3]);
    }
};
template <> struct Pack<__half> {
    static constexpr int V = 8;
    static __host__ __device__ constexpr int words(int nv) { return nv / 2 + 1; }
    template <int NV> static TS_D void unpack(const unsigned* w, int hs, float* out) {
#pragma unroll
        for (int k = 0; k < (NV + 1) / 2; ++k) {
            const unsigned v = __funnelshift_r(w[k], w[k + 1], hs);
            const float2 f = __half22float2(*(const __half2*)&v);
            out[2 * k] = f.x;
            if (2 * k + 1 < NV) out[2 * k + 1] = f.y;
        }
    }
    template <int NV, int HS> static TS_D void unpack_c(const unsigned* w, float* out) {
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            const int h = t + (HS ? 1 : 0);
            const __half2 v = *(const __half2*)&w[h >> 1];
            out[t] = (h & 1) ? __high2float(v) : __low2float(v);
        }
    }
    static TS_D uint4 pack(const float* o) {
        unsigned r[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const __half2 v = __floats2half2_rn(o[2 * k], o[2 * k + 1]);
            r[k] = *(const unsigned*)&v;
        }
        return make_uint4(r[0], r[1], r[2], r[3]);
    }
};


// window of NV elements whose first element sits PH bytes (compile-time, a multiple of sizeof(ST)) into the
// 16-byte group at shared address `group`: exactly the words the window touches are loaded, no run-time realignment
template <typename ST, int PH, int NV>
TS_D void load_window_c(unsigned group, float* out) {
    constexpr int WS = PH >> 2, HS = (PH & 2) * 8;
    constexpr int NW = sizeof(ST) == 4 ? NV : (NV + (HS ? 1 : 0) + 1) / 2;
    unsigned w[NW];
    load_words<WS, NW>(group, 0, w);
    Pack<ST>::template unpack_c<NV, HS>(w, out);
}
#endif

// ------------------------------------------------------------------------------------------
// Which work units (channel, chunk of the batch) a persistent CTA processes, shared by the producer and the
// consumers of a CTA.  order 1 (default): round-robin over (chunk, channel) -- the CTAs of one wave stream
// neighbouring planes.  order 0: the CTA owns a CONTIGUOUS range of the channel-major unit list, so consecutive units
// share the channel (same unrolled code variant, warm weights); tuning knob `unit_order`.
#ifdef __CUDACC__
struct UnitRange { int u, end, step; };
TS_D UnitRange unit_range(int units, int order) {
    UnitRange r;
    if (order) { r.u = (int)blockIdx.x; r.end = units; r.step = (int)gridDim.x; return r; }
    const long long b = blockIdx.x, G = gridDim.x;
    r.u = (int)((long long)units * b / G);
    r.end = (int)((long long)units * (b + 1) / G);
    r.step = 1;
    return r;
}
TS_D void unit_decode(int u, int C, int chunks, int order, int& c, int& chunk) {
    if (order) { chunk = u / C; c = u - chunk * C; }
    else { c = u / chunks; chunk = u - c * chunks; }
}
#endif

// ------------------------------------------------------------------------------------------
// Programmatic dependent launch.  A kernel launched with launch_pdl() may start while its predecessor in the stream is
// still draining: its CTAs are scheduled, set up their barriers and then block in pdl_wait() until the predecessor
// has completed and flushed -- so NOTHING that touches global memory may precede pdl_wait().  pdl_trigger() at the
// top of a kernel lets its successor do the same.  Hides ~2 us of launch latency and ramp per kernel boundary, which is
// 5 % of the three-kernel step of a 32-image shard (8-GPU strong scaling); also inside captured CUDA graphs.
#ifdef __CUDACC__
TS_D void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
TS_D void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg;
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}
#endif

// ------------------------------------------------------------------------------------------
// Launch bookkeeping shared by the translation units.
void note_launch(int n = 1);
void note_error(const char* text);  // text returned by ts_last_cuda_error() for non-CUDA-runtime failures
int check_launch();               // cudaGetLastError -> ts_status
// cudaFuncAttributeMaxDynamicSharedMemorySize >= bytes for `func` on the current device; the attribute call is
// made only when a kernel needs more than it was last given (not on every launch)
bool ensure_dynamic_smem(const void* func, size_t bytes);

#ifdef __CUDACC__
// One launch of a kernel with `smem` bytes of dynamic shared memory, counted and checked.  pdl: programmatic dependent
// launch (a plain launch where that is refused) -- only for kernels that call pdl_wait() before touching global memory.
template <typename... KArgs, typename... Args>
int launch_persistent(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args... args) {
    if (!ensure_dynamic_smem((const void*)kernel, smem)) return check_launch();
    if (!pdl || launch_pdl(kernel, grid, block, smem, stream, args...) != cudaSuccess) {
        if (pdl) (void)cudaGetLastError();
        kernel<<<grid, block, smem, stream>>>(args...);
    }
    note_launch();
    return check_launch();
}
#endif

}  // namespace ts

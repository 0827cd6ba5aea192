// ts_nhwc_float.cu -- channels-last FLOAT forward and backward (ts_shift_forward_nhwc / ts_shift_backward_nhwc): 2-D,
// fp32 / fp16 / bf16, every padding, border crops, C a multiple of 32.  Input and output keep the channel axis innermost,
// so a Shift2d between two channels-last convolutions pays one read and one write per tensor and no layout pass.
//
// Work layout.  A CTA owns (image n, slice of 128 bytes of channels, segment of rows).  Lane <-> 32-bit word of the
// slice (1 fp32 channel or 2 16-bit channels): the channel's shift parameters are registers for the CTA's lifetime and a
// warp store of one pixel is one 128-byte line.  Rows of the slice (all pixels of an input row, 128 bytes each) are
// staged in a K-slot shared-memory ring (slot = row mod K) with 16-byte cp.async copies; a lane's gather from a staged
// row reads the word of ITS bank whatever pixel its shift selects, so the scattered per-channel taps are conflict-free
// shared-memory loads instead of one L1 sector access each.
//
// Pipeline.  The CTA walks its segment in steps of G output rows (the forward) or input rows (the backward).  Step j
// needs the input rows [lo_j, hi_j] its rows can reach (the slice's min / max shift), capped at WIN rows.  The copies of
// step j + D are issued as one cp.async group before step j is computed, so D steps of loads are in flight while the
// CTA gathers.  lo_j and hi_j never decrease and lo grows by at most G per step, and WIN = K - (D + 1) G: the rows
// written by the copies of any step in flight never alias a row some warp still reads, so a step needs one
// __syncthreads (after its copies land) and no release barrier.  A tap whose (remapped) row is not in the window --
// wrap-around paddings at the image edges, shifts spread wider than WIN -- is read from global memory: the window
// only ever affects speed.  A row outside the tensor under zeros padding is no tap at all.
//
// Arithmetic.  The forward and grad_input use the reference's operations in its order (ts_common.cuh: lerp / interp2,
// each product and sum rounded separately), fp32 for the 16-bit types with one rounding at the store, so fp32 is
// bit-exact against the reference CPU kernels.  grad_weight: a thread owns its channels at every pixel it visits, so it accumulates
// the per-element products in fp64 registers with no cross-lane reduction; the warps of a CTA are summed in fixed order
// into one fp64 partial slot per (image, segment) -- the layout launch_reduce_partials<ST> reads -- and that pass 2
// (with its fused all-reduce) is reused unchanged.  Results are bit-identical from run to run.
#include "ts_kernels.h"
#include "ts_ptx.cuh"

namespace ts {

namespace {

using namespace ptx;

constexpr int CL_D = 2;            // default steps of copies in flight ahead of the gather (tuning knob cl_ahead: 1..4)
constexpr int CL_G = 2;            // default rows per step (tuning knob cl_rows: 1, 2, 4 or 8)
constexpr int CL_PIX = 128;        // bytes of a staged pixel (one channel slice)
constexpr int CL_FWD_THREADS = 256, CL_BWD_THREADS = 512;

struct ClPlan {
    int D, G;                      // steps of copies in flight, rows per step
    int K, WIN;                    // ring slots per staged tensor, window rows
    int seg_rows, segs, slices;    // rows per unit, units per image, channel slices
    unsigned ring_x, ring_g;       // bytes of one ring (x / grad)
    unsigned off_red, smem_bytes;
};

template <typename ST> struct Bits { using type = unsigned short; };
template <> struct Bits<float> { using type = unsigned; };

template <typename ST> TS_D float from_bits(unsigned b);
template <> TS_D float from_bits<float>(unsigned b) { return __uint_as_float(b); }
template <> TS_D float from_bits<__half>(unsigned b) { return __half2float(__ushort_as_half((unsigned short)b)); }
template <> TS_D float from_bits<__nv_bfloat16>(unsigned b) { return __bfloat162float(__ushort_as_bfloat16((unsigned short)b)); }
template <typename ST> TS_D unsigned to_bits(float v);
template <> TS_D unsigned to_bits<float>(float v) { return __float_as_uint(v); }
template <> TS_D unsigned to_bits<__half>(float v) { return __half_as_ushort(__float2half_rn(v)); }
template <> TS_D unsigned to_bits<__nv_bfloat16>(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }

template <typename ST> TS_D unsigned lds_bits(unsigned addr) {
    unsigned v;
    if constexpr (sizeof(ST) == 4) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    else asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
template <typename ST> TS_D unsigned ldg_bits(const ST* p) {
    return (unsigned)__ldg(reinterpret_cast<const typename Bits<ST>::type*>(p));
}

TS_D void cp_async_wait_n(int n) {      // wait_group takes an immediate
    switch (n) {
    case 1: cp_async_wait<1>(); break;
    case 2: cp_async_wait<2>(); break;
    case 3: cp_async_wait<3>(); break;
    default: cp_async_wait<4>(); break;
    }
}

TS_D int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Rows [lo, hi] of step j of a ring: raw reach [a, b] clamped to the tensor's rows, capped at WIN rows.
TS_D void cl_window(int a, int b, int rows, int WIN, int& lo, int& hi) {
    lo = clampi(a, 0, rows - 1);
    hi = clampi(b, 0, rows - 1);
    if (hi > lo + WIN - 1) hi = lo + WIN - 1;
    if (hi < lo) hi = lo;
}

// Issue the copies of rows [r0, r1] of one tensor's channel slice into their ring slots.  src: pixel (n, row 0, col 0)
// at the slice's first channel; width pixels per row, C elements per pixel; chunks (16 bytes) per pixel = 1 << lgc.
template <typename ST>
TS_D void cl_stage(unsigned ring, int K, const ST* src, int width, long long C, int lgc, int r0, int r1) {
    const int per_row = width << lgc;
    for (int row = r0; row <= r1; ++row) {
        const unsigned dst = ring + (unsigned)((row % K) * width) * CL_PIX;
        const ST* s = src + (long long)row * width * C;
        for (int f = (int)threadIdx.x; f < per_row; f += (int)blockDim.x) {
            const int px = f >> lgc, ch = f & ((1 << lgc) - 1);
            cp_async16(dst + (unsigned)px * CL_PIX + (unsigned)ch * 16u, reinterpret_cast<const char*>(s + (long long)px * C) + ch * 16);
        }
    }
}

// One tap row of a lane's channel: not a tap (outside, zeros padding), a staged row, or a global-memory row.
template <typename ST> struct TapRow {
    int kind;                      // 0 zero, 1 shared memory, 2 global memory
    unsigned sa;                   // kind 1: shared address of pixel 0 of the lane's word
    const ST* gp;                  // kind 2: pixel 0 of the lane's channel
};
template <typename ST>
TS_D TapRow<ST> tap_row(int t, int lo, int hi, unsigned ring, int K, int width, unsigned lane_off, const ST* g0, long long C) {
    TapRow<ST> r;
    r.kind = t < 0 ? 0 : (t >= lo && t <= hi ? 1 : 2);
    r.sa = ring + (unsigned)(((t < 0 ? 0 : t) % K) * width) * CL_PIX + lane_off;
    r.gp = g0 + (long long)(t < 0 ? 0 : t) * width * C;
    return r;
}
template <typename ST> TS_D float tap(const TapRow<ST>& r, int col, long long C) {
    if (col < 0 || r.kind == 0) return 0.f;
    if (r.kind == 1) return from_bits<ST>(lds_bits<ST>(r.sa + (unsigned)col * CL_PIX));
    return from_bits<ST>(ldg_bits<ST>(r.gp + (long long)col * C));
}

// min / max over the lanes' channels (every warp holds the same slice, so every warp gets the same result)
TS_D void warp_minmax(int& mn, int& mx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const int a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
        mn = a < mn ? a : mn;
        mx = b > mx ? b : mx;
    }
}

// ---- forward -------------------------------------------------------------------------------------------------------
template <typename ST, int PAD, bool ACTIVE>
__global__ void __launch_bounds__(CL_FWD_THREADS, 2) k_cl_forward(Geo g, ClPlan pl, const ST* __restrict__ x, const ST* __restrict__ w,
                                                                  ST* __restrict__ y) {
    constexpr int VEC = 4 / (int)sizeof(ST), CPW = 32 * VEC, A = ACTIVE ? 1 : 0;
    extern __shared__ __align__(128) unsigned char csm[];
    const unsigned ring = shared_addr(csm);
    const int lane = (int)threadIdx.x & 31, warp = (int)threadIdx.x >> 5, NW = (int)blockDim.x >> 5, WPR = NW / pl.G;
    const int n = (int)blockIdx.x / pl.segs, seg = (int)blockIdx.x - n * pl.segs;
    const long long C = g.C, c0 = (long long)blockIdx.y * CPW;
    const int cw = C - c0 < CPW ? (int)(C - c0) : CPW;
    const int lgc = cw * (int)sizeof(ST) == 128 ? 3 : 2;
    const int S0 = g.S[0], S1 = g.S[1], OS0 = g.OS[0], OW = g.OS[1], lb0 = g.lb[0], lb1 = g.lb[1];

    int s0[VEC], s1[VEC];
    float d0[VEC], d1[VEC];
    bool on[VEC];
    int mn = 0x7fffffff, mx = -0x7fffffff;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        on[v] = lane * VEC + v < cw;
        s0[v] = s1[v] = 0;
        d0[v] = d1[v] = 0.f;
        if (on[v]) {
            const ShiftParams<float, 2> p = load_params<ST, 2>(w, c0 + lane * VEC + v, g, ACTIVE, false);
            s0[v] = p.sx[0]; s1[v] = p.sx[1]; d0[v] = p.d[0]; d1[v] = p.d[1];
            mn = s0[v] < mn ? s0[v] : mn;
            mx = s0[v] > mx ? s0[v] : mx;
        }
    }
    warp_minmax(mn, mx);

    const int o_a = seg * pl.seg_rows, o_b = o_a + pl.seg_rows < OS0 ? o_a + pl.seg_rows : OS0;
    const int steps = (o_b - o_a + pl.G - 1) / pl.G;
    const ST* xs = x + (long long)n * S0 * S1 * C + c0;
    int loaded = -1;
    auto issue = [&](int j) {
        if (j < steps) {
            const int fa = o_a + j * pl.G, fb = (fa + pl.G < o_b ? fa + pl.G : o_b) - 1;
            int lo, hi;
            cl_window(fa + lb0 - mx, fb + lb0 - mn + A, S0, pl.WIN, lo, hi);
            cl_stage<ST>(ring, pl.K, xs, S1, C, lgc, loaded + 1 > lo ? loaded + 1 : lo, hi);
            loaded = hi > loaded ? hi : loaded;
        }
        cp_async_commit();
    };
    for (int j = 0; j < pl.D; ++j) issue(j);

    const unsigned lane_off = (unsigned)(lane * VEC * (int)sizeof(ST));
    for (int j = 0; j < steps; ++j) {
        issue(j + pl.D);
        cp_async_wait_n(pl.D);
        __syncthreads();
        const int fa = o_a + j * pl.G, fb = (fa + pl.G < o_b ? fa + pl.G : o_b) - 1;
        int lo, hi;
        cl_window(fa + lb0 - mx, fb + lb0 - mn + A, S0, pl.WIN, lo, hi);
        const int o = fa + warp / WPR;
        if (o > fb) continue;
        TapRow<ST> ra[VEC], rb[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const unsigned lo_v = lane_off + (unsigned)(v * (int)sizeof(ST));
            ra[v] = tap_row<ST>(axis_index(o + lb0 - s0[v], S0, PAD), lo, hi, ring, pl.K, S1, lo_v, xs + lane * VEC + v, C);
            if (ACTIVE) rb[v] = tap_row<ST>(axis_index(o + lb0 - s0[v] + 1, S0, PAD), lo, hi, ring, pl.K, S1, lo_v, xs + lane * VEC + v, C);
        }
        if (lane * VEC >= cw) continue;
        unsigned* yrow = reinterpret_cast<unsigned*>(y + (((long long)n * OS0 + o) * OW) * C + c0) + lane;
        for (int p = warp % WPR; p < OW; p += WPR) {
            unsigned out = 0;
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const int i1 = p + lb1 - s1[v];
                const int ca = axis_index(i1, S1, PAD);
                float r;
                if (ACTIVE) {
                    const int cb = axis_index(i1 + 1, S1, PAD);
                    const float vv[4] = {tap(ra[v], ca, C), tap(rb[v], ca, C), tap(ra[v], cb, C), tap(rb[v], cb, C)};
                    const float dd[2] = {d0[v], d1[v]};
                    r = interpolate<float, 2>(vv, dd);
                } else {
                    r = tap(ra[v], ca, C);
                }
                out |= to_bits<ST>(r) << (16 * v);
            }
            yrow[(long long)p * C / VEC] = out;
        }
    }
}

// ---- backward ------------------------------------------------------------------------------------------------------
// Step j covers input rows (rows of grad_input).  x ring: the rows of x the weight partials read (pos - sx, +1);
// grad ring: the rows of grad the grad_input gather reads (o - sg, +1 interpolating; o + sg sparse), o = pos - lb.
// The gradient at the output position itself is one coalesced global load per pixel.
template <typename ST, int PAD, bool ACTIVE>
__global__ void __launch_bounds__(CL_BWD_THREADS, 1) k_cl_backward(Geo g, ClPlan pl, const ST* __restrict__ grad, const ST* __restrict__ x,
                                                                     const ST* __restrict__ w, ST* __restrict__ gi, double* __restrict__ partials) {
    constexpr int VEC = 4 / (int)sizeof(ST), CPW = 32 * VEC;
    extern __shared__ __align__(128) unsigned char csm[];
    const unsigned ring_x = shared_addr(csm), ring_g = ring_x + pl.ring_x;
    const int lane = (int)threadIdx.x & 31, warp = (int)threadIdx.x >> 5, NW = (int)blockDim.x >> 5, WPR = NW / pl.G;
    const int n = (int)blockIdx.x / pl.segs, seg = (int)blockIdx.x - n * pl.segs;
    const long long C = g.C, c0 = (long long)blockIdx.y * CPW;
    const int cw = C - c0 < CPW ? (int)(C - c0) : CPW;
    const int lgc = cw * (int)sizeof(ST) == 128 ? 3 : 2;
    const int S0 = g.S[0], S1 = g.S[1], OS0 = g.OS[0], OS1 = g.OS[1], lb0 = g.lb[0], lb1 = g.lb[1];

    int sx0[VEC], sx1[VEC], sg0[VEC], sg1[VEC];
    float d[VEC][2];
    bool on[VEC];
    double acc[VEC][2];
    int xmn = 0x7fffffff, xmx = -0x7fffffff, gmn = 0x7fffffff, gmx = -0x7fffffff;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        on[v] = lane * VEC + v < cw;
        sx0[v] = sx1[v] = sg0[v] = sg1[v] = 0;
        d[v][0] = d[v][1] = 0.f;
        acc[v][0] = acc[v][1] = 0.0;
        if (on[v]) {
            const ShiftParams<float, 2> p = load_params<ST, 2>(w, c0 + lane * VEC + v, g, ACTIVE, true);
            sx0[v] = p.sx[0]; sx1[v] = p.sx[1]; sg0[v] = p.sg[0]; sg1[v] = p.sg[1]; d[v][0] = p.d[0]; d[v][1] = p.d[1];
            xmn = sx0[v] < xmn ? sx0[v] : xmn;
            xmx = sx0[v] > xmx ? sx0[v] : xmx;
            gmn = sg0[v] < gmn ? sg0[v] : gmn;
            gmx = sg0[v] > gmx ? sg0[v] : gmx;
        }
    }
    warp_minmax(xmn, xmx);
    warp_minmax(gmn, gmx);

    const int i_a = seg * pl.seg_rows, i_b = i_a + pl.seg_rows < S0 ? i_a + pl.seg_rows : S0;
    const int steps = (i_b - i_a + pl.G - 1) / pl.G;
    const ST* xs = x + (long long)n * S0 * S1 * C + c0;
    const ST* gs = grad + (long long)n * OS0 * OS1 * C + c0;
    auto windows = [&](int j, int& xlo, int& xhi, int& glo, int& ghi) {
        const int fa = i_a + j * pl.G, fb = (fa + pl.G < i_b ? fa + pl.G : i_b) - 1;
        cl_window(fa - xmx, fb - xmn + 1, S0, pl.WIN, xlo, xhi);
        if (ACTIVE) cl_window(fa - lb0 - gmx, fb - lb0 - gmn + 1, OS0, pl.WIN, glo, ghi);
        else cl_window(fa - lb0 + gmn, fb - lb0 + gmx, OS0, pl.WIN, glo, ghi);
    };
    int xloaded = -1, gloaded = -1;
    auto issue = [&](int j) {
        if (j < steps) {
            int xlo, xhi, glo, ghi;
            windows(j, xlo, xhi, glo, ghi);
            cl_stage<ST>(ring_x, pl.K, xs, S1, C, lgc, xloaded + 1 > xlo ? xloaded + 1 : xlo, xhi);
            cl_stage<ST>(ring_g, pl.K, gs, OS1, C, lgc, gloaded + 1 > glo ? gloaded + 1 : glo, ghi);
            xloaded = xhi > xloaded ? xhi : xloaded;
            gloaded = ghi > gloaded ? ghi : gloaded;
        }
        cp_async_commit();
    };
    for (int j = 0; j < pl.D; ++j) issue(j);

    const unsigned lane_off = (unsigned)(lane * VEC * (int)sizeof(ST));
    for (int j = 0; j < steps; ++j) {
        issue(j + pl.D);
        cp_async_wait_n(pl.D);
        __syncthreads();
        int xlo, xhi, glo, ghi;
        windows(j, xlo, xhi, glo, ghi);
        const int fa = i_a + j * pl.G, fb = (fa + pl.G < i_b ? fa + pl.G : i_b) - 1;
        const int i = fa + warp / WPR;
        if (i > fb || lane * VEC >= cw) continue;
        const int o = i - lb0;
        const bool row_ok = o >= 0 && o < OS0;
        unsigned* girow = reinterpret_cast<unsigned*>(gi + (((long long)n * S0 + i) * S1) * C + c0) + lane;
        if (!row_ok) {
            for (int p = warp % WPR; p < S1; p += WPR) girow[(long long)p * C / VEC] = 0u;
            continue;
        }
        TapRow<ST> xa[VEC], xb[VEC], ga[VEC], gb[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const unsigned lo_v = lane_off + (unsigned)(v * (int)sizeof(ST));
            xa[v] = tap_row<ST>(axis_index(i - sx0[v], S0, PAD), xlo, xhi, ring_x, pl.K, S1, lo_v, xs + lane * VEC + v, C);
            xb[v] = tap_row<ST>(axis_index(i - sx0[v] + 1, S0, PAD), xlo, xhi, ring_x, pl.K, S1, lo_v, xs + lane * VEC + v, C);
            if (ACTIVE) {
                ga[v] = tap_row<ST>(axis_index(o - sg0[v], OS0, PAD), glo, ghi, ring_g, pl.K, OS1, lo_v, gs + lane * VEC + v, C);
                gb[v] = tap_row<ST>(axis_index(o - sg0[v] + 1, OS0, PAD), glo, ghi, ring_g, pl.K, OS1, lo_v, gs + lane * VEC + v, C);
            } else {
                ga[v] = tap_row<ST>(axis_index(o + sg0[v], OS0, PAD), glo, ghi, ring_g, pl.K, OS1, lo_v, gs + lane * VEC + v, C);
            }
        }
        const ST* gvrow = gs + (long long)o * OS1 * C + lane * VEC;
        for (int p = warp % WPR; p < S1; p += WPR) {
            const int o1 = p - lb1;
            unsigned out = 0;
            if (o1 >= 0 && o1 < OS1) {
                const unsigned gbits = __ldg(reinterpret_cast<const unsigned*>(gvrow + (long long)o1 * C));
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    if (!on[v]) continue;
                    const float gv = from_bits<ST>(VEC == 1 ? gbits : (gbits >> (16 * v)) & 0xffffu);
                    const int ca = axis_index(p - sx1[v], S1, PAD), cb = axis_index(p - sx1[v] + 1, S1, PAD);
                    const float xv[4] = {tap(xa[v], ca, C), tap(xb[v], ca, C), tap(xa[v], cb, C), tap(xb[v], cb, C)};
                    float wg[3];
                    weight_partials<float, 2>(xv, d[v], wg);
                    acc[v][0] += (double)Arith<float>::mul(gv, wg[0]);
                    acc[v][1] += (double)Arith<float>::mul(gv, wg[1]);
                    float r;
                    if (ACTIVE) {
                        const int ga_c = axis_index(o1 - sg1[v], OS1, PAD), gb_c = axis_index(o1 - sg1[v] + 1, OS1, PAD);
                        const float gv4[4] = {tap(ga[v], ga_c, C), tap(gb[v], ga_c, C), tap(ga[v], gb_c, C), tap(gb[v], gb_c, C)};
                        r = interpolate<float, 2>(gv4, d[v]);
                    } else {
                        r = tap(ga[v], axis_index(o1 + sg1[v], OS1, PAD), C);
                    }
                    out |= to_bits<ST>(r) << (16 * v);
                }
            }
            girow[(long long)p * C / VEC] = out;
        }
    }

    // grad_weight: the warps' accumulators summed in warp order, one fp64 partial slot per (image, segment)
    double* red = reinterpret_cast<double*>(csm + pl.off_red);
    __syncthreads();
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        red[((long long)warp * CPW + lane * VEC + v) * 2 + 0] = acc[v][0];
        red[((long long)warp * CPW + lane * VEC + v) * 2 + 1] = acc[v][1];
    }
    __syncthreads();
    for (int t = (int)threadIdx.x; t < cw * 2; t += (int)blockDim.x) {
        double s = 0.0;
        for (int k = 0; k < NW; ++k) s += red[(long long)k * CPW * 2 + t];
        partials[(long long)blockIdx.x * (C * 2) + c0 * 2 + t] = s;
    }
}

// ---- host ----------------------------------------------------------------------------------------------------------
bool dense_nhwc(const Geo& g) {
    return g.dim == 2 && (g.C == 1 || g.xs[1] == 1) && (g.S[1] == 1 || g.xs[3] == g.C) && (g.S[0] == 1 || g.xs[2] == g.C * g.S[1]) &&
           (g.N == 1 || g.xs[0] == g.C * g.in_plane);
}

bool plan_cl(const Geo& g, int dtype, bool backward, int sm_count, ClPlan* out) {
    if (dtype != TS_F32 && dtype != TS_F16 && dtype != TS_BF16) return false;
    if (!dense_nhwc(g) || g.C % 32 != 0 || g.N * g.C == 0 || g.in_plane == 0 || g.out_plane == 0) return false;
    const int cpw = dtype == TS_F32 ? 32 : 64, threads = backward ? CL_BWD_THREADS : CL_FWD_THREADS;
    ClPlan pl;
    pl.slices = (int)((g.C + cpw - 1) / cpw);
    if (pl.slices > 65535) return false;
    const long long slot_x = (long long)g.S[1] * CL_PIX, slot_g = backward ? (long long)g.OS[1] * CL_PIX : 0;
    const long long red = backward ? (long long)(threads / 32) * cpw * 2 * 8 : 0;
    // forward: two CTAs per SM; backward (two rings): one CTA of 16 warps
    const long long budget = backward ? 220LL * 1024 : 110LL * 1024;
    long long K = (budget - red) / (slot_x + slot_g);
    if (K > 24) K = 24;
    pl.D = tuning().cl_ahead > 0 ? tuning().cl_ahead : CL_D;
    pl.G = tuning().cl_rows > 0 ? tuning().cl_rows : CL_G;
    const int WIN = (int)K - (pl.D + 1) * pl.G;
    if (WIN < pl.G + 2) return false;     // rows too wide to stage a useful window: the planar path serves them
    pl.K = (int)K;
    pl.WIN = WIN;
    pl.ring_x = (unsigned)(K * slot_x);
    pl.ring_g = (unsigned)(K * slot_g);
    pl.off_red = pl.ring_x + pl.ring_g;
    pl.smem_bytes = pl.off_red + (unsigned)red;
    // segments of rows: enough CTAs to fill the machine twice over, segments of at least 8 rows (each pays its halo once)
    const long long rows = backward ? g.S[0] : g.OS[0];
    long long segs = 1;
    const long long target = 2LL * sm_count * (backward ? 1 : 2);
    while (g.N * pl.slices * segs < target && rows / (segs * 2) >= 8) segs *= 2;
    pl.seg_rows = (int)((rows + segs - 1) / segs);
    pl.segs = (int)((rows + pl.seg_rows - 1) / pl.seg_rows);
    if (g.N * pl.segs >= 0x7fffffffLL) return false;
    *out = pl;
    return true;
}

template <typename ST, int PAD>
int cl_forward_t(const Geo& g, const ClPlan& pl, int active, const void* x, const void* w, void* y, cudaStream_t s) {
    auto k = active ? k_cl_forward<ST, PAD, true> : k_cl_forward<ST, PAD, false>;
    const dim3 grid((unsigned)(g.N * pl.segs), (unsigned)pl.slices, 1);
    return launch_persistent(k, grid, CL_FWD_THREADS, pl.smem_bytes, s, false, g, pl, (const ST*)x, (const ST*)w, (ST*)y);
}

template <typename ST, int PAD>
int cl_backward_t(const Geo& g, const ClPlan& pl, int active, const void* grad, const void* x, const void* w, void* gi,
                  double* partials, cudaStream_t s) {
    auto k = active ? k_cl_backward<ST, PAD, true> : k_cl_backward<ST, PAD, false>;
    const dim3 grid((unsigned)(g.N * pl.segs), (unsigned)pl.slices, 1);
    return launch_persistent(k, grid, CL_BWD_THREADS, pl.smem_bytes, s, false, g, pl, (const ST*)grad, (const ST*)x, (const ST*)w, (ST*)gi,
                             partials);
}

template <typename ST>
int cl_forward_pad(const Geo& g, const ClPlan& pl, int active, const void* x, const void* w, void* y, cudaStream_t s) {
    switch (g.pad) {
    case TS_PAD_BORDER: return cl_forward_t<ST, TS_PAD_BORDER>(g, pl, active, x, w, y, s);
    case TS_PAD_PERIODIC: return cl_forward_t<ST, TS_PAD_PERIODIC>(g, pl, active, x, w, y, s);
    case TS_PAD_REFLECT: return cl_forward_t<ST, TS_PAD_REFLECT>(g, pl, active, x, w, y, s);
    case TS_PAD_SYMMETRIC: return cl_forward_t<ST, TS_PAD_SYMMETRIC>(g, pl, active, x, w, y, s);
    default: return cl_forward_t<ST, TS_PAD_ZEROS>(g, pl, active, x, w, y, s);
    }
}

template <typename ST>
int cl_backward_pad(const Geo& g, const ClPlan& pl, int active, const void* grad, const void* x, const void* w, void* gi,
                    double* partials, cudaStream_t s) {
    switch (g.pad) {
    case TS_PAD_BORDER: return cl_backward_t<ST, TS_PAD_BORDER>(g, pl, active, grad, x, w, gi, partials, s);
    case TS_PAD_PERIODIC: return cl_backward_t<ST, TS_PAD_PERIODIC>(g, pl, active, grad, x, w, gi, partials, s);
    case TS_PAD_REFLECT: return cl_backward_t<ST, TS_PAD_REFLECT>(g, pl, active, grad, x, w, gi, partials, s);
    case TS_PAD_SYMMETRIC: return cl_backward_t<ST, TS_PAD_SYMMETRIC>(g, pl, active, grad, x, w, gi, partials, s);
    default: return cl_backward_t<ST, TS_PAD_ZEROS>(g, pl, active, grad, x, w, gi, partials, s);
    }
}

}  // namespace

size_t cl_backward_workspace_bytes(const Geo& g, int dtype, int sm_count) {
    ClPlan pl;
    if (!plan_cl(g, dtype, true, sm_count, &pl)) return 16;
    return (size_t)(g.N * pl.segs) * (size_t)(g.C * 2) * sizeof(double) + 16;
}

int cl_forward(const Geo& g, int dtype, int active, const void* x, const void* w, void* y, int sm_count, cudaStream_t s) {
    ClPlan pl;
    if (!plan_cl(g, dtype, false, sm_count, &pl) || ((uintptr_t)x & 15u) || ((uintptr_t)y & 15u)) return TS_ERR_UNSUPPORTED;
    switch (dtype) {
    case TS_F32: return cl_forward_pad<float>(g, pl, active, x, w, y, s);
    case TS_F16: return cl_forward_pad<__half>(g, pl, active, x, w, y, s);
    default: return cl_forward_pad<__nv_bfloat16>(g, pl, active, x, w, y, s);
    }
}

int cl_backward(const Geo& g, int dtype, int active, const void* grad, const void* x, const void* w, void* gi, double* partials,
                size_t workspace_bytes, int sm_count, int* slots, cudaStream_t s) {
    ClPlan pl;
    if (!plan_cl(g, dtype, true, sm_count, &pl) || ((uintptr_t)x & 15u) || ((uintptr_t)grad & 15u) || ((uintptr_t)gi & 15u))
        return TS_ERR_UNSUPPORTED;
    if (workspace_bytes < (size_t)(g.N * pl.segs) * (size_t)(g.C * 2) * sizeof(double)) return TS_ERR_WORKSPACE;
    *slots = (int)(g.N * pl.segs);
    switch (dtype) {
    case TS_F32: return cl_backward_pad<float>(g, pl, active, grad, x, w, gi, partials, s);
    case TS_F16: return cl_backward_pad<__half>(g, pl, active, grad, x, w, gi, partials, s);
    default: return cl_backward_pad<__nv_bfloat16>(g, pl, active, grad, x, w, gi, partials, s);
    }
}

}  // namespace ts

// ts_flat.cu -- zero-padded sparse / quantized forward of 1-D / 2-D tensors as a FLAT shifted copy (the cfg5 byte
// mover).
//
// Under zeros padding (BIPadding::Zeros, ops/kernels/shifts_kernels.h:10-54, :532-571) and without a border crop the
// gather of one dense (n, c) plane (rows x row_bytes, contiguous in NCHW) is a LINEAR shifted copy plus a validity
// mask:      out[o] = valid(o) ? in[o - delta] : pad_value,      delta = s_row * row_bytes + s_col * elem_bytes
// for every byte offset o of the plane, with valid(o) <=> source row AND source column inside the plane.
//
//  * A dense NCHW tensor is ONE contiguous array of N*C planes, so a stage is K CONSECUTIVE planes moved by ONE 1-D
//    bulk copy (cp.async.bulk -> UBLKCP; cfg5: 8 planes = 25 KB) instead of one 3 KB copy per plane: the per-copy
//    and per-hand-off costs that bounded the round-1 byte movers at ~50 % of the roofline are paid per 25 KB.
//  * The planes of a stage belong to different channels: lane l of every consumer warp computes the shift of plane
//    l of the stage in its registers and the warp reads it back with a shuffle per item -- no shared table, no
//    barrier.
//  * Every thread-iteration emits 16 output bytes from one unaligned 16-byte window of the staged plane (two
//    LDS.128, a word-select network and funnel shifts), whatever the row length: 56-byte qint8 rows no longer force
//    8-byte items, an item simply spans two rows.  The pad value (the input zero point,
//    quantized/shifts_quantized.cpp:113) is blended in with byte masks derived from the item's offset; items
//    without an invalid byte skip that.
//
// CTA = nw consumer warps + 1 producer warp (one CTA of 15 warps per SM by default, `flat_ctas` for several smaller
// ones); stages are dealt round-robin.
#include <cstring>

#include "ts_kernels.h"
#include "ts_ptx.cuh"

namespace ts {

namespace {

using namespace ptx;

constexpr int GUARD = 32;
constexpr int MAX_K = 32;          // planes per stage: one lane of a warp per plane

// (row shift, column shift in bytes) of channel c; a size-1 axis ignores its shift (reduce_shift)
TS_D void flat_shift(const FArgs& a, long long c, int& sr, int& scb) {
    int s[2] = {0, 0};
#pragma unroll
    for (int lev = 0; lev < 2; ++lev) {
        const int ax = lev - (2 - a.dim);
        if (ax < 0) continue;
        s[lev] = reduce_shift(sparse_shift(a.w, a.wk, a.qkind, a.wzp, c * a.dim + ax), a.g.S[ax], TS_PAD_ZEROS);      // |s| <= len + 1
    }
    sr = s[0];
    scb = s[1] * a.es;
}

TS_D void producer(const FArgs& a, unsigned char* smem, uint64_t* full, uint64_t* empty) {
    int s = 0, k = 0;
    for (int t = blockIdx.x; t < a.nstages; t += gridDim.x) {
        const long long p0 = (long long)t * a.K;
        const int np = a.planes - p0 < a.K ? (int)(a.planes - p0) : a.K;
        if (k > 0) mbar_wait(&empty[s], (unsigned)((k - 1) & 1));
        unsigned char* st = smem + (size_t)s * a.stage_stride + GUARD;
        const unsigned bytes = (unsigned)np * (unsigned)a.plane_bytes;
        mbar_expect_tx(&full[s], bytes);
        bulk_g2s(st, a.x + p0 * a.plane_bytes, bytes, &full[s]);
        if (++s == a.stages) { s = 0; ++k; }
    }
}

TS_D unsigned bits_range(int lo, int hi) {       // bits [lo, hi) of a 16-bit mask, 0 <= lo, hi <= 16
    return hi > lo ? (((1u << hi) - 1u) & ~((1u << lo) - 1u)) : 0u;
}
TS_D unsigned spread_nibble(unsigned nib) { return ((nib * 0x00204081u) & 0x01010101u) * 0xffu; }

__global__ void __launch_bounds__(512, 1) k_flat_gather(const __grid_constant__ FArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t* full = (uint64_t*)(smem + (size_t)a.stages * a.stage_stride);
    uint64_t* empty = full + a.stages;
    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], (unsigned)a.nw); }
        fence_barrier_init();
    }
    __syncthreads();
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wid == a.nw) { if (lane == 0) producer(a, smem, full, empty); return; }
    const int tid = threadIdx.x, nt = a.nw * 32;
    const int Lb = a.Lb, B = a.B, C = (int)a.g.C;
    const unsigned fillw = a.fillw;
    int s = 0;
    unsigned phase = 0;
    for (int t = blockIdx.x; t < a.nstages; t += gridDim.x) {
        const long long p0 = (long long)t * a.K;
        const int np = a.planes - p0 < a.K ? (int)(a.planes - p0) : a.K;
        // lane l holds the shift of plane p0 + l of this stage
        int my_sr = 0, my_scb = 0;
        if (lane < np) flat_shift(a, (p0 + lane) % C, my_sr, my_scb);
        const unsigned sbase = shared_addr(smem + (size_t)s * a.stage_stride + GUARD);
        unsigned char* dst0 = a.y + p0 * a.plane_bytes;
        const int total = np * a.ipp;
        mbar_wait(&full[s], phase);
        for (int i0 = 0; i0 < total; i0 += nt) {       // warp-uniform trip count: the shuffles below need every lane
            const int i = i0 + tid;
            const bool live = i < total;
            const int q = live ? (int)fdiv((unsigned)i, a.d_ipp) : 0;
            const int sr = __shfl_sync(0xffffffffu, my_sr, q), scb = __shfl_sync(0xffffffffu, my_scb, q);
            if (!live) continue;
            const int m = i - q * a.ipp;
            const int delta = sr * Lb + scb;
            const int o = 16 * m;
            const int r0 = (int)fdiv((unsigned)o, a.d_Lb), c0 = o - r0 * Lb;
            const int n0b = Lb - c0 < 16 ? Lb - c0 : 16;
            const int lo = scb > 0 ? scb : 0, hi = scb < 0 ? Lb + scb : Lb;          // valid byte columns of a row
            unsigned mask = 0u;
            if ((unsigned)(r0 - sr) < (unsigned)B) {
                const int l = lo - c0 > 0 ? lo - c0 : 0, h = hi - c0 < n0b ? hi - c0 : n0b;
                mask |= bits_range(l, h);
            }
            if (n0b < 16 && (unsigned)(r0 + 1 - sr) < (unsigned)B) {
                const int h = n0b + hi < 16 ? n0b + hi : 16;
                mask |= bits_range(n0b + lo, h);
            }
            uint4 out = make_uint4(fillw, fillw, fillw, fillw);
            if (mask) {
                const int so = o - delta;                  // >= -15 whenever a byte is valid
                const unsigned addr = sbase + (unsigned)(q * a.plane_bytes + (so & ~15));
                const uint4 A = lds128(addr), Bv = lds128(addr + 16);
                const unsigned W[8] = {A.x, A.y, A.z, A.w, Bv.x, Bv.y, Bv.z, Bv.w};
                const int ws = (so & 15) >> 2, bs8 = (so & 3) * 8;
                unsigned U[7], V[5], v[4];
#pragma unroll
                for (int k = 0; k < 7; ++k) U[k] = (ws & 1) ? W[k + 1] : W[k];
#pragma unroll
                for (int k = 0; k < 5; ++k) V[k] = (ws & 2) ? U[k + 2] : U[k];
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] = __funnelshift_r(V[k], V[k + 1], bs8);
                if (mask != 0xffffu) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const unsigned wm = spread_nibble((mask >> (4 * k)) & 15u);
                        v[k] = (v[k] & wm) | (fillw & ~wm);
                    }
                }
                out = make_uint4(v[0], v[1], v[2], v[3]);
            }
            __stcs((uint4*)(dst0 + (size_t)q * a.plane_bytes + 16 * m), out);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        if (++s == a.stages) { s = 0; phase ^= 1u; }
    }
}

// ---- variant 2: a WARP owns whole planes ----------------------------------------------------------
// The plane's shift is warp-uniform, so the window misalignment is a compile-time constant of the inner loop (no
// select network, no shuffles) and everything that depends on the shift only is hoisted out of it; the per-channel
// shifts come from a table every CTA builds once in shared memory.
template <int WS>
TS_D void plane_items(const FArgs& a, unsigned src_plane, unsigned char* dst, int sr, int scb, int lane) {
    const int Lb = a.Lb, B = a.B;
    const unsigned fillw = a.fillw;
    const int delta = sr * Lb + scb;
    const int bs8 = ((-delta) & 3) * 8;
    const int lo = scb > 0 ? scb : 0, hi = scb < 0 ? Lb + scb : Lb;          // valid byte columns of a row
    const int base = (-delta) & ~15;                                            // so & ~15 = 16 m + base  (16 m is a multiple of 16)
    for (int m = lane; m < a.ipp; m += 32) {
        const int o = 16 * m;
        const int r0 = (int)fdiv((unsigned)o, a.d_Lb), c0 = o - r0 * Lb;
        const int n0b = Lb - c0 < 16 ? Lb - c0 : 16;
        unsigned mask = 0u;
        if ((unsigned)(r0 - sr) < (unsigned)B) {
            const int l = lo - c0 > 0 ? lo - c0 : 0, h = hi - c0 < n0b ? hi - c0 : n0b;
            mask |= bits_range(l, h);
        }
        if (n0b < 16 && (unsigned)(r0 + 1 - sr) < (unsigned)B) {
            const int h = n0b + hi < 16 ? n0b + hi : 16;
            mask |= bits_range(n0b + lo, h);
        }
        uint4 out = make_uint4(fillw, fillw, fillw, fillw);
        if (mask) {
            const unsigned addr = src_plane + (unsigned)(o + base);
            const uint4 A = lds128(addr), Bv = lds128(addr + 16);
            const unsigned W[9] = {A.x, A.y, A.z, A.w, Bv.x, Bv.y, Bv.z, Bv.w, 0u};
            unsigned v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = __funnelshift_r(W[k + WS], W[k + WS + 1], bs8);
            if (mask != 0xffffu) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const unsigned wm = spread_nibble((mask >> (4 * k)) & 15u);
                    v[k] = (v[k] & wm) | (fillw & ~wm);
                }
            }
            out = make_uint4(v[0], v[1], v[2], v[3]);
        }
        __stcs((uint4*)(dst + o), out);
    }
}

__global__ void __launch_bounds__(512, 1) k_flat_gather_wp(const __grid_constant__ FArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t* full = (uint64_t*)(smem + (size_t)a.stages * a.stage_stride);
    uint64_t* empty = full + a.stages;
    int2* tbl = (int2*)(empty + a.stages);
    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], (unsigned)a.nw); }
        fence_barrier_init();
    }
    const int C = (int)a.g.C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        int sr, scb;
        flat_shift(a, c, sr, scb);
        tbl[c] = make_int2(sr, scb);
    }
    __syncthreads();
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wid == a.nw) { if (lane == 0) producer(a, smem, full, empty); return; }
    int s = 0;
    unsigned phase = 0;
    for (int t = blockIdx.x; t < a.nstages; t += gridDim.x) {
        const long long p0 = (long long)t * a.K;
        const int np = a.planes - p0 < a.K ? (int)(a.planes - p0) : a.K;
        const unsigned sbase = shared_addr(smem + (size_t)s * a.stage_stride + GUARD);
        unsigned char* dst0 = a.y + p0 * a.plane_bytes;
        int c0;                                  // channel of the stage's first plane
        if (a.planes < 0x7fffffffLL) { const unsigned pu = (unsigned)p0; c0 = (int)(pu - fdiv(pu, a.d_C) * (unsigned)C); }
        else c0 = (int)(p0 % C);
        mbar_wait(&full[s], phase);
        for (int q = wid; q < np; q += a.nw) {
            int c = c0 + q;
            while (c >= C) c -= C;
            const int2 sh = tbl[c];
            const int ws = ((-(sh.x * a.Lb + sh.y)) & 15) >> 2;
            const unsigned src = sbase + (unsigned)(q * a.plane_bytes);
            unsigned char* dst = dst0 + (size_t)q * a.plane_bytes;
            switch (ws) {
            case 0: plane_items<0>(a, src, dst, sh.x, sh.y, lane); break;
            case 1: plane_items<1>(a, src, dst, sh.x, sh.y, lane); break;
            case 2: plane_items<2>(a, src, dst, sh.x, sh.y, lane); break;
            default: plane_items<3>(a, src, dst, sh.x, sh.y, lane); break;
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        if (++s == a.stages) { s = 0; phase ^= 1u; }
    }
}

}  // namespace

FlatPlan plan_flat(const Geo& g, int esize, bool dense_x, const void* x, const void* y, int sm_count, bool forced) {
    FlatPlan p;
    memset(&p, 0, sizeof(p));
    p.ok = false;
    if (g.pad != TS_PAD_ZEROS || !dense_x) return p;
    if (esize != 1 && esize != 2 && esize != 4) return p;
    if (g.N * g.C == 0 || g.in_plane == 0) return p;
    const int d = g.dim;
    if (d > 2) return p;                                                // 3-D volumes: the slab axis needs the producer remap (staged family)
    for (int ax = 0; ax < d; ++ax)
        if (g.lb[ax] != 0 || g.OS[ax] != g.S[ax]) return p;            // a crop breaks the constant source offset
    const long long B = d == 2 ? g.S[0] : 1;
    const long long Lb = (long long)g.S[d - 1] * esize;
    const long long plane = B * Lb;
    if (Lb < 16 || plane % 16 || plane >= (1 << 19)) return p;
    if (((uintptr_t)x & 15) || ((uintptr_t)y & 15)) return p;
    if (g.N * g.C >= (1ll << 40)) return p;
    const Tuning& t = tuning();
    // defaults from tools/knob_sweep.py cfg5 on B200: one CTA of 15 warps per SM, 4 stages of 48 KB (74 us; two CTAs of 8 warps
    // with 24 KB stages: 80 us; three with 16 KB: 77 us)
    const int ctas = t.flat_ctas > 0 ? t.flat_ctas : 1;
    const bool wp = g.C <= TABLE_MAX_C;                // warp-per-plane variant with the shift table
    const long long table_bytes = wp ? g.C * 8 : 0;
    const long long budget = SMEM_LIMIT / ctas - 1024 - table_bytes;
    const long long target = (long long)(t.flat_stage_kb > 0 ? t.flat_stage_kb : (ctas == 1 ? 48 : 24)) * 1024;
    long long K = target / plane;
    if (K < 1) K = 1;
    if (K > MAX_K) K = MAX_K;
    if (K > g.N * g.C) K = g.N * g.C;
    auto stride_of = [&](long long n) { return round_up(n * plane + 2 * GUARD + 32, 128); };
    int stages = t.flat_stages > 0 ? t.flat_stages : 4;
    while (stages * (stride_of(K) + 16) + 64 > budget) {
        if (K > 1) --K;
        else if (stages > 2) --stages;
        else return p;
    }
    if (K * plane >= (1 << 20)) return p;                              // mbarrier tx-count range
    if (!forced && K * (plane / 16) < 64) return p;
    const long long nstages = (g.N * g.C + K - 1) / K;
    if (nstages > 0x7fffffffLL) return p;
    const long long grid_max = (long long)sm_count * ctas;
    int warps = t.flat_warps > 0 ? t.flat_warps : (ctas >= 2 ? (wp ? 8 : 7) : 15);
    if (warps > 15) warps = 15;
    FArgs& a = p.a;
    a.g = g;
    a.planes = g.N * g.C;
    a.es = esize; a.dim = d;
    a.B = (int)B;
    a.Lb = (int)Lb;
    a.plane_bytes = (int)plane;
    a.ipp = a.plane_bytes / 16;
    a.K = (int)K; a.stages = stages; a.stage_stride = (int)stride_of(K); a.nw = warps;
    a.nstages = (int)nstages;
    a.table = wp ? 1 : 0;
    a.d_ipp = make_fastdiv((unsigned)a.ipp);
    a.d_Lb = make_fastdiv((unsigned)a.Lb);
    a.d_C = make_fastdiv((unsigned)g.C);
    p.ok = true;
    p.grid = (int)(nstages < grid_max ? nstages : grid_max);
    p.smem_bytes = (size_t)(stages * stride_of(K) + 16 * stages + 64 + table_bytes);
    return p;
}

int flat_gather(const Geo& g, const FlatPlan& p, int wk, const void* x, void* y, unsigned long long fill, int esize, const void* w,
                int qkind, long long wzp, cudaStream_t s) {
    FArgs a = p.a;
    a.x = (const unsigned char*)x; a.y = (unsigned char*)y; a.w = w; a.wzp = wzp;
    a.fillw = esize == 1 ? 0x01010101u * (unsigned)(fill & 0xffu) : esize == 2 ? 0x00010001u * (unsigned)(fill & 0xffffu) : (unsigned)fill;
    a.qkind = qkind; a.wk = wk;
    return launch_persistent(a.table ? k_flat_gather_wp : k_flat_gather, p.grid, (a.nw + 1) * 32, p.smem_bytes, s, false, a);
}

}  // namespace ts

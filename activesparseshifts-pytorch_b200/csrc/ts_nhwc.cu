// ts_nhwc.cu -- channels-last (NHWC / NDHWC) support.
//
//  * Quantized gather with input AND output channels-last (ts_qshift_forward_nhwc), so a quantized
//    channels-last pipeline pays one read and one write of the tensor instead of the three passes
//    (to-NCHW copy, NCHW kernel, to-NHWC copy) the planar families would need.  Two kernels:
//      k_gather_nhwc_ring  2-D, 1-byte elements, C % 32 == 0: input rows staged in a shared-memory ring,
//      k_gather_nhwc       everything else (3-D, 4-byte elements, odd channel counts): direct global loads.
//    Semantics: reference body  ops/kernels/shifts_kernels.h:574-624 (shift_forward_kernel_nhwdc_q),
//               driver          ops/quantized/shifts_quantized.cpp:107-130 (output allocated in the
//                               input's memory format, :119-122).
//  * k_nhwc_to_nchw (ts_nhwc_to_nchw): the layout pass of the FLOAT path, whose outputs are planar in the
//    reference too (ops/cpu/shifts_cpu.cpp:55-75 reads NHWC, :221 returns NCHW).
//
// Both gather kernels' thread programs are host+device code: ts_debug_nhwc_emulate walks them on the host,
// barrier phase by barrier phase, so the CPU-side tests can check the index logic without a GPU.
//
// Direct kernel, layout of the work.  In NHWC the per-channel shift is a per-lane gather: the channel vector
// of one output pixel takes each of its channels from a different input pixel.  Consecutive lanes own
// consecutive 4-byte words of the channel vector (4 channels of a 1-byte type, 1 channel of a 4-byte
// type), so every warp store is one contiguous 128-byte line; the loads are one byte each and land in
// (nearly) as many 32-byte sectors as there are lanes, re-used by the neighbouring pixels through L1/L2.
// A CTA owns a few consecutive output rows of one image and its threads keep their channel group for
// the whole CTA lifetime: the shifts, the remapped outer-axis offsets and the validity flags are
// registers, and the inner loop over the pixels of a row is one remap + one byte load per channel.
#include "ts_kernels.h"
#include "ts_ptx.cuh"

namespace ts {

namespace {

constexpr int NHWC_THREADS = 256;

struct NhwcPlan {
    int vec;            // elements per thread item (vec * esize == 4 when possible)
    int cg;             // channel groups = C / vec
    int tc, tp;         // threads along the channel groups / along the pixels of a row
    unsigned rows;      // N * prod(OS[0..dim-2])
    int rows_per_cta;
    unsigned groups;    // ceil(rows / rows_per_cta)
    int segs, seg_len;  // split of the last axis across blockIdx.y
    unsigned grid_x;    // CTAs along x (row groups are grid-strided when there are more)
};

template <typename E, int VEC> struct PackOut;
template <> struct PackOut<uint8_t, 4> {
    static TS_HD void store(uint8_t* p, const uint8_t* v) {
        *reinterpret_cast<uint32_t*>(p) = (uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) | ((uint32_t)v[3] << 24);
    }
};
template <typename E> struct PackOut<E, 1> {
    static TS_HD void store(E* p, const E* v) { *p = v[0]; }
};

// A size-1 axis needs no special case here: its reduced shift is 0 (reduce_shift), so the index is 0 and
// every padding mode maps 0 to 0.
template <int PAD> TS_HD int axis_index_c(int idx, int len) { return remap_bounded(idx, len, PAD); }

template <typename E> TS_HD E load_ro(const E* p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

// The whole per-thread program, host+device so the CPU-side tests can run the very same index logic
// over every (block, thread) of a small launch (ts_debug_nhwc_emulate) without a GPU.
template <typename E, int DIM, int VEC, int PAD>
TS_HD void nhwc_thread(const Geo& g, const NhwcPlan& pl, int tid, unsigned bx, unsigned by, unsigned grid_x,
                       const E* __restrict__ x, E* __restrict__ y, E fill, const void* __restrict__ w, int qkind, long long wzp) {
    constexpr int LAST = DIM - 1;
    const int cgi = tid % pl.tc;
    const int pw = tid / pl.tc;
    const int L = g.OS[LAST];
    const int p_begin = (int)by * pl.seg_len;
    const int p_end = L < p_begin + pl.seg_len ? L : p_begin + pl.seg_len;
    const unsigned xs_last_bytes = (unsigned)(g.xs[2 + LAST] * (long long)sizeof(E));   // < 2^31, checked by the launcher
    const int lb_last = g.lb[LAST], s_last = g.S[LAST];

    for (int cg = cgi; cg < pl.cg; cg += pl.tc) {
        const int c0 = cg * VEC;
        int sx[VEC][DIM];
#pragma unroll
        for (int v = 0; v < VEC; ++v) load_qshifts<DIM>(w, qkind, wzp, (long long)(c0 + v), g, sx[v]);

        for (unsigned grp = bx; grp < pl.groups; grp += grid_x) {
            const unsigned r_begin = grp * (unsigned)pl.rows_per_cta;
            const unsigned r_stop = r_begin + (unsigned)pl.rows_per_cta;
            const unsigned r_end = pl.rows < r_stop ? pl.rows : r_stop;
            for (unsigned row = r_begin; row < r_end; ++row) {
                // row -> (n, o0[, o1]) in output coordinates
                unsigned n = row;
                int o[2] = {0, 0};
                if (DIM == 2) {
                    n = row / (unsigned)g.OS[0];
                    o[0] = (int)(row - n * (unsigned)g.OS[0]);
                } else if (DIM == 3) {
                    const unsigned t = row / (unsigned)g.OS[1];
                    o[1] = (int)(row - t * (unsigned)g.OS[1]);
                    n = t / (unsigned)g.OS[0];
                    o[0] = (int)(t - n * (unsigned)g.OS[0]);
                }
                const char* xp[VEC];     // start of the source row of each channel (byte pointer)
                bool ok[VEC];
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    long long base = (long long)n * g.xs[0] + (long long)(c0 + v) * g.xs[1];
                    ok[v] = true;
#pragma unroll
                    for (int a = 0; a < LAST; ++a) {
                        const int t = axis_index_c<PAD>(o[a] + g.lb[a] - sx[v][a], g.S[a]);
                        ok[v] = ok[v] && (t >= 0);
                        base += (long long)(t < 0 ? 0 : t) * g.xs[2 + a];
                    }
                    xp[v] = reinterpret_cast<const char*>(x + base);
                }
                E* yp = y + ((long long)row * L + (p_begin + pw)) * g.C + c0;
                const long long y_step = (long long)pl.tp * g.C;
#pragma unroll 2
                for (int p = p_begin + pw; p < p_end; p += pl.tp, yp += y_step) {
                    E val[VEC];
#pragma unroll
                    for (int v = 0; v < VEC; ++v) {
                        const int t = axis_index_c<PAD>(p + lb_last - sx[v][LAST], s_last);
                        const bool valid = ok[v] && (t >= 0);
                        // the load is unconditional (an invalid tap reads the row start, always inside x): no predicated
                        // address arithmetic in the loop, one select after the load
                        const unsigned long long off = (unsigned long long)(valid ? (unsigned)t : 0u) * xs_last_bytes;
                        const E got = load_ro(reinterpret_cast<const E*>(xp[v] + off));
                        val[v] = valid ? got : fill;
                    }
                    PackOut<E, VEC>::store(yp, val);
                }
            }
        }
    }
}

template <typename E, int DIM, int VEC, int PAD>
__global__ void __launch_bounds__(NHWC_THREADS) k_gather_nhwc(Geo g, NhwcPlan pl, const E* __restrict__ x, E* __restrict__ y,
                                                              E fill, const void* __restrict__ w, int qkind, long long wzp) {
    nhwc_thread<E, DIM, VEC, PAD>(g, pl, (int)threadIdx.x, blockIdx.x, blockIdx.y, gridDim.x, x, y, fill, w, qkind, wzp);
}

NhwcPlan make_plan(const Geo& g, int esize, const void* y, int sm_count, int max_grid_x) {
    NhwcPlan pl;
    pl.vec = (esize == 1 && g.C % 4 == 0 && ((uintptr_t)y & 3u) == 0) ? 4 : 1;
    pl.cg = (int)(g.C / pl.vec);
    if (pl.cg >= NHWC_THREADS) { pl.tc = NHWC_THREADS; pl.tp = 1; }
    else { pl.tc = pl.cg; pl.tp = NHWC_THREADS / pl.cg; }
    long long rows = g.N;
    for (int a = 0; a < g.dim - 1; ++a) rows *= g.OS[a];
    pl.rows = (unsigned)rows;
    const int L = g.OS[g.dim - 1];
    const long long want_ctas = (long long)sm_count * 16;
    long long rb = rows / want_ctas;
    if (rb < 1) rb = 1;
    if (rb > 8) rb = 8;
    const long long items_per_row = (long long)L * pl.cg;
    while (rb * items_per_row < 16 * NHWC_THREADS && rb < 64 && rb < rows) rb *= 2;
    pl.rows_per_cta = (int)rb;
    pl.groups = (unsigned)((rows + rb - 1) / rb);
    long long segs = 1;
    if ((long long)pl.groups < (long long)sm_count * 8) {
        segs = ((long long)sm_count * 8 + pl.groups - 1) / pl.groups;
        const long long max_segs = (L + pl.tp - 1) / pl.tp;
        if (segs > max_segs) segs = max_segs;
        if (segs > 65535) segs = 65535;
        if (segs < 1) segs = 1;
    }
    pl.seg_len = (int)((L + segs - 1) / segs);
    pl.segs = (L + pl.seg_len - 1) / pl.seg_len;
    const unsigned cap = max_grid_x > 0 ? (unsigned)max_grid_x : (1u << 20);
    pl.grid_x = pl.groups > cap ? cap : pl.groups;
    return pl;
}

// ------------------------------------------------------------------------------------------
// Ring kernel (2-D, 1-byte elements): the same gather, fed from shared memory.
//
// Through L1 every gathered byte costs one 32-byte sector access (neighbouring channels have different
// shifts, so the 32 lanes of a request land in ~28 different sectors: measured with ncu, 184 M sector
// accesses for 205 M output bytes, L1 throughput-bound at 0.28 ms).  Shared memory serves 32 scattered
// bytes per cycle as long as the lanes hit different banks, and with lane <-> word-of-the-channel-slice
// the bank IS the lane whatever pixel each lane's shift selects.  So a CTA owns (image, slice of <= 128
// channels, segment of output rows), walks down the rows and keeps the input rows the current group of
// output rows can reach in a ring of K row slots: every input row slice is fetched from global memory
// exactly once per unit, with 16-byte cp.async copies of whole sectors.  The ring is a software cache,
// not a contract: a tap whose (remapped) row is not in the ring -- wrap-around paddings at the image
// edges, shifts spread wider than the ring -- is read from global memory instead, so the choice of
// window only ever affects speed.
struct RingPlan {
    int cs, slices;       // channels per slice (power of two, 32..128), C / cs
    int k;                // ring slots (input rows of one slice)
    int segs, seg_rows;   // output rows are split into segs segments of seg_rows rows
    int tw;               // lanes along the words of a slice (cs / 4); a warp covers 32 / tw pixels at a time
    int chunk_shift;      // log2(cs / 16): 16-byte chunks per pixel slice
    unsigned units, grid;
    unsigned smem_bytes;  // ring + 16 (the last 16 bytes hold the fill byte)
};
constexpr int RING_THREADS = 256;
constexpr int RING_MAX_CS = 128;
constexpr int RING_WARPS = RING_THREADS / 32;
static_assert(RING_WARPS == 8, "ring_compute splits rows across 8 warps with shifts");

struct RingUnit { unsigned n; int c_base, o_begin, o_end; };
struct RingThread { int s0[4], s1[4], smin, smax; };   // lives in registers across the phases of a unit
struct RingStep { int o_a, o_b, lo, hi, new_lo, slot_lo, rb; };

TS_HD int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

TS_HD RingUnit ring_unit(const Geo& g, const RingPlan& pl, unsigned unit) {
    RingUnit u;
    const unsigned seg = unit % (unsigned)pl.segs;
    const unsigned t = unit / (unsigned)pl.segs;
    const unsigned k = t % (unsigned)pl.slices;
    u.n = t / (unsigned)pl.slices;
    u.c_base = (int)k * pl.cs;
    u.o_begin = (int)seg * pl.seg_rows;
    u.o_end = u.o_begin + pl.seg_rows < g.OS[0] ? u.o_begin + pl.seg_rows : g.OS[0];
    return u;
}

// Phase 1: one thread per channel of the slice reduces its two shifts into sh[0..cs) / sh[128..128+cs).
TS_HD void ring_phase_shifts(const Geo& g, const RingPlan& pl, const RingUnit& u, int tid, const void* __restrict__ w, int qkind,
                             long long wzp, int* sh, uint8_t* ring, uint8_t fill) {
    if (tid == 0) ring[pl.smem_bytes - 16u] = fill;      // the pad value, addressable like any ring byte
    if (tid < pl.cs) {
        int sx[2];
        load_qshifts<2>(w, qkind, wzp, (long long)(u.c_base + tid), g, sx);
        sh[tid] = sx[0];
        sh[RING_MAX_CS + tid] = sx[1];
    }
}

// Phase 2 (after a barrier): every thread picks up the shifts of its 4 channels and the slice-wide range
// of the axis-0 shifts (identical in every thread: it sizes the groups of output rows).
TS_HD void ring_phase_regs(const RingPlan& pl, int tid, const int* sh, RingThread& th) {
    const int wi = (tid & 31) % pl.tw;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        th.s0[v] = sh[4 * wi + v];
        th.s1[v] = sh[RING_MAX_CS + 4 * wi + v];
    }
    int mn = sh[0], mx = sh[0];
    for (int i = 1; i < pl.cs; ++i) {
        const int s = sh[i];
        mn = s < mn ? s : mn;
        mx = s > mx ? s : mx;
    }
    th.smin = mn;
    th.smax = mx;
}

// The walk down the output rows of a unit, identical in every thread.
struct RingWalk {
    int o_next, o_end, rb, phi, smin, smax, lb0, s0, k, prev_lo, prev_slot;
    TS_HD RingWalk(const Geo& g, const RingPlan& pl, const RingUnit& u, const RingThread& th) {
        o_next = u.o_begin;
        o_end = u.o_end;
        smin = th.smin;
        smax = th.smax;
        lb0 = g.lb[0];
        s0 = g.S[0];
        k = pl.k;
        const int span = smax - smin;
        rb = k - span > 1 ? k - span : 1;         // output rows per step: their reach, rb + span rows, fits the ring
        if (rb >= RING_WARPS) rb -= rb % RING_WARPS;  // a warp owns one output row at a time: keep the warps level
        else rb = rb >= 4 ? 4 : (rb >= 2 ? 2 : 1);    // fewer rows than warps: 2 / 4 / 8 warps share a row (ring_compute)
        phi = -1;                                  // highest input row fetched so far in this unit
        prev_lo = 0;                               // row 0 lives in slot 0: slot(row) = row mod k
        prev_slot = 0;
    }
    TS_HD bool next(RingStep& s) {
        if (o_next >= o_end) return false;
        s.o_a = o_next;
        s.rb = rb;
        s.o_b = o_next + rb < o_end ? o_next + rb : o_end;
        o_next = s.o_b;
        s.lo = clampi(s.o_a + lb0 - smax, 0, s0 - 1);
        s.hi = clampi(s.o_b - 1 + lb0 - smin, 0, s0 - 1);
        if (s.hi - s.lo + 1 > k) s.hi = s.lo + k - 1;
        s.new_lo = s.lo > phi + 1 ? s.lo : phi + 1;
        if (s.hi > phi) phi = s.hi;
        // lo only moves forward: one division for the first step, a short catch-up afterwards
        const int adv = s.lo - prev_lo;
        if (adv >= 2 * k) prev_slot = s.lo % k;
        else { prev_slot += adv; if (prev_slot >= k) prev_slot -= k; if (prev_slot >= k) prev_slot -= k; }
        prev_lo = s.lo;
        s.slot_lo = prev_slot;
        return true;
    }
};

TS_HD int ring_slot(const RingStep& st, int k, int row) {   // row in [st.lo, st.hi]
    const int s = row - st.lo + st.slot_lo;
    return s >= k ? s - k : s;
}

TS_HD void copy16(uint8_t* dst_ring, const uint8_t* src_global) {
#ifdef __CUDA_ARCH__
    ptx::cp_async16(shared_addr(dst_ring), src_global);
#else
    for (int i = 0; i < 16; ++i) dst_ring[i] = src_global[i];
#endif
}

// One byte of the ring.  On the device the ring is addressed through its 32-bit shared-window address and an
// opaque ld.shared.u8 (written as `ring[off]` the compiler re-derives the window base, half a dozen
// instructions, next to every load).
TS_HD unsigned ring_base(const uint8_t* ring) {
#ifdef __CUDA_ARCH__
    return shared_addr(ring);
#else
    (void)ring;
    return 0u;
#endif
}
TS_HD unsigned ring_byte(const uint8_t* ring, unsigned addr) {      // zero-extended
#ifdef __CUDA_ARCH__
    unsigned v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
#else
    return ring[addr];
#endif
}
// Four zero-extended bytes -> one little-endian word (three PRMTs on the device).
TS_HD void store4(uint8_t* p, const unsigned* v) {
#ifdef __CUDA_ARCH__
    const unsigned lo = __byte_perm(v[0], v[1], 0x0040), hi = __byte_perm(v[2], v[3], 0x0040);
    *reinterpret_cast<uint32_t*>(p) = __byte_perm(lo, hi, 0x5410);
#else
    *reinterpret_cast<uint32_t*>(p) = (v[0] & 0xffu) | ((v[1] & 0xffu) << 8) | ((v[2] & 0xffu) << 16) | ((v[3] & 0xffu) << 24);
#endif
}

// Fetch the input rows [st.new_lo, st.hi] of this unit's channel slice into their ring slots.
TS_HD void ring_load(const Geo& g, const RingPlan& pl, const RingUnit& u, const RingStep& st, int tid, int threads,
                     const uint8_t* __restrict__ x, uint8_t* ring) {
    const int nrows = st.hi - st.new_lo + 1;
    if (nrows <= 0) return;
    // A thread keeps its chunk position(s) inside the row slice and walks down the rows: per copy one
    // 64-bit add for the source and an add-with-wrap for the ring slot.
    const int per_row = g.S[1] << pl.chunk_shift;       // 16-byte chunks of one row slice
    const unsigned row_bytes = (unsigned)g.S[1] * (unsigned)pl.cs;
    const unsigned ring_bytes = (unsigned)pl.k * row_bytes;
    const int slot0 = ring_slot(st, pl.k, st.new_lo);
    const uint8_t* src0 = x + (long long)u.n * g.xs[0] + u.c_base + (long long)st.new_lo * g.xs[2];
    for (int j = tid; j < per_row; j += threads) {
        const int q = j >> pl.chunk_shift;
        const int part = j & ((1 << pl.chunk_shift) - 1);
        const uint8_t* src = src0 + (long long)q * g.xs[3] + part * 16;
        unsigned d = (unsigned)slot0 * row_bytes + (unsigned)q * (unsigned)pl.cs + (unsigned)part * 16u;
        for (int r = 0; r < nrows; ++r) {
            copy16(ring + d, src);
            src += g.xs[2];
            d += row_bytes;
            if (d >= ring_bytes) d -= ring_bytes;
        }
    }
}

template <int OFF> TS_HD unsigned ring_byte_at(const uint8_t* ring, unsigned addr) {   // ring_byte with an immediate offset
#ifdef __CUDA_ARCH__
    unsigned v;
    asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
    return v;
#else
    return ring[addr + OFF];
#endif
}

// 8 consecutive pixel steps of a warp (one step = 32 words = 128 ring bytes whatever the slice width) with
// the ring offsets as immediates: 4 loads, 3 PRMTs and one store per 4 output bytes.  All 32 loads are
// issued before the first pack, so the warp waits for the shared-memory latency once per 8 pixels.
template <int I> struct Span8 {
    static TS_HD void load(const uint8_t* ring, const unsigned* a, unsigned (*val)[4]) {
#pragma unroll
        for (int v = 0; v < 4; ++v) val[I][v] = ring_byte_at<I * 128>(ring, a[v]);
        Span8<I + 1>::load(ring, a, val);
    }
};
template <> struct Span8<8> {
    static TS_HD void load(const uint8_t*, const unsigned*, unsigned (*)[4]) {}
};

// Gather phase.  A warp owns one output row at a time: its lanes are the words of the channel slice (and,
// for slices narrower than 128 channels, 2 or 4 neighbouring pixels), so the per-row work -- remapping the
// source row of each of the thread's 4 channels, locating it in the ring -- is paid once per 56-pixel row,
// not once per handful of pixels.  Per (output row, channel) the source is one of three: a ring row (the
// common case), the fill byte (the whole source row is outside the image: zeros padding), or global memory
// (a valid row the ring does not hold).  The fill byte lives in shared memory right behind the ring, so
// "outside" is just another address; rows with a global-memory channel take a separate, slower loop.
template <int PAD>
TS_HD void ring_compute(const Geo& g, const RingPlan& pl, const RingUnit& u, const RingStep& st, const RingThread& th, int tid,
                        const uint8_t* __restrict__ x, uint8_t* __restrict__ y, uint8_t fill, const uint8_t* ring) {
    const int lane = tid & 31, warp = tid >> 5;
    const int wi = lane % pl.tw;              // word of the slice
    const int pw = lane / pl.tw;              // pixel lane inside the warp
    const int ppw = 32 / pl.tw;               // pixels a warp covers per step; ppw * cs == 128
    const int c0 = u.c_base + 4 * wi;
    const int s1 = g.S[1], lb1 = g.lb[1], ow = g.OS[1];
    const unsigned base = ring_base(ring);
    const unsigned fill_addr = base + pl.smem_bytes - 16u;
    const unsigned cs = (unsigned)pl.cs;
    const unsigned long long xs3 = (unsigned long long)g.xs[3];
    const long long y_step = (long long)ppw * g.C;
    // output pixels [p_lo, p_hi] whose taps p + lb1 - s1[v] fall inside the source row for all 4 channels
    int s1_max = th.s1[0], s1_min = th.s1[0];
#pragma unroll
    for (int v = 1; v < 4; ++v) {
        s1_max = th.s1[v] > s1_max ? th.s1[v] : s1_max;
        s1_min = th.s1[v] < s1_min ? th.s1[v] : s1_min;
    }
    const int p_lo = s1_max - lb1 > 0 ? s1_max - lb1 : 0;
    const int p_hi = s1 - 1 - lb1 + s1_min < ow - 1 ? s1 - 1 - lb1 + s1_min : ow - 1;
    // rows of the step over the warps; with fewer rows than warps, `parts` warps share a row (pixel ranges)
    // (st.rb is a multiple of the warp count, or 4 / 2 / 1: everything here is a shift)
    const int part_shift = st.rb >= RING_WARPS ? 0 : (st.rb == 4 ? 1 : (st.rb == 2 ? 2 : 3));
    const int rows_in_flight = RING_WARPS >> part_shift;
    const int part = warp >> (3 - part_shift);
    const int part_len = (ow + (1 << part_shift) - 1) >> part_shift;
    const int pa = part * part_len < ow ? part * part_len : ow;
    const int pb = pa + part_len < ow ? pa + part_len : ow;
    const int p_hi_w = p_hi < pb - 1 ? p_hi : pb - 1;
    for (int o = st.o_a + (warp & (rows_in_flight - 1)); o < st.o_b; o += rows_in_flight) {
        unsigned row_addr[4], pitch[4];     // ring address of pixel 0 of the source row, bytes between its pixels
        bool from_global = false, all_ring = true;
        int t0s[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int t0 = axis_index_c<PAD>(o + g.lb[0] - th.s0[v], g.S[0]);
            t0s[v] = t0;
            const bool inw = t0 >= st.lo && t0 <= st.hi;           // implies t0 >= 0
            row_addr[v] = inw ? base + (unsigned)(ring_slot(st, pl.k, t0) * s1) * cs + (unsigned)(4 * wi + v) : fill_addr;
            pitch[v] = inw ? cs : 0u;
            from_global = from_global || (t0 >= 0 && !inw);
            all_ring = all_ring && inw;
        }
        int p = pa + pw;
        uint8_t* yp = y + (((long long)u.n * g.OS[0] + o) * ow + p) * g.C + c0;
        if (!from_global) {
            for (; p < p_lo && p < pb; p += ppw, yp += y_step) {            // leading pixels: some tap is left of the row
                unsigned val[4];
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int t1 = axis_index_c<PAD>(p + lb1 - th.s1[v], s1);
                    val[v] = ring_byte(ring, t1 >= 0 ? row_addr[v] + (unsigned)t1 * pitch[v] : fill_addr);
                }
                store4(yp, val);
            }
            // interior: every tap of the 4 channels is inside its source row, the addresses just advance
            unsigned addr[4], step[4];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                addr[v] = row_addr[v] + (unsigned)(p + lb1 - th.s1[v]) * pitch[v];
                step[v] = (unsigned)ppw * pitch[v];
            }
            if (all_ring) {
                for (; p + 7 * ppw <= p_hi_w; p += 8 * ppw) {
                    unsigned val[8][4];
                    Span8<0>::load(ring, addr, val);
#pragma unroll
                    for (int i = 0; i < 8; ++i, yp += y_step) store4(yp, val[i]);
#pragma unroll
                    for (int v = 0; v < 4; ++v) addr[v] += 8u * 128u;
                }
            }
            for (; p <= p_hi_w; p += ppw, yp += y_step) {
                unsigned val[4];
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    val[v] = ring_byte(ring, addr[v]);
                    addr[v] += step[v];
                }
                store4(yp, val);
            }
            for (; p < pb; p += ppw, yp += y_step) {                        // trailing pixels
                unsigned val[4];
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int t1 = axis_index_c<PAD>(p + lb1 - th.s1[v], s1);
                    val[v] = ring_byte(ring, t1 >= 0 ? row_addr[v] + (unsigned)t1 * pitch[v] : fill_addr);
                }
                store4(yp, val);
            }
        } else {
            for (; p < pb; p += ppw, yp += y_step) {
                unsigned val[4];
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int t1 = axis_index_c<PAD>(p + lb1 - th.s1[v], s1);
                    if (t0s[v] >= 0 && pitch[v] == 0u) {     // valid row, not in the ring
                        const uint8_t* src = x + (long long)u.n * g.xs[0] + (long long)t0s[v] * g.xs[2] + (c0 + v);
                        val[v] = t1 >= 0 ? (unsigned)load_ro(src + (unsigned long long)(unsigned)t1 * xs3) : (unsigned)fill;
                    } else {
                        val[v] = ring_byte(ring, t1 >= 0 ? row_addr[v] + (unsigned)t1 * pitch[v] : fill_addr);
                    }
                }
                store4(yp, val);
            }
        }
    }
}

template <int PAD>
__global__ void __launch_bounds__(RING_THREADS, 3) k_gather_nhwc_ring(Geo g, RingPlan pl, const uint8_t* __restrict__ x,
                                                                   uint8_t* __restrict__ y, uint8_t fill,
                                                                   const void* __restrict__ w, int qkind, long long wzp) {
    extern __shared__ uint4 ring_store[];
    __shared__ int sh[2 * RING_MAX_CS];
    uint8_t* ring = reinterpret_cast<uint8_t*>(ring_store);
    const int tid = (int)threadIdx.x;
    for (unsigned unit = blockIdx.x; unit < pl.units; unit += gridDim.x) {
        const RingUnit u = ring_unit(g, pl, unit);
        ring_phase_shifts(g, pl, u, tid, w, qkind, wzp, sh, ring, fill);
        __syncthreads();
        RingThread th;
        ring_phase_regs(pl, tid, sh, th);
        RingWalk walk(g, pl, u, th);
        RingStep st;
        while (walk.next(st)) {
            ring_load(g, pl, u, st, tid, RING_THREADS, x, ring);
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncthreads();             // the new rows are visible to every thread
            ring_compute<PAD>(g, pl, u, st, th, tid, x, y, fill, ring);
            __syncthreads();             // every thread is done with the rows the next step overwrites (and with sh)
        }
    }
}

// Host walk of the same CTA program: phases separated by the kernel's barriers, threads in turn.
template <int PAD>
void ring_emulate(const Geo& g, const RingPlan& pl, const uint8_t* x, uint8_t* y, uint8_t fill, const void* w, int qkind,
                  long long wzp) {
    uint8_t* ring = new uint8_t[pl.smem_bytes];
    RingThread* th = new RingThread[RING_THREADS];
    int sh[2 * RING_MAX_CS];
    for (unsigned b = 0; b < pl.grid; ++b) {
        for (unsigned unit = b; unit < pl.units; unit += pl.grid) {
            const RingUnit u = ring_unit(g, pl, unit);
            for (unsigned i = 0; i < pl.smem_bytes; ++i) ring[i] = 0xEE;   // a slot read before it is fetched shows up as a mismatch
            for (int tid = 0; tid < RING_THREADS; ++tid) ring_phase_shifts(g, pl, u, tid, w, qkind, wzp, sh, ring, fill);
            for (int tid = 0; tid < RING_THREADS; ++tid) ring_phase_regs(pl, tid, sh, th[tid]);
            RingWalk walk(g, pl, u, th[0]);
            RingStep st;
            while (walk.next(st)) {
                for (int tid = 0; tid < RING_THREADS; ++tid) ring_load(g, pl, u, st, tid, RING_THREADS, x, ring);
                for (int tid = 0; tid < RING_THREADS; ++tid) ring_compute<PAD>(g, pl, u, st, th[tid], tid, x, y, fill, ring);
            }
        }
    }
    delete[] th;
    delete[] ring;
}

bool plan_ring(const Geo& g, int esize, const void* x, const void* y, int sm_count, int max_grid_x, int ring_rows, RingPlan* out) {
    if (g.dim != 2 || esize != 1 || g.xs[1] != 1 || g.C % 32 != 0) return false;
    if (((uintptr_t)x & 15u) || ((uintptr_t)y & 3u)) return false;
    if ((g.xs[0] & 15) || (g.xs[2] & 15) || (g.xs[3] & 15) || g.xs[0] < 0 || g.xs[2] < 0 || g.xs[3] < 0) return false;
    if (g.xs[3] * (long long)g.S[1] >= 0x7fffffffLL) return false;
    RingPlan pl;
    const int cs_first = g.C % 128 == 0 ? 128 : (g.C % 64 == 0 ? 64 : 32);
    // Ring size: several CTAs per SM overlap one CTA's fetch phase with the others' gather phase (measured on
    // cfg5: 3 CTAs x 10 rows beat 2 x 15), but the ring must still hold the rows a group of output rows can reach.
    bool found = false;
    for (int min_k = 8; min_k >= 4 && !found; min_k -= 4) {
        for (int cs = cs_first; cs >= 32 && !found; cs >>= 1) {
            for (int ctas = 3; ctas >= 1 && !found; --ctas) {
                const long long avail = (227LL * 1024) / ctas - 1024 - 2048 - 16;   // reserved per CTA, static shared, fill tail
                long long k = avail / ((long long)g.S[1] * cs);
                if (k > g.S[0]) k = g.S[0];
                if (ring_rows > 0 && k > ring_rows) k = ring_rows;        // tuning / tests: force a small ring
                if (k >= min_k || (k >= 1 && (k == g.S[0] || ring_rows > 0))) {
                    pl.cs = cs;
                    pl.k = (int)k;
                    found = true;
                }
            }
        }
    }
    if (!found) return false;
    pl.slices = (int)(g.C / pl.cs);
    pl.tw = pl.cs / 4;
    pl.chunk_shift = pl.cs == 128 ? 3 : (pl.cs == 64 ? 2 : 1);
    pl.smem_bytes = (unsigned)((long long)pl.k * g.S[1] * pl.cs) + 16u;   // + the fill byte's 16-byte tail
    const long long base_units = g.N * pl.slices;
    long long fit = (228LL * 1024) / ((long long)pl.smem_bytes + 2048 + 1024);       // CTAs of this size one SM holds
    fit = fit < 1 ? 1 : (fit > 8 ? 8 : fit);
    const long long slots = (long long)sm_count * fit;
    double best = -1.0;
    int best_rows = g.OS[0];
    for (int segs = 1; segs <= 8 && segs <= g.OS[0]; ++segs) {
        int rows = (g.OS[0] + segs - 1) / segs;
        if (segs > 1 && rows > RING_WARPS) rows = (rows + RING_WARPS - 1) / RING_WARPS * RING_WARPS;   // whole rounds of the warps
        const int real_segs = (g.OS[0] + rows - 1) / rows;
        const long long units = base_units * real_segs;
        const long long waves = (units + slots - 1) / slots;
        const double eff = (double)units / (double)(waves * slots) * (double)rows / (double)(rows + 2);   // wave tail x halo re-reads
        if (eff > best * 1.02) { best = eff; best_rows = rows; }
    }
    pl.seg_rows = best_rows;
    pl.segs = (g.OS[0] + best_rows - 1) / best_rows;
    const long long units = base_units * pl.segs;
    if (units >= 0x7fffffffLL) return false;
    pl.units = (unsigned)units;
    long long grid = units < slots ? units : slots;
    if (max_grid_x > 0 && grid > max_grid_x) grid = max_grid_x;
    pl.grid = (unsigned)grid;
    *out = pl;
    return true;
}

template <int PAD>
int ring_launch(const Geo& g, const RingPlan& pl, const void* x, void* y, uint8_t fill, const void* w, int qkind, long long wzp,
                cudaStream_t s, bool emulate) {
    if (emulate) {
        ring_emulate<PAD>(g, pl, (const uint8_t*)x, (uint8_t*)y, fill, w, qkind, wzp);
        return TS_OK;
    }
    return launch_persistent(k_gather_nhwc_ring<PAD>, pl.grid, RING_THREADS, pl.smem_bytes, s, false, g, pl, (const uint8_t*)x, (uint8_t*)y,
                             fill, w, qkind, wzp);
}

int ring_run(const Geo& g, const RingPlan& pl, const void* x, void* y, uint8_t fill, const void* w, int qkind, long long wzp,
             cudaStream_t s, bool emulate) {
    switch (g.pad) {
    case TS_PAD_BORDER: return ring_launch<TS_PAD_BORDER>(g, pl, x, y, fill, w, qkind, wzp, s, emulate);
    case TS_PAD_PERIODIC: return ring_launch<TS_PAD_PERIODIC>(g, pl, x, y, fill, w, qkind, wzp, s, emulate);
    case TS_PAD_REFLECT: return ring_launch<TS_PAD_REFLECT>(g, pl, x, y, fill, w, qkind, wzp, s, emulate);
    case TS_PAD_SYMMETRIC: return ring_launch<TS_PAD_SYMMETRIC>(g, pl, x, y, fill, w, qkind, wzp, s, emulate);
    default: return ring_launch<TS_PAD_ZEROS>(g, pl, x, y, fill, w, qkind, wzp, s, emulate);
    }
}


// ------------------------------------------------------------------------------------------
// Row-pipelined kernel (2-D, 1-byte elements, dense pixels, C a multiple of 128; compile-time pixel pitch for 128 / 256 / 512): the ring kernel's gather fed by a
// producer warp instead of load / barrier / gather / barrier rounds.
//
// In NHWC a whole input row (S1 pixels x C channels) is CONTIGUOUS, so it is ONE bulk copy (cp.async.bulk, 14 KB for
// cfg5) into a slot of a K-row ring, announced on that slot's `full` mbarrier.  A CTA owns a contiguous range of the
// global list of output rows (N x OS0 rows dealt evenly: no wave tail, halo rows re-read only where a range starts); its W
// consumer warps take output rows round-robin.  A warp that is about to gather output row o waits (in row order) until
// the highest input row of o's window has landed, gathers, and releases every row below the window of its NEXT output
// row by arriving on those slots' `empty` mbarriers (W arrivals free a slot for the producer).  Nothing ever waits for
// a CTA-wide barrier: fetch, gather and store of different rows overlap inside one CTA (the ring kernel needed three
// CTAs per SM to overlap its phases and still stalled on cp.async.wait_all + two __syncthreads per step).
// The window of an output row is capped at WIN = K - W - 1 rows, so the rows in use never fill the ring; a tap whose
// (remapped) row lies outside the window -- wrap-around paddings at the image edges, axis-0 shifts spread wider than WIN --
// is read from global memory, exactly like in the ring kernel: the window only ever affects speed.
struct RowsPlan {
    int K, W, WIN;
    unsigned grid, row_bytes, smem_bytes, off_bar, off_tab;
};
constexpr int ROWS_MAX_W = 12;

struct RowsSeg { unsigned n; int o_a, o_b, lo, hi; };
// the s-th piece of the CTA's range [r0, r1) of global output rows: one image's rows and the input rows it can reach
TS_D bool rows_segment(const Geo& g, int WIN, unsigned& r, unsigned r1, int smin, int smax, RowsSeg& sg) {
    if (r >= r1) return false;
    const unsigned os0 = (unsigned)g.OS[0];
    sg.n = r / os0;
    sg.o_a = (int)(r - sg.n * os0);
    const unsigned left = r1 - r;
    sg.o_b = (unsigned)sg.o_a + left < os0 ? sg.o_a + (int)left : (int)os0;
    r += (unsigned)(sg.o_b - sg.o_a);
    const int top = sg.o_b - 1 + g.lb[0] - smax + WIN - 1, reach = sg.o_b - 1 + g.lb[0] - smin;
    sg.lo = clampi(sg.o_a + g.lb[0] - smax, 0, g.S[0] - 1);
    sg.hi = clampi(top < reach ? top : reach, 0, g.S[0] - 1);
    if (sg.hi < sg.lo) sg.hi = sg.lo;
    return true;
}
TS_D void rows_window(const Geo& g, int WIN, const RowsSeg& sg, int o, int smin, int smax, int& wlo, int& whi) {
    const int a = o + g.lb[0] - smax, top = a + WIN - 1, reach = o + g.lb[0] - smin;
    wlo = clampi(a, sg.lo, sg.hi);
    whi = clampi(top < reach ? top : reach, sg.lo, sg.hi);
    if (whi < wlo) whi = wlo;
}

template <int I, int CB> struct SpanRows {
    static TS_D void load(const unsigned* a, unsigned (*val)[4]) {
#pragma unroll
        for (int v = 0; v < 4; ++v) asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(val[I][v]) : "r"(a[v]), "n"(I * CB));
        SpanRows<I + 1, CB>::load(a, val);
    }
};
template <int CB> struct SpanRows<8, CB> {
    static TS_D void load(const unsigned*, unsigned (*)[4]) {}
};

template <int PAD, int CB>
__global__ void __launch_bounds__((ROWS_MAX_W + 1) * 32, 1) k_gather_nhwc_rows(Geo g, RowsPlan pl, const uint8_t* __restrict__ x,
                                                                                  uint8_t* __restrict__ y, uint8_t fill,
                                                                                  const void* __restrict__ w, int qkind, long long wzp) {
    extern __shared__ __align__(128) unsigned char rsm[];
    using namespace ptx;
    uint64_t* full = (uint64_t*)(rsm + pl.off_bar);
    uint64_t* empty = full + pl.K;
    int* s0t = (int*)(rsm + pl.off_tab);        // axis-0 shift per channel
    const int cb = CB > 0 ? CB : (int)g.C;      // bytes of a pixel = channels (CB == 0: any multiple of 128, run-time pitch)
    int* s1t = s0t + cb;                        // axis-1 shift per channel
    int* red = s1t + cb;                        // [0] min, [1] max of the axis-0 shifts
    const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) rsm[pl.smem_bytes - 16u] = fill;       // the pad value, addressable like any ring byte
    for (int c = tid; c < cb; c += (int)blockDim.x) {
        int sx[2];
        load_qshifts<2>(w, qkind, wzp, (long long)c, g, sx);
        s0t[c] = sx[0];
        s1t[c] = sx[1];
    }
    __syncthreads();
    if (warp == 0) {
        int mn = s0t[lane], mx = mn;
        for (int c = lane + 32; c < cb; c += 32) { const int v = s0t[c]; mn = v < mn ? v : mn; mx = v > mx ? v : mx; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const int a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
            mn = a < mn ? a : mn; mx = b > mx ? b : mx;
        }
        if (lane == 0) { red[0] = mn; red[1] = mx; }
    }
    __syncthreads();
    const int smin = red[0], smax = red[1];
    // Shifts spread wider than the planned window: fewer consumer warps, wider windows (the rows in flight plus one free
    // slot must fit the ring) as long as that covers the whole reach; beyond that the taps outside the window are read
    // from global memory (slow: 2.3 ms for cfg5 with shifts in +-6 -- like the ring kernel, this kernel is built for the
    // shifts layers learn).
    int W = pl.W, WIN = pl.WIN;
    {
        const int PP = cb / 128;
        const int rows_fit = pl.K - 2 - (smax - smin);                   // rows in flight that leave the whole reach in the ring
        if (smax - smin + 1 > WIN && rows_fit * PP >= 3) {               // (below 3 warps the global-memory fall-back is the lesser evil)
            W = rows_fit * PP < W ? rows_fit * PP : W;
            WIN = pl.K - (W + PP - 1) / PP - 1;
        }
    }
    if (tid == 0) {
        for (int k = 0; k < pl.K; ++k) { mbar_init(&full[k], 1); mbar_init(&empty[k], (unsigned)W); }
        fence_barrier_init();
    }
    __syncthreads();
    const unsigned long long R = (unsigned long long)g.N * (unsigned long long)g.OS[0];
    const unsigned r_begin = (unsigned)(R * blockIdx.x / gridDim.x), r_end = (unsigned)(R * (blockIdx.x + 1) / gridDim.x);
    const int K = pl.K;
    const unsigned row_bytes = pl.row_bytes;

    if (warp == pl.W) {                        // ---- producer: one lane, one bulk copy per input row ----
        if (lane != 0) return;
        int slot = 0, round = 0;
        unsigned r = r_begin;
        RowsSeg sg;
        while (rows_segment(g, WIN, r, r_end, smin, smax, sg)) {
            const uint8_t* src = x + (long long)sg.n * g.xs[0] + (long long)sg.lo * g.xs[2];
            for (int row = sg.lo; row <= sg.hi; ++row, src += g.xs[2]) {
                if (round > 0) mbar_wait_relaxed(&empty[slot], (unsigned)((round - 1) & 1), 64);
                mbar_expect_tx(&full[slot], row_bytes);
                bulk_g2s(rsm + (size_t)slot * row_bytes, src, row_bytes, &full[slot]);
                if (++slot == K) { slot = 0; ++round; }
            }
        }
        return;
    }
    if (warp >= W) return;

    // ---- consumers ----
    const int P = cb / 128;                    // passes (tasks) per output row
    const unsigned base = shared_addr(rsm);
    const unsigned fill_addr = base + pl.smem_bytes - 16u;
    const int s1n = g.S[1], lb1 = g.lb[1], ow = g.OS[1];
    const unsigned long long xs3 = (unsigned long long)g.xs[3];
    int ready_slot = 0;                        // slot / phase of the next row this warp has not seen land yet
    unsigned ready_phase = 0;
    int ready_q = 0;                           // rows seen landed so far (q index of the next one)
    int rel_slot = 0, rel_q = 0;               // next row to release
    int qbase = 0;                             // q index of the current segment's first row
    unsigned r = r_begin;
    RowsSeg sg;
    while (rows_segment(g, WIN, r, r_end, smin, smax, sg)) {
        // a task is (output row, pass of 128 channels): consecutive warps share a row, so W warps hold W / P rows
        for (int t = warp; t < (sg.o_b - sg.o_a) * P; t += W) {
            const int o = sg.o_a + t / P, ps = t % P;
            int wlo, whi;
            rows_window(g, WIN, sg, o, smin, smax, wlo, whi);
            const int q_lo = qbase + (wlo - sg.lo), q_hi = qbase + (whi - sg.lo);
            // Rows below this window are never touched by this warp again: release them -- but only after having SEEN
            // each of them land.  (Releasing a row it has not observed yet would let the producer refill the slot, and
            // a refill that lands before the warp gets to that slot's barrier flips its parity twice: the wait for the
            // older phase would then block for ever.  Observe-then-release keeps every warp at most one phase behind
            // any barrier, and the warp never holds a row below the one it waits for, so the producer is never stuck.)
            if (rel_q < q_lo) {
                __syncwarp();
                while (rel_q < q_lo) {
                    if (ready_q <= rel_q) {
                        mbar_wait_parked(&full[ready_slot], ready_phase);
                        ++ready_q;
                        if (++ready_slot == K) { ready_slot = 0; ready_phase ^= 1u; }
                    }
                    if (lane == 0) mbar_arrive(&empty[rel_slot]);
                    ++rel_q;
                    if (++rel_slot == K) rel_slot = 0;
                }
            }
            while (ready_q <= q_hi) {
                mbar_wait_parked(&full[ready_slot], ready_phase);
                ++ready_q;
                if (++ready_slot == K) { ready_slot = 0; ready_phase ^= 1u; }
            }
            int slot_lo = rel_slot;            // == q_lo mod K (rel_q == q_lo here)
            uint8_t* yrow = y + (((long long)sg.n * g.OS[0] + o) * ow) * g.C;
            {
                const int cw = 128 * ps + 4 * lane;      // first of the thread's 4 channels in this pass
                const int4 a0 = *reinterpret_cast<const int4*>(s0t + cw), a1 = *reinterpret_cast<const int4*>(s1t + cw);
                const int s0v[4] = {a0.x, a0.y, a0.z, a0.w}, s1v[4] = {a1.x, a1.y, a1.z, a1.w};
                unsigned row_addr[4], pitch[4];
                int t0s[4];
                bool from_global = false, all_ring = true;
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int t0 = axis_index_c<PAD>(o + g.lb[0] - s0v[v], g.S[0]);
                    t0s[v] = t0;
                    const bool inw = t0 >= wlo && t0 <= whi;           // implies t0 >= 0
                    int sl = slot_lo + (t0 - wlo);
                    sl = sl >= K ? sl - K : sl;
                    row_addr[v] = inw ? base + (unsigned)sl * row_bytes + (unsigned)(cw + v) : fill_addr;
                    pitch[v] = inw ? (unsigned)cb : 0u;
                    from_global = from_global || (t0 >= 0 && !inw);
                    all_ring = all_ring && inw;
                }
                int s1_max = s1v[0], s1_min = s1v[0];
#pragma unroll
                for (int v = 1; v < 4; ++v) { s1_max = s1v[v] > s1_max ? s1v[v] : s1_max; s1_min = s1v[v] < s1_min ? s1v[v] : s1_min; }
                const int p_lo = s1_max - lb1 > 0 ? s1_max - lb1 : 0;
                const int p_hi = s1n - 1 - lb1 + s1_min < ow - 1 ? s1n - 1 - lb1 + s1_min : ow - 1;
                uint8_t* yp = yrow + cw;
                int p = 0;
                if (!from_global) {
                    for (; p < p_lo && p < ow; ++p, yp += cb) {            // leading pixels: some tap is left of the row
                        unsigned val[4];
#pragma unroll
                        for (int v = 0; v < 4; ++v) {
                            const int t1 = axis_index_c<PAD>(p + lb1 - s1v[v], s1n);
                            val[v] = ring_byte(nullptr, t1 >= 0 ? row_addr[v] + (unsigned)t1 * pitch[v] : fill_addr);
                        }
                        store4(yp, val);
                    }
                    unsigned addr[4];
#pragma unroll
                    for (int v = 0; v < 4; ++v) addr[v] = row_addr[v] + (unsigned)(p + lb1 - s1v[v]) * pitch[v];
                    if (all_ring) {
                        for (; p + 7 <= p_hi; p += 8) {
                            unsigned val[8][4];
                            if constexpr (CB > 0) {
                                SpanRows<0, CB>::load(addr, val);
                            } else {
#pragma unroll
                                for (int i = 0; i < 8; ++i)
#pragma unroll
                                    for (int v = 0; v < 4; ++v) val[i][v] = ring_byte(nullptr, addr[v] + (unsigned)(i * cb));
                            }
#pragma unroll
                            for (int i = 0; i < 8; ++i, yp += cb) store4(yp, val[i]);
#pragma unroll
                            for (int v = 0; v < 4; ++v) addr[v] += 8u * (unsigned)cb;
                        }
                    }
                    for (; p <= p_hi; ++p, yp += cb) {
                        unsigned val[4];
#pragma unroll
                        for (int v = 0; v < 4; ++v) { val[v] = ring_byte(nullptr, addr[v]); addr[v] += pitch[v]; }
                        store4(yp, val);
                    }
                    for (; p < ow; ++p, yp += cb) {                        // trailing pixels
                        unsigned val[4];
#pragma unroll
                        for (int v = 0; v < 4; ++v) {
                            const int t1 = axis_index_c<PAD>(p + lb1 - s1v[v], s1n);
                            val[v] = ring_byte(nullptr, t1 >= 0 ? row_addr[v] + (unsigned)t1 * pitch[v] : fill_addr);
                        }
                        store4(yp, val);
                    }
                } else {
                    for (; p < ow; ++p, yp += cb) {
                        unsigned val[4];
#pragma unroll
                        for (int v = 0; v < 4; ++v) {
                            const int t1 = axis_index_c<PAD>(p + lb1 - s1v[v], s1n);
                            if (t0s[v] >= 0 && pitch[v] == 0u) {     // valid row, not in this row's window
                                const uint8_t* src = x + (long long)sg.n * g.xs[0] + (long long)t0s[v] * g.xs[2] + (cw + v);
                                val[v] = t1 >= 0 ? (unsigned)load_ro(src + (unsigned long long)(unsigned)t1 * xs3) : (unsigned)fill;
                            } else {
                                val[v] = ring_byte(nullptr, t1 >= 0 ? row_addr[v] + (unsigned)t1 * pitch[v] : fill_addr);
                            }
                        }
                        store4(yp, val);
                    }
                }
            }
        }
        qbase += sg.hi - sg.lo + 1;
    }
    // rows this warp never needed (or no longer needs): see each of them land, then release it
    __syncwarp();
    while (rel_q < qbase) {
        if (ready_q <= rel_q) {
            mbar_wait_parked(&full[ready_slot], ready_phase);
            ++ready_q;
            if (++ready_slot == K) { ready_slot = 0; ready_phase ^= 1u; }
        }
        if (lane == 0) mbar_arrive(&empty[rel_slot]);
        ++rel_q;
        if (++rel_slot == K) rel_slot = 0;
    }
}

bool plan_rows(const Geo& g, int esize, const void* x, const void* y, int sm_count, int max_grid_x, int ring_rows, RowsPlan* out) {
    if (!tma_available()) return false;
    if (g.dim != 2 || esize != 1 || g.xs[1] != 1) return false;
    if (g.C % 128 != 0 || g.C > 2048) return false;
    if (g.xs[3] != g.C || g.xs[2] != g.C * (long long)g.S[1] || (g.xs[0] & 15) || g.xs[0] < 0) return false;   // dense rows
    if (((uintptr_t)x & 15u) || ((uintptr_t)y & 3u)) return false;
    const long long row_bytes = (long long)g.S[1] * g.C;
    if (row_bytes % 16 || row_bytes >= (1 << 20)) return false;
    if (g.N * (long long)g.OS[0] >= 0x7fffffffLL || g.N * (long long)g.S[0] >= 0x7fffffffLL) return false;
    RowsPlan pl;
    const long long tab = 2 * g.C * 4 + 16, avail = 227LL * 1024 - 1024 - tab - 16;
    long long K = avail / (row_bytes + 16);
    if (ring_rows > 0 && K > ring_rows) K = ring_rows;
    if (K > 64) K = 64;
    if (K < 7) return false;
    // consumer warps: a task is (output row, pass of 128 channels), so W warps hold W / P rows; the windows of the rows in
    // flight plus the prefetched rows must fit the ring, and a window should hold the reach of the shifts layers learn
    // (|shift| <= 3: 7 rows) -- wider ones fall back to global loads.  Measured on cfg5 (K = 15): more warps win until the
    // ring has fewer than ~3 free slots for the producer.
    const int P = (int)(g.C / 128);
    int W = K >= 20 ? 8 * P : (K >= 14 ? 6 * P : ((int)K - 5) * P);
    if (tuning().nhwc_rows_warps > 0) W = tuning().nhwc_rows_warps;
    if (W > ROWS_MAX_W) W = ROWS_MAX_W;
    if ((W + P - 1) / P > (int)K - 3) W = ((int)K - 3) * P;
    if (W < 2) W = 2;
    pl.K = (int)K;
    pl.W = W;
    pl.WIN = (int)K - (W + P - 1) / P - 1;
    if (pl.WIN < 2) return false;
    pl.row_bytes = (unsigned)row_bytes;
    pl.off_bar = (unsigned)(K * row_bytes);
    pl.off_tab = pl.off_bar + (unsigned)(2 * K * 8);
    pl.smem_bytes = pl.off_tab + (unsigned)tab + 16u;
    long long grid = sm_count;
    const long long rows = g.N * (long long)g.OS[0];
    if (grid > rows) grid = rows;
    if (max_grid_x > 0 && grid > max_grid_x) grid = max_grid_x;
    pl.grid = (unsigned)grid;
    *out = pl;
    return true;
}

template <int PAD, int CB>
int rows_launch(const Geo& g, const RowsPlan& pl, const void* x, void* y, uint8_t fill, const void* w, int qkind, long long wzp,
                cudaStream_t s) {
    return launch_persistent(k_gather_nhwc_rows<PAD, CB>, pl.grid, (pl.W + 1) * 32, pl.smem_bytes, s, false, g, pl, (const uint8_t*)x,
                             (uint8_t*)y, fill, w, qkind, wzp);
}
template <int PAD>
int rows_run_c(const Geo& g, const RowsPlan& pl, const void* x, void* y, uint8_t fill, const void* w, int qkind, long long wzp, cudaStream_t s) {
    switch ((int)g.C) {
    case 128: return rows_launch<PAD, 128>(g, pl, x, y, fill, w, qkind, wzp, s);
    case 256: return rows_launch<PAD, 256>(g, pl, x, y, fill, w, qkind, wzp, s);
    case 512: return rows_launch<PAD, 512>(g, pl, x, y, fill, w, qkind, wzp, s);
    default: return rows_launch<PAD, 0>(g, pl, x, y, fill, w, qkind, wzp, s);        // any other multiple of 128: run-time pixel pitch
    }
}
int rows_run(const Geo& g, const RowsPlan& pl, const void* x, void* y, uint8_t fill, const void* w, int qkind, long long wzp, cudaStream_t s) {
    switch (g.pad) {
    case TS_PAD_BORDER: return rows_run_c<TS_PAD_BORDER>(g, pl, x, y, fill, w, qkind, wzp, s);
    case TS_PAD_PERIODIC: return rows_run_c<TS_PAD_PERIODIC>(g, pl, x, y, fill, w, qkind, wzp, s);
    case TS_PAD_REFLECT: return rows_run_c<TS_PAD_REFLECT>(g, pl, x, y, fill, w, qkind, wzp, s);
    case TS_PAD_SYMMETRIC: return rows_run_c<TS_PAD_SYMMETRIC>(g, pl, x, y, fill, w, qkind, wzp, s);
    default: return rows_run_c<TS_PAD_ZEROS>(g, pl, x, y, fill, w, qkind, wzp, s);
    }
}

template <typename E, int DIM, int VEC, int PAD>
void run_dim(const Geo& g, const NhwcPlan& pl, const void* x, void* y, E fill, const void* w, int qkind, long long wzp, cudaStream_t s,
             bool emulate) {
    const int threads = pl.tc * pl.tp;
    if (emulate) {      // host mirror: the same per-thread program, every (block, thread) in turn
        for (unsigned by = 0; by < (unsigned)pl.segs; ++by)
            for (unsigned bx = 0; bx < pl.grid_x; ++bx)
                for (int tid = 0; tid < threads; ++tid)
                    nhwc_thread<E, DIM, VEC, PAD>(g, pl, tid, bx, by, pl.grid_x, (const E*)x, (E*)y, fill, w, qkind, wzp);
        return;
    }
    const dim3 grid(pl.grid_x, (unsigned)pl.segs, 1);
    k_gather_nhwc<E, DIM, VEC, PAD><<<grid, threads, 0, s>>>(g, pl, (const E*)x, (E*)y, fill, w, qkind, wzp);
}

template <typename E, int VEC, int PAD>
void run_pad(const Geo& g, const NhwcPlan& pl, const void* x, void* y, E fill, const void* w, int qkind, long long wzp, cudaStream_t s,
             bool emulate) {
    switch (g.dim) {
    case 1: run_dim<E, 1, VEC, PAD>(g, pl, x, y, fill, w, qkind, wzp, s, emulate); break;
    case 2: run_dim<E, 2, VEC, PAD>(g, pl, x, y, fill, w, qkind, wzp, s, emulate); break;
    default: run_dim<E, 3, VEC, PAD>(g, pl, x, y, fill, w, qkind, wzp, s, emulate); break;
    }
}

template <typename E, int VEC>
int run_type(const Geo& g, const NhwcPlan& pl, const void* x, void* y, E fill, const void* w, int qkind, long long wzp, cudaStream_t s,
             bool emulate) {
    switch (g.pad) {
    case TS_PAD_BORDER: run_pad<E, VEC, TS_PAD_BORDER>(g, pl, x, y, fill, w, qkind, wzp, s, emulate); break;
    case TS_PAD_PERIODIC: run_pad<E, VEC, TS_PAD_PERIODIC>(g, pl, x, y, fill, w, qkind, wzp, s, emulate); break;
    case TS_PAD_REFLECT: run_pad<E, VEC, TS_PAD_REFLECT>(g, pl, x, y, fill, w, qkind, wzp, s, emulate); break;
    case TS_PAD_SYMMETRIC: run_pad<E, VEC, TS_PAD_SYMMETRIC>(g, pl, x, y, fill, w, qkind, wzp, s, emulate); break;
    default: run_pad<E, VEC, TS_PAD_ZEROS>(g, pl, x, y, fill, w, qkind, wzp, s, emulate); break;
    }
    if (emulate) return TS_OK;
    note_launch();
    return check_launch();
}

// ------------------------------------------------------------------------------------------
// Layout adapter for the float path: dense channels-last -> dense planar (per image a [P, C] -> [C, P]
// transpose through a padded shared-memory tile; both sides move whole 128-byte lines).  The reference
// returns planar tensors for channels-last float inputs (cpu/shifts_cpu.cpp:221), so the planar bandwidth
// kernels serve them after this one pass; torch's own .contiguous() does the same job at 1.9 TB/s.
// 64 x 64 tiles, 16 independent 4-byte loads in flight per thread (a 32 x 32 tile leaves too few bytes in
// flight per SM: 2.9 TB/s measured); row pitch 65 keeps both the row-wise fill and the column-wise drain
// of the tile conflict-free.
constexpr int TT = 64;
template <typename E>
__global__ void __launch_bounds__(256) k_nhwc_to_nchw(const E* __restrict__ x, E* __restrict__ y, int C, int P, unsigned ptiles) {
    __shared__ E tile[TT][TT + 1];
    const unsigned n = blockIdx.x / ptiles;
    const int p0 = (int)(blockIdx.x - n * ptiles) * TT;
    const int c0 = (int)blockIdx.y * TT;
    const E* xi = x + (long long)n * P * C;
    E* yo = y + (long long)n * P * C;
    const int tx = threadIdx.x, ty = threadIdx.y;
    E v[TT / 8][TT / 32];            // all 16 loads are issued before the first shared-memory store
#pragma unroll
    for (int i = 0; i < TT / 8; ++i) {
        const int p = p0 + ty + 8 * i;
#pragma unroll
        for (int h = 0; h < TT / 32; ++h) {
            const int c = c0 + tx + 32 * h;
            v[i][h] = (p < P && c < C) ? xi[(long long)p * C + c] : (E)0;
        }
    }
#pragma unroll
    for (int i = 0; i < TT / 8; ++i)
#pragma unroll
        for (int h = 0; h < TT / 32; ++h) tile[ty + 8 * i][tx + 32 * h] = v[i][h];
    __syncthreads();
#pragma unroll
    for (int j = ty; j < TT; j += 8) {
        const int c = c0 + j;
#pragma unroll
        for (int h = 0; h < TT; h += 32) {
            const int p = p0 + tx + h;
            if (c < C && p < P) yo[(long long)c * P + p] = tile[tx + h][j];
        }
    }
}

template <typename E>
int to_planar_t(const void* x, void* y, long long N, long long C, long long P, cudaStream_t s) {
    const long long ptiles = (P + TT - 1) / TT, ctiles = (C + TT - 1) / TT;
    if (N * ptiles >= 0x7fffffffLL || ctiles > 65535) return TS_ERR_TOO_LARGE;
    const dim3 grid((unsigned)(N * ptiles), (unsigned)ctiles, 1), block(32, 8, 1);
    k_nhwc_to_nchw<E><<<grid, block, 0, s>>>((const E*)x, (E*)y, (int)C, (int)P, (unsigned)ptiles);
    note_launch();
    return check_launch();
}

}  // namespace

int nhwc_to_planar(const void* x, void* y, long long N, long long C, long long P, int esize, cudaStream_t s) {
    if (N == 0 || C == 0 || P == 0) return TS_OK;
    if (C >= 0x7fffffffLL || P >= 0x7fffffffLL) return TS_ERR_TOO_LARGE;
    switch (esize) {
    case 2: return to_planar_t<uint16_t>(x, y, N, C, P, s);
    case 4: return to_planar_t<uint32_t>(x, y, N, C, P, s);
    case 8: return to_planar_t<unsigned long long>(x, y, N, C, P, s);
    }
    return TS_ERR_UNSUPPORTED;
}

// x: any strides (g.xs), meant for channel stride 1; y: dense [N, OS0(,OS1(,OS2)), C].
// emulate: x / y / w are HOST pointers and the launch is walked on the host (tests only, no GPU work).
// variant: 0 automatic (row-pipelined kernel, else ring kernel, else direct), 1 direct only, 2 ring only, 3 row-pipelined only;
// ring_rows > 0 caps the ring.
int nhwc_gather(const Geo& g, const void* x, void* y, unsigned long long fill, int esize, const void* w, int qkind,
                long long wzp, int sm_count, int max_grid_x, int variant, int ring_rows, bool emulate, cudaStream_t s) {
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    if (!emulate && (variant == 0 || variant == 3)) {      // row-pipelined kernel (no host emulation: GPU tests only)
        RowsPlan wp;
        if (plan_rows(g, esize, x, y, sm_count, max_grid_x, ring_rows, &wp))
            return rows_run(g, wp, x, y, (uint8_t)fill, w, qkind, wzp, s);
        if (variant == 3) return TS_ERR_UNSUPPORTED;
    }
    if (variant != 1) {
        RingPlan rp;
        if (plan_ring(g, esize, x, y, sm_count, max_grid_x, ring_rows, &rp))
            return ring_run(g, rp, x, y, (uint8_t)fill, w, qkind, wzp, s, emulate);
        if (variant == 2) return TS_ERR_UNSUPPORTED;
    }
    long long rows = g.N;
    for (int a = 0; a < g.dim - 1; ++a) rows *= g.OS[a];
    if (rows >= 0x7fffffffLL || g.C >= 0x7fffffffLL) return TS_ERR_TOO_LARGE;
    const long long xsl = g.xs[2 + g.dim - 1];
    if (xsl < 0 || xsl * (long long)esize * g.S[g.dim - 1] >= 0x7fffffffLL) return TS_ERR_UNSUPPORTED;   // 32-bit row offsets
    const NhwcPlan pl = make_plan(g, esize, y, sm_count, max_grid_x);
    if (esize == 1) {
        if (pl.vec == 4) return run_type<uint8_t, 4>(g, pl, x, y, (uint8_t)fill, w, qkind, wzp, s, emulate);
        return run_type<uint8_t, 1>(g, pl, x, y, (uint8_t)fill, w, qkind, wzp, s, emulate);
    }
    if (esize == 4) return run_type<uint32_t, 1>(g, pl, x, y, (uint32_t)fill, w, qkind, wzp, s, emulate);
    return TS_ERR_UNSUPPORTED;
}

}  // namespace ts

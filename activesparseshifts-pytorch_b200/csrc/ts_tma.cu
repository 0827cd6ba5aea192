// ts_tma.cu -- the zero-padding fast path, built on TMA *tensor* copies (cp.async.bulk.tensor.5d,
// SASS UTMALDG).
//
// Idea.  A tiled TMA load whose box starts at the (possibly negative) coordinates
//     (col0 - s_col rounded down to 16 bytes, row0 - s_row, slab0 - s_slab, c, n0)
// delivers a tile of the plane(s) already SHIFTED along every axis, with every element that lies
// outside the tensor filled with zero by the copy engine.  That is the reference's zero-padded
// gather (ops/kernels/shifts_kernels.h:10-54 with BIPadding::Zeros) done by hardware, so the
// consumers have no index remapping, no validity masks and no edge cases at all: every item reads
// aligned 16-byte groups from shared memory and only resolves the residual sub-16-byte column
// misalignment (0..3 fp32 or 0..7 16-bit elements; the copy engine requires the innermost coordinate to be a
// multiple of 16 bytes -- measured: an unaligned inner coordinate raises "illegal instruction").
// The box carries one extra 16-byte group per row (and one extra row / slab for the arithmetic
// kernels) for the residual window and the +1 interpolation neighbours.
//
//   mode 0  sparse / quantized forward (pad value 0): y item = funnel-shifted pair of groups
//   mode 1  active forward:  x box (TA+1, TB+1, TG+1 groups) -> exact unfused lerp nest
//   mode 2  backward (no border crop): x box as mode 1, grad box unshifted (gv), and grad box
//           shifted by +s (sparse: grad_input is a gather) or by -s with +1 neighbours (active)
//
// CTA = `nw` consumer warps + 1 producer warp (one elected lane issues the TMA loads), persistent,
// one CTA per SM, ring of `stages` stages with full/empty mbarriers; grad_weight partials are
// per-(unit, warp) in fp64, fixed shuffle tree, second pass in ts_generic.cu -> deterministic.
//
// Applicability (plan_tma): zeros padding, dense NCHW x, row bytes a multiple of 16, pad value 0,
// no border crop for the backward; the arithmetic modes take fp32, and 2-D fp16 / bf16 tensors whose weights are
// fp32 (TS_WEIGHTS_F32: an item is then 8 elements, fp32 arithmetic, one rounding at the store).  Everything else runs
// on the other families.
#include <cuda.h>

#include <cstdio>
#include <type_traits>

#include "ts_kernels.h"
#include "ts_ptx.cuh"

namespace ts {

namespace {

using namespace ptx;

constexpr int MAXT_TMA_GATHER = 1024, MAXT_TMA_ARITH = 512;

// ---- driver entry point (no libcuda link dependency) ------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) p = nullptr;
        (void)cudaGetLastError();
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// rank-5 map over a dense [N][C][A][B][L] tensor of `es`-byte elements, box {bl, bb, ba, 1, bn}.
// Encoded maps are memoised per thread (a training loop presents the same few (pointer, geometry) pairs every
// step; the descriptor is a pure function of these arguments).
struct MapKey {
    const void* base;
    long long N, C;
    int es, dtype, A, B, L, bl, bb, ba, bn;
};
struct MapSlot { MapKey key; CUtensorMap map; bool used; };
constexpr int MAP_CACHE = 32;

// dtype: TS_F16 / TS_BF16 name the 16-bit element type of the arithmetic kernels' maps; anything else copies raw words.
bool make_map(CUtensorMap* map, const void* base, int es, long long N, long long C, int A, int B, int L, int bl, int bb, int ba,
              int bn, int dtype = -1) {
    static thread_local MapSlot cache[MAP_CACHE];
    static thread_local int next_victim = 0;
    MapKey key;
    memset(&key, 0, sizeof(key));
    key.base = base; key.N = N; key.C = C; key.es = es; key.dtype = dtype; key.A = A; key.B = B; key.L = L; key.bl = bl; key.bb = bb; key.ba = ba; key.bn = bn;
    for (int i = 0; i < MAP_CACHE; ++i)
        if (cache[i].used && !memcmp(&cache[i].key, &key, sizeof(key))) { *map = cache[i].map; return true; }
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    // cuTensorMapEncodeTiled is a DRIVER call: it needs the primary context current on the calling
    // thread.  A thread that has only used cached allocations so far (PyTorch's autograd worker on
    // its first backward) has none yet (CUDA_ERROR_INVALID_CONTEXT); cudaFree(0) binds it.
    static thread_local bool ctx_bound = false;
    if (!ctx_bound) { (void)cudaFree(nullptr); ctx_bound = true; }
    const CUtensorMapDataType dt = es == 2 && dtype == TS_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                 : es == 2 && dtype == TS_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                 : es == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : es == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16
                                 : es == 4 ? CU_TENSOR_MAP_DATA_TYPE_UINT32 : CU_TENSOR_MAP_DATA_TYPE_UINT64;
    cuuint64_t dims[5] = {(cuuint64_t)L, (cuuint64_t)B, (cuuint64_t)A, (cuuint64_t)C, (cuuint64_t)N};
    const cuuint64_t row = (cuuint64_t)L * es;
    cuuint64_t strides[4] = {row, row * B, row * B * A, row * B * A * (cuuint64_t)C};
    cuuint32_t box[5] = {(cuuint32_t)bl, (cuuint32_t)bb, (cuuint32_t)ba, 1u, (cuuint32_t)bn};
    cuuint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
    const CUresult r = enc(map, dt, 5, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        char msg[240];
        snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled -> %d: es %d dims {%d,%d,%d,%lld,%lld} box {%d,%d,%d,1,%d} base %p", (int)r, es, L, B,
                 A, C, N, bl, bb, ba, bn, base);
        note_error(msg);
        return false;
    }
    MapSlot& slot = cache[next_victim];
    next_victim = (next_victim + 1) % MAP_CACHE;
    slot.key = key; slot.map = *map; slot.used = true;
    return true;
}

TS_D int floor_to(int v, int q) { return v & ~(q - 1); }      // q is a power of two (elements per 16 bytes)

struct UnitShift {
    int sh[3];     // integer shift per level (0 slab, 1 row, 2 column); absent levels 0
    float d[3];    // fractional part per TENSOR AXIS (reference order), 0 for the sparse forward
};

TS_D UnitShift compute_unit_shift(const TArgs& a, long long c) {
    UnitShift u;
    const int dim = a.g.dim;
    u.d[0] = u.d[1] = u.d[2] = 0.f;
#pragma unroll
    for (int lev = 0; lev < 3; ++lev) {
        const int ax = level_axis(lev, dim);
        long long iw = 0;
        if (ax >= 0) {
            const long long idx = c * dim + ax;
            if (a.mode == 0) {
                iw = sparse_shift(a.w, a.wk, a.qkind, a.wzp, idx);
            } else {             // fp32 weights: fp32 layers, and 16-bit layers under TS_WEIGHTS_F32 (the only ones planned)
                float d;
                if (a.mode == 1) split_forward<float>(((const float*)a.w)[idx], true, iw, d);
                else split_backward<float>(((const float*)a.w)[idx], a.active != 0, iw, d);
                u.d[ax] = d;
            }
            u.sh[lev] = reduce_shift(iw, a.g.S[ax], TS_PAD_ZEROS);
        } else {
            u.sh[lev] = 0;
        }
    }
    return u;
}

// The per-channel parameters cost a few hundred dependent instructions (64-bit conversions, saturation, the reduced
// shift): computed per work unit by the single producer thread they bounded small batches (one stage per unit).
// Every CTA tabulates them once in shared memory instead; a unit then costs one 24-byte read.
TS_D UnitShift unit_shift(const TArgs& a, const UnitShift* tbl, long long c) { return a.table ? tbl[c] : compute_unit_shift(a, c); }

// u -> (channel, chunk) without an integer division
TS_D void decode_unit(const TArgs& a, int u, int& c, int& chunk) {
    if (a.unit_order) { chunk = (int)fdiv((unsigned)u, a.d_C); c = u - chunk * (int)a.g.C; }
    else { c = (int)fdiv((unsigned)u, a.d_chunks); chunk = u - c * a.chunks; }
}

struct Tile { int a0, b0, g0; };
TS_D Tile tile_of(const TArgs& a, int t) {
    Tile tl;
    const int tg = (int)fdiv((unsigned)t, a.d_tg);          // t / tiles_g
    tl.g0 = (t - tg * a.tiles_g) * a.TG;
    const int ta = (int)fdiv((unsigned)tg, a.d_tb);         // (t / tiles_g) / tiles_b
    tl.b0 = (tg - ta * a.tiles_b) * a.TB;
    tl.a0 = ta * a.TA;
    return tl;
}

// ---- producer ---------------------------------------------------------------------------------
TS_D void producer(const TArgs& a, unsigned char* smem, uint64_t* full, uint64_t* empty, const UnitShift* tbl) {
    int s = 0, k = 0;
    const long long N = a.g.N;
    const int dim = a.g.dim;
    const UnitRange ur = unit_range(a.units, a.unit_order);
    for (int u = ur.u; u < ur.end; u += ur.step) {
        int ci, chunki;
        decode_unit(a, u, ci, chunki);
        const long long c = ci, chunk = chunki;
        const long long n0 = chunk * a.n_per_unit;
        const long long n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
        const UnitShift us = unit_shift(a, tbl, c);
        for (long long nb = n0; nb < n1; nb += a.np) {
            for (int t = 0; t < a.tiles; ++t) {
                if (k > 0) mbar_wait(&empty[s], (unsigned)((k - 1) & 1));
                const Tile tl = tile_of(a, t);
                unsigned char* st = smem + (size_t)s * a.stage_stride;
                mbar_expect_tx(&full[s], (unsigned)a.tx_bytes);
                const int l0 = tl.g0 * a.vec;
                // x box: source coordinates of the tile's first output element, column rounded down to a group
                const int xc = floor_to(l0 + a.lbL - us.sh[2], a.vec);
                const int xr = dim >= 2 ? tl.b0 + a.lbB - us.sh[1] : 0;
                const int xs = dim == 3 ? tl.a0 + a.lbA - us.sh[0] : 0;
                tma_load_5d(st, &a.map_x, xc, xr, xs, (int)c, (int)nb, &full[s]);
                if (a.mode == 2) {
                    tma_load_5d(st + a.off_gv, &a.map_gs, l0, dim >= 2 ? tl.b0 : 0, dim == 3 ? tl.a0 : 0, (int)c, (int)nb, &full[s]);
                    if (a.active) {      // grad at (o - s) with +1 neighbours: same geometry as the x box
                        tma_load_5d(st + a.off_g2, &a.map_gb, xc, xr, xs, (int)c, (int)nb, &full[s]);
                    } else {             // grad_input of the sparse shift gathers grad at (o + s)
                        tma_load_5d(st + a.off_g2, &a.map_gs, floor_to(l0 + us.sh[2], a.vec), dim >= 2 ? tl.b0 + us.sh[1] : 0,
                                    dim == 3 ? tl.a0 + us.sh[0] : 0, (int)c, (int)nb, &full[s]);
                    }
                }
                if (++s == a.stages) { s = 0; ++k; }
            }
        }
    }
}

// ---- consumer skeleton -----------------------------------------------------------------------
// Everything a body needs about the current stage; all values are CTA-uniform.
struct Stage {
    const unsigned char* st;   // stage base in shared memory
    unsigned char* dst;        // output address of (first image of the stage, channel c, tile origin)
    int npl;                   // images in this stage
    int total;                 // items of this stage in the padded index space: images * img_items
    int an, bn, gn;            // valid extents of this tile (slabs, rows, groups)
};

template <class Body>
TS_D void consumer_loop(const TArgs& a, unsigned char* smem, uint64_t* full, uint64_t* empty, int lane, Body& body) {
    int s = 0;
    unsigned phase = 0;
    const int C = (int)a.g.C, N = (int)a.g.N, np = a.np, tiles = a.tiles, stages = a.stages;
    const long long plane_bytes = (a.mode == 2 ? a.g.in_plane : a.g.out_plane) * a.es;
    const UnitRange ur = unit_range(a.units, a.unit_order);
    for (int u = ur.u; u < ur.end; u += ur.step) {
        int chunk, c;
        decode_unit(a, u, c, chunk);
        const int n0 = chunk * a.n_per_unit;
        const int n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
        body.begin_unit(c);
        for (int nb = n0; nb < n1; nb += np) {
            Stage sg;
            sg.npl = n1 - nb < np ? n1 - nb : np;
            sg.total = sg.npl * a.img_items;
            unsigned char* img = a.out + ((long long)nb * C + c) * plane_bytes;
            for (int t = 0; t < tiles; ++t) {
                sg.an = a.TA; sg.bn = a.TB; sg.gn = a.TG;
                sg.dst = img;
                if (tiles > 1) {
                    const Tile tl = tile_of(a, t);
                    sg.an = a.OA - tl.a0 < a.TA ? a.OA - tl.a0 : a.TA;
                    sg.bn = a.OB - tl.b0 < a.TB ? a.OB - tl.b0 : a.TB;
                    sg.gn = a.OGR - tl.g0 < a.TG ? a.OGR - tl.g0 : a.TG;
                    sg.dst = img + ((long long)(tl.a0 * a.OB + tl.b0) * a.OGR + tl.g0) * 16;
                }
                sg.st = smem + (size_t)s * a.stage_stride;
                mbar_wait(&full[s], phase);
                body.step(sg);
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
                if (++s == stages) { s = 0; phase ^= 1u; }
            }
        }
        body.end_unit(c, chunk);
    }
}

// item (padded index space: [image][slab][row][GP groups]) -> position inside the tile.  The
// padded row length GP is a multiple of 8 when that wastes <= 15 % of the lanes: a quarter-warp
// then never straddles two box rows, which keeps the 128-bit shared-memory loads conflict-free.
struct Item { int pl, a, b, cg; };
template <bool SLABS>
TS_D bool decode_item(const TArgs& a, const Stage& sg, int item, Item& p) {
    p.pl = 0;
    int rem = item;
    if (a.np > 1) { p.pl = (int)fdiv((unsigned)item, a.d_img); rem = item - p.pl * a.img_items; }
    const int row = (int)fdiv((unsigned)rem, a.d_GP);
    p.cg = rem - row * a.GP;
    p.a = 0;
    p.b = row;
    if (SLABS) { p.a = (int)fdiv((unsigned)row, a.d_TB); p.b = row - p.a * a.TB; }
    return p.cg < sg.gn && p.b < sg.bn && p.a < sg.an;
}
// 16-byte offset of the item's output inside the stage's destination
TS_D unsigned char* item_dst(const TArgs& a, const Stage& sg, const Item& p) {
    const int off16 = p.pl * a.img_stride16 + (p.a * a.OB + p.b) * a.OGR + p.cg;
    return sg.dst + (size_t)(unsigned)off16 * 16;
}

// ================================================================================================
// mode 0: sparse / quantized forward.  WS = word misalignment of the source window (0..3); SUB =
// elements narrower than 4 bytes, whose residual byte shift is a run-time funnel-shift amount.
template <bool SLABS>
struct GatherBody {
    const TArgs& a;
    const int tid, nt;
    int ws, bs8;

    const UnitShift* tbl;
    TS_D GatherBody(const TArgs& a_, int tid_, int nt_, const UnitShift* tbl_) : a(a_), tid(tid_), nt(nt_), ws(0), bs8(0), tbl(tbl_) {}
    TS_D void begin_unit(int c) {
        const UnitShift us = unit_shift(a, tbl, c);
        const int mb = pmod((a.lbL - us.sh[2]) * a.es, 16);    // tiles start at multiples of 16 bytes
        ws = mb >> 2;
        bs8 = (mb & 3) * 8;
    }
    TS_D void end_unit(int, int) {}

    template <int WS, bool SUB>
    TS_D void run(const Stage& sg) const {
        const unsigned box = shared_addr(sg.st);
        const int pitch = a.TG + 1, ximg = a.x_img_chunks, xb = a.xb;
        for (int item = tid; item < sg.total; item += nt) {
            Item p;
            if (!decode_item<SLABS>(a, sg, item, p)) continue;
            const int ch = p.pl * ximg + (p.a * xb + p.b) * pitch + p.cg;
            const uint4 A = lds128(box + ch * 16);
            unsigned W[8] = {A.x, A.y, A.z, A.w, 0u, 0u, 0u, 0u};
            if (WS > 0 || SUB) { const uint4 B = lds128(box + ch * 16 + 16); W[4] = B.x; W[5] = B.y; W[6] = B.z; W[7] = B.w; }
            unsigned o[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) o[k] = SUB ? __funnelshift_r(W[k + WS], W[(k + WS + 1) & 7], bs8) : W[k + WS];
            __stcs((uint4*)item_dst(a, sg, p), make_uint4(o[0], o[1], o[2], o[3]));
        }
    }
    TS_D void step(const Stage& sg) const {
        if (bs8 == 0) {
            switch (ws) {
            case 0: run<0, false>(sg); break;
            case 1: run<1, false>(sg); break;
            case 2: run<2, false>(sg); break;
            default: run<3, false>(sg); break;
            }
        } else {
            switch (ws) {
            case 0: run<0, true>(sg); break;
            case 1: run<1, true>(sg); break;
            case 2: run<2, true>(sg); break;
            default: run<3, true>(sg); break;
            }
        }
    }
};

// ================================================================================================
// Arithmetic bodies, fp32 arithmetic on ST elements (fp32, or fp16 / bf16 rounded once at the store).  An item is one
// 16-byte group: V = 4 or 8 elements.  A window of NV consecutive elements starting M elements into the aligned group
// `ch` of a staged box (compile-time word select, plus a half-word shift for 16-bit elements).
template <typename ST, int M, int NV>
TS_D void load_win(unsigned box, int ch, float* out) {
    load_window_c<ST, M * (int)sizeof(ST), NV>(box + ch * 16, out);
}

// group offset of the +1 neighbour rows inside a box with `rows` rows per slab, `pitch` groups per row
template <int DIM>
TS_D int neighbour_row_offset(int rv, int rows, int pitch) {
    if (DIM == 1) return 0;
    if (DIM == 2) return (rv & 1) * pitch;
    return ((rv & 1) * rows + ((rv >> 1) & 1)) * pitch;
}

template <int DIM, int NVW>
TS_D void neighbours_from_rows(const float (*X)[NVW], int t, float* v) {
    constexpr int NR = 1 << (DIM - 1);
#pragma unroll
    for (int q = 0; q < (1 << DIM); ++q) v[q] = X[q & (NR - 1)][t + (q >> (DIM - 1))];
}

// The reference's per-element weight-gradient factors (ts_common.cuh weight_partials) written with
// ordinary, contractable arithmetic: grad_weight is tolerance-checked (rtol 1e-5 vs an fp64 CPU
// evaluation of the reference formulas), only forward / grad_input have to be bit-exact.
template <int DIM>
TS_D void weight_partials_fast(const float* v, const float* d, float* g) {
    if (DIM == 1) { g[0] = v[1] - v[0]; return; }
    if (DIM == 2) {
        const float p = v[2] - v[0], q = (v[3] - v[1]) - p;   // both factors are p + frac * q (see DESIGN.md)
        g[0] = fmaf(d[1], q, p);
        g[1] = fmaf(d[0], q, p);
        return;
    }
    const float p0 = v[2] - v[0], q0 = (v[3] - v[1]) - p0, p1 = v[6] - v[4], q1 = (v[7] - v[5]) - p1;
    const float x0 = fmaf(d[1], q0, p0), x1 = fmaf(d[1], q1, p1);
    const float y0 = fmaf(d[0], q0, p0), y1 = fmaf(d[0], q1, p1);
    g[0] = fmaf(d[2], x1 - x0, x0);
    g[1] = fmaf(d[2], y1 - y0, y0);
    const float i0 = fmaf(d[0], v[1] - v[0], v[0]), i1 = fmaf(d[0], v[3] - v[2], v[2]);
    const float i2 = fmaf(d[0], v[5] - v[4], v[4]), i3 = fmaf(d[0], v[7] - v[6], v[6]);
    g[2] = fmaf(d[1], i3 - i2, i2) - fmaf(d[1], i1 - i0, i0);
}

// f(integral_constant<M>) for the run-time window phase m in [0, V): the bodies are instantiated per phase
template <int V, class F>
TS_D void with_phase(int m, F&& f) {
    using std::integral_constant;
    if constexpr (V == 8) {
        switch (m) {
        case 4: f(integral_constant<int, 4>()); return;
        case 5: f(integral_constant<int, 5>()); return;
        case 6: f(integral_constant<int, 6>()); return;
        case 7: f(integral_constant<int, 7>()); return;
        }
    }
    switch (m) {
    case 0: f(integral_constant<int, 0>()); return;
    case 1: f(integral_constant<int, 1>()); return;
    case 2: f(integral_constant<int, 2>()); return;
    default: f(integral_constant<int, 3>()); return;
    }
}

template <typename ST, int DIM>
struct ActiveFwdBody {
    static constexpr int V = Pack<ST>::V, NVW = V + 1;   // elements per item, window with the +1 neighbour
    const TArgs& a;
    const int tid, nt;
    UnitShift us;
    int m;

    const UnitShift* tbl;
    TS_D ActiveFwdBody(const TArgs& a_, int tid_, int nt_, const UnitShift* tbl_) : a(a_), tid(tid_), nt(nt_), m(0), tbl(tbl_) {}
    TS_D void begin_unit(int c) {
        us = unit_shift(a, tbl, c);
        m = pmod(a.lbL - us.sh[2], V);
    }
    TS_D void end_unit(int, int) {}

    template <int M>
    TS_D void run(const Stage& sg) const {
        constexpr int NR = 1 << (DIM - 1);
        const unsigned box = shared_addr(sg.st);
        const int pitch = a.TG + 1, ximg = a.x_img_chunks, xb = a.xb;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        for (int item = tid; item < sg.total; item += nt) {
            Item p;
            if (!decode_item<DIM == 3>(a, sg, item, p)) continue;
            const int base = p.pl * ximg + (p.a * xb + p.b) * pitch + p.cg;
            float X[NR][NVW];
#pragma unroll
            for (int rv = 0; rv < NR; ++rv) load_win<ST, M, NVW>(box, base + neighbour_row_offset<DIM>(rv, xb, pitch), X[rv]);
            float o[V];
#pragma unroll
            for (int t = 0; t < V; ++t) {
                float v[8];
                neighbours_from_rows<DIM>(X, t, v);
                o[t] = interpolate<float, DIM>(v, d);
            }
            __stcs((uint4*)item_dst(a, sg, p), Pack<ST>::pack(o));
        }
    }
    // strip-mined variant, used for 3-D (see BackwardBody::run_strip)
    template <int M>
    TS_D void run_strip(const Stage& sg) const {
        constexpr int NR = 1 << (DIM - 1);
        constexpr int S = DIM == 3 ? 2 : 1;
        const unsigned box = shared_addr(sg.st);
        const int pitch = a.TG + 1, ximg = a.x_img_chunks, xb = a.xb;
        const int xslab = xb * pitch;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        const int R = a.R, nchunk = a.nchunk, TG = a.TG, TA = a.TA;
        const int strips = sg.npl * TA * nchunk * TG;
        const int orow = a.OGR * 16;
        for (int sidx = tid; sidx < strips; sidx += nt) {
            const int r = (int)fdiv((unsigned)sidx, a.d_TG), cg = sidx - r * TG;
            const int r2 = (int)fdiv((unsigned)r, a.d_nchunk), kc = r - r2 * nchunk;
            int pl = r2, ia = 0;
            if (TA > 1) { pl = (int)fdiv((unsigned)r2, a.d_TA); ia = r2 - pl * TA; }
            const int b0 = kc * R;
            if (cg >= sg.gn || ia >= sg.an || b0 >= sg.bn) continue;
            const int bend = b0 + R < sg.bn ? b0 + R : sg.bn;
            Item p;
            p.pl = pl; p.a = ia; p.b = b0; p.cg = cg;
            int xch = pl * ximg + (ia * xb + b0) * pitch + cg;
            unsigned char* dst = item_dst(a, sg, p);
            float Xlo[S][NVW];
#pragma unroll
            for (int q = 0; q < S; ++q) load_win<ST, M, NVW>(box, xch + q * xslab, Xlo[q]);
            for (int b = b0; b < bend; ++b) {
                float X[NR][NVW];
#pragma unroll
                for (int q = 0; q < S; ++q) {
                    load_win<ST, M, NVW>(box, xch + pitch + q * xslab, X[S + q]);
#pragma unroll
                    for (int t = 0; t < NVW; ++t) X[q][t] = Xlo[q][t];
                }
                float o[V];
#pragma unroll
                for (int t = 0; t < V; ++t) {
                    float v[8];
                    neighbours_from_rows<DIM>(X, t, v);
                    o[t] = interpolate<float, DIM>(v, d);
                }
                __stcs((uint4*)dst, Pack<ST>::pack(o));
#pragma unroll
                for (int q = 0; q < S; ++q)
#pragma unroll
                    for (int t = 0; t < NVW; ++t) Xlo[q][t] = X[S + q][t];
                xch += pitch; dst += orow;
            }
        }
    }
    template <int M>
    TS_D void run_any(const Stage& sg) const {
        if constexpr (DIM == 3) run_strip<M>(sg); else run<M>(sg);   // 2-D is HBM-bound either way and the flat,
                                                                     // padded index space is measurably faster there
    }
    TS_D void step(const Stage& sg) const {
        with_phase<V>(m, [&](auto M) { this->template run_any<decltype(M)::value>(sg); });
    }
};

template <typename ST, int DIM, bool ACTIVE>
struct BackwardBody {
    static constexpr int V = Pack<ST>::V, NVW = V + 1;
    const TArgs& a;
    const int tid, nt, wid, lane;
    UnitShift us;
    int m;
    double acc[DIM];

    const UnitShift* tbl;
    TS_D BackwardBody(const TArgs& a_, int tid_, int nt_, int wid_, int lane_, const UnitShift* tbl_)
        : a(a_), tid(tid_), nt(nt_), wid(wid_), lane(lane_), m(0), tbl(tbl_) {}
    TS_D void begin_unit(int c) {
        us = unit_shift(a, tbl, c);
        m = pmod(-us.sh[2], V);
#pragma unroll
        for (int d = 0; d < DIM; ++d) acc[d] = 0.0;
    }
    // one partial per (unit, consumer warp): fixed shuffle tree, no atomics
    TS_D void end_unit(int c, int chunk) {
#pragma unroll
        for (int d = 0; d < DIM; ++d) {
            double v = acc[d];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) a.partials[((long long)chunk * a.nw + wid) * (a.g.C * DIM) + (long long)c * DIM + d] = v;
        }
    }

    template <int M>
    TS_D void run(const Stage& sg) {
        constexpr int NR = 1 << (DIM - 1);
        constexpr int MG = ACTIVE ? M : ((V - M) & (V - 1));      // misalignment of the grad window used for grad_input
        const unsigned xbox = shared_addr(sg.st);
        const unsigned gv_box = xbox + a.off_gv;
        const unsigned g2_box = xbox + a.off_g2;
        const int pitch = a.TG + 1, ximg = a.x_img_chunks, gimg = a.g_img_chunks, xb = a.xb, tb = a.TB;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        float ts[DIM];
#pragma unroll
        for (int k = 0; k < DIM; ++k) ts[k] = 0.f;
        for (int item = tid; item < sg.total; item += nt) {
            Item p;
            if (!decode_item<DIM == 3>(a, sg, item, p)) continue;
            const int gch = p.pl * gimg + (p.a * tb + p.b) * pitch + p.cg;
            const int xch = p.pl * ximg + (p.a * xb + p.b) * pitch + p.cg;
            float gv[V];
            load_win<ST, 0, V>(gv_box, gch, gv);
            // ---- grad_weight terms ----
            float X[NR][NVW];
#pragma unroll
            for (int rv = 0; rv < NR; ++rv) load_win<ST, M, NVW>(xbox, xch + neighbour_row_offset<DIM>(rv, xb, pitch), X[rv]);
#pragma unroll
            for (int t = 0; t < V; ++t) {
                float v[8], wg[3];
                neighbours_from_rows<DIM>(X, t, v);
                weight_partials_fast<DIM>(v, d, wg);
#pragma unroll
                for (int k = 0; k < DIM; ++k) ts[k] = fmaf(gv[t], wg[k], ts[k]);
            }
            // ---- grad_input ----
            float o[V];
            if (ACTIVE) {
                float G[NR][NVW];
#pragma unroll
                for (int rv = 0; rv < NR; ++rv) load_win<ST, MG, NVW>(g2_box, xch + neighbour_row_offset<DIM>(rv, xb, pitch), G[rv]);
#pragma unroll
                for (int t = 0; t < V; ++t) {
                    float v[8];
                    neighbours_from_rows<DIM>(G, t, v);
                    o[t] = interpolate<float, DIM>(v, d);
                }
            } else {
                load_win<ST, MG, V>(g2_box, gch, o);
            }
            __stcs((uint4*)item_dst(a, sg, p), Pack<ST>::pack(o));
        }
#pragma unroll
        for (int k = 0; k < DIM; ++k) acc[k] += (double)ts[k];   // fp32 inside a stage, fp64 across stages
    }
    // Strip-mined variant (used for 3-D, where the kernels are instruction-bound): a thread owns (image, slab, group, chunk of R rows); the "+1 row"
    // windows of one item are the "+0 row" windows of the next and stay in registers.
    template <int M>
    TS_D void run_strip(const Stage& sg) {
        constexpr int NR = 1 << (DIM - 1);
        constexpr int S = DIM == 3 ? 2 : 1;
        constexpr int MG = ACTIVE ? M : ((V - M) & (V - 1));
        const unsigned xbox = shared_addr(sg.st);
        const unsigned gv_box = xbox + a.off_gv;
        const unsigned g2_box = xbox + a.off_g2;
        const int pitch = a.TG + 1, ximg = a.x_img_chunks, gimg = a.g_img_chunks, xb = a.xb, tb = a.TB;
        const int xslab = xb * pitch;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        float ts[DIM];
#pragma unroll
        for (int k = 0; k < DIM; ++k) ts[k] = 0.f;
        const int R = a.R, nchunk = a.nchunk, TG = a.TG, TA = a.TA;
        const int strips = sg.npl * TA * nchunk * TG;
        const int orow = a.OGR * 16;
        for (int sidx = tid; sidx < strips; sidx += nt) {
            const int r = (int)fdiv((unsigned)sidx, a.d_TG), cg = sidx - r * TG;
            const int r2 = (int)fdiv((unsigned)r, a.d_nchunk), kc = r - r2 * nchunk;
            int pl = r2, ia = 0;
            if (TA > 1) { pl = (int)fdiv((unsigned)r2, a.d_TA); ia = r2 - pl * TA; }
            const int b0 = kc * R;
            if (cg >= sg.gn || ia >= sg.an || b0 >= sg.bn) continue;
            const int bend = b0 + R < sg.bn ? b0 + R : sg.bn;
            Item p;
            p.pl = pl; p.a = ia; p.b = b0; p.cg = cg;
            int gch = pl * gimg + (ia * tb + b0) * pitch + cg;
            int xch = pl * ximg + (ia * xb + b0) * pitch + cg;
            unsigned char* dst = item_dst(a, sg, p);
            float Xlo[S][NVW], Glo[S][NVW];
#pragma unroll
            for (int q = 0; q < S; ++q) load_win<ST, M, NVW>(xbox, xch + q * xslab, Xlo[q]);
            if (ACTIVE) {
#pragma unroll
                for (int q = 0; q < S; ++q) load_win<ST, MG, NVW>(g2_box, xch + q * xslab, Glo[q]);
            }
            for (int b = b0; b < bend; ++b) {
                float gv[V];
                load_win<ST, 0, V>(gv_box, gch, gv);
                float X[NR][NVW];
#pragma unroll
                for (int q = 0; q < S; ++q) {
                    load_win<ST, M, NVW>(xbox, xch + pitch + q * xslab, X[S + q]);
#pragma unroll
                    for (int t = 0; t < NVW; ++t) X[q][t] = Xlo[q][t];
                }
#pragma unroll
                for (int t = 0; t < V; ++t) {
                    float v[8], wg[3];
                    neighbours_from_rows<DIM>(X, t, v);
                    weight_partials_fast<DIM>(v, d, wg);
#pragma unroll
                    for (int k = 0; k < DIM; ++k) ts[k] = fmaf(gv[t], wg[k], ts[k]);
                }
                float o[V];
                if (ACTIVE) {
                    float G[NR][NVW];
#pragma unroll
                    for (int q = 0; q < S; ++q) {
                        load_win<ST, MG, NVW>(g2_box, xch + pitch + q * xslab, G[S + q]);
#pragma unroll
                        for (int t = 0; t < NVW; ++t) G[q][t] = Glo[q][t];
                    }
#pragma unroll
                    for (int t = 0; t < V; ++t) {
                        float v[8];
                        neighbours_from_rows<DIM>(G, t, v);
                        o[t] = interpolate<float, DIM>(v, d);
                    }
#pragma unroll
                    for (int q = 0; q < S; ++q)
#pragma unroll
                        for (int t = 0; t < NVW; ++t) Glo[q][t] = G[S + q][t];
                } else {
                    load_win<ST, MG, V>(g2_box, gch, o);
                }
                __stcs((uint4*)dst, Pack<ST>::pack(o));
#pragma unroll
                for (int q = 0; q < S; ++q)
#pragma unroll
                    for (int t = 0; t < NVW; ++t) Xlo[q][t] = X[S + q][t];
                xch += pitch; gch += pitch; dst += orow;
            }
        }
#pragma unroll
        for (int k = 0; k < DIM; ++k) acc[k] += (double)ts[k];
    }
    template <int M>
    TS_D void run_any(const Stage& sg) {
        if constexpr (DIM == 3) run_strip<M>(sg); else run<M>(sg);   // 2-D is HBM-bound either way and the flat,
                                                                     // padded index space is measurably faster there
    }
    TS_D void step(const Stage& sg) {
        with_phase<V>(m, [&](auto M) { this->template run_any<decltype(M)::value>(sg); });
    }
};

// ---- kernels -----------------------------------------------------------------------------------
TS_D const UnitShift* setup_barriers(const TArgs& a, unsigned char* smem, uint64_t*& full, uint64_t*& empty) {
    full = (uint64_t*)(smem + (size_t)a.stages * a.stage_stride);
    empty = full + a.stages;
    UnitShift* tbl = (UnitShift*)(empty + a.stages);
    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], (unsigned)a.nw); }
        fence_barrier_init();
    }
    pdl_trigger();          // the next kernel of the stream may be scheduled as soon as SMs free up
    pdl_wait();             // nothing above touches global memory; everything below may depend on the previous kernel
    if (a.table)
        for (int c = threadIdx.x; c < (int)a.g.C; c += blockDim.x) tbl[c] = compute_unit_shift(a, c);
    __syncthreads();
    return tbl;
}

template <bool SLABS>
__global__ void __launch_bounds__(MAXT_TMA_GATHER, 1) k_tma_gather(const __grid_constant__ TArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *full, *empty;
    const UnitShift* tbl = setup_barriers(a, smem, full, empty);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wid == a.nw) { if (lane == 0) producer(a, smem, full, empty, tbl); return; }
    GatherBody<SLABS> body(a, threadIdx.x, a.nw * 32, tbl);
    consumer_loop(a, smem, full, empty, lane, body);
}

template <typename ST, int DIM>
__global__ void __launch_bounds__(MAXT_TMA_ARITH, 1) k_tma_active_forward(const __grid_constant__ TArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *full, *empty;
    const UnitShift* tbl = setup_barriers(a, smem, full, empty);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wid == a.nw) { if (lane == 0) producer(a, smem, full, empty, tbl); return; }
    ActiveFwdBody<ST, DIM> body(a, threadIdx.x, a.nw * 32, tbl);
    consumer_loop(a, smem, full, empty, lane, body);
}

template <typename ST, int DIM, bool ACTIVE>
__global__ void __launch_bounds__(MAXT_TMA_ARITH, 1) k_tma_backward(const __grid_constant__ TArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *full, *empty;
    const UnitShift* tbl = setup_barriers(a, smem, full, empty);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wid == a.nw) { if (lane == 0) producer(a, smem, full, empty, tbl); return; }
    BackwardBody<ST, DIM, ACTIVE> body(a, threadIdx.x, a.nw * 32, wid, lane, tbl);
    consumer_loop(a, smem, full, empty, lane, body);
}

// every TMA kernel calls pdl_wait() before it touches global memory
int launch(void (*kernel)(TArgs), const TArgs& a, const TmaPlan& p, cudaStream_t s) {
    return launch_persistent(kernel, p.grid, (a.nw + 1) * 32, p.smem_bytes, s, true, a);
}

}  // namespace

bool tma_available() { return encode_tiled() != nullptr; }
bool make_tensor_map5(void* map, const void* base, int es, long long N, long long C, int A, int B, int L, int bl, int bb, int ba, int bn) {
    return make_map((CUtensorMap*)map, base, es, N, C, A, B, L, bl, bb, ba, bn);
}

// ---- planning -----------------------------------------------------------------------------------
TmaPlan plan_tma(const Geo& g, int mode, int active, int esize, int dtype, bool dense_x, unsigned long long fill, const void* x,
                 const void* out, const void* grad, int sm_count) {
    TmaPlan p;
    memset(&p, 0, sizeof(p));
    p.ok = false;
    if (!encode_tiled()) return p;
    if (g.pad != TS_PAD_ZEROS || !dense_x || fill != 0ull) return p;
    if (g.N * g.C == 0 || g.in_plane == 0 || g.out_plane == 0) return p;
    // arithmetic kernels: fp32, or 2-D fp16 / bf16 whose weights are fp32 (same-dtype 16-bit layers keep their families)
    const bool arith16 = g.wf32 && g.dim == 2 && (dtype == TS_F16 || dtype == TS_BF16);
    if (mode != 0 && dtype != TS_F32 && !arith16) return p;
    if (mode != 0) esize = dtype == TS_F32 ? 4 : 2;
    if (esize != 1 && esize != 2 && esize != 4 && esize != 8) return p;
    const int d = g.dim;
    if (mode == 2)                                       // the backward tiles assume output space == input space
        for (int ax = 0; ax < d; ++ax)
            if (g.lb[ax] != 0 || g.OS[ax] != g.S[ax]) return p;
    if (mode != 0)                                       // a size-1 axis ignores its shift AND its +1 neighbour is the element
        for (int ax = 0; ax < d; ++ax)                   // itself (shifts_kernels.h:40-50), not the zero the copy engine would fill
            if (g.S[ax] == 1) return p;
    const int vec = 16 / esize;
    const Levels lv(g);
    const int L = lv.L, OL = lv.OL, OB = lv.OB, OA = lv.OA;
    if (((long long)L * esize) % 16 || ((long long)OL * esize) % 16) return p;   // global strides / output rows: 16-byte multiples
    if (((uintptr_t)x & 15) || ((uintptr_t)out & 15) || ((uintptr_t)grad & 15)) return p;
    if (g.N >= (1ll << 31) || g.C >= (1ll << 31)) return p;
    if (g.in_plane * esize >= (1ll << 40) / (g.C > 0 ? g.C : 1)) return p;       // tensor-map strides < 2^40

    const Tuning& t = tuning();
    TArgs& a = p.a;
    a.g = g;
    a.es = esize;
    a.vec = vec;
    a.mode = mode;
    a.active = active ? 1 : 0;
    a.OA = OA;    a.lbA = lv.lbA;
    a.OB = OB;    a.lbB = lv.lbB;
    const int OGR = a.OGR = OL / vec;
    a.lbL = lv.lbL;
    const int max_groups = 256 / vec - 1;               // box inner extent (TG+1)*vec <= 256 elements
    const int tiles_g = a.tiles_g = (OGR + max_groups - 1) / max_groups;
    const int TG = a.TG = (OGR + tiles_g - 1) / tiles_g;
    const int ex = mode != 0 ? 1 : 0;                   // +1 neighbour row / slab in the arithmetic boxes
    const int exb = d >= 2 ? ex : 0, exa = d == 3 ? ex : 0;
    long long TB = OB < 256 - exb ? OB : 256 - exb;
    long long TA = OA < 256 - exa ? OA : 256 - exa;
    auto image_bytes = [&](long long ta, long long tb, int* off_gv, int* off_g2) {
        const long long xbytes = round_up((ta + exa) * (tb + exb) * (TG + 1) * 16, 128);
        const long long gsbytes = round_up(ta * tb * (TG + 1) * 16, 128);
        if (off_gv) *off_gv = (int)xbytes;
        if (off_g2) *off_g2 = (int)(xbytes + gsbytes);
        if (mode != 2) return xbytes;
        return xbytes + gsbytes + (active ? xbytes : gsbytes);
    };
    const long long table_bytes = g.C <= TABLE_MAX_C ? g.C * 24 : 0;
    const long long budget = SMEM_LIMIT - 1024 - table_bytes;
    // defaults from the cfg3 sweep on B200 (tools/tune.py --tma): forward 6 x 28 KB, backward 5 x 42 KB
    // 3-D volumes: few large stages (deep slab tiles re-read fewer +1 neighbour slabs)
    // Ring depth, 1-D / 2-D: re-tuned in round 2 (tools/tma_sweep.py, cfg3, CUDA-graph replays).  Once the producer stopped
    // computing the shift parameters per unit it ran a full ring ahead, and MORE stages in flight made the kernels slower
    // (HBM page locality: forward 293 us with 6 stages, 256 us with 3; sparse backward 409 us with 5, 372 us with 4).
    const int want_stages = t.tma_stages > 0 ? t.tma_stages : d == 3 ? (mode == 2 ? 2 : 3) : (mode == 0 ? 3 : mode == 1 ? 4 : (active ? 5 : 4));
    const long long auto_target = d == 3 ? (mode == 2 ? 108 * 1024 : 72 * 1024) : (mode == 2 ? 42 * 1024 : 28 * 1024);
    const long long target = t.tma_stage_kb > 0 ? (long long)t.tma_stage_kb * 1024
                                                : (auto_target < budget / want_stages - 64 ? auto_target : budget / want_stages - 64);
    while (image_bytes(TA, TB, nullptr, nullptr) > target) {
        if (TA > 1) TA = (TA + 1) / 2;
        else if (TB > 1) TB = (TB + 1) / 2;
        else return p;
    }
    a.TA = (int)TA; a.TB = (int)TB;
    a.xa = (int)(TA + exa); a.xb = (int)(TB + exb);
    const int tiles_a = (int)((OA + TA - 1) / TA), tiles_b = a.tiles_b = (int)((OB + TB - 1) / TB);
    const long long tiles = (long long)tiles_a * tiles_b * tiles_g;
    if (tiles > 0x7fffffffLL) return p;
    a.tiles = (int)tiles;
    long long np = 1;
    if (tiles == 1) {
        // several images per stage only through a rank-5 box; the sub-box offsets then scale with np
        np = target / image_bytes(TA, TB, nullptr, nullptr);
        if (np < 1) np = 1;
        if (np > 256) np = 256;
        if (np > g.N) np = g.N;
    }
    a.np = (int)np;
    a.x_img_chunks = a.xa * a.xb * (TG + 1);
    a.g_img_chunks = a.TA * a.TB * (TG + 1);
    // with np images the three regions are [np x-boxes][np gv-boxes][np g2-boxes]
    const long long xbytes1 = (TA + exa) * (TB + exb) * (TG + 1) * 16, gsbytes1 = TA * TB * (TG + 1) * 16;
    const long long xreg = round_up(np * xbytes1, 128), gsreg = round_up(np * gsbytes1, 128);
    a.off_gv = (int)xreg;
    a.off_g2 = (int)(xreg + gsreg);
    long long stage_bytes = xreg, tx = np * xbytes1;
    if (mode == 2) {
        stage_bytes += gsreg + (active ? xreg : gsreg);
        tx += np * gsbytes1 + np * (active ? xbytes1 : gsbytes1);
    }
    const long long stride = round_up(stage_bytes, 1024);
    long long stages = budget / (stride + 16);
    if (stages > want_stages) stages = want_stages;
    if (stages < 2) return p;
    if (tx >= (1 << 20)) return p;                       // mbarrier tx-count range
    a.tx_bytes = (int)tx;
    a.stages = (int)stages;
    a.stage_stride = (int)stride;

    const int GP = a.GP = padded_groups(TG);
    const long long plane16 = g.C * (mode == 2 ? g.in_plane : g.out_plane) * esize / 16;
    if (np * plane16 >= 0x7fffffffLL || np * TA * TB * (long long)GP >= 0x7fffffffLL) return p;
    a.img_items = a.TA * a.TB * GP;
    a.img_stride16 = (int)plane16;
    // consumer warps: fill the last pass over a stage's items as well as possible
    const long long items = np * TA * TB * GP;
    const int max_warps = mode == 0 ? MAXT_TMA_GATHER / 32 - 1 : MAXT_TMA_ARITH / 32 - 1;
    int warps = t.tma_warps > 0 ? (t.tma_warps < max_warps ? t.tma_warps : max_warps) : 0;
    if (!warps) {
        auto eff = [&](int w) {
            const long long nt = 32ll * w, passes = (items + nt - 1) / nt;
            return (double)items / (double)(passes * nt);
        };
        // best fill of the last pass over a stage's items, preferring 8..16 warps: on cfg3 more
        // consumer warps never helped (the kernels are HBM-bound) and 25+ were measurably slower
        const int lo = 8, hi = 15;
        int best = lo;
        for (int w = lo; w <= hi && w <= max_warps; ++w)
            if (eff(w) >= eff(best) - 1e-9) best = w;
        int best_all = 8;
        for (int w = 8; w <= max_warps; ++w)
            if (eff(w) >= eff(best_all) - 1e-9) best_all = w;
        warps = eff(best) >= eff(best_all) - 0.08 ? best : best_all;
    }
    a.nw = warps;
    {   // strips: about three per thread and stage, at least two rows each (the row reuse is the point)
        const long long nt = 32ll * warps;
        long long R = (np * TA * TB * TG + 3 * nt - 1) / (3 * nt);
        if (R < 2) R = 2;
        if (R > TB) R = TB;
        a.R = (int)R;
        a.nchunk = (a.TB + a.R - 1) / a.R;
    }
    const UnitPlan up = plan_units(np, t.chunk_planes > 0 ? t.chunk_planes : pick_unit_images(g.N, g.C, np, sm_count, mode == 2 ? 0.4 : 0.1),
                                   g.N, g.C, sm_count, warps);
    if (!up.ok) return p;
    a.n_per_unit = up.n_per_unit;
    a.units = up.units;
    a.chunks = up.chunks;
    a.unit_order = t.unit_order;
    a.table = g.C <= TABLE_MAX_C ? 1 : 0;
    a.d_img = make_fastdiv((unsigned)a.img_items);
    a.d_GP = make_fastdiv((unsigned)GP);
    a.d_TB = make_fastdiv((unsigned)a.TB);
    a.d_tg = make_fastdiv((unsigned)tiles_g);
    a.d_tb = make_fastdiv((unsigned)tiles_b);
    a.d_TG = make_fastdiv((unsigned)TG);
    a.d_nchunk = make_fastdiv((unsigned)a.nchunk);
    a.d_TA = make_fastdiv((unsigned)a.TA);
    a.d_C = make_fastdiv((unsigned)g.C);
    a.d_chunks = make_fastdiv((unsigned)a.chunks);

    p.ok = true;
    p.grid = up.grid;
    p.slots = up.slots;
    p.smem_bytes = (size_t)(stages * stride + 16 * stages + 64 + table_bytes);
    return p;
}

int tma_gather(const Geo& g, const TmaPlan& p, int wk, const void* x, void* y, int esize, const void* w, int qkind, long long wzp,
               cudaStream_t s) {
    TArgs a = p.a;
    const Levels lv(g);
    a.out = (unsigned char*)y;
    a.w = w;
    a.wk = wk;
    a.qkind = qkind;
    a.wzp = wzp;
    if (!make_map(&a.map_x, x, esize, g.N, g.C, lv.A, lv.B, lv.L, (a.TG + 1) * a.vec, a.xb, a.xa, a.np))
        return TS_ERR_UNSUPPORTED;
    return a.TA > 1 ? launch(k_tma_gather<true>, a, p, s) : launch(k_tma_gather<false>, a, p, s);
}

template <typename ST>
static int active_forward_t(const Geo& g, const TArgs& a, const TmaPlan& p, cudaStream_t s) {
    switch (g.dim) {
    case 1: return launch(k_tma_active_forward<ST, 1>, a, p, s);
    case 2: return launch(k_tma_active_forward<ST, 2>, a, p, s);
    default: return launch(k_tma_active_forward<ST, 3>, a, p, s);
    }
}

int tma_active_forward(const Geo& g, const TmaPlan& p, int dtype, const void* x, const void* w, void* y, cudaStream_t s) {
    TArgs a = p.a;
    const Levels lv(g);
    a.out = (unsigned char*)y;
    a.w = w;
    if (!make_map(&a.map_x, x, a.es, g.N, g.C, lv.A, lv.B, lv.L, (a.TG + 1) * a.vec, a.xb, a.xa, a.np, dtype)) return TS_ERR_UNSUPPORTED;
    switch (dtype) {      // 16-bit: planned for 2-D only
    case TS_F16: return launch(k_tma_active_forward<__half, 2>, a, p, s);
    case TS_BF16: return launch(k_tma_active_forward<__nv_bfloat16, 2>, a, p, s);
    }
    return active_forward_t<float>(g, a, p, s);
}

template <typename ST>
static int backward_t(const Geo& g, const TArgs& a, const TmaPlan& p, int active, cudaStream_t s) {
    switch (g.dim * 2 + (active ? 1 : 0)) {
    case 2: return launch(k_tma_backward<ST, 1, false>, a, p, s);
    case 3: return launch(k_tma_backward<ST, 1, true>, a, p, s);
    case 4: return launch(k_tma_backward<ST, 2, false>, a, p, s);
    case 5: return launch(k_tma_backward<ST, 2, true>, a, p, s);
    case 6: return launch(k_tma_backward<ST, 3, false>, a, p, s);
    default: return launch(k_tma_backward<ST, 3, true>, a, p, s);
    }
}

int tma_backward(const Geo& g, const TmaPlan& p, int dtype, int active, const void* grad, const void* x, const void* w, void* gi,
                 double* partials, cudaStream_t s) {
    TArgs a = p.a;
    const Levels lv(g);
    const int A = lv.A, B = lv.B, L = lv.L, es = a.es, bl = (a.TG + 1) * a.vec;
    a.out = (unsigned char*)gi;
    a.w = w;
    a.partials = partials;
    if (!make_map(&a.map_x, x, es, g.N, g.C, A, B, L, bl, a.xb, a.xa, a.np, dtype)) return TS_ERR_UNSUPPORTED;
    if (!make_map(&a.map_gs, grad, es, g.N, g.C, A, B, L, bl, a.TB, a.TA, a.np, dtype)) return TS_ERR_UNSUPPORTED;
    if (active && !make_map(&a.map_gb, grad, es, g.N, g.C, A, B, L, bl, a.xb, a.xa, a.np, dtype)) return TS_ERR_UNSUPPORTED;
    switch (dtype) {      // 16-bit: planned for 2-D only
    case TS_F16: return active ? launch(k_tma_backward<__half, 2, true>, a, p, s) : launch(k_tma_backward<__half, 2, false>, a, p, s);
    case TS_BF16:
        return active ? launch(k_tma_backward<__nv_bfloat16, 2, true>, a, p, s) : launch(k_tma_backward<__nv_bfloat16, 2, false>, a, p, s);
    }
    return backward_t<float>(g, a, p, active, s);
}

}  // namespace ts

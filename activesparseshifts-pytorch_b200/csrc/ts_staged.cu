// ts_staged.cu -- the general bandwidth path (every padding mode, border crops, 1-/2-/4-/8-byte
// elements, fp32 / fp16 / bf16 arithmetic, 3-D volumes): persistent, warp-specialised kernels that
// stage whole slabs of the (n,c) planes in shared memory with 1-D bulk async copies
// (cp.async.bulk -> SASS UBLKCP) signalled through mbarriers, resolve the per-channel shift while
// READING shared memory and write global memory with 128-bit streaming stores.
//
//   CTA  = `nw` consumer warps + 1 producer warp (one elected lane), one CTA per SM, persistent.
//   Unit = (channel c, chunk of the batch), dealt round-robin to CTAs; the shift parameters are
//          registers for the whole unit and (backward) the grad_weight terms accumulate in
//          per-thread registers; every consumer warp writes ONE fp64 partial per unit -> no atomics.
//   Step = one ring stage = `np` images x one slab tile.  A slab (all rows x columns of one index of
//          the first of three axes; the whole plane for 1-D / 2-D) is contiguous in NCHW, so it is
//          ONE bulk copy.  The PRODUCER resolves the shift along the slab axis: slot k of a stage
//          holds source slab P(a0 - s + k), so consumers never remap that axis and 3-D volumes are
//          tiled over it (16x56x56 fp32 does not fit a stage).
//   Item = 16 bytes of output.  Each stage is processed in two passes:
//          (1) INTERIOR items -- every source window lies inside its row and every source row
//              inside its slab, so there is no index remapping, no validity mask, no padding rule:
//              aligned LDS.128 pairs + a compile-time word select (the column shift misaligns the
//              source by a unit-uniform amount).  This is the padding-independent fast path.
//          (2) EDGE items (rows / columns whose windows touch a border, ~10 % on 56x56 planes),
//              enumerated COMPACTLY so warps stay full, run the element-wise path with the
//              reference's remapping rules (ops/kernels/shifts_kernels.h:10-54).
//
// Semantics: ops/kernels/shifts_kernels.h:156-327, :532-571; the arithmetic helpers are the shared
// ones of ts_common.cuh (unfused lerp nest), so forward and grad_input are bit-identical to the
// generic family and to the CPU reference; grad_weight terms are summed in fp32 per stage, fp64
// across stages.
#include <cstring>

#include "ts_kernels.h"
#include "ts_ptx.cuh"

namespace ts {

namespace {

using namespace ptx;

constexpr int GUARD = 32;            // readable slack around the slabs of a stage (second group of a window pair)
constexpr int MAXT_GATHER = 1024, MAXT_ARITH = 512;   // 512 threads -> 128 registers per thread

// Per-unit shift parameters by LEVEL (0 slab, 1 row, 2 column).
struct UnitShift {
    int sx[3];     // integer shift reduced against the input sizes
    int sg[3];     // integer shift reduced against the output sizes (fetches from grad)
    float d[3];    // fractional parts per TENSOR AXIS (reference order)
};

TS_D UnitShift unit_shift(const SArgs& a, long long c) {
    UnitShift u;
    const int dim = a.g.dim;
    u.d[0] = u.d[1] = u.d[2] = 0.f;
#pragma unroll
    for (int lev = 0; lev < 3; ++lev) {
        const int ax = level_axis(lev, dim);
        u.sx[lev] = u.sg[lev] = 0;
        if (ax < 0) continue;
        const long long idx = c * dim + ax;
        long long iw = 0;
        if (a.mode == 0) {
            iw = sparse_shift(a.w, a.wk, a.qkind, a.wzp, idx);
        } else {
            float wv;
            if (a.wk == WK_F16) wv = __half2float(((const __half*)a.w)[idx]);
            else if (a.wk == WK_BF16) wv = __bfloat162float(((const __nv_bfloat16*)a.w)[idx]);
            else wv = ((const float*)a.w)[idx];
            float d;
            if (a.mode == 1) split_forward<float>(wv, true, iw, d);
            else split_backward<float>(wv, a.active != 0, iw, d);
            u.d[ax] = d;
        }
        u.sx[lev] = reduce_shift(iw, a.g.S[ax], a.g.pad);
        u.sg[lev] = reduce_shift(iw, a.g.OS[ax], a.g.pad);
    }
    return u;
}

// Tabulated once per CTA (like the TMA and halo families): the split + reduction of a weight is a few hundred dependent
// instructions (64-bit conversions and a 64-bit modulo), paid per UNIT by every consumer warp and -- on the critical path of
// the pipeline -- by the producer, whose next copies waited for it at every unit boundary.
TS_D UnitShift unit_shift_t(const SArgs& a, const UnitShift* tbl, long long c) { return tbl ? tbl[c] : unit_shift(a, c); }

// ---- producer ---------------------------------------------------------------------------------
// slab held by slot k of the three regions for tile origin a0 (negative: nothing to copy -> zeros padding)
TS_D int x_slot_slab(const SArgs& a, const UnitShift& us, int a0, int k) {
    if (a.g.dim < 3) return 0;
    const int j = (a.mode == 2 ? a0 : a0 + a.lbA) - us.sx[0] + k;
    return axis_index(j, a.A, a.g.pad);
}
TS_D int gv_slot_slab(const SArgs& a, int a0, int k) {
    if (a.g.dim < 3) return 0;
    const int oa = a0 - a.lbA + k;
    return (oa >= 0 && oa < a.OA) ? oa : -1;
}
TS_D int gi_slot_slab(const SArgs& a, const UnitShift& us, int a0, int k) {
    if (a.g.dim < 3) return 0;
    const int oa = a0 - a.lbA + k;              // output slab of the iteration slab (k may include the +1 neighbour)
    if (a.active) return axis_index(oa - us.sg[0], a.OA, a.g.pad);
    return axis_index(oa + us.sg[0], a.OA, a.g.pad);
}

// The whole producer WARP runs this: lane 0 waits for the slot and posts the byte count, then the copies of a stage are
// dealt to the lanes (one elected thread spent ~40 instructions per copy on addresses at single-thread issue rates:
// with many small slabs per stage -- 16-bit rows, 12 copies of 8 KB -- the consumers waited for the producer, not for HBM).
// TBL: the shift table exists (arithmetic kernels).  A template, not a run-time test: the byte mover's instantiation must stay
// the code it was -- the same source with a dead `tbl ? ... : ...` in it made ptxas schedule k_staged_gather 10 % slower.
template <bool TBL>
TS_D void producer(const SArgs& a, unsigned char* smem, uint64_t* full, uint64_t* empty, int lane, const UnitShift* tbl) {
    int s = 0, k = 0;
    const int C = (int)a.g.C, N = (int)a.g.N;
    const int per_img = a.xs + (a.mode == 2 ? a.gvs + a.gis : 0);
    const UnitRange ur = unit_range(a.units, a.unit_order);
    for (int u = ur.u; u < ur.end; u += ur.step) {
        int chunk, c;
        unit_decode(u, C, a.chunks, a.unit_order, c, chunk);
        const int n0 = chunk * a.n_per_unit;
        const int n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
        UnitShift us;
        if constexpr (TBL) us = unit_shift_t(a, tbl, c); else us = unit_shift(a, c);
        for (int nb = n0; nb < n1; nb += a.np) {
            const int npl = n1 - nb < a.np ? n1 - nb : a.np;
            for (int t = 0; t < a.tiles; ++t) {
                const int a0 = t * a.TA;
                unsigned char* st = smem + (size_t)s * a.stage_stride + GUARD;
                if (lane == 0) {
                    if (k > 0) mbar_wait(&empty[s], (unsigned)((k - 1) & 1));
                    // bytes first (slots outside the tensor under zeros padding are not copied)
                    int vx = 0, vgv = 0, vgi = 0;
                    for (int q = 0; q < a.xs; ++q) vx += x_slot_slab(a, us, a0, q) >= 0;
                    if (a.mode == 2) {
                        for (int q = 0; q < a.gvs; ++q) vgv += gv_slot_slab(a, a0, q) >= 0;
                        for (int q = 0; q < a.gis; ++q) vgi += gi_slot_slab(a, us, a0, q) >= 0;
                    }
                    mbar_expect_tx(&full[s], (unsigned)npl * ((unsigned)vx * a.slab_x + (unsigned)(vgv + vgi) * a.slab_g));
                }
                __syncwarp();        // the slot is free (lane 0 saw empty[s]) before any lane writes into it
                for (int job = lane; job < npl * per_img; job += 32) {
                    const int pl = job / per_img;
                    int q = job - pl * per_img;
                    const long long plane = (long long)(nb + pl) * C + c;
                    if (q < a.xs) {
                        const int slab = x_slot_slab(a, us, a0, q);
                        if (slab >= 0)
                            bulk_g2s(st + (size_t)(pl * a.xs + q) * a.slab_x, a.x + (plane * a.A + slab) * a.slab_x, (unsigned)a.slab_x, &full[s]);
                    } else if ((q -= a.xs) < a.gvs) {
                        const int slab = gv_slot_slab(a, a0, q);
                        if (slab >= 0)
                            bulk_g2s(st + a.off_gv + (size_t)(pl * a.gvs + q) * a.slab_g, a.grad + (plane * a.OA + slab) * a.slab_g,
                                     (unsigned)a.slab_g, &full[s]);
                    } else {
                        q -= a.gvs;
                        const int slab = gi_slot_slab(a, us, a0, q);
                        if (slab >= 0)
                            bulk_g2s(st + a.off_gi + (size_t)(pl * a.gis + q) * a.slab_g, a.grad + (plane * a.OA + slab) * a.slab_g,
                                     (unsigned)a.slab_g, &full[s]);
                    }
                }
                if (++s == a.stages) { s = 0; ++k; }
            }
        }
    }
}

// ---- consumer skeleton -----------------------------------------------------------------------
struct Stage {
    const unsigned char* st;   // stage base (after GUARD)
    unsigned char* dst;        // output address of (first image of the stage, channel c, slab a0)
    int npl, a0, an;           // images in the stage, tile origin, valid slabs of the tile
};

template <class Body>
TS_D void consumer_loop(const SArgs& a, unsigned char* smem, uint64_t* full, uint64_t* empty, int lane, Body& body) {
    int s = 0;
    unsigned phase = 0;
    const int C = (int)a.g.C, N = (int)a.g.N;
    const long long plane_bytes = a.img_stride / C;
    const long long out_slab = (long long)a.IB * a.gpr * a.VB;
    const UnitRange ur = unit_range(a.units, a.unit_order);
    for (int u = ur.u; u < ur.end; u += ur.step) {
        int chunk, c;
        unit_decode(u, C, a.chunks, a.unit_order, c, chunk);
        const int n0 = chunk * a.n_per_unit;
        const int n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
        body.begin_unit(c);
        for (int nb = n0; nb < n1; nb += a.np) {
            Stage sg;
            sg.npl = n1 - nb < a.np ? n1 - nb : a.np;
            unsigned char* img = a.out + ((long long)nb * C + c) * plane_bytes;
            for (int t = 0; t < a.tiles; ++t) {
                sg.a0 = t * a.TA;
                sg.an = a.IA - sg.a0 < a.TA ? a.IA - sg.a0 : a.TA;
                sg.dst = img + sg.a0 * out_slab;
                sg.st = smem + (size_t)s * a.stage_stride + GUARD;
                mbar_wait(&full[s], phase);
                body.step(sg);
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
                if (++s == a.stages) { s = 0; phase ^= 1u; }
            }
        }
        body.end_unit(c, chunk);
    }
}

// item of the padded index space -> (image, tile-local slab, row, group)
struct Item { int pl, a, b, cg; };
TS_D void decode_item(const SArgs& a, int item, Item& p) {
    p.pl = 0;
    int rem = item;
    if (a.np > 1) { p.pl = (int)fdiv((unsigned)item, a.d_img); rem = item - p.pl * a.img_items; }
    const int row = (int)fdiv((unsigned)rem, a.d_GP);
    p.cg = rem - row * a.GP;
    p.a = 0;
    p.b = row;
    if (a.TA > 1) { p.a = (int)fdiv((unsigned)row, a.d_IB); p.b = row - p.a * a.IB; }
}
// np * img_stride < 2^31 (plan_staged), so the offset inside a stage's destination fits 32 bits
TS_D unsigned char* item_dst(const SArgs& a, const Stage& sg, const Item& p) {
    const unsigned off = (unsigned)p.pl * (unsigned)a.img_stride + (unsigned)(((p.a * a.IB + p.b) * a.gpr + p.cg) * a.VB);
    return sg.dst + off;
}
// (unsigned)(v - lo) < (unsigned)(hi - lo)  <=>  lo <= v < hi
TS_D bool in_range(int v, int lo, int hi) { return (unsigned)(v - lo) < (unsigned)(hi - lo); }

// Interior box of a unit (rows, groups): items inside need no remap / mask.
struct Interior { int b_lo, b_hi, c_lo, c_hi; };
TS_D int ceil_div(int n, int d) { return n >= 0 ? (n + d - 1) / d : -((-n) / d); }
TS_D int floor_div(int n, int d) { return n >= 0 ? n / d : -((-n + d - 1) / d); }
TS_D void clamp_range(int& lo, int& hi, int n) {
    lo = lo < 0 ? 0 : lo;
    hi = hi > n ? n : hi;
    if (hi < lo) hi = lo;
}

// exact n / d for a divisor that is uniform over a unit: one real division per unit, then umulhi
// (exact for n * d < 2^32; here n < 2^20 items, d < 2^11)
struct UDiv { unsigned m; int d; };
TS_D UDiv make_udiv(int d) {
    UDiv u;
    u.d = d > 0 ? d : 1;
    u.m = u.d == 1 ? 0u : (unsigned)(0xFFFFFFFFu / (unsigned)u.d) + 1u;
    return u;
}
TS_D int udiv(int n, const UDiv& u) { return u.d == 1 ? n : (int)__umulhi((unsigned)n, u.m); }

// compact enumeration of the items OUTSIDE the interior box of a tile:
//   E1: every slab, every row, edge groups            E2: every slab, edge rows, interior groups
//   E3: edge slabs, interior rows, interior groups
struct EdgeSets {
    int b_lo, b_hi, c_lo, c_hi;               // interior box (rows, groups): per unit
    int B, G;                                 // rows, groups of the iteration space
    UDiv d_ce, d_ci, d_be, d_bi, d_B;
    int a_lo, a_hi, A;                        // interior slabs / valid slabs of the tile: per stage
    int n1, n2, n3;                           // set sizes per image (per stage)
    UDiv d_per;                               // divisor "edge items per image", recomputed only when it changes
    TS_D void init_unit(const Interior& in, int rows, int groups) {
        b_lo = in.b_lo; b_hi = in.b_hi; c_lo = in.c_lo; c_hi = in.c_hi;
        B = rows; G = groups;
        d_ce = make_udiv(c_lo + (G - c_hi));
        d_ci = make_udiv(c_hi - c_lo);
        d_be = make_udiv(b_lo + (B - b_hi));
        d_bi = make_udiv(b_hi - b_lo);
        d_B = make_udiv(B);
        d_per.d = -1;
    }
    TS_D void init_stage(int alo, int ahi, int an) {
        a_lo = alo; a_hi = ahi; A = an;
        const int ce = c_lo + (G - c_hi), ci = c_hi - c_lo;
        const int be = b_lo + (B - b_hi), bi = b_hi - b_lo;
        const int ae = a_lo + (A - a_hi);
        n1 = A * B * ce;
        n2 = A * be * ci;
        n3 = ae * bi * ci;
        if (n1 + n2 + n3 != d_per.d) d_per = make_udiv(n1 + n2 + n3);
    }
    TS_D int per_image() const { return n1 + n2 + n3; }
    TS_D int image_of(int e) const { return udiv(e, d_per); }
    static TS_D int pick(int k, int lo, int hi) { return k < lo ? k : hi + (k - lo); }
    TS_D void decode(int e, Item& p) const {
        if (e < n1) {
            const int r = udiv(e, d_ce), k = e - r * d_ce.d;
            p.cg = pick(k, c_lo, c_hi);
            p.a = udiv(r, d_B);
            p.b = r - p.a * B;
        } else if (e < n1 + n2) {
            e -= n1;
            const int r = udiv(e, d_ci), j = e - r * d_ci.d;
            p.cg = c_lo + j;
            p.a = udiv(r, d_be);
            p.b = pick(r - p.a * d_be.d, b_lo, b_hi);
        } else {
            e -= n1 + n2;
            const int r = udiv(e, d_ci), j = e - r * d_ci.d;
            p.cg = c_lo + j;
            const int ka = udiv(r, d_bi);
            p.b = b_lo + (r - ka * d_bi.d);
            p.a = pick(ka, a_lo, a_hi);
        }
    }
};

// Edge items are few (~10 %), compact (so a warp that has any is full of them) and several times
// more expensive than interior items: hand them to a DIFFERENT group of warps every stage, so that
// over the ring depth every consumer warp does the same amount of work.
struct EdgeRotor {
    int rot;
    TS_D EdgeRotor() : rot(0) {}
    // first edge index of this thread for a stage with `total` edge items
    TS_D int first(int tid, int nt, int total) {
        const int span = ((total + 31) >> 5) << 5;
        rot += span;                       // running offset modulo nt (span <= a few thousand)
        while (rot >= nt) rot -= nt;
        int vt = tid - rot;
        if (vt < 0) vt += nt;
        return vt;
    }
};

// rows per strip (about three strips per thread and stage) and strips per column of the interior box
TS_D void strip_plan(const Interior& in, int images_x_slabs, int nt, int& R, int& nchunk, UDiv& d_nchunk) {
    const int ci = in.c_hi - in.c_lo, bi = in.b_hi - in.b_lo;
    const unsigned items = (unsigned)images_x_slabs * (unsigned)(bi > 0 ? bi : 0) * (unsigned)(ci > 0 ? ci : 0);   // < 2^31 (plan_staged)
    R = (int)((items + 3u * (unsigned)nt - 1u) / (3u * (unsigned)nt));
    if (R < 2) R = 2;                  // a strip of one row reuses nothing
    R = R > bi ? (bi > 0 ? bi : 1) : R;
    nchunk = bi > 0 ? (bi + R - 1) / R : 1;
    d_nchunk = make_udiv(nchunk);
}

// ---- window loads -----------------------------------------------------------------------------
template <int NW>
TS_D void load_words_rt(unsigned base, int off, int ws, unsigned* w) {
    switch (ws) {
    case 0: load_words<0, NW>(base, off, w); break;
    case 1: load_words<1, NW>(base, off, w); break;
    case 2: load_words<2, NW>(base, off, w); break;
    default: load_words<3, NW>(base, off, w); break;
    }
}

// window of NV elements starting at element index `e0` (>= 0, window inside the region) of a staged region
// (`region` = 32-bit shared-window address)
template <typename ST, int WS, int NV>
TS_D void load_window(unsigned region, int e0, float* out) {
    constexpr int NW = Pack<ST>::words(NV);
    const int byte = e0 * (int)sizeof(ST);
    unsigned w[NW + 1];
    load_words<WS, NW>(region, byte & ~15, w);
    w[NW] = 0u;
    Pack<ST>::template unpack<NV>(w, (byte & 2) * 8, out);
}
template <typename ST, int NV>
TS_D void load_window_rt(unsigned region, int e0, float* out) {
    constexpr int NW = Pack<ST>::words(NV);
    const int byte = e0 * (int)sizeof(ST);
    unsigned w[NW + 1];
    load_words_rt<NW>(region, byte & ~15, (byte >> 2) & 3, w);
    w[NW] = 0u;
    Pack<ST>::template unpack<NV>(w, (byte & 2) * 8, out);
}

// 1-D tensors (an image is ONE row): per-unit stepping of the flat (image, interior group) loop of a thread
struct LineWalk {
    int ci, pl0, j0, dpl, dj;
    TS_D void init(int ci_, int tid, int nt) {
        ci = ci_;
        pl0 = j0 = dpl = dj = 0;
        if (ci > 0) { pl0 = tid / ci; j0 = tid - pl0 * ci; dpl = nt / ci; dj = nt - dpl * ci; }
    }
    TS_D void next(int& pl, int& j) const {
        pl += dpl; j += dj;
        if (j >= ci) { j -= ci; ++pl; }
    }
};

// Column part of an edge item's window, shared by all its rows: either fully inside the row (vector
// loads with a run-time misalignment) or remapped element by element (hoisted out of the row loop).
template <typename ST, int NV>
struct EdgeCols {
    bool inside;
    int c0;
    int cols[NV];
    TS_D void init(int c0_, int L, int pad) {
        c0 = c0_;
        inside = c0 >= 0 && c0 + NV <= L;
        if (!inside) {
#pragma unroll
            for (int t = 0; t < NV; ++t) cols[t] = axis_index(c0 + t, L, pad);
        }
    }
    // row: flat row index inside `region` or -1 (zeros)
    TS_D void load(const unsigned char* region, int row, int L, float* out) const {
        if (row < 0) {
#pragma unroll
            for (int t = 0; t < NV; ++t) out[t] = 0.f;
        } else if (inside) {
            load_window_rt<ST, NV>(shared_addr(region), row * L + c0, out);
        } else {
#pragma unroll
            for (int t = 0; t < NV; ++t) out[t] = cols[t] >= 0 ? Elem<ST>::ld(((const ST*)region)[row * L + cols[t]]) : 0.f;
        }
    }
};

template <int DIM, int NVW>
TS_D void neighbours_from_rows(const float (*X)[NVW], int t, float* v) {
    constexpr int NR = 1 << (DIM - 1);
#pragma unroll
    for (int q = 0; q < (1 << DIM); ++q) v[q] = X[q & (NR - 1)][t + (q >> (DIM - 1))];
}

// grad_weight factors with ordinary (contractable) arithmetic: tolerance-checked only
template <int DIM>
TS_D void weight_partials_fast(const float* v, const float* d, float* g) {
    if (DIM == 1) { g[0] = v[1] - v[0]; return; }
    if (DIM == 2) {
        const float p = v[2] - v[0], q = (v[3] - v[1]) - p;
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

// flat row (slot * rows + row) of neighbour variant rv for an edge item, or -1 (zeros).  DIM 3:
// bit0 of rv = +1 slab slot (the producer resolved that axis), bit1 = +1 row; DIM 2: bit0 = +1 row.
template <int DIM>
TS_D int edge_row(int slot, bool slot1_ok, bool slot0_ok, int rowv, int rv, int rows, int pad) {
    if (DIM == 1) return 0;
    if (DIM == 2) return axis_index(rowv + (rv & 1), rows, pad);
    const bool ok = (rv & 1) ? slot1_ok : slot0_ok;
    const int r = axis_index(rowv + ((rv >> 1) & 1), rows, pad);
    return (ok && r >= 0) ? (slot + (rv & 1)) * rows + r : -1;
}
// same for an interior item: plain arithmetic
template <int DIM>
TS_D int interior_row(int row0, int rv, int rows) {
    if (DIM == 1) return row0;
    if (DIM == 2) return row0 + (rv & 1);
    return row0 + (rv & 1) * rows + ((rv >> 1) & 1);
}

// ================================================================================================
// mode 0: sparse / quantized forward -- a byte mover.  G = 32-bit words per item (4/2/1), ES =
// element bytes.
template <int G, int ES>
struct GatherBody {
    static constexpr int VB = 4 * G, V = VB / ES;
    const SArgs& a;
    const int tid, nt;
    UnitShift us;
    Interior in;
    EdgeSets es;
    EdgeRotor rotor;
    int mb;
    int R, nchunk;        // rows per strip / strips per column of the interior box (per unit)
    UDiv d_nchunk;

    TS_D GatherBody(const SArgs& a_, int tid_, int nt_) : a(a_), tid(tid_), nt(nt_), mb(0), R(1), nchunk(1) {}
    TS_D void begin_unit(int c) {
        us = unit_shift(a, c);
        mb = pmod((a.lbL - us.sx[2]) * ES, VB);
        // rows: 0 <= ob + lbB - s1 < B ; groups: 0 <= V*cg + lbL - s2, V*cg + lbL - s2 + V <= L
        in.b_lo = us.sx[1] - a.lbB;
        in.b_hi = a.B - a.lbB + us.sx[1];
        clamp_range(in.b_lo, in.b_hi, a.OB);
        in.c_lo = ceil_div(us.sx[2] - a.lbL, V);
        in.c_hi = floor_div(a.L - V - a.lbL + us.sx[2], V) + 1;
        clamp_range(in.c_lo, in.c_hi, a.gpr);
        es.init_unit(in, a.OB, a.gpr);
        strip_plan(in, a.np * a.TA, nt, R, nchunk, d_nchunk);
    }
    TS_D void end_unit(int, int) {}

    // slots whose slab lies outside the tensor (zeros padding) make the tile slab an edge slab
    TS_D void slab_range(const Stage& sg, int& a_lo, int& a_hi) const {
        a_lo = 0;
        a_hi = sg.an;
        if (a.g.dim == 3 && a.g.pad == TS_PAD_ZEROS && a.A > 1) {
            a_lo = us.sx[0] - a.lbA - sg.a0;                 // a0 + a + lbA - s0 >= 0
            a_hi = a.A - a.lbA + us.sx[0] - sg.a0;           // ... < A
            clamp_range(a_lo, a_hi, sg.an);
        }
    }

    // Interior pass, strip-mined: a thread owns (image, slab, group, chunk of `R` consecutive rows) and
    // walks down the rows with two pointer increments per item -- no per-item index decoding.
    template <int WS, bool SUB>
    TS_D void interior(const Stage& sg, int a_lo, int a_hi) const {
        const int ci = in.c_hi - in.c_lo, bi = in.b_hi - in.b_lo, ai = a_hi - a_lo;
        if (ci <= 0 || bi <= 0 || ai <= 0) return;
        const int bs8 = (mb & 3) * 8;
        const int rowb = a.L * ES, orowb = a.gpr * VB;
        const int img_bytes = a.xs * a.slab_x;
        const int col0 = (a.lbL - us.sx[2]) * ES - mb;        // aligned byte offset of group 0's window inside its row
        const int rsh = a.lbB - us.sx[1];
        const int strips = sg.npl * ai * nchunk * ci;
        const UDiv d_ai = make_udiv(ai);
        const unsigned sst = shared_addr(sg.st);
        for (int sidx = tid; sidx < strips; sidx += nt) {
            const int r = udiv(sidx, es.d_ci), j = sidx - r * ci;
            const int r2 = udiv(r, d_nchunk), k = r - r2 * nchunk;
            int pl = r2, ia = 0;
            if (ai > 1) { pl = udiv(r2, d_ai); ia = r2 - pl * ai; }
            Item p;
            p.pl = pl; p.a = a_lo + ia; p.b = in.b_lo + k * R; p.cg = in.c_lo + j;
            const int bend = p.b + R < in.b_hi ? p.b + R : in.b_hi;
            unsigned src = sst + p.pl * img_bytes + (p.a * a.B + p.b + rsh) * rowb + col0 + p.cg * VB;
            unsigned char* dst = item_dst(a, sg, p);
            for (int b = p.b; b < bend; ++b, src += rowb, dst += orowb) {
                unsigned W[2 * G + 1];
                if constexpr (G == 4) {
                    const uint4 A = lds128(src);
                    W[0] = A.x; W[1] = A.y; W[2] = A.z; W[3] = A.w;
                    if (WS > 0 || SUB) { const uint4 Bv = lds128(src + 16); W[4] = Bv.x; W[5] = Bv.y; W[6] = Bv.z; W[7] = Bv.w; }
                } else if constexpr (G == 2) {
                    const uint2 A = lds64(src);
                    W[0] = A.x; W[1] = A.y;
                    if (WS > 0 || SUB) { const uint2 Bv = lds64(src + 8); W[2] = Bv.x; W[3] = Bv.y; }
                } else {
                    W[0] = lds32(src);
                    if (WS > 0 || SUB) W[1] = lds32(src + 4);
                }
                W[2 * G] = 0u;
                unsigned o[G];
#pragma unroll
                for (int q = 0; q < G; ++q) o[q] = SUB ? __funnelshift_r(W[q + WS], W[q + WS + 1], bs8) : W[q + WS];
                if constexpr (G == 4) __stcs((uint4*)dst, make_uint4(o[0], o[1], o[2], o[3]));
                else if constexpr (G == 2) __stcs((uint2*)dst, make_uint2(o[0], o[1]));
                else __stcs((unsigned*)dst, o[0]);
            }
        }
    }

    // Edge items: rows remapped per item; a window that lies inside its row (edge ROWS) or any
    // window under zeros padding takes the same aligned-pair load as the interior (zeros: the pad
    // value is blended in with byte masks); only windows that wrap / reflect / clamp at a row end
    // are gathered element by element.
    template <int WS, bool SUB>
    TS_D void edges(const Stage& sg, int a_lo, int a_hi, int first, int total, int per) const {
        const int pad = a.g.pad;
        const int bs8 = (mb & 3) * 8;
        unsigned fillw[G];
#pragma unroll
        for (int k = 0; k < G; ++k) {
            if (ES == 1) fillw[k] = 0x01010101u * (unsigned)(a.fill & 0xffu);
            else if (ES == 2) fillw[k] = 0x00010001u * (unsigned)(a.fill & 0xffffu);
            else if (ES == 4) fillw[k] = (unsigned)a.fill;
            else fillw[k] = (k & 1) ? (unsigned)(a.fill >> 32) : (unsigned)a.fill;
        }
        for (int e = first; e < total; e += nt) {
            Item p;
            p.pl = a.np > 1 ? es.image_of(e) : 0;
            es.decode(e - p.pl * per, p);
            const bool slab_ok = x_slot_slab(a, us, sg.a0, p.a) >= 0;     // the producer already applied the slab shift
            const int rb = a.g.dim >= 2 ? axis_index(p.b + a.lbB - us.sx[1], a.B, pad) : 0;
            const int cs = p.cg * V + a.lbL - us.sx[2];
            const unsigned char* slab = sg.st + (size_t)(p.pl * a.xs + p.a) * a.slab_x;
            const bool inside = cs >= 0 && cs + V <= a.L;
            unsigned o[G];
            if (!slab_ok || rb < 0 || (pad == TS_PAD_ZEROS && (cs + V <= 0 || cs >= a.L))) {
#pragma unroll
                for (int k = 0; k < G; ++k) o[k] = fillw[k];
            } else if (inside || pad == TS_PAD_ZEROS) {
                const unsigned char* src = slab + ((long long)rb * a.L + cs) * ES - mb;       // aligned to VB by construction
                unsigned W[2 * G + 1];
                if constexpr (G == 4) {
                    const uint4 A = *(const uint4*)src, Bv = *(const uint4*)(src + 16);
                    W[0] = A.x; W[1] = A.y; W[2] = A.z; W[3] = A.w; W[4] = Bv.x; W[5] = Bv.y; W[6] = Bv.z; W[7] = Bv.w;
                } else if constexpr (G == 2) {
                    const uint2 A = *(const uint2*)src, Bv = *(const uint2*)(src + 8);
                    W[0] = A.x; W[1] = A.y; W[2] = Bv.x; W[3] = Bv.y;
                } else {
                    W[0] = *(const unsigned*)src; W[1] = *(const unsigned*)(src + 4);
                }
                W[2 * G] = 0u;
#pragma unroll
                for (int q = 0; q < G; ++q) o[q] = SUB ? __funnelshift_r(W[q + WS], W[q + WS + 1], bs8) : W[q + WS];
                if (!inside) {          // zeros padding, partially outside: blend the pad value in
                    const int lo_b = (cs < 0 ? -cs : 0) * ES;
                    const int hi_b = (a.L - cs < V ? a.L - cs : V) * ES;
#pragma unroll
                    for (int k = 0; k < G; ++k) {
                        int l = lo_b - 4 * k, h = hi_b - 4 * k;
                        l = l < 0 ? 0 : (l > 4 ? 4 : l);
                        h = h < 0 ? 0 : (h > 4 ? 4 : h);
                        const unsigned m = h > l ? ((0xffffffffu >> (8 * (4 - h))) & (0xffffffffu << (8 * l))) : 0u;
                        o[k] = (o[k] & m) | (fillw[k] & ~m);
                    }
                }
            } else {
#pragma unroll
                for (int k = 0; k < G; ++k) o[k] = 0u;
#pragma unroll
                for (int t = 0; t < V; ++t) {
                    const int col = axis_index(cs + t, a.L, pad);
                    const unsigned char* ep = slab + ((long long)rb * a.L + col) * ES;
                    if (ES == 1) o[(t / 4) % G] |= (unsigned)(*ep) << (8 * (t % 4));
                    else if (ES == 2) o[(t / 2) % G] |= (unsigned)(*(const unsigned short*)ep) << (16 * (t % 2));
                    else if (ES == 4) o[t % G] = *(const unsigned*)ep;
                    else { const uint2 v = *(const uint2*)ep; o[(2 * t) % G] = v.x; o[(2 * t + 1) % G] = v.y; }
                }
            }
            unsigned char* dst = item_dst(a, sg, p);
            if constexpr (G == 4) __stcs((uint4*)dst, make_uint4(o[0], o[1], o[2], o[3]));
            else if constexpr (G == 2) __stcs((uint2*)dst, make_uint2(o[0], o[1]));
            else __stcs((unsigned*)dst, o[0]);
        }
    }

    template <int WS, bool SUB>
    TS_D void both(const Stage& sg, int a_lo, int a_hi, int first, int total, int per) const {
        interior<WS, SUB>(sg, a_lo, a_hi);
        edges<WS, SUB>(sg, a_lo, a_hi, first, total, per);
    }

    TS_D void step(const Stage& sg) {
        int a_lo, a_hi;
        slab_range(sg, a_lo, a_hi);
        es.init_stage(a_lo, a_hi, sg.an);
        const int per = es.per_image(), total = sg.npl * per;
        const int first = rotor.first(tid, nt, total);
        const int ws = mb >> 2;
        if ((mb & 3) == 0) {
            switch (ws) {
            case 0: both<0, false>(sg, a_lo, a_hi, first, total, per); break;
            case 1: both<1 % G, false>(sg, a_lo, a_hi, first, total, per); break;
            case 2: both<2 % G, false>(sg, a_lo, a_hi, first, total, per); break;
            default: both<3 % G, false>(sg, a_lo, a_hi, first, total, per); break;
            }
        } else {
            switch (ws) {
            case 0: both<0, true>(sg, a_lo, a_hi, first, total, per); break;
            case 1: both<1 % G, true>(sg, a_lo, a_hi, first, total, per); break;
            case 2: both<2 % G, true>(sg, a_lo, a_hi, first, total, per); break;
            default: both<3 % G, true>(sg, a_lo, a_hi, first, total, per); break;
            }
        }
    }
};

// ================================================================================================
// mode 1: active (interpolating) forward.
template <typename ST, int DIM>
struct ActiveFwdBody {
    static constexpr int V = Pack<ST>::V, ES = (int)sizeof(ST), NVW = V + 1, NR = 1 << (DIM - 1);
    const SArgs& a;
    const int tid, nt;
    UnitShift us;
    Interior in;
    EdgeSets es;
    EdgeRotor rotor;
    bool any_interior;
    int R, nchunk;        // rows per strip / strips per column of the interior box (per unit)
    UDiv d_nchunk;
    LineWalk lw;          // DIM == 1 only
    const UnitShift* tbl = nullptr;

    TS_D ActiveFwdBody(const SArgs& a_, int tid_, int nt_) : a(a_), tid(tid_), nt(nt_), any_interior(false), R(1), nchunk(1) {}
    TS_D void begin_unit(int c) {
        us = unit_shift_t(a, tbl, c);
        // rows: 0 <= ob + lbB - s1, ob + lbB - s1 + 1 <= B-1 ; groups: 0 <= cs, cs + V + 1 <= L
        in.b_lo = us.sx[1] - a.lbB;
        in.b_hi = a.B - 1 - a.lbB + us.sx[1];
        if (DIM == 1) { in.b_lo = 0; in.b_hi = 1; }
        clamp_range(in.b_lo, in.b_hi, a.OB);
        in.c_lo = ceil_div(us.sx[2] - a.lbL, V);
        in.c_hi = floor_div(a.L - V - 1 - a.lbL + us.sx[2], V) + 1;
        clamp_range(in.c_lo, in.c_hi, a.gpr);
        // a size-1 axis ignores its shift and its +1 neighbour is the element itself: edge path only
        any_interior = a.L > 1 && (DIM < 2 || a.B > 1) && (DIM < 3 || a.A > 1);
        if (!any_interior) in.b_hi = in.b_lo = in.c_hi = in.c_lo = 0;
        es.init_unit(in, a.OB, a.gpr);
        strip_plan(in, a.np * a.TA, nt, R, nchunk, d_nchunk);
        if constexpr (DIM == 1) lw.init(in.c_hi - in.c_lo, tid, nt);
    }
    TS_D void end_unit(int, int) {}

    // 1-D tensors: an image is ONE row, so there is nothing to decode and nothing to carry between rows -- a flat
    // loop over (image, interior group) with every address term hoisted out; PH = byte phase of the x window inside
    // its 16-byte group (unit-uniform), compile-time here: a window costs its loads + one conversion per element.
    template <int PH>
    TS_D void interior_line(const Stage& sg) const {
        if (lw.ci <= 0) return;
        const int xb = (a.lbL - us.sx[2] + in.c_lo * V) * ES;            // >= 0 (interior); xb & 15 == PH
        const unsigned x0 = shared_addr(sg.st) + (unsigned)(xb & ~15);
        const int ximg = a.xs * a.slab_x;
        unsigned char* dst0 = sg.dst + in.c_lo * 16;
        const unsigned istr = (unsigned)a.img_stride;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        int pl = lw.pl0, j = lw.j0;
        while (pl < sg.npl) {
            float X[NVW], o[V];
            load_window_c<ST, PH, NVW>(x0 + (unsigned)(pl * ximg + j * 16), X);
#pragma unroll
            for (int t = 0; t < V; ++t) o[t] = interpolate<float, 1>(X + t, d);
            __stcs((uint4*)(dst0 + ((unsigned)pl * istr + (unsigned)(j * 16))), Pack<ST>::pack(o));
            lw.next(pl, j);
        }
    }

    TS_D void slab_range(const Stage& sg, int& a_lo, int& a_hi) const {
        a_lo = 0;
        a_hi = sg.an;
        if (DIM == 3 && a.g.pad == TS_PAD_ZEROS) {
            a_lo = us.sx[0] - a.lbA - sg.a0;
            a_hi = a.A - 1 - a.lbA + us.sx[0] - sg.a0;        // the +1 slot must exist as well
            clamp_range(a_lo, a_hi, sg.an);
        }
        if (!any_interior) a_lo = a_hi = 0;
    }

    // strip-mined interior (fp32, DIM >= 2): see BackwardBody::interior_strip
    template <int WS>
    TS_D void interior_strip(const Stage& sg, int a_lo, int a_hi) const {
        constexpr int S = DIM == 3 ? 2 : 1;
        const int ci = in.c_hi - in.c_lo, bi = in.b_hi - in.b_lo, ai = a_hi - a_lo;
        if (ci <= 0 || bi <= 0 || ai <= 0) return;
        const int img_bytes = a.xs * a.slab_x;
        const int col0 = a.lbL - us.sx[2];
        const int rsh = a.lbB - us.sx[1];
        const unsigned sst = shared_addr(sg.st);
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        const int L = a.L, xslab = a.B * a.L, orowb = a.gpr * 16;
        const int strips = sg.npl * ai * nchunk * ci;
        const UDiv d_ai = make_udiv(ai);
        for (int sidx = tid; sidx < strips; sidx += nt) {
            const int r = udiv(sidx, es.d_ci), j = sidx - r * ci;
            const int r2 = udiv(r, d_nchunk), k = r - r2 * nchunk;
            int pl = r2, ia = 0;
            if (ai > 1) { pl = udiv(r2, d_ai); ia = r2 - pl * ai; }
            Item p;
            p.pl = pl; p.a = a_lo + ia; p.b = in.b_lo + k * R; p.cg = in.c_lo + j;
            const int bend = p.b + R < in.b_hi ? p.b + R : in.b_hi;
            const unsigned img = sst + p.pl * img_bytes;
            int xe = (p.a * a.B + p.b + rsh) * L + col0 + p.cg * V;
            unsigned char* dst = item_dst(a, sg, p);
            float Xlo[S][NVW];
#pragma unroll
            for (int q = 0; q < S; ++q) load_window<ST, WS, NVW>(img, xe + q * xslab, Xlo[q]);
            for (int b = p.b; b < bend; ++b) {
                float X[NR][NVW];
#pragma unroll
                for (int q = 0; q < S; ++q) {
                    load_window<ST, WS, NVW>(img, xe + L + q * xslab, X[S + q]);
#pragma unroll
                    for (int t = 0; t < NVW; ++t) X[q][t] = Xlo[q][t];
                }
                float o[V];
#pragma unroll
                for (int t = 0; t < V; ++t) {
                    float v[8];
                    neighbours_from_rows<DIM, NVW>(X, t, v);
                    o[t] = interpolate<float, DIM>(v, d);
                }
                __stcs((uint4*)dst, Pack<ST>::pack(o));
#pragma unroll
                for (int q = 0; q < S; ++q)
#pragma unroll
                    for (int t = 0; t < NVW; ++t) Xlo[q][t] = X[S + q][t];
                xe += L; dst += orowb;
            }
        }
    }

    template <int WS>
    TS_D void interior(const Stage& sg, int a_lo, int a_hi) const {
        if constexpr (sizeof(ST) == 4 && DIM >= 2) interior_strip<WS>(sg, a_lo, a_hi);
        else interior_flat<WS>(sg, a_lo, a_hi);
    }

    template <int WS>
    TS_D void interior_flat(const Stage& sg, int a_lo, int a_hi) const {
        const int total = sg.npl * a.img_items;
        const int img_bytes = a.xs * a.slab_x;
        const int col0 = a.lbL - us.sx[2];
        const int rsh = DIM >= 2 ? a.lbB - us.sx[1] : 0;
        const unsigned sst = shared_addr(sg.st);
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        for (int item = tid; item < total; item += nt) {
            Item p;
            decode_item(a, item, p);
            if (!(in_range(p.cg, in.c_lo, in.c_hi) && in_range(p.b, in.b_lo, in.b_hi) && in_range(p.a, a_lo, a_hi))) continue;
            const unsigned img = sst + p.pl * img_bytes;
            const int row0 = p.a * a.B + p.b + rsh;
            float X[NR][NVW];
#pragma unroll
            for (int rv = 0; rv < NR; ++rv) load_window<ST, WS, NVW>(img, interior_row<DIM>(row0, rv, a.B) * a.L + col0 + p.cg * V, X[rv]);
            float o[V];
#pragma unroll
            for (int t = 0; t < V; ++t) {
                float v[8];
                neighbours_from_rows<DIM, NVW>(X, t, v);
                o[t] = interpolate<float, DIM>(v, d);
            }
            __stcs((uint4*)item_dst(a, sg, p), Pack<ST>::pack(o));
        }
    }

    // (an element-per-thread edge pass like the backward's was measured slower here: the forward gathers
    // only the x windows, whole items amortise the remapping better)
    TS_D void edges(const Stage& sg, int a_lo, int a_hi) {
        es.init_stage(a_lo, a_hi, sg.an);
        const int per = es.per_image(), total = sg.npl * per;
        const int pad = a.g.pad;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        for (int e = rotor.first(tid, nt, total); e < total; e += nt) {
            Item p;
            p.pl = a.np > 1 ? es.image_of(e) : 0;
            es.decode(e - p.pl * per, p);
            const unsigned char* img = sg.st + (size_t)p.pl * a.xs * a.slab_x;
            const bool ok0 = DIM < 3 || x_slot_slab(a, us, sg.a0, p.a) >= 0;
            const bool ok1 = DIM < 3 || x_slot_slab(a, us, sg.a0, p.a + 1) >= 0;
            EdgeCols<ST, NVW> xc;
            xc.init(p.cg * V + a.lbL - us.sx[2], a.L, pad);
            float X[NR][NVW];
#pragma unroll
            for (int rv = 0; rv < NR; ++rv) xc.load(img, edge_row<DIM>(p.a, ok1, ok0, p.b + a.lbB - us.sx[1], rv, a.B, pad), a.L, X[rv]);
            float o[V];
#pragma unroll
            for (int t = 0; t < V; ++t) {
                float v[8];
                neighbours_from_rows<DIM, NVW>(X, t, v);
                o[t] = interpolate<float, DIM>(v, d);
            }
            __stcs((uint4*)item_dst(a, sg, p), Pack<ST>::pack(o));
        }
    }

    TS_D void step(const Stage& sg) {
        int a_lo, a_hi;
        slab_range(sg, a_lo, a_hi);
        if constexpr (DIM == 1) {
            switch (pmod((a.lbL - us.sx[2]) * ES, 16)) {
            case 0: interior_line<0>(sg); break;
            case 4: interior_line<4>(sg); break;
            case 8: interior_line<8>(sg); break;
            case 12: interior_line<12>(sg); break;
            default:
                if constexpr (ES == 2) {
                    switch (pmod((a.lbL - us.sx[2]) * ES, 16)) {
                    case 2: interior_line<2>(sg); break;
                    case 6: interior_line<6>(sg); break;
                    case 10: interior_line<10>(sg); break;
                    default: interior_line<14>(sg); break;
                    }
                }
            }
            edges(sg, a_lo, a_hi);
            return;
        }
        const int ws = (pmod((a.lbL - us.sx[2]) * ES, 16)) >> 2;
        switch (ws) {
        case 0: interior<0>(sg, a_lo, a_hi); break;
        case 1: interior<1>(sg, a_lo, a_hi); break;
        case 2: interior<2>(sg, a_lo, a_hi); break;
        default: interior<3>(sg, a_lo, a_hi); break;
        }
        edges(sg, a_lo, a_hi);
    }
};

// ================================================================================================
// mode 2: backward (grad_input + grad_weight partials); iterates the INPUT space.
template <typename ST, int DIM, bool ACTIVE>
struct BackwardBody {
    static constexpr int V = Pack<ST>::V, ES = (int)sizeof(ST), NVW = V + 1, NR = 1 << (DIM - 1);
    const SArgs& a;
    const int tid, nt, wid, lane;
    UnitShift us;
    Interior in;
    EdgeSets es;
    EdgeRotor rotor;
    bool any_interior;
    int R, nchunk;        // rows per strip / strips per column of the interior box (per unit)
    UDiv d_nchunk;
    LineWalk lw;          // DIM == 1 only
    const UnitShift* tbl = nullptr;
    double acc[DIM];

    TS_D BackwardBody(const SArgs& a_, int tid_, int nt_, int wid_, int lane_)
        : a(a_), tid(tid_), nt(nt_), wid(wid_), lane(lane_), any_interior(false) {}

    TS_D void begin_unit(int c) {
        us = unit_shift_t(a, tbl, c);
#pragma unroll
        for (int k = 0; k < DIM; ++k) acc[k] = 0.0;
        // rows (input row ib, output row ob = ib - lbB):
        //   inside the crop          lbB <= ib < lbB + OB
        //   x window                 0 <= ib - sx1,  ib - sx1 + 1 <= B - 1
        //   grad window  sparse      0 <= ob + sg1 < OB          active   0 <= ob - sg1, ob - sg1 + 1 <= OB - 1
        int lo = a.lbB, hi = a.lbB + a.OB;
        if (DIM >= 2) {
            lo = max(lo, us.sx[1]);
            hi = min(hi, a.B - 1 + us.sx[1]);
            if (ACTIVE) { lo = max(lo, a.lbB + us.sg[1]); hi = min(hi, a.lbB + a.OB - 1 + us.sg[1]); }
            else { lo = max(lo, a.lbB - us.sg[1]); hi = min(hi, a.lbB + a.OB - us.sg[1]); }
        }
        in.b_lo = lo; in.b_hi = hi;
        clamp_range(in.b_lo, in.b_hi, a.B);
        // groups (input columns V*cg .. V*cg+V-1, output column oj0 = V*cg - lbL):
        //   inside the crop          lbL <= V*cg, V*cg + V <= lbL + OL
        //   x window                 0 <= V*cg - sx2,  V*cg - sx2 + V + 1 <= L
        //   grad window  sparse      0 <= oj0 + sg2, oj0 + sg2 + V <= OL     active  0 <= oj0 - sg2, oj0 - sg2 + V + 1 <= OL
        int clo = ceil_div(a.lbL, V), chi = floor_div(a.lbL + a.OL - V, V) + 1;
        clo = max(clo, ceil_div(us.sx[2], V));
        chi = min(chi, floor_div(a.L - V - 1 + us.sx[2], V) + 1);
        if (ACTIVE) { clo = max(clo, ceil_div(a.lbL + us.sg[2], V)); chi = min(chi, floor_div(a.lbL + a.OL - V - 1 + us.sg[2], V) + 1); }
        else { clo = max(clo, ceil_div(a.lbL - us.sg[2], V)); chi = min(chi, floor_div(a.lbL + a.OL - V - us.sg[2], V) + 1); }
        in.c_lo = clo; in.c_hi = chi;
        clamp_range(in.c_lo, in.c_hi, a.gpr);
        // the fast path needs the unshifted grad window 16-byte aligned and no size-1 axis
        any_interior = (a.lbL * ES) % 16 == 0 && a.L > 1 && (DIM < 2 || a.B > 1) && (DIM < 3 || a.A > 1);
        if (!any_interior) in.b_hi = in.b_lo = in.c_hi = in.c_lo = 0;
        es.init_unit(in, a.B, a.gpr);
        strip_plan(in, a.np * a.TA, nt, R, nchunk, d_nchunk);
        if constexpr (DIM == 1) lw.init(in.c_hi - in.c_lo, tid, nt);
    }

    // 1-D tensors (see ActiveFwdBody::interior_line).  PH / GPH: byte phases of the x window and of the grad_input
    // window inside their 16-byte groups; GPH = -1 when it does not follow from PH (crops): run-time realignment.
    template <int PH, int GPH>
    TS_D void interior_line(const Stage& sg, float* ts) const {
        if (lw.ci <= 0) return;
        constexpr int NG = ACTIVE ? NVW : V;
        const unsigned sst = shared_addr(sg.st);
        const int ximg = a.xs * a.slab_x, gvimg = a.gvs * a.slab_g, giimg = (a.gis ? a.gis : a.gvs) * a.slab_g;
        const int xb = (in.c_lo * V - us.sx[2]) * ES;                                // >= 0 (interior); xb & 15 == PH
        const int gvb = (in.c_lo * V - a.lbL) * ES;                                  // a multiple of 16 (any_interior)
        const int gie = in.c_lo * V - a.lbL + (ACTIVE ? -us.sg[2] : us.sg[2]);       // >= 0 (interior)
        const unsigned x0 = sst + (unsigned)(xb & ~15), gv0 = sst + (unsigned)(a.off_gv + gvb);
        const unsigned gireg = sst + (unsigned)(a.gis ? a.off_gi : a.off_gv), gi0 = gireg + (unsigned)((gie * ES) & ~15);
        unsigned char* dst0 = sg.dst + in.c_lo * 16;
        const unsigned istr = (unsigned)a.img_stride;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        float t0 = ts[0];
        int pl = lw.pl0, j = lw.j0;
        while (pl < sg.npl) {
            const int o16 = j * 16;
            float gv[V], X[NVW], G[NG], o[V];
            load_window_c<ST, 0, V>(gv0 + (unsigned)(pl * gvimg + o16), gv);
            load_window_c<ST, PH, NVW>(x0 + (unsigned)(pl * ximg + o16), X);
            if constexpr (GPH >= 0) load_window_c<ST, GPH, NG>(gi0 + (unsigned)(pl * giimg + o16), G);
            else load_window_rt<ST, NG>(gireg + (unsigned)(pl * giimg), gie + j * V, G);
#pragma unroll
            for (int t = 0; t < V; ++t) t0 = fmaf(gv[t], X[t + 1] - X[t], t0);
#pragma unroll
            for (int t = 0; t < V; ++t) {
                if constexpr (ACTIVE) o[t] = interpolate<float, 1>(G + t, d);
                else o[t] = G[t];
            }
            __stcs((uint4*)(dst0 + ((unsigned)pl * istr + (unsigned)o16)), Pack<ST>::pack(o));
            lw.next(pl, j);
        }
        ts[0] = t0;
    }
    template <int PH>
    TS_D void interior_line_x(const Stage& sg, float* ts) const {
        // the grad_input window's phase follows from the x window's when both shifts agree and nothing is cropped
        if (a.lbL == 0 && us.sg[2] == us.sx[2]) interior_line<PH, ACTIVE ? PH : ((16 - PH) & 15)>(sg, ts);
        else interior_line<PH, -1>(sg, ts);
    }
    // one partial per (unit, consumer warp): fixed shuffle tree, no atomics
    TS_D void end_unit(int c, int chunk) {
#pragma unroll
        for (int k = 0; k < DIM; ++k) {
            double v = acc[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) a.partials[((long long)chunk * a.nw + wid) * (a.g.C * DIM) + (long long)c * DIM + k] = v;
        }
    }

    // tile-local slabs whose x slots (a, a+1), gv slot and grad_input slots are all real slabs
    TS_D void slab_range(const Stage& sg, int& a_lo, int& a_hi) const {
        a_lo = 0;
        a_hi = sg.an;
        if (DIM == 3) {
            int lo = a.lbA - sg.a0, hi = a.lbA + a.OA - sg.a0;          // inside the crop
            if (a.g.pad == TS_PAD_ZEROS) {
                lo = max(lo, us.sx[0] - sg.a0);
                hi = min(hi, a.A - 1 + us.sx[0] - sg.a0);
                if (ACTIVE) { lo = max(lo, a.lbA + us.sg[0] - sg.a0); hi = min(hi, a.lbA + a.OA - 1 + us.sg[0] - sg.a0); }
                else { lo = max(lo, a.lbA - us.sg[0] - sg.a0); hi = min(hi, a.lbA + a.OA - us.sg[0] - sg.a0); }
            }
            a_lo = lo; a_hi = hi;
            clamp_range(a_lo, a_hi, sg.an);
        }
        if (!any_interior) a_lo = a_hi = 0;
    }

    // Strip-mined interior (fp32): a thread owns (image, slab, group, chunk of R consecutive rows).
    // Walking down the rows, the "+1 row" windows of one item are the "+0 row" windows of the next:
    // they stay in registers, so an item loads half of its x / grad windows and no index is decoded.
    // WSG: word misalignment of the grad_input window, or -1 when it is only known at run time.
    template <int WS, int WSG>
    TS_D void interior_strip(const Stage& sg, int a_lo, int a_hi, float* ts) const {
        constexpr int S = DIM == 3 ? 2 : 1;                 // slab variants of a window: slot a (and a + 1)
        const int ci = in.c_hi - in.c_lo, bi = in.b_hi - in.b_lo, ai = a_hi - a_lo;
        if (ci <= 0 || bi <= 0 || ai <= 0) return;
        const int ximg = a.xs * a.slab_x, gvimg = a.gvs * a.slab_g, giimg = (a.gis ? a.gis : a.gvs) * a.slab_g;
        const unsigned sst = shared_addr(sg.st), gibase = sst + (a.gis ? a.off_gi : a.off_gv);
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        const int gsh = ACTIVE ? -us.sg[2] : us.sg[2];
        const int grow_sh = DIM >= 2 ? (ACTIVE ? -us.sg[1] : us.sg[1]) : 0;
        const int xrsh = DIM >= 2 ? -us.sx[1] : 0;
        const int L = a.L, OL = a.OL, xslab = a.B * a.L, gslab = a.OB * a.OL, orowb = a.gpr * 16;
        const int strips = sg.npl * ai * nchunk * ci;
        const UDiv d_ai = make_udiv(ai);
        auto load_g = [&](unsigned base, int e0, float* out) {
            if constexpr (WSG >= 0) load_window<ST, WSG, NVW>(base, e0, out); else load_window_rt<ST, NVW>(base, e0, out);
        };
        for (int sidx = tid; sidx < strips; sidx += nt) {
            const int r = udiv(sidx, es.d_ci), j = sidx - r * ci;
            const int r2 = udiv(r, d_nchunk), k = r - r2 * nchunk;
            int pl = r2, ia = 0;
            if (ai > 1) { pl = udiv(r2, d_ai); ia = r2 - pl * ai; }
            Item p;
            p.pl = pl; p.a = a_lo + ia; p.b = in.b_lo + k * R; p.cg = in.c_lo + j;
            const int bend = p.b + R < in.b_hi ? p.b + R : in.b_hi;
            const unsigned x_p = sst + p.pl * ximg;
            const unsigned gv_p = sst + a.off_gv + p.pl * gvimg;
            const unsigned gi_p = gibase + p.pl * giimg;
            int xe = (p.a * a.B + p.b + xrsh) * L + p.cg * V - us.sx[2];
            int gve = (p.a * a.OB + p.b - a.lbB) * OL + p.cg * V - a.lbL;
            int gie = gve + grow_sh * OL + gsh;
            unsigned char* dst = item_dst(a, sg, p);
            float Xlo[S][NVW], Glo[S][NVW];
            if (DIM >= 2) {
#pragma unroll
                for (int q = 0; q < S; ++q) load_window<ST, WS, NVW>(x_p, xe + q * xslab, Xlo[q]);
                if (ACTIVE) {
#pragma unroll
                    for (int q = 0; q < S; ++q) load_g(gi_p, gie + q * gslab, Glo[q]);
                }
            }
            for (int b = p.b; b < bend; ++b) {
                float gv[V];
                load_window<ST, 0, V>(gv_p, gve, gv);
                // ---- grad_weight terms ----
                float X[NR][NVW];
                if (DIM == 1) {
                    load_window<ST, WS, NVW>(x_p, xe, X[0]);
                } else {
#pragma unroll
                    for (int q = 0; q < S; ++q) {
                        load_window<ST, WS, NVW>(x_p, xe + L + q * xslab, X[S + q]);
#pragma unroll
                        for (int t = 0; t < NVW; ++t) X[q][t] = Xlo[q][t];
                    }
                }
#pragma unroll
                for (int t = 0; t < V; ++t) {
                    float v[8], wg[3];
                    neighbours_from_rows<DIM, NVW>(X, t, v);
                    weight_partials_fast<DIM>(v, d, wg);
#pragma unroll
                    for (int q = 0; q < DIM; ++q) ts[q] = fmaf(gv[t], wg[q], ts[q]);
                }
                // ---- grad_input ----
                float o[V];
                if (ACTIVE) {
                    float Gw[NR][NVW];
                    if (DIM == 1) {
                        load_g(gi_p, gie, Gw[0]);
                    } else {
#pragma unroll
                        for (int q = 0; q < S; ++q) {
                            load_g(gi_p, gie + OL + q * gslab, Gw[S + q]);
#pragma unroll
                            for (int t = 0; t < NVW; ++t) Gw[q][t] = Glo[q][t];
                        }
                    }
#pragma unroll
                    for (int t = 0; t < V; ++t) {
                        float v[8];
                        neighbours_from_rows<DIM, NVW>(Gw, t, v);
                        o[t] = interpolate<float, DIM>(v, d);
                    }
                    if (DIM >= 2) {
#pragma unroll
                        for (int q = 0; q < S; ++q)
#pragma unroll
                            for (int t = 0; t < NVW; ++t) Glo[q][t] = Gw[S + q][t];
                    }
                } else {
                    if constexpr (WSG >= 0) load_window<ST, WSG, V>(gi_p, gie, o); else load_window_rt<ST, V>(gi_p, gie, o);
                }
                __stcs((uint4*)dst, Pack<ST>::pack(o));
                if (DIM >= 2) {
#pragma unroll
                    for (int q = 0; q < S; ++q)
#pragma unroll
                        for (int t = 0; t < NVW; ++t) Xlo[q][t] = X[S + q][t];
                }
                xe += L; gve += OL; gie += OL; dst += orowb;
            }
        }
    }

    template <int WS>
    TS_D void interior(const Stage& sg, int a_lo, int a_hi, float* ts) const {
        if constexpr (sizeof(ST) == 4) {
            // the grad_input window's misalignment follows from the x window's when both shifts agree
            if (a.lbL == 0 && us.sg[2] == us.sx[2]) interior_strip<WS, ACTIVE ? WS : ((4 - WS) & 3)>(sg, a_lo, a_hi, ts);
            else interior_strip<WS, -1>(sg, a_lo, a_hi, ts);
        } else {
            interior_flat<WS>(sg, a_lo, a_hi, ts);
        }
    }

    template <int WS>
    TS_D void interior_flat(const Stage& sg, int a_lo, int a_hi, float* ts) const {
        const int total = sg.npl * a.img_items;
        const int ximg = a.xs * a.slab_x, gvimg = a.gvs * a.slab_g, giimg = (a.gis ? a.gis : a.gvs) * a.slab_g;
        const unsigned sst = shared_addr(sg.st), gibase = sst + (a.gis ? a.off_gi : a.off_gv);
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        const int gsh = ACTIVE ? -us.sg[2] : us.sg[2];
        const int grow_sh = DIM >= 2 ? (ACTIVE ? -us.sg[1] : us.sg[1]) : 0;
        const int xrsh = DIM >= 2 ? -us.sx[1] : 0;
        for (int item = tid; item < total; item += nt) {
            Item p;
            decode_item(a, item, p);
            if (!(in_range(p.cg, in.c_lo, in.c_hi) && in_range(p.b, in.b_lo, in.b_hi) && in_range(p.a, a_lo, a_hi))) continue;
            const unsigned x_p = sst + p.pl * ximg;
            const unsigned gv_p = sst + a.off_gv + p.pl * gvimg;
            const unsigned gi_p = gibase + p.pl * giimg;
            const int ob = p.b - a.lbB, oj0 = p.cg * V - a.lbL;
            float gv[V];
            load_window<ST, 0, V>(gv_p, (p.a * a.OB + ob) * a.OL + oj0, gv);
            // ---- grad_weight terms ----
            const int xrow0 = p.a * a.B + p.b + xrsh;
            float X[NR][NVW];
#pragma unroll
            for (int rv = 0; rv < NR; ++rv) load_window<ST, WS, NVW>(x_p, interior_row<DIM>(xrow0, rv, a.B) * a.L + p.cg * V - us.sx[2], X[rv]);
#pragma unroll
            for (int t = 0; t < V; ++t) {
                float v[8], wg[3];
                neighbours_from_rows<DIM, NVW>(X, t, v);
                weight_partials_fast<DIM>(v, d, wg);
#pragma unroll
                for (int k = 0; k < DIM; ++k) ts[k] = fmaf(gv[t], wg[k], ts[k]);
            }
            // ---- grad_input ----
            float o[V];
            const int grow0 = p.a * a.OB + ob + grow_sh;
            if (ACTIVE) {
                float Gw[NR][NVW];
#pragma unroll
                for (int rv = 0; rv < NR; ++rv) load_window_rt<ST, NVW>(gi_p, interior_row<DIM>(grow0, rv, a.OB) * a.OL + oj0 + gsh, Gw[rv]);
#pragma unroll
                for (int t = 0; t < V; ++t) {
                    float v[8];
                    neighbours_from_rows<DIM, NVW>(Gw, t, v);
                    o[t] = interpolate<float, DIM>(v, d);
                }
            } else {
                load_window_rt<ST, V>(gi_p, grow0 * a.OL + oj0 + gsh, o);
            }
            __stcs((uint4*)item_dst(a, sg, p), Pack<ST>::pack(o));
        }
    }

    // Edge pass, fp32: ONE ELEMENT per thread-iteration (4 per item).  An edge item's windows are gathered
    // element by element anyway; with whole items per thread the lanes of a warp sit on consecutive ROWS at
    // the same column, and a row pitch of 56 words puts them on 4 banks (8-way conflicts on ~44 scalar loads
    // per item; measured: 10 % of the items cost 55 % of the 3-D backward).  With the element index fastest,
    // 4 consecutive lanes read 4 consecutive words (2-way conflicts), four times as many threads share the
    // edge work and the dependent chain per thread is one element instead of four.
    TS_D void edges_elem(const Stage& sg, int a_lo, int a_hi, float* ts) {
        es.init_stage(a_lo, a_hi, sg.an);
        const int per = es.per_image(), total = sg.npl * per * V;
        const int pad = a.g.pad;
        const int ximg = a.xs * a.slab_x, gvimg = a.gvs * a.slab_g, giimg = (a.gis ? a.gis : a.gvs) * a.slab_g;
        const unsigned char* gibase = sg.st + (a.gis ? a.off_gi : a.off_gv);
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        for (int task = rotor.first(tid, nt, total); task < total; task += nt) {
            const int e = task / V, t = task - e * V;
            Item p;
            p.pl = a.np > 1 ? es.image_of(e) : 0;
            es.decode(e - p.pl * per, p);
            const ST* x_p = (const ST*)(sg.st + (size_t)p.pl * ximg);
            const ST* gv_p = (const ST*)(sg.st + a.off_gv + (size_t)p.pl * gvimg);
            const ST* gi_p = (const ST*)(gibase + (size_t)p.pl * giimg);
            ST* dst = (ST*)item_dst(a, sg, p) + t;
            const int col = p.cg * V + t;
            const int oa = sg.a0 + p.a - a.lbA, ob = p.b - a.lbB, oj = col - a.lbL;
            const bool pass = ob >= 0 && ob < a.OB && (DIM < 3 || (oa >= 0 && oa < a.OA)) && oj >= 0 && oj < a.OL;
            if (!pass) { __stcs(dst, Elem<ST>::st(0.f)); continue; }
            const float gvv = Elem<ST>::ld(gv_p[((DIM == 3 ? p.a * a.OB : 0) + ob) * a.OL + oj]);
            // per-level index pairs (index, index of the +1 neighbour); -1 = outside (zeros padding)
            int xs[3][2], gs[3][2];
            xs[0][0] = xs[0][1] = gs[0][0] = gs[0][1] = 0;
            xs[1][0] = xs[1][1] = gs[1][0] = gs[1][1] = 0;
            if (DIM == 3) {
                xs[0][0] = x_slot_slab(a, us, sg.a0, p.a) >= 0 ? p.a : -1;
                xs[0][1] = x_slot_slab(a, us, sg.a0, p.a + 1) >= 0 ? p.a + 1 : -1;
                gs[0][0] = gi_slot_slab(a, us, sg.a0, p.a) >= 0 ? p.a : -1;
                gs[0][1] = ACTIVE ? (gi_slot_slab(a, us, sg.a0, p.a + 1) >= 0 ? p.a + 1 : -1) : -1;
            }
            if (DIM >= 2) {
                xs[1][0] = axis_index(p.b - us.sx[1], a.B, pad);
                xs[1][1] = axis_index(p.b - us.sx[1] + 1, a.B, pad);
                gs[1][0] = axis_index(ACTIVE ? ob - us.sg[1] : ob + us.sg[1], a.OB, pad);
                gs[1][1] = ACTIVE ? axis_index(ob - us.sg[1] + 1, a.OB, pad) : -1;
            }
            xs[2][0] = axis_index(col - us.sx[2], a.L, pad);
            xs[2][1] = axis_index(col - us.sx[2] + 1, a.L, pad);
            gs[2][0] = axis_index(ACTIVE ? oj - us.sg[2] : oj + us.sg[2], a.OL, pad);
            gs[2][1] = ACTIVE ? axis_index(oj - us.sg[2] + 1, a.OL, pad) : -1;
            // neighbour q: bit k = +1 on TENSOR axis k; tensor axis k lives on level k + (3 - DIM)
            float v[8], wg[3];
#pragma unroll
            for (int q = 0; q < (1 << DIM); ++q) {
                const int ia = DIM == 3 ? xs[0][q & 1] : 0;
                const int ib = DIM == 3 ? xs[1][(q >> 1) & 1] : DIM == 2 ? xs[1][q & 1] : 0;
                const int ic = xs[2][(q >> (DIM - 1)) & 1];
                v[q] = (ia >= 0 && ib >= 0 && ic >= 0) ? Elem<ST>::ld(x_p[(ia * a.B + ib) * a.L + ic]) : 0.f;
            }
            weight_partials_fast<DIM>(v, d, wg);
#pragma unroll
            for (int k = 0; k < DIM; ++k) ts[k] = fmaf(gvv, wg[k], ts[k]);
            float o;
            if (ACTIVE) {
#pragma unroll
                for (int q = 0; q < (1 << DIM); ++q) {
                    const int ia = DIM == 3 ? gs[0][q & 1] : 0;
                    const int ib = DIM == 3 ? gs[1][(q >> 1) & 1] : DIM == 2 ? gs[1][q & 1] : 0;
                    const int ic = gs[2][(q >> (DIM - 1)) & 1];
                    v[q] = (ia >= 0 && ib >= 0 && ic >= 0) ? Elem<ST>::ld(gi_p[(ia * a.OB + ib) * a.OL + ic]) : 0.f;
                }
                o = interpolate<float, DIM>(v, d);
            } else {
                const int ia = gs[0][0], ib = gs[1][0], ic = gs[2][0];
                o = (ia >= 0 && ib >= 0 && ic >= 0) ? Elem<ST>::ld(gi_p[(ia * a.OB + ib) * a.OL + ic]) : 0.f;
            }
            __stcs(dst, Elem<ST>::st(o));
        }
    }

    TS_D void edges(const Stage& sg, int a_lo, int a_hi, float* ts) {
        // 2-D / 1-D sparse items gather few words: whole items win there (measured on cfg3 with reflect padding)
        if constexpr (sizeof(ST) == 4 && (ACTIVE || DIM == 3)) { edges_elem(sg, a_lo, a_hi, ts); return; }
        es.init_stage(a_lo, a_hi, sg.an);
        const int per = es.per_image(), total = sg.npl * per;
        const int pad = a.g.pad;
        const int ximg = a.xs * a.slab_x, gvimg = a.gvs * a.slab_g, giimg = (a.gis ? a.gis : a.gvs) * a.slab_g;
        const unsigned char* gibase = sg.st + (a.gis ? a.off_gi : a.off_gv);
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        for (int e = rotor.first(tid, nt, total); e < total; e += nt) {
            Item p;
            p.pl = a.np > 1 ? es.image_of(e) : 0;
            es.decode(e - p.pl * per, p);
            const unsigned char* x_p = sg.st + (size_t)p.pl * ximg;
            const unsigned char* gv_p = sg.st + a.off_gv + (size_t)p.pl * gvimg;
            const unsigned char* gi_p = gibase + (size_t)p.pl * giimg;
            const int oa = sg.a0 + p.a - a.lbA, ob = p.b - a.lbB, oj0 = p.cg * V - a.lbL;
            const bool row_ok = ob >= 0 && ob < a.OB && (DIM < 3 || (oa >= 0 && oa < a.OA));
            float o[V];
            if (!row_ok || oj0 + V <= 0 || oj0 >= a.OL) {
#pragma unroll
                for (int t = 0; t < V; ++t) o[t] = 0.f;
                __stcs((uint4*)item_dst(a, sg, p), Pack<ST>::pack(o));
                continue;
            }
            bool okc[V];
#pragma unroll
            for (int t = 0; t < V; ++t) okc[t] = oj0 + t >= 0 && oj0 + t < a.OL;
            // gv: unshifted grad, zero outside the crop (slot p.a of the gv region holds output slab oa)
            float gv[V];
            {
                EdgeCols<ST, V> gc;
                gc.init(oj0, a.OL, TS_PAD_ZEROS);
                gc.load(gv_p, (DIM == 3 ? p.a * a.OB : 0) + ob, a.OL, gv);
            }
            // ---- grad_weight terms ----
            const bool xok0 = DIM < 3 || x_slot_slab(a, us, sg.a0, p.a) >= 0;
            const bool xok1 = DIM < 3 || x_slot_slab(a, us, sg.a0, p.a + 1) >= 0;
            float X[NR][NVW];
            {
                EdgeCols<ST, NVW> xc;
                xc.init(p.cg * V - us.sx[2], a.L, pad);
#pragma unroll
                for (int rv = 0; rv < NR; ++rv) xc.load(x_p, edge_row<DIM>(p.a, xok1, xok0, p.b - us.sx[1], rv, a.B, pad), a.L, X[rv]);
            }
#pragma unroll
            for (int t = 0; t < V; ++t) {
                float v[8], wg[3];
                neighbours_from_rows<DIM, NVW>(X, t, v);
                weight_partials_fast<DIM>(v, d, wg);
#pragma unroll
                for (int k = 0; k < DIM; ++k) ts[k] += okc[t] ? gv[t] * wg[k] : 0.f;
            }
            // ---- grad_input ----
            const bool gok0 = DIM < 3 || gi_slot_slab(a, us, sg.a0, p.a) >= 0;
            if (ACTIVE) {
                const bool gok1 = DIM < 3 || gi_slot_slab(a, us, sg.a0, p.a + 1) >= 0;
                float Gw[NR][NVW];
                EdgeCols<ST, NVW> gc;
                gc.init(oj0 - us.sg[2], a.OL, pad);
#pragma unroll
                for (int rv = 0; rv < NR; ++rv) gc.load(gi_p, edge_row<DIM>(p.a, gok1, gok0, ob - us.sg[1], rv, a.OB, pad), a.OL, Gw[rv]);
#pragma unroll
                for (int t = 0; t < V; ++t) {
                    float v[8];
                    neighbours_from_rows<DIM, NVW>(Gw, t, v);
                    o[t] = okc[t] ? interpolate<float, DIM>(v, d) : 0.f;
                }
            } else {
                int row = 0;
                if (DIM >= 2) {
                    const int r = axis_index(ob + us.sg[1], a.OB, pad);
                    row = (gok0 && r >= 0) ? (DIM == 3 ? p.a * a.OB : 0) + r : -1;
                }
                float Gs[V];
                EdgeCols<ST, V> gc;
                gc.init(oj0 + us.sg[2], a.OL, pad);
                gc.load(gi_p, row, a.OL, Gs);
#pragma unroll
                for (int t = 0; t < V; ++t) o[t] = okc[t] ? Gs[t] : 0.f;
            }
            __stcs((uint4*)item_dst(a, sg, p), Pack<ST>::pack(o));
        }
    }

    TS_D void step(const Stage& sg) {
        int a_lo, a_hi;
        slab_range(sg, a_lo, a_hi);
        float ts[DIM];
#pragma unroll
        for (int k = 0; k < DIM; ++k) ts[k] = 0.f;
        if constexpr (DIM == 1) {
            switch (pmod(-us.sx[2] * ES, 16)) {
            case 0: interior_line_x<0>(sg, ts); break;
            case 4: interior_line_x<4>(sg, ts); break;
            case 8: interior_line_x<8>(sg, ts); break;
            case 12: interior_line_x<12>(sg, ts); break;
            default:
                if constexpr (ES == 2) {
                    switch (pmod(-us.sx[2] * ES, 16)) {
                    case 2: interior_line_x<2>(sg, ts); break;
                    case 6: interior_line_x<6>(sg, ts); break;
                    case 10: interior_line_x<10>(sg, ts); break;
                    default: interior_line_x<14>(sg, ts); break;
                    }
                }
            }
        } else {
            const int ws = (pmod(-us.sx[2] * ES, 16)) >> 2;
            switch (ws) {
            case 0: interior<0>(sg, a_lo, a_hi, ts); break;
            case 1: interior<1>(sg, a_lo, a_hi, ts); break;
            case 2: interior<2>(sg, a_lo, a_hi, ts); break;
            default: interior<3>(sg, a_lo, a_hi, ts); break;
            }
        }
        edges(sg, a_lo, a_hi, ts);
#pragma unroll
        for (int k = 0; k < DIM; ++k) acc[k] += (double)ts[k];   // fp32 inside a stage, fp64 across stages
    }
};

// ---- kernels -----------------------------------------------------------------------------------
template <bool TBL>
TS_D const UnitShift* setup_barriers(const SArgs& a, unsigned char* smem, uint64_t*& full, uint64_t*& empty) {
    full = (uint64_t*)(smem + (size_t)a.stages * a.stage_stride);
    empty = full + a.stages;
    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], (unsigned)a.nw); }
        fence_barrier_init();
    }
    UnitShift* tbl = nullptr;
    if constexpr (TBL) {
        if (a.table) {
            tbl = (UnitShift*)(empty + a.stages);
            for (int c = threadIdx.x; c < (int)a.g.C; c += blockDim.x) tbl[c] = unit_shift(a, c);
        }
    }
    __syncthreads();
    return tbl;
}

template <int G, int ES>
__global__ void __launch_bounds__(MAXT_GATHER, 1) k_staged_gather(const __grid_constant__ SArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *full, *empty;
    setup_barriers<false>(a, smem, full, empty);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wid == a.nw) { producer<false>(a, smem, full, empty, lane, nullptr); return; }
    GatherBody<G, ES> body(a, threadIdx.x, a.nw * 32);
    consumer_loop(a, smem, full, empty, lane, body);
}

template <typename ST, int DIM>
__global__ void __launch_bounds__(MAXT_ARITH, 1) k_staged_active_forward(const __grid_constant__ SArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *full, *empty;
    const UnitShift* tbl = setup_barriers<true>(a, smem, full, empty);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wid == a.nw) { producer<true>(a, smem, full, empty, lane, tbl); return; }
    ActiveFwdBody<ST, DIM> body(a, threadIdx.x, a.nw * 32);
    body.tbl = tbl;
    consumer_loop(a, smem, full, empty, lane, body);
}

template <typename ST, int DIM, bool ACTIVE>
__global__ void __launch_bounds__(MAXT_ARITH, 1) k_staged_backward(const __grid_constant__ SArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t *full, *empty;
    const UnitShift* tbl = setup_barriers<true>(a, smem, full, empty);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (wid == a.nw) { producer<true>(a, smem, full, empty, lane, tbl); return; }
    BackwardBody<ST, DIM, ACTIVE> body(a, threadIdx.x, a.nw * 32, wid, lane);
    body.tbl = tbl;
    consumer_loop(a, smem, full, empty, lane, body);
}

int launch(void (*kernel)(SArgs), const SArgs& a, const StagedPlan& p, cudaStream_t s) {
    return launch_persistent(kernel, p.grid, (a.nw + 1) * 32, p.smem_bytes, s, false, a);
}

}  // namespace

// ---- planning -----------------------------------------------------------------------------------
StagedPlan plan_staged(const Geo& g, int mode, int active, int esize, int dtype, bool dense_x, const void* x, const void* y_or_gi,
                       const void* grad, int sm_count) {
    StagedPlan p;
    memset(&p, 0, sizeof(p));
    p.ok = false;
    if (!dense_x || g.N * g.C == 0 || g.in_plane == 0 || g.out_plane == 0) return p;
    if (mode != 0) {
        if (dtype != TS_F32 && dtype != TS_F16 && dtype != TS_BF16) return p;     // fp64 arithmetic: generic family
        esize = dtype == TS_F32 ? 4 : 2;
    }
    if (g.N >= (1ll << 31) || g.C >= (1ll << 31)) return p;
    const int d = g.dim;
    const Levels lv(g);
    const int A = lv.A, OA = lv.OA;
    const long long B = lv.B, OB = lv.OB;
    const long long Lb = (long long)lv.L * esize, OLb = (long long)lv.OL * esize;
    int vb = 0;
    if (mode == 0) {
        for (int cand : {16, 8, 4})
            if (cand >= esize && Lb % cand == 0 && OLb % cand == 0) { vb = cand; break; }
    } else if (Lb % 16 == 0 && OLb % 16 == 0) vb = 16;
    if (!vb) return p;
    const long long slab_x = B * Lb, slab_g = OB * OLb;
    if (slab_x % 16 || (mode == 2 && slab_g % 16)) return p;                      // bulk copies: 16-byte granules
    if (slab_x >= (1 << 20) || slab_g >= (1 << 20)) return p;
    if (((uintptr_t)x & 15) || ((uintptr_t)grad & 15) || ((uintptr_t)y_or_gi & (uintptr_t)(vb - 1))) return p;

    const Tuning& t = tuning();
    SArgs& a = p.a;
    a.g = g;
    a.es = esize;
    a.mode = mode;
    a.active = active ? 1 : 0;
    a.A = lv.A;    a.OA = lv.OA;    a.lbA = lv.lbA;
    a.B = lv.B;    a.OB = lv.OB;    a.lbB = lv.lbB;
    a.L = lv.L;    a.OL = lv.OL;    a.lbL = lv.lbL;
    a.VB = vb;
    a.V = vb / esize;
    a.gpr = (mode == 2 ? a.L : a.OL) / a.V;
    a.slab_x = (int)slab_x;
    a.slab_g = (int)slab_g;
    const int IA = a.IA = mode == 2 ? A : OA;
    const long long IB = mode == 2 ? B : OB;
    a.IB = (int)IB;
    const int ex = mode != 0 ? 1 : 0;                       // +1 neighbour slab for the arithmetic kernels
    const int ctas = (mode == 0 && t.ctas_per_sm > 1) ? t.ctas_per_sm : 1;     // byte mover only: several small pipelines per SM
    const long long table_bytes = (mode != 0 && g.C <= TABLE_MAX_C) ? (g.C * 36 + 15) / 16 * 16 : 0;     // per-channel shift table
    const long long budget = SMEM_LIMIT / ctas - 1024 - table_bytes;
    // bytes of one image's slots for a tile of `ta` slabs
    auto slots = [&](long long ta, int* xs, int* gvs, int* gis) {
        const int x_ = (int)(d == 3 ? ta + ex : 1);
        int gv_ = 0, gi_ = 0;
        if (mode == 2) {
            gv_ = (int)(d == 3 ? ta : 1);
            gi_ = d == 3 ? (int)(active ? ta + 1 : ta) : 0;  // 1-D / 2-D: grad_input reads the same grad plane
        }
        if (xs) { *xs = x_; *gvs = gv_; *gis = gi_; }
        return x_ * slab_x + (gv_ + gi_) * slab_g;
    };
    // defaults from the B200 sweeps (tools/tune.py cfg2 / cfg3r / cfg4r): few, large stages -- the
    // per-stage hand-off is what limits these kernels, not the bytes in flight
    int stages = t.stages > 0 ? t.stages : (mode == 2 ? 2 : 3);
    long long TA = IA;
    long long stage_kb = mode == 2 ? 108 : 72;
    // 1-D interpolating forward (flat row loop): tools/knob_sweep.py cfg2 / cfg2h -- fp32 173 us with 2 x 64 KB (187 with the
    // general default), 16-bit 90 us with 4 x 32 KB (97)
    if (mode == 1 && d == 1) {
        if (t.stages <= 0) stages = esize == 4 ? 2 : 4;
        stage_kb = esize == 4 ? 64 : 32;
    }
    const long long stage_target = (long long)(t.stage_kb > 0 ? t.stage_kb : stage_kb) * 1024;
    // shrink the slab tile until it meets the stage target (or is a single slab) and double-buffers
    for (;;) {
        const long long need = round_up(slots(TA, nullptr, nullptr, nullptr) + 2 * GUARD, 128);
        if (need * 2 + 64 <= budget && (need <= stage_target * 2 || TA == 1)) break;
        if (TA > 1) TA = (TA + 1) / 2;
        else return p;                                        // not even one slab (+ neighbours) double-buffers: generic family
    }
    const int tiles = a.tiles = (int)((IA + TA - 1) / TA);
    a.TA = (int)TA;
    const long long per_image = slots(TA, &a.xs, &a.gvs, &a.gis);
    a.img_stride = g.C * (mode == 2 ? g.in_plane : g.out_plane) * esize;
    long long np = 1;
    if (tiles == 1) {
        np = stage_target / per_image;
        if (np < 1) np = 1;
        if (np > g.N) np = g.N;
        while (np > 1 && np * a.img_stride >= 0x7fffffffLL) --np;      // 32-bit offsets inside a stage's destination
    }
    auto stride_of = [&](long long n) { return round_up(n * per_image + 2 * GUARD, 128); };
    for (;;) {
        if (stages * stride_of(np) + 16 * stages + 64 <= budget) break;
        if (np > 1) --np;
        else if (stages > 2) --stages;
        else return p;
    }
    if (np * per_image >= (1 << 20)) return p;                // mbarrier tx-count range
    a.np = (int)np;
    a.stages = stages;
    a.stage_stride = (int)stride_of(np);
    a.off_gv = (int)(np * a.xs * slab_x);
    a.off_gi = (int)(np * a.xs * slab_x + np * a.gvs * slab_g);

    const int GP = a.GP = padded_groups((int)((mode == 2 ? Lb : OLb) / vb));
    const long long img_items = TA * IB * GP;
    if (np * img_items >= 0x7fffffffLL) return p;
    if ((long long)a.xs * slab_x * np >= 0x7fffffffLL) return p;
    a.img_items = (int)img_items;

    const long long planes = g.N * g.C;
    const long long grid_max = (long long)sm_count * ctas;
    // images per unit: the per-unit setup (shift split, interior box, magic divisors) is amortised over
    // >= 4 stages while every CTA still gets >= 8 units
    long long npu = t.chunk_planes > 0 ? t.chunk_planes : planes / (grid_max * 32);
    if (t.chunk_planes <= 0) {
        if (npu < 4 * np) npu = 4 * np;
        while (npu > np && ((g.N + npu - 1) / npu) * g.C < 8 * grid_max) npu -= np;
    }
    int warps = t.warps;
    const int max_warps = ((mode == 0 ? MAXT_GATHER : MAXT_ARITH) / 32) / ctas - 1;
    if (warps > max_warps) warps = max_warps;
    const UnitPlan up = plan_units(np, npu, g.N, g.C, grid_max, warps);
    if (!up.ok) return p;
    a.nw = warps;
    a.n_per_unit = up.n_per_unit;
    a.units = up.units;
    a.chunks = up.chunks;
    a.unit_order = t.unit_order;
    a.table = table_bytes != 0;
    a.d_img = make_fastdiv((unsigned)a.img_items);
    a.d_GP = make_fastdiv((unsigned)GP);
    a.d_IB = make_fastdiv((unsigned)IB);

    p.ok = true;
    p.grid = up.grid;
    p.slots = up.slots;
    p.smem_bytes = (size_t)(stages * stride_of(np) + 16 * stages + 64 + table_bytes);
    return p;
}

// ---- launchers ----------------------------------------------------------------------------------
int staged_gather(const Geo& g, const StagedPlan& p, int wk, const void* x, void* y, unsigned long long fill, int esize,
                  const void* w, int qkind, long long wzp, cudaStream_t s) {
    SArgs a = p.a;
    a.x = (const unsigned char*)x;
    a.out = (unsigned char*)y;
    a.w = w;
    a.wk = wk;
    a.qkind = qkind;
    a.wzp = wzp;
    a.fill = fill;
    const int G = a.VB / 4;
#define TS_GATHER(GG, EE) if (G == GG && esize == EE) return launch(k_staged_gather<GG, EE>, a, p, s);
    TS_GATHER(4, 1) TS_GATHER(2, 1) TS_GATHER(1, 1)
    TS_GATHER(4, 2) TS_GATHER(2, 2) TS_GATHER(1, 2)
    TS_GATHER(4, 4) TS_GATHER(2, 4) TS_GATHER(1, 4)
    TS_GATHER(4, 8) TS_GATHER(2, 8)
#undef TS_GATHER
    return TS_ERR_UNSUPPORTED;
}

template <typename ST>
static int active_forward_t(const Geo& g, const SArgs& a, const StagedPlan& p, cudaStream_t s) {
    switch (g.dim) {
    case 1: return launch(k_staged_active_forward<ST, 1>, a, p, s);
    case 2: return launch(k_staged_active_forward<ST, 2>, a, p, s);
    default: return launch(k_staged_active_forward<ST, 3>, a, p, s);
    }
}

int staged_active_forward(const Geo& g, const StagedPlan& p, int dtype, const void* x, const void* w, void* y, cudaStream_t s) {
    SArgs a = p.a;
    a.x = (const unsigned char*)x;
    a.out = (unsigned char*)y;
    a.w = w;
    a.wk = dtype == TS_F32 || g.wf32 ? WK_F32 : dtype == TS_F16 ? WK_F16 : WK_BF16;
    switch (dtype) {
    case TS_F32: return active_forward_t<float>(g, a, p, s);
    case TS_F16: return active_forward_t<__half>(g, a, p, s);
    default: return active_forward_t<__nv_bfloat16>(g, a, p, s);
    }
}

template <typename ST>
static int backward_t(const Geo& g, const SArgs& a, const StagedPlan& p, int active, cudaStream_t s) {
    switch (g.dim * 2 + (active ? 1 : 0)) {
    case 2: return launch(k_staged_backward<ST, 1, false>, a, p, s);
    case 3: return launch(k_staged_backward<ST, 1, true>, a, p, s);
    case 4: return launch(k_staged_backward<ST, 2, false>, a, p, s);
    case 5: return launch(k_staged_backward<ST, 2, true>, a, p, s);
    case 6: return launch(k_staged_backward<ST, 3, false>, a, p, s);
    default: return launch(k_staged_backward<ST, 3, true>, a, p, s);
    }
}

int staged_backward(const Geo& g, const StagedPlan& p, int dtype, int active, const void* grad, const void* x, const void* w,
                    void* gi, double* partials, cudaStream_t s) {
    SArgs a = p.a;
    a.x = (const unsigned char*)x;
    a.grad = (const unsigned char*)grad;
    a.out = (unsigned char*)gi;
    a.w = w;
    a.wk = dtype == TS_F32 || g.wf32 ? WK_F32 : dtype == TS_F16 ? WK_F16 : WK_BF16;
    a.partials = partials;
    switch (dtype) {
    case TS_F32: return backward_t<float>(g, a, p, active, s);
    case TS_F16: return backward_t<__half>(g, a, p, active, s);
    default: return backward_t<__nv_bfloat16>(g, a, p, active, s);
    }
}

}  // namespace ts

// ts_halo.cu -- the fp32 arithmetic kernels (active forward, backward) for EVERY padding mode and border crop on
// 2-D planes and 3-D volumes: whole slabs are staged in shared memory WITH a halo, the halo is filled according to
// the padding rule, and after that every item is an interior item -- no index remapping, no validity masks, no
// edge pass in the arithmetic loop.
//
// Layout of a staged slab ("tile"): (hr + rows + hr) x pitch fp32, the slab's rows at [hr, hr + rows), its columns at
// [hc, hc + cols).  ONE TMA tensor load (cp.async.bulk.tensor.5d, box {pitch, hr + rows + hr, 1, 1, 1} at coordinates
// (-hc, -hr, slab, c, n)) delivers it: the copy engine lays the rows out at the padded pitch and fills everything
// outside the tensor with zeros -- which IS the halo under zeros padding.  For border / periodic / reflect /
// symmetric the consumer warps overwrite the halo cells the unit's shift can reach with tile[P(r)][P(c)]
// (reference index remap, ops/kernels/shifts_kernels.h:10-29; ~3 % of the cells for |shift| <= 1) and meet at a
// named barrier; the slab axis of 3-D volumes is resolved by the PRODUCER, which loads slab P(a - s) into the stage
// of iteration a (a slab coordinate outside the tensor makes the copy engine deliver a zero tile).
//
// 3-D volumes stream slab by slab through the ring: stage k of an image holds source slab k of x and of grad (plus
// the unshifted grad slab k-1); a thread owns one (row pair, 16-byte column group) of the slab for the whole image,
// keeps the windows of slab k-1 in REGISTERS and combines them with the windows of slab k: every slab is fetched
// from L2/HBM once (the round-1 kernels re-read the +1 neighbour slab per tile) and read from shared memory once.
// The trilinear arithmetic is evaluated separably per column of the 5-wide window (slab lerp, row lerp, then the
// column lerp between adjacent columns): the reference's operations in the reference's order for forward /
// grad_input (bit-exact, unfused: ops/kernels/interpolation.h:3-38), an FMA form for the tolerance-checked
// grad_weight factors (interpolation.h:9-61, shifts_kernels.h:132-154).
//
// A channel whose shift reaches beyond the halo (|shift| > hr/hc, default 4) is served by an element-wise routine
// inside the same kernel (global loads with the literal remap): always correct, fast for the shifts layers learn.
//
// CTA = nw consumer warps + 1 producer warp, persistent, one per SM; unit = (channel, chunk of images); grad_weight
// partials per (chunk, warp) in fp64, fixed shuffle tree, pass 2 in ts_generic.cu -> deterministic, no atomics.
#include <cuda.h>

#include <cstring>

#include "ts_kernels.h"
#include "ts_ptx.cuh"

namespace ts {

namespace {

using namespace ptx;

constexpr int MAXT = 512;
constexpr int GUARD = 128;          // readable slack before / after the tiles of a stage (window pairs may start 16 bytes early)

struct UnitShift {
    int sx[3], sg[3];      // per level; absent levels 0
    float d[3];            // per TENSOR axis
};

TS_D UnitShift compute_unit_shift(const HArgs& a, long long c) {
    UnitShift u;
    u.d[0] = u.d[1] = u.d[2] = 0.f;
#pragma unroll
    for (int lev = 0; lev < 3; ++lev) {
        const int ax = level_axis(lev, a.dim);
        u.sx[lev] = u.sg[lev] = 0;
        if (ax < 0) continue;
        long long iw;
        float d;
        const float wv = a.w[c * a.dim + ax];
        if (a.mode != 2) split_forward<float>(wv, a.mode == 1, iw, d);
        else split_backward<float>(wv, a.active != 0, iw, d);
        u.d[ax] = d;
        u.sx[lev] = reduce_shift(iw, a.g.S[ax], a.g.pad);
        u.sg[lev] = reduce_shift(iw, a.g.OS[ax], a.g.pad);
    }
    return u;
}

// computed once per CTA into shared memory (a few hundred dependent instructions per channel otherwise paid per unit by
// the single producer thread); a unit then costs one 36-byte read
TS_D UnitShift unit_shift(const HArgs& a, const UnitShift* tbl, long long c) { return a.table ? tbl[c] : compute_unit_shift(a, c); }

// Where a unit's windows sit inside the tiles, and whether they fit the halo.
struct UnitGeom {
    int xr0, xc0;          // tile row / column of the x window of iteration (row 0, column 0)
    int gr0, gc0;          // same for the grad window that feeds grad_input (backward)
    int vr0, vc0;          // same for the unshifted grad window (2-D: inside the grad tile; 3-D: inside the dense tile)
    bool fits;
};

TS_D UnitGeom unit_geom(const HArgs& a, const UnitShift& us) {
    UnitGeom u;
    const bool bwd = a.mode == 2;
    u.xr0 = (bwd ? 0 : a.lbB) - us.sx[1] + a.hr;
    u.xc0 = (bwd ? 0 : a.lbL) - us.sx[2] + a.hc;
    // rows r .. r+1 for r in [0, IB), columns xc0 .. xc0 + 4*IG (the +1 neighbour of the last element)
    bool ok = u.xr0 >= 0 && u.xr0 + a.IB <= a.bpx - 1 && u.xc0 >= 0 && u.xc0 + 4 * a.IG <= a.px - 1;
    u.gr0 = u.gc0 = u.vr0 = u.vc0 = 0;
    if (bwd) {
        const int sgr = a.active ? -us.sg[1] : us.sg[1], sgc = a.active ? -us.sg[2] : us.sg[2];
        const int ex = a.active ? 1 : 0;
        u.gr0 = -a.lbB + sgr + a.hr;          // + input row b
        u.gc0 = -a.lbL + sgc + a.hc;          // + input column
        // only rows / columns inside the crop read the tile: ob in [0, OB), oj in [0, OL)
        ok = ok && sgr + a.hr >= 0 && a.OB - 1 + sgr + a.hr + ex <= a.bpg - 1 && sgc + a.hc >= 0 && a.OL - 1 + sgc + a.hc + ex <= a.pg - 1;
        if (a.dim == 3) { u.vr0 = -a.lbB; u.vc0 = -a.lbL; }
        else { u.vr0 = -a.lbB + a.hr; u.vc0 = -a.lbL + a.hc; }
    }
    u.fits = ok;
    return u;
}

// ---- units ordered by window-misalignment class -------------------------------------------------
// The misalignment of a unit's windows inside their 16-byte groups (0..3 words) is a property of the CHANNEL.  A body
// with compile-time misalignment is free of select instructions (12 FSEL per 5-wide window otherwise, 72 per slab step
// of the 3-D backward), but a switch over four inlined bodies per image group made ptxas spill.  So every CTA sorts the
// channels by class once (class k < 4: every window's misalignment follows from the x window's = k; class 4: crops that
// untie the windows, or a shift beyond the halo) and the persistent loop walks the units CLASS BY CLASS: one body per
// class, each with its own unit loop, run one after the other -- nothing is live across them but the ring position.
constexpr int NCLS = 5;
TS_D int classify(const HArgs& a, const UnitShift& us) {
    const UnitGeom ug = unit_geom(a, us);
    if (!ug.fits) return 4;
    const int wsx = ug.xc0 & 3;
    if (a.mode == 2 && !((ug.vc0 & 3) == 0 && (ug.gc0 & 3) == (a.active ? wsx : ((4 - wsx) & 3)))) return 4;
    return wsx;
}
struct UnitOrder {
    const unsigned short* order;     // channels sorted by class (nullptr: identity, everything in class 4)
    const int* cend;                 // cend[k] = units in classes 0..k
    const int* coff;                 // coff[k] = channels in classes 0..k-1
    int chunks, C;
    // u is monotonic per caller: k only moves forward
    TS_D void decode(int u, int& k, int& c, int& chunk, int unit_order) const {
        while (u >= cend[k]) ++k;
        const int base = k ? cend[k - 1] : 0, cnt = coff[k + 1] - coff[k], v = u - base;
        int j;
        if (unit_order) { chunk = v / cnt; j = v - chunk * cnt; }
        else { j = v / chunks; chunk = v - j * chunks; }
        c = order ? (int)order[coff[k] + j] : j;
    }
};

// ---- window loads -----------------------------------------------------------------------------
// 5 (or 4) consecutive fp32 starting `ws` words into the aligned 16-byte group at shared address `addr`.
// WS >= 0: compile-time misalignment (free register renaming); WS = -1: run-time, a two-level select network.
template <int WS>
TS_D void load5(unsigned addr, int ws, float* out) {
    const uint4 A = lds128(addr), B = lds128(addr + 16);
    const float W[8] = {__uint_as_float(A.x), __uint_as_float(A.y), __uint_as_float(A.z), __uint_as_float(A.w),
                        __uint_as_float(B.x), __uint_as_float(B.y), __uint_as_float(B.z), __uint_as_float(B.w)};
    if constexpr (WS >= 0) {
#pragma unroll
        for (int t = 0; t < 5; ++t) out[t] = W[t + WS];
    } else {
        float U[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) U[i] = (ws & 1) ? W[i + 1] : W[i];
#pragma unroll
        for (int t = 0; t < 5; ++t) out[t] = (ws & 2) ? U[t + 2] : U[t];
    }
}
template <int WS>
TS_D void load4(unsigned addr, int ws, float* out) {
    if (WS == 0 || (WS < 0 && ws == 0)) {         // (run-time: the unshifted grad window is aligned unless the crop is not)
        const uint4 A = lds128(addr);
        out[0] = __uint_as_float(A.x); out[1] = __uint_as_float(A.y); out[2] = __uint_as_float(A.z); out[3] = __uint_as_float(A.w);
    } else {
        float t5[5];
        load5<WS>(addr, ws, t5);
#pragma unroll
        for (int t = 0; t < 4; ++t) out[t] = t5[t];
    }
}

// ---- halo fill --------------------------------------------------------------------------------
// Cells of the needed extended range [rn_lo, rn_hi] x [cn_lo, cn_hi] that lie outside [0, rows) x [0, cols) take
// tile[P(r)][P(c)].  Writers touch halo cells only, readers interior cells only: one pass, no ordering inside.
// The (destination, source) word offsets are the same for every stage of a work unit, so the fixer warp lists them
// ONCE per unit in shared memory (16 + 16 bits per cell) and a stage costs one list read, one LDS and one STS per cell.
TS_D int remap_any(int idx, int len, int pad, bool bounded) { return bounded ? axis_index(idx, len, pad) : axis_index_literal(idx, len, pad); }

constexpr int FIXCAP = 1536;       // cells per tile list; a unit that needs more is patched without a list

struct HaloRange { int rn_lo, rn_hi, cn_lo, cn_hi; };

TS_D int halo_cells(const HaloRange& h, int rows, int cols) {
    const int nr = (h.rn_lo < 0 ? -h.rn_lo : 0) + (h.rn_hi > rows - 1 ? h.rn_hi - (rows - 1) : 0);
    const int nc = (h.cn_lo < 0 ? -h.cn_lo : 0) + (h.cn_hi > cols - 1 ? h.cn_hi - (cols - 1) : 0);
    return nr * (h.cn_hi - h.cn_lo + 1) + rows * nc;
}

// list != nullptr: write the cell list (entry = dst | src << 16, word offsets inside the tile); else copy in `tile`
TS_D void halo_walk(unsigned* list, float* tile, int pitch, int rows, int cols, int hr, int hc, int pad, const HaloRange& h, int lane) {
    const int nrt = h.rn_lo < 0 ? -h.rn_lo : 0, nrb = h.rn_hi > rows - 1 ? h.rn_hi - (rows - 1) : 0;
    const int nct = h.cn_lo < 0 ? -h.cn_lo : 0, ncb = h.cn_hi > cols - 1 ? h.cn_hi - (cols - 1) : 0;
    const int wc = h.cn_hi - h.cn_lo + 1;
    // the division-free remap is valid for indices within one period of the axis: halo <= hr (hc) < len
    const bool rb = rows > hr + 1, cb = cols > hc + 1;
    for (int ri = 0; ri < nrt + nrb; ++ri) {
        const int r = ri < nrt ? h.rn_lo + ri : rows + (ri - nrt);
        const int sr = remap_any(r, rows, pad, rb);
        for (int c = h.cn_lo + lane; c <= h.cn_hi; c += 32) {
            const unsigned dst = (unsigned)((r + hr) * pitch + c + hc), src = (unsigned)((sr + hr) * pitch + remap_any(c, cols, pad, cb) + hc);
            if (list) list[ri * wc + (c - h.cn_lo)] = dst | (src << 16); else tile[dst] = tile[src];
        }
    }
    const int nA = (nrt + nrb) * wc;
    for (int k = 0; k < nct + ncb; ++k) {
        const int c = k < nct ? h.cn_lo + k : cols + (k - nct);
        const int sc = remap_any(c, cols, pad, cb);
        for (int r = lane; r < rows; r += 32) {
            const unsigned dst = (unsigned)((r + hr) * pitch + c + hc), src = (unsigned)((r + hr) * pitch + sc + hc);
            if (list) list[nA + k * rows + r] = dst | (src << 16); else tile[dst] = tile[src];
        }
    }
}


// pooled-gradient kernels: the same walk, with a mode that CLEARS the cells (zeros padding of a tile that was written by
// pool_expand, not by the copy engine)
TS_D void halo_walk_z(unsigned* list, float* tile, int pitch, int rows, int cols, int hr, int hc, int pad, const HaloRange& h, int lane,
                    bool zero = false) {
    const int nrt = h.rn_lo < 0 ? -h.rn_lo : 0, nrb = h.rn_hi > rows - 1 ? h.rn_hi - (rows - 1) : 0;
    const int nct = h.cn_lo < 0 ? -h.cn_lo : 0, ncb = h.cn_hi > cols - 1 ? h.cn_hi - (cols - 1) : 0;
    const int wc = h.cn_hi - h.cn_lo + 1;
    // the division-free remap is valid for indices within one period of the axis: halo <= hr (hc) < len
    const bool rb = rows > hr + 1, cb = cols > hc + 1;
    for (int ri = 0; ri < nrt + nrb; ++ri) {
        const int r = ri < nrt ? h.rn_lo + ri : rows + (ri - nrt);
        const int sr = remap_any(r, rows, pad, rb);
        for (int c = h.cn_lo + lane; c <= h.cn_hi; c += 32) {
            const unsigned dst = (unsigned)((r + hr) * pitch + c + hc);
            const unsigned src = zero ? dst : (unsigned)((sr + hr) * pitch + remap_any(c, cols, pad, cb) + hc);
            if (list) list[ri * wc + (c - h.cn_lo)] = dst | (src << 16); else tile[dst] = zero ? 0.f : tile[src];
        }
    }
    const int nA = (nrt + nrb) * wc;
    for (int k = 0; k < nct + ncb; ++k) {
        const int c = k < nct ? h.cn_lo + k : cols + (k - nct);
        const int sc = remap_any(c, cols, pad, cb);
        for (int r = lane; r < rows; r += 32) {
            const unsigned dst = (unsigned)((r + hr) * pitch + c + hc), src = zero ? dst : (unsigned)((r + hr) * pitch + sc + hc);
            if (list) list[nA + k * rows + r] = dst | (src << 16); else tile[dst] = zero ? 0.f : tile[src];
        }
    }
}

// ZERO: the listed cells are cleared (zeros padding of a tile the copy engine did not fill)
TS_D void halo_apply(const unsigned* list, int n, float* tile, int lane) {
    // four independent cells in flight per lane in EVERY pass: indices past the end repeat the last cell (the same copy
    // twice is harmless), so a tile costs ceil(n / 128) dependent list -> load -> store round trips, not one per 32 cells
    for (int e = lane; e < n; e += 128) {
        const int last = n - 1;
        const unsigned e0 = list[e], e1 = list[min(e + 32, last)], e2 = list[min(e + 64, last)], e3 = list[min(e + 96, last)];
        const float v0 = tile[e0 >> 16], v1 = tile[e1 >> 16], v2 = tile[e2 >> 16], v3 = tile[e3 >> 16];
        tile[e0 & 0xffffu] = v0; tile[e1 & 0xffffu] = v1; tile[e2 & 0xffffu] = v2; tile[e3 & 0xffffu] = v3;
    }
}


// pooled-gradient kernels: the cells of a list dealt to `stride` threads (several fixer warps); ZERO clears them
template <bool ZERO>
TS_D void halo_apply_m(const unsigned* list, int n, float* tile, int lane, const int stride = 32) {
    // four independent cells in flight per lane in EVERY pass: indices past the end repeat the last cell (the same copy
    // twice is harmless), so a tile costs ceil(n / 128) dependent list -> load -> store round trips, not one per 32 cells
    // (lane: index among the `stride` threads that share the list)
    for (int e = lane; e < n; e += 4 * stride) {
        const int last = n - 1;
        const unsigned e0 = list[e], e1 = list[min(e + stride, last)], e2 = list[min(e + 2 * stride, last)], e3 = list[min(e + 3 * stride, last)];
        const float v0 = ZERO ? 0.f : tile[e0 >> 16], v1 = ZERO ? 0.f : tile[e1 >> 16], v2 = ZERO ? 0.f : tile[e2 >> 16],
                    v3 = ZERO ? 0.f : tile[e3 >> 16];
        tile[e0 & 0xffffu] = v0; tile[e1 & 0xffffu] = v1; tile[e2 & 0xffffu] = v2; tile[e3 & 0xffffu] = v3;
    }
}

// Adjoint of avg_pool2d(kernel 2, stride 2, ceil_mode=True) while staging: every element of a pooling window receives the
// pooled gradient divided by the window's element count (ATen's avg_pool2d_backward: 4, or 2 for the last row of an odd
// height; /4 and /2 are exact as multiplications).  pooled: dense [PH][PW]; tile: the grad tile, data at (hr, hc).
TS_D void sts64(unsigned addr, float a, float b) { asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory"); }
TS_D void pool_expand(const float* pooled, float* tile, int PH, int PW, int OB, int pitch, int hr, int hc, int lane, int stride,
                      const FastDiv& dPW) {
    // A few warps expand a plane between the copy engine and the arithmetic warps, so they must not crawl: shared-window
    // addresses (no generic stores), a flat index over the pooled cells, four independent cells in flight per thread
    // (lane: index among the `stride` expanding threads)
    const unsigned src = shared_addr(pooled), dst = shared_addr(tile) + (unsigned)((hr * pitch + hc) * 4);
    const int n = PH * PW, pb = pitch * 4;
    for (int p0 = lane; p0 < n; p0 += 4 * stride) {
        float v[4];
        unsigned o[4];
        bool two[4], on[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int p = p0 + stride * i;
            on[i] = p < n;
            const int q = on[i] ? p : 0;
            const int pr = (int)fdiv((unsigned)q, dPW), pc = q - pr * PW;
            two[i] = 2 * pr + 1 < OB;
            o[i] = dst + (unsigned)(2 * pr * pb + 8 * pc);
            v[i] = __uint_as_float(lds32(src + 4u * (unsigned)q)) * (two[i] ? 0.25f : 0.5f);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (!on[i]) continue;
            sts64(o[i], v[i], v[i]);
            if (two[i]) sts64(o[i] + (unsigned)pb, v[i], v[i]);
        }
    }
}

// ---- arithmetic -------------------------------------------------------------------------------
// exact (unfused) column values of the reference's interpolation nest: rows / slabs first, columns last.
// 3-D: V00 (slab a, row r), V10 (slab a+1, row r), V01 (slab a, row r+1), V11 (slab a+1, row r+1)
TS_D float col3(float v00, float v10, float v01, float v11, float d0, float d1) {
    return lerp<float>(lerp<float>(v00, v10, d0), lerp<float>(v01, v11, d0), d1);
}

// grad_weight terms of one item, 3-D, FMA form (tolerance-checked): windows of x over 5 columns, gv over 4
TS_D void wp3(const float* x00, const float* x10, const float* x01, const float* x11, const float* gv, const float* d, float* ts) {
    float hv[5], kv[5];
    const float omd2 = 1.f - d[2];
    hv[0] = omd2 * gv[0]; kv[0] = -gv[0];
#pragma unroll
    for (int c = 1; c < 4; ++c) { hv[c] = fmaf(d[2], gv[c - 1], omd2 * gv[c]); kv[c] = gv[c - 1] - gv[c]; }
    hv[4] = d[2] * gv[3]; kv[4] = gv[3];
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        const float a0 = fmaf(d[0], x10[c] - x00[c], x00[c]), a1 = fmaf(d[0], x11[c] - x01[c], x01[c]);
        const float g1c = a1 - a0, pc = fmaf(d[1], g1c, a0);
        const float e0 = x01[c] - x00[c], e1 = x11[c] - x10[c];
        const float g0c = fmaf(d[1], e1 - e0, e0);
        ts[0] = fmaf(g0c, hv[c], ts[0]);
        ts[1] = fmaf(g1c, hv[c], ts[1]);
        ts[2] = fmaf(pc, kv[c], ts[2]);
    }
}
// 2-D: x0 (row r), x1 (row r+1)
TS_D void wp2(const float* x0, const float* x1, const float* gv, const float* d, float* ts) {
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const float p = x0[t + 1] - x0[t], q = (x1[t + 1] - x1[t]) - p;
        ts[0] = fmaf(gv[t], fmaf(d[1], q, p), ts[0]);
        ts[1] = fmaf(gv[t], fmaf(d[0], q, p), ts[1]);
    }
}

// ---- element-wise routine for channels whose shift does not fit the halo ------------------------
// (global loads, literal remap; mirrors ts_generic.cu.  All consumer threads of the CTA share the unit.)
template <int DIM, class Load>
TS_D void fetch8f(Load ld, const int* idx, const int* sizes, int pad, float* v) {
    int t[DIM][2];
#pragma unroll
    for (int ax = 0; ax < DIM; ++ax) {
        t[ax][0] = axis_index_literal(idx[ax], sizes[ax], pad);
        t[ax][1] = axis_index_literal(idx[ax] + 1, sizes[ax], pad);
    }
#pragma unroll
    for (int q = 0; q < (1 << DIM); ++q) {
        bool ok = true;
        long long off = 0;
#pragma unroll
        for (int ax = 0; ax < DIM; ++ax) {
            const int i = t[ax][(q >> ax) & 1];
            ok = ok && i >= 0;
            off = off * sizes[ax] + i;
        }
        v[q] = ok ? ld(off) : 0.f;
    }
}
template <int DIM>
TS_D void fetch8(const float* __restrict__ vol, const int* idx, const int* sizes, int pad, float* v) {
    fetch8f<DIM>([vol](long long off) { return vol[off]; }, idx, sizes, pad, v);
}

template <int DIM, bool ACTIVE>
TS_D float slow_forward_value(const Geo& g, const float* xp, const int* o, const int* sx, const float* d) {
    int idx[DIM];
#pragma unroll
    for (int ax = 0; ax < DIM; ++ax) idx[ax] = o[ax] + g.lb[ax] - sx[ax];
    if (ACTIVE) {
        float v[8];
        fetch8<DIM>(xp, idx, g.S, g.pad, v);
        return interpolate<float, DIM>(v, d);
    }
    bool ok = true;
    long long off = 0;
#pragma unroll
    for (int ax = 0; ax < DIM; ++ax) {
        const int t = axis_index_literal(idx[ax], g.S[ax], g.pad);
        ok = ok && t >= 0;
        off = off * g.S[ax] + t;
    }
    return ok ? xp[off] : 0.f;
}

template <int DIM, bool ACTIVE, bool POOL>
TS_D void slow_forward(const HArgs& a, int c, int n0, int n1, const UnitShift& us, int tid, int nt) {
    const Geo& g = a.g;
    int sx[DIM];
    float d[3] = {us.d[0], us.d[1], us.d[2]};
#pragma unroll
    for (int ax = 0; ax < DIM; ++ax) sx[ax] = us.sx[ax + 3 - DIM];
    for (int n = n0; n < n1; ++n) {
        const float* xp = a.x + ((long long)n * g.C + c) * g.in_plane;
        float* yp = (float*)((unsigned char*)a.out + ((long long)n * g.C + c) * a.out_plane_bytes);
        if (POOL && DIM == 2) {
            const int PH = (g.OS[0] + 1) / 2, PW = g.OS[1] / 2;
            for (int e = tid; e < PH * PW; e += nt) {
                const int ph = e / PW, pw = e - ph * PW;
                float sum = 0.f;
                int cnt = 0;
                for (int i = 0; i < 2; ++i)
                    for (int j = 0; j < 2; ++j) {
                        int o[DIM];
                        o[0] = 2 * ph + i; o[DIM - 1] = 2 * pw + j;
                        if (o[0] >= g.OS[0]) continue;
                        const float v = slow_forward_value<DIM, ACTIVE>(g, xp, o, sx, d);
                        sum = cnt ? __fadd_rn(sum, v) : v;
                        ++cnt;
                    }
                yp[e] = __fdiv_rn(sum, (float)cnt);
            }
        } else if constexpr (POOL && DIM == 3) {
            // avg_pool3d(kernel = stride = (sA, 2, 2), ceil_mode): one running sum in (slab, row, column) order, as ATen's kernel
            const int PH = a.PH, PW = a.PW, sA = a.sA;
            for (int e = tid; e < a.PA * PH * PW; e += nt) {
                const int pa = e / (PH * PW), rem = e - pa * (PH * PW), ph = rem / PW, pw = rem - ph * PW;
                float sum = 0.f;
                int cnt = 0;
                for (int s = 0; s < sA; ++s)
                    for (int i = 0; i < 2; ++i)
                        for (int j = 0; j < 2; ++j) {
                            const int o[3] = {sA * pa + s, 2 * ph + i, 2 * pw + j};
                            if (o[0] >= g.OS[0] || o[1] >= g.OS[1]) continue;
                            const float v = slow_forward_value<DIM, ACTIVE>(g, xp, o, sx, d);
                            sum = cnt ? __fadd_rn(sum, v) : v;
                            ++cnt;
                        }
                yp[e] = __fdiv_rn(sum, (float)cnt);
            }
        } else {
            const int plane = (int)g.out_plane;
            for (int e = tid; e < plane; e += nt) {
                int o[DIM], rem = e;
#pragma unroll
                for (int ax = DIM - 1; ax >= 0; --ax) { o[ax] = rem % g.OS[ax]; rem /= g.OS[ax]; }
                yp[e] = slow_forward_value<DIM, ACTIVE>(g, xp, o, sx, d);
            }
        }
    }
}

template <int DIM, bool ACTIVE, bool PBWD>
TS_D void slow_backward(const HArgs& a, int c, int n0, int n1, const UnitShift& us, int tid, int nt, double* acc) {
    const Geo& g = a.g;
    const int plane = (int)g.in_plane;
    int sx[DIM], sg[DIM];
    float d[3] = {us.d[0], us.d[1], us.d[2]};
#pragma unroll
    for (int ax = 0; ax < DIM; ++ax) { sx[ax] = us.sx[ax + 3 - DIM]; sg[ax] = us.sg[ax + 3 - DIM]; }
    constexpr bool pool = PBWD;                 // a.grad is the POOLED gradient, expanded on the fly
    const int PW = a.PW, OL = a.OL, OB = a.OB;
    for (int n = n0; n < n1; ++n) {
        const float* xp = a.x + ((long long)n * g.C + c) * g.in_plane;
        const float* gp = a.grad + ((long long)n * g.C + c) * (pool ? (DIM == 3 ? (long long)a.PA : 1ll) * a.PH * a.PW : g.out_plane);
        float* gip = a.out + ((long long)n * g.C + c) * g.in_plane;
        // gradient of the shift's output at linear offset `off` of the (cropped) output plane
        auto gld = [gp, PW, OL, OB](long long off) {
            if (!pool) return gp[off];
            const int r = (int)(off / OL), cc = (int)(off - (long long)r * OL), pr = r >> 1;
            return gp[pr * PW + (cc >> 1)] * (2 * pr + 1 < OB ? 0.25f : 0.5f);
        };
        // 3-D: grad / count of the (sA, 2, 2) window (a power of two: the product is the quotient)
        const int PH = a.PH, OA = a.OA, sA = a.sA;
        auto gld3 = [gp, PW, PH, OL, OB, OA, sA](long long off) {
            const int plane = OB * OL, o0 = (int)(off / plane), rem = (int)(off - (long long)o0 * plane), r = rem / OL, cc = rem - r * OL;
            const int pa = sA == 2 ? o0 >> 1 : o0, pr = r >> 1;
            const float f = (sA == 2 && 2 * pa + 1 < OA ? 0.5f : 1.f) * (2 * pr + 1 < OB ? 0.25f : 0.5f);
            return gp[((long long)pa * PH + pr) * PW + (cc >> 1)] * f;
        };
        auto gsel = [&](long long off) {
            if constexpr (pool && DIM == 3) return gld3(off);
            else return gld(off);
        };
        for (int e = tid; e < plane; e += nt) {
            int pos[DIM], rem = e, o[DIM];
#pragma unroll
            for (int ax = DIM - 1; ax >= 0; --ax) { pos[ax] = rem % g.S[ax]; rem /= g.S[ax]; }
            bool pass = true;
            long long goff = 0;
#pragma unroll
            for (int ax = 0; ax < DIM; ++ax) {
                o[ax] = pos[ax] - g.lb[ax];
                pass = pass && o[ax] >= 0 && o[ax] < g.OS[ax];
                goff = goff * g.OS[ax] + o[ax];
            }
            float r = 0.f;
            if (pass) {
                const float gv = gsel(goff);
                int idx[DIM];
#pragma unroll
                for (int ax = 0; ax < DIM; ++ax) idx[ax] = pos[ax] - sx[ax];
                float v[8], wg[3];
                fetch8<DIM>(xp, idx, g.S, g.pad, v);
                weight_partials<float, DIM>(v, d, wg);
#pragma unroll
                for (int ax = 0; ax < DIM; ++ax) acc[ax] += (double)(gv * wg[ax]);
                if (ACTIVE) {
#pragma unroll
                    for (int ax = 0; ax < DIM; ++ax) idx[ax] = o[ax] - sg[ax];
                    fetch8f<DIM>(gsel, idx, g.OS, g.pad, v);
                    r = interpolate<float, DIM>(v, d);
                } else {
                    bool in = true;
                    long long off = 0;
#pragma unroll
                    for (int ax = 0; ax < DIM; ++ax) {
                        const int t = axis_index_literal(o[ax] + sg[ax], g.OS[ax], g.pad);
                        in = in && t >= 0;
                        off = off * g.OS[ax] + t;
                    }
                    r = in ? gsel(off) : 0.f;
                }
            }
            gip[e] = r;
        }
    }
}

// ---- producer ---------------------------------------------------------------------------------
TS_D int slab_coord(int idx, int len, int pad) {
    // ONE thread evaluates this two or three times per stage: the literal remap (integer divisions, ~120 dependent
    // instructions for reflect) made the producer the slowest stage of the 3-D pipeline under periodic / reflect /
    // symmetric padding (measured: 0.66 ms against 0.56 ms with border padding).  Indices within one period of the axis --
    // everything a slab inside the crop can ask for after reduce_shift -- take the division-free form.
    const int P = remap_period(len, pad);
    const int t = (P == 0 || (idx > -P && idx < len + P)) ? axis_index(idx, len, pad) : axis_index_literal(idx, len, pad);
    return t < 0 ? -1 : t;                 // outside under zeros padding: the copy engine delivers a zero tile
}

// The whole producer WARP runs this.  The slab coordinates of a unit's steps depend on the channel only: lane k works them
// out for step k once per unit (one elected thread evaluating the remaps every stage was near the critical path of the 3-D
// pipeline: reflect / symmetric padding ran 8 % behind border padding for ~20 extra dependent instructions per stage), and the
// (up to three) tensor copies of an image are issued by three different lanes.
// POOL3 (3-D backward fused with avg_pool3d): both grad copies are slabs of the POOLED gradient, the one that feeds
// grad_input lands in the second dense tile of the image (after the a.np tiles at off_v) and the fixer warp expands it.
TS_D int pooled_slab(int s, int sA) { return s < 0 ? -1 : (sA == 2 ? s >> 1 : s); }

template <bool POOL3>
TS_D void producer(const HArgs& a, unsigned char* smem, uint64_t* full, uint64_t* empty, const UnitShift* tbl, const UnitOrder& uo, int lane) {
    int s = 0, kk = 0, cls = 0;
    const int N = (int)a.g.N;
    const bool bwd = a.mode == 2;
    const int steps = a.dim == 3 ? a.IA + 1 : 1;
    const UnitRange ur = unit_range(a.units, a.unit_order);
    for (int u = ur.u; u < ur.end; u += ur.step) {
        int chunk, c;
        uo.decode(u, cls, c, chunk, a.unit_order);
        const int n0 = chunk * a.n_per_unit;
        const int n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
        const UnitShift us = unit_shift(a, tbl, c);
        if (!unit_geom(a, us).fits) continue;              // consumers take the element-wise routine for this unit
        for (int nb = n0; nb < n1; nb += a.np) {
            const int npl = n1 - nb < a.np ? n1 - nb : a.np;
            int xs_l = 0, gs_l = 0, vs_l = 0;              // coordinates of step (k & ~31) + lane
            for (int k = 0; k < steps; ++k) {
                if (a.dim == 3 && (k & 31) == 0) {
                    const int kl = k + lane;
                    xs_l = slab_coord((bwd ? kl : kl + a.lbA) - us.sx[0], a.A, a.g.pad);
                    if (bwd) {
                        gs_l = a.active ? slab_coord(kl - a.lbA - us.sg[0], a.OA, a.g.pad) : slab_coord(kl - 1 - a.lbA + us.sg[0], a.OA, a.g.pad);
                        const int oa = kl - 1 - a.lbA;
                        vs_l = (oa >= 0 && oa < a.OA) ? oa : -1;
                        if constexpr (POOL3) { gs_l = pooled_slab(gs_l, a.sA); vs_l = pooled_slab(vs_l, a.sA); }
                    }
                }
                const int xs = __shfl_sync(0xffffffffu, xs_l, k & 31), gs = __shfl_sync(0xffffffffu, gs_l, k & 31),
                          vs = __shfl_sync(0xffffffffu, vs_l, k & 31);
                unsigned char* st = smem + (size_t)s * a.stage_stride + GUARD;
                const bool has_g = bwd && (a.dim == 2 || a.active || k >= 1);
                const bool has_v = bwd && a.dim == 3 && k >= 1;
                if (lane == 0) {
                    if (kk > 0) mbar_wait_parked(&empty[s], (unsigned)((kk - 1) & 1));
                    mbar_expect_tx(&full[s], (unsigned)npl * (unsigned)(a.box_x + (has_g ? (a.pool_bwd ? a.box_v : a.box_g) : 0) + (has_v ? a.box_v : 0)));
                }
                __syncwarp();                              // the slot is free and its byte count posted before any lane copies into it
                for (int job = lane; job < 3 * npl; job += 32) {
                    const int pl = job / 3, what = job - 3 * pl;
                    if (what == 0) tma_load_5d(st + (size_t)pl * a.tile_x, &a.map_x, -a.hc, -a.hr, xs, c, nb + pl, &full[s]);
                    else if (what == 1) {
                        if constexpr (POOL3) {
                            if (has_g) tma_load_5d(st + a.off_v + (size_t)(a.np + pl) * a.tile_v, &a.map_v, 0, 0, gs, c, nb + pl, &full[s]);
                        } else if (has_g && a.pool_bwd) tma_load_5d(st + a.off_v + (size_t)pl * a.tile_v, &a.map_v, 0, 0, 0, c, nb + pl, &full[s]);   // pooled grad, dense
                        else if (has_g) tma_load_5d(st + a.off_g + (size_t)pl * a.tile_g, &a.map_g, -a.hc, -a.hr, gs, c, nb + pl, &full[s]);
                    }
                    else if (has_v) tma_load_5d(st + a.off_v + (size_t)pl * a.tile_v, &a.map_v, 0, 0, vs, c, nb + pl, &full[s]);
                }
                if (++s == a.stages) { s = 0; ++kk; }
            }
        }
    }
}

// ---- fixer warp -------------------------------------------------------------------------------
// One warp fills the halo cells of every stage (paddings other than zeros) between the copy engine and the consumers:
// it waits for full[s], patches the tiles and arrives on ready[s]; the consumers wait for ready[s] instead of full[s].
// It runs ahead of the consumers by the ring depth, so the arithmetic warps never meet at a barrier.
TS_D void fixer(const HArgs& a, unsigned char* smem, uint64_t* full, uint64_t* ready, int lane, const UnitShift* tbl, unsigned* lists,
                const UnitOrder& uo) {
    int s = 0, cls = 0;
    unsigned phase = 0;
    const int N = (int)a.g.N;
    const bool bwd = a.mode == 2;
    const int steps = a.dim == 3 ? a.IA + 1 : 1;
    unsigned* list_x = lists;
    unsigned* list_g = lists + FIXCAP;
    const bool listable = a.px * a.bpx < 65536 && a.pg * a.bpg < 65536;
    const UnitRange ur = unit_range(a.units, a.unit_order);
    for (int u = ur.u; u < ur.end; u += ur.step) {
        int chunk, c;
        uo.decode(u, cls, c, chunk, a.unit_order);
        const int n0 = chunk * a.n_per_unit;
        const int n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
        const UnitShift us = unit_shift(a, tbl, c);
        if (!unit_geom(a, us).fits) continue;
        const int xr_lo = (bwd ? 0 : a.lbB) - us.sx[1], xc_lo = (bwd ? 0 : a.lbL) - us.sx[2];
        const int sgr = a.active ? -us.sg[1] : us.sg[1], sgc = a.active ? -us.sg[2] : us.sg[2], ex = a.active ? 1 : 0;
        const HaloRange hx = {xr_lo, xr_lo + a.IB, xc_lo, xc_lo + 4 * a.IG};
        const HaloRange hg = {sgr, a.OB - 1 + sgr + ex, sgc, a.OL - 1 + sgc + ex};
        const int nx = halo_cells(hx, a.B, a.L), ng = bwd ? halo_cells(hg, a.OB, a.OL) : 0;
        const bool use_list = listable && nx <= FIXCAP && ng <= FIXCAP;
        if (use_list) {
            __syncwarp();                       // every lane is done with the previous unit's lists
            halo_walk(list_x, nullptr, a.px, a.B, a.L, a.hr, a.hc, a.g.pad, hx, lane);
            if (bwd) halo_walk(list_g, nullptr, a.pg, a.OB, a.OL, a.hr, a.hc, a.g.pad, hg, lane);
            __syncwarp();
        }
        for (int nb = n0; nb < n1; nb += a.np) {
            const int npl = n1 - nb < a.np ? n1 - nb : a.np;
            for (int k = 0; k < steps; ++k) {
                unsigned char* st = smem + (size_t)s * a.stage_stride + GUARD;
                const bool has_g = bwd && (a.dim == 2 || a.active || k >= 1);
                mbar_wait_parked(&full[s], phase);
                for (int pl = 0; pl < npl; ++pl) {
                    float* tx = (float*)(st + (size_t)pl * a.tile_x);
                    float* tg = (float*)(st + a.off_g + (size_t)pl * a.tile_g);
                    if (use_list) {
                        halo_apply(list_x, nx, tx, lane);
                        if (has_g) halo_apply(list_g, ng, tg, lane);
                    } else {
                        halo_walk(nullptr, tx, a.px, a.B, a.L, a.hr, a.hc, a.g.pad, hx, lane);
                        if (has_g) halo_walk(nullptr, tg, a.pg, a.OB, a.OL, a.hr, a.hc, a.g.pad, hg, lane);
                    }
                }
                fence_proxy_async();             // the next TMA load of this stage must not overtake these generic-proxy writes
                __syncwarp();
                if (lane == 0) mbar_arrive(&ready[s]);
                if (++s == a.stages) { s = 0; phase ^= 1u; }
            }
        }
    }
}


// MULTI: several fixer warps (the pooled-gradient expansion); the single-warp instantiation keeps compile-time strides
// (with run-time ones the forward of cfg4 lost 20 %: that kernel runs at the pace of its fixer warp).
template <bool MULTI>
TS_D void fixer_pool(const HArgs& a, unsigned char* smem, uint64_t* full, uint64_t* ready, int lane, int fw, const UnitShift* tbl, unsigned* lists,
                const UnitOrder& uo) {
    // fw: index of this warp among the a.nfix fixer warps (1, or 4 when the pooled gradient is expanded here: they split
    // the cells of every tile and meet at a named barrier between the expansion and the halo copies that read it)
    int s = 0, cls = 0;
    unsigned phase = 0;
    const int N = (int)a.g.N;
    const bool bwd = a.mode == 2;
    const int steps = a.dim == 3 ? a.IA + 1 : 1;
    const int nf = MULTI ? a.nfix : 1, fl = MULTI ? fw * 32 + lane : lane, fstride = MULTI ? 32 * nf : 32;
    auto fsync = [nf]() { if (MULTI) named_barrier(1, 32 * nf); else __syncwarp(); };
    unsigned* list_x = lists;
    unsigned* list_g = lists + FIXCAP;
    const bool listable = a.px * a.bpx < 65536 && a.pg * a.bpg < 65536;
    const UnitRange ur = unit_range(a.units, a.unit_order);
    for (int u = ur.u; u < ur.end; u += ur.step) {
        int chunk, c;
        uo.decode(u, cls, c, chunk, a.unit_order);
        const int n0 = chunk * a.n_per_unit;
        const int n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
        const UnitShift us = unit_shift(a, tbl, c);
        if (!unit_geom(a, us).fits) continue;
        const int xr_lo = (bwd ? 0 : a.lbB) - us.sx[1], xc_lo = (bwd ? 0 : a.lbL) - us.sx[2];
        const int sgr = a.active ? -us.sg[1] : us.sg[1], sgc = a.active ? -us.sg[2] : us.sg[2], ex = a.active ? 1 : 0;
        const HaloRange hx = {xr_lo, xr_lo + a.IB, xc_lo, xc_lo + 4 * a.IG};
        const HaloRange hg = {sgr, a.OB - 1 + sgr + ex, sgc, a.OL - 1 + sgc + ex};
        const int nx = halo_cells(hx, a.B, a.L), ng = bwd ? halo_cells(hg, a.OB, a.OL) : 0;
        const bool use_list = listable && nx <= FIXCAP && ng <= FIXCAP;
        // x tile: the copy engine's zero fill IS the zeros padding.  grad tile of the fused avg-pool backward: written by
        // pool_expand below, so its reachable halo is cleared (zeros padding) or patched like any other tile.
        const bool fix_x = a.g.pad != TS_PAD_ZEROS, fix_g = bwd && (fix_x || a.pool_bwd), zero_g = a.pool_bwd && !fix_x;
        if (use_list) {
            fsync();                            // every fixer thread is done with the previous unit's lists
            if (fw == 0) {
                if (fix_x) halo_walk_z(list_x, nullptr, a.px, a.B, a.L, a.hr, a.hc, a.g.pad, hx, lane);
                if (fix_g) halo_walk_z(list_g, nullptr, a.pg, a.OB, a.OL, a.hr, a.hc, a.g.pad, hg, lane, zero_g);
            }
            fsync();
        }
        for (int nb = n0; nb < n1; nb += a.np) {
            const int npl = n1 - nb < a.np ? n1 - nb : a.np;
            for (int k = 0; k < steps; ++k) {
                unsigned char* st = smem + (size_t)s * a.stage_stride + GUARD;
                const bool has_g = bwd && (a.dim == 2 || a.active || k >= 1);
                mbar_wait_parked(&full[s], phase);
                if (MULTI && a.pool_bwd) {
                    for (int pl = 0; pl < npl; ++pl)
                        pool_expand((const float*)(st + a.off_v + (size_t)pl * a.tile_v), (float*)(st + a.off_g + (size_t)pl * a.tile_g), a.PH, a.PW,
                                    a.OB, a.pg, a.hr, a.hc, fl, fstride, a.d_PW);
                    fsync();                     // the halo cells below copy from cells other fixer threads have just written
                }
                for (int pl = 0; pl < npl; ++pl) {
                    float* tx = (float*)(st + (size_t)pl * a.tile_x);
                    float* tg = (float*)(st + a.off_g + (size_t)pl * a.tile_g);
                    if (use_list) {
                        if (MULTI) {
                            if (fix_x) halo_apply_m<false>(list_x, nx, tx, fl, fstride);
                            if (has_g && fix_g) { if (zero_g) halo_apply_m<true>(list_g, ng, tg, fl, fstride); else halo_apply_m<false>(list_g, ng, tg, fl, fstride); }
                        } else {
                            if (fix_x) halo_apply_m<false>(list_x, nx, tx, lane);
                            if (has_g && fix_g) halo_apply_m<false>(list_g, ng, tg, lane);
                        }
                    } else if (fw == 0) {
                        if (fix_x) halo_walk_z(nullptr, tx, a.px, a.B, a.L, a.hr, a.hc, a.g.pad, hx, lane);
                        if (has_g && fix_g) halo_walk_z(nullptr, tg, a.pg, a.OB, a.OL, a.hr, a.hc, a.g.pad, hg, lane, zero_g);
                    }
                }
                fence_proxy_async();             // the next TMA load of this stage must not overtake these generic-proxy writes
                __syncwarp();
                if (lane == 0) mbar_arrive(&ready[s]);
                if (++s == a.stages) { s = 0; phase ^= 1u; }
            }
        }
    }
}

// 3-D backward fused with avg_pool3d (kernel = stride = (sA, 2, 2), ceil_mode): ONE fixer warp -- a cfg4 slab (28 row pairs x 16
// groups) takes all 448 consumer threads the CTA has left, so the four expansion warps of the 2-D kernels do not fit.  It
// expands the pooled slab that feeds grad_input into the padded grad tile (every element of a window receives grad / count,
// as ATen's avg_pool3d_backward; the count is a power of two, so the product is the quotient) and then clears (zeros
// padding) or patches the tile's reachable halo: the padding rule applies to the EXPANDED gradient.  The consumers read the
// unshifted gradient for grad_weight straight from the image's other pooled tile.
TS_D void sts128(unsigned addr, float a, float b, float c, float d) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
TS_D void pool_expand3(unsigned src, unsigned dst, int PH, int PW, int OB, int pitch, float fa, int lane, const FastDiv& dPW) {
    // item: 4 pooled values of a row (16 bytes) -> 8 columns of one or two rows of the tile (dst: its element (hr, hc))
    const int n = PH * PW, pb = pitch * 4;
    for (int e = 4 * lane; e < n; e += 128) {
        const int pr = (int)fdiv((unsigned)e, dPW), pc = e - pr * PW;
        const uint4 v = lds128(src + 4u * (unsigned)e);
        const bool two = 2 * pr + 1 < OB;
        const float f = fa * (two ? 0.25f : 0.5f);
        const float v0 = __uint_as_float(v.x) * f, v1 = __uint_as_float(v.y) * f, v2 = __uint_as_float(v.z) * f, v3 = __uint_as_float(v.w) * f;
        const unsigned o = dst + (unsigned)(2 * pr * pb + 8 * pc);
        sts128(o, v0, v0, v1, v1);
        sts128(o + 16, v2, v2, v3, v3);
        if (two) { sts128(o + pb, v0, v0, v1, v1); sts128(o + pb + 16, v2, v2, v3, v3); }
    }
}

TS_D void fixer_pool3(const HArgs& a, unsigned char* smem, uint64_t* full, uint64_t* ready, int lane, const UnitShift* tbl, unsigned* lists,
                      const UnitOrder& uo) {
    int s = 0, cls = 0;
    unsigned phase = 0;
    const int N = (int)a.g.N;
    const int steps = a.IA + 1;
    unsigned* list_x = lists;
    unsigned* list_g = lists + FIXCAP;
    const bool listable = a.px * a.bpx < 65536 && a.pg * a.bpg < 65536;
    const bool fix_x = a.g.pad != TS_PAD_ZEROS, zero_g = !fix_x;
    const UnitRange ur = unit_range(a.units, a.unit_order);
    for (int u = ur.u; u < ur.end; u += ur.step) {
        int chunk, c;
        uo.decode(u, cls, c, chunk, a.unit_order);
        const int n0 = chunk * a.n_per_unit;
        const int n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
        const UnitShift us = unit_shift(a, tbl, c);
        if (!unit_geom(a, us).fits) continue;
        const int xr_lo = -us.sx[1], xc_lo = -us.sx[2];
        const int sgr = a.active ? -us.sg[1] : us.sg[1], sgc = a.active ? -us.sg[2] : us.sg[2], ex = a.active ? 1 : 0;
        const HaloRange hx = {xr_lo, xr_lo + a.IB, xc_lo, xc_lo + 4 * a.IG};
        const HaloRange hg = {sgr, a.OB - 1 + sgr + ex, sgc, a.OL - 1 + sgc + ex};
        const int nx = halo_cells(hx, a.B, a.L), ng = halo_cells(hg, a.OB, a.OL);
        const bool use_list = listable && nx <= FIXCAP && ng <= FIXCAP;
        if (use_list) {
            __syncwarp();                       // every lane is done with the previous unit's lists
            if (fix_x) halo_walk_z(list_x, nullptr, a.px, a.B, a.L, a.hr, a.hc, a.g.pad, hx, lane);
            halo_walk_z(list_g, nullptr, a.pg, a.OB, a.OL, a.hr, a.hc, a.g.pad, hg, lane, zero_g);
            __syncwarp();
        }
        for (int nb = n0; nb < n1; nb += a.np) {
            const int npl = n1 - nb < a.np ? n1 - nb : a.np;
            int gs_l = 0;                                   // pooled grad slab of step (k & ~31) + lane, as the producer loads it
            for (int k = 0; k < steps; ++k) {
                if ((k & 31) == 0) {
                    const int kl = k + lane;
                    gs_l = pooled_slab(a.active ? slab_coord(kl - a.lbA - us.sg[0], a.OA, a.g.pad) : slab_coord(kl - 1 - a.lbA + us.sg[0], a.OA, a.g.pad),
                                       a.sA);
                }
                const int gs = __shfl_sync(0xffffffffu, gs_l, k & 31);
                unsigned char* st = smem + (size_t)s * a.stage_stride + GUARD;
                const bool has_g = a.active || k >= 1;
                mbar_wait_parked(&full[s], phase);
                if (has_g) {
                    const float fa = a.sA == 2 && 2 * gs + 1 < a.OA ? 0.5f : 1.f;      // slabs in the window (a zero tile for gs < 0)
                    for (int pl = 0; pl < npl; ++pl)
                        pool_expand3(shared_addr(st + a.off_v + (size_t)(a.np + pl) * a.tile_v),
                                     shared_addr(st + a.off_g + (size_t)pl * a.tile_g) + (unsigned)((a.hr * a.pg + a.hc) * 4), a.PH, a.PW, a.OB, a.pg,
                                     fa, lane, a.d_PW);
                    __syncwarp();                    // the halo copies below read cells other lanes have just written
                }
                for (int pl = 0; pl < npl; ++pl) {
                    float* tx = (float*)(st + (size_t)pl * a.tile_x);
                    float* tg = (float*)(st + a.off_g + (size_t)pl * a.tile_g);
                    if (use_list) {
                        if (fix_x) halo_apply_m<false>(list_x, nx, tx, lane);
                        if (has_g) { if (zero_g) halo_apply_m<true>(list_g, ng, tg, lane); else halo_apply_m<false>(list_g, ng, tg, lane); }
                    } else {
                        if (fix_x) halo_walk_z(nullptr, tx, a.px, a.B, a.L, a.hr, a.hc, a.g.pad, hx, lane);
                        if (has_g) halo_walk_z(nullptr, tg, a.pg, a.OB, a.OL, a.hr, a.hc, a.g.pad, hg, lane, zero_g);
                    }
                }
                fence_proxy_async();             // the next TMA load of this stage must not overtake these generic-proxy writes
                __syncwarp();
                if (lane == 0) mbar_arrive(&ready[s]);
                if (++s == a.stages) { s = 0; phase ^= 1u; }
            }
        }
    }
}

// ---- consumers ----------------------------------------------------------------------------------
// pair index -> (image of the stage, first row of the pair, column group); false = padding lane
struct Pair { int pl, r, cg; };
TS_D bool decode_pair(const HArgs& a, int p, Pair& q) {
    q.pl = 0;
    int rem = p;
    if (a.np > 1) { q.pl = (int)fdiv((unsigned)p, a.d_img); rem = p - q.pl * a.img_pairs; }
    const int rp = (int)fdiv((unsigned)rem, a.d_GP);
    q.cg = rem - rp * a.GP;
    q.r = 2 * rp;
    return q.cg < a.IG;
}

// Everything about one pair that does not change from stage to stage of a unit.
struct PairCtx {
    unsigned xo, go, vo;       // byte offsets (from the stage base) of the aligned group of the pair's FIRST row in the x / grad / unshifted-grad tile
    long long out_off;         // byte offset of the first row's 16-byte output from the output of (first image of the stage, slab 0)
    int rows;                  // rows of the pair that exist (1 or 2), 0: padding lane
    unsigned cmask;            // bit t of nibble j: element t of row j takes part (inside the crop)
};

template <int MODE, bool CROP>
TS_D PairCtx pair_ctx(const HArgs& a, const UnitGeom& ug, const Pair& q, bool valid) {
    PairCtx p;
    p.rows = !valid ? 0 : (q.r + 1 < a.IB ? 2 : 1);
    p.xo = (unsigned)(q.pl * a.tile_x + ((q.r + ug.xr0) * a.px + ((4 * q.cg + ug.xc0) & ~3)) * 4);
    p.out_off = (long long)q.pl * (a.g.C * a.out_plane_bytes) + (a.pool ? (long long)(((q.r >> 1) * a.IG + q.cg) * 8) : (long long)((q.r * a.IG + q.cg) * 16));
    p.go = p.vo = 0;
    p.cmask = 0xffu;
    if (MODE == 2) {
        unsigned m = p.rows == 2 ? 0xffu : (p.rows == 1 ? 0x0fu : 0u);
        if (CROP) m = 0;
#pragma unroll
        for (int j = 0; CROP && j < 2; ++j) {
            const int ob = q.r + j - a.lbB;
            if (ob < 0 || ob >= a.OB) continue;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int oj = 4 * q.cg + t - a.lbL;
                if (oj >= 0 && oj < a.OL) m |= 1u << (4 * j + t);
            }
        }
        p.cmask = m;
        // A pair with no row inside the crop never reads the grad tiles.  Otherwise the addresses are exact: a row of
        // the pair outside the crop (masked) may then lie one row before / after its tile -- still inside the stage
        // (tiles are preceded by other tiles or the head guard and followed by a tail of one row pitch).
        if (m) {
            p.go = (unsigned)(a.off_g + q.pl * a.tile_g + ((q.r + ug.gr0) * a.pg + ((4 * q.cg + ug.gc0) & ~3)) * 4);
            if (a.dim == 3) p.vo = (unsigned)(a.off_v + q.pl * a.tile_v + ((q.r + ug.vr0) * a.OL + ((4 * q.cg + ug.vc0) & ~3)) * 4);
            else p.vo = (unsigned)(a.off_g + q.pl * a.tile_g + ((q.r + ug.vr0) * a.pg + ((4 * q.cg + ug.vc0) & ~3)) * 4);
        }
    }
    return p;
}

struct Ring {
    int s;
    unsigned phase;
};

// CROP (backward only): the call has a border crop, so grad values outside the crop are masked element by element; without
// one every mask is full and the mask code (48 of 510 instructions per slab step of the 3-D backward) is compiled out.
template <int DIM, int MODE, bool ACTIVE, bool POOL, bool CROP>
struct Body {
    const HArgs& a;
    const int tid, nt, wid, lane;
    uint64_t* const wait_bar;      // ready[] when a fixer warp patches the stages, else full[]
    uint64_t* const empty;
    UnitShift us;
    UnitGeom ug;
    int wsx, wsg, wsv;
    double acc[3];

    const UnitShift* const tbl;
    TS_D Body(const HArgs& a_, int tid_, int nt_, int wid_, int lane_, uint64_t* wait_, uint64_t* empty_, const UnitShift* tbl_)
        : a(a_), tid(tid_), nt(nt_), wid(wid_), lane(lane_), wait_bar(wait_), empty(empty_), tbl(tbl_) {}

    TS_D void begin_unit(int c) {
        us = unit_shift(a, tbl, c);
        ug = unit_geom(a, us);
        wsx = ug.xc0 & 3; wsg = ug.gc0 & 3; wsv = ug.vc0 & 3;
        acc[0] = acc[1] = acc[2] = 0.0;
    }
    TS_D void end_unit(int c, int chunk) {
        if (MODE != 2) return;
#pragma unroll
        for (int k = 0; k < DIM; ++k) {
            double v = acc[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) a.partials[((long long)chunk * a.nw + wid) * (a.g.C * DIM) + (long long)c * DIM + k] = v;
        }
    }
    TS_D void release(Ring& ring) const {
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[ring.s]);
        if (++ring.s == a.stages) { ring.s = 0; ring.phase ^= 1u; }
    }

    // ---------------------------------------------------------------------------------------------
    // 2-D: a stage = np images, every pair is independent
    template <int WSX, int WSG, int WSV>
    TS_D void pair2(unsigned sb, unsigned char* dst, const PairCtx& pc, float* ts) const {
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        unsigned char* o = dst + pc.out_off;
        const unsigned xa = sb + pc.xo;
        const int orow = a.IG * 16;
        float X[3][5];
        load5<WSX>(xa, wsx, X[0]);
        load5<WSX>(xa + a.px * 4, wsx, X[1]);
        if (pc.rows == 2 && MODE != 0) load5<WSX>(xa + 2 * a.px * 4, wsx, X[2]);
        if (MODE != 2) {
            float y[2][4];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                if (j < pc.rows) {
                    if (MODE == 1) {
                        float R[5];
#pragma unroll
                        for (int t = 0; t < 5; ++t) R[t] = lerp<float>(X[j][t], X[j + 1][t], d[0]);
#pragma unroll
                        for (int t = 0; t < 4; ++t) y[j][t] = lerp<float>(R[t], R[t + 1], d[1]);
                    } else {
#pragma unroll
                        for (int t = 0; t < 4; ++t) y[j][t] = X[j][t];
                    }
                    if (!POOL) __stcs((float4*)(o + j * orow), make_float4(y[j][0], y[j][1], y[j][2], y[j][3]));
                }
            }
            if (POOL) {
                // avg_pool2d(kernel 2, stride 2, ceil_mode) of the row pair: the window's elements are added in
                // row-major order and divided by their count, like ATen's kernel (modules/shifts.py:85-89)
                float q0, q1;
                if (pc.rows == 2) {
                    q0 = __fdiv_rn(__fadd_rn(__fadd_rn(__fadd_rn(y[0][0], y[0][1]), y[1][0]), y[1][1]), 4.f);
                    q1 = __fdiv_rn(__fadd_rn(__fadd_rn(__fadd_rn(y[0][2], y[0][3]), y[1][2]), y[1][3]), 4.f);
                } else {
                    q0 = __fdiv_rn(__fadd_rn(y[0][0], y[0][1]), 2.f);
                    q1 = __fdiv_rn(__fadd_rn(y[0][2], y[0][3]), 2.f);
                }
                __stcs((float2*)o, make_float2(q0, q1));
            }
            return;
        }
        const unsigned ga = sb + pc.go, va = sb + pc.vo;
        float G[3][5];
        if (ACTIVE && pc.cmask) {
            load5<WSG>(ga, wsg, G[0]);
            load5<WSG>(ga + a.pg * 4, wsg, G[1]);
            if (pc.rows == 2) load5<WSG>(ga + 2 * a.pg * 4, wsg, G[2]);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (j >= pc.rows) continue;
            const unsigned m = CROP ? (pc.cmask >> (4 * j)) & 15u : 15u;
            float y[4] = {0.f, 0.f, 0.f, 0.f};
            if (m) {
                float gv[4];
                load4<WSV>(va + j * a.pg * 4, wsv, gv);
                if (CROP && m != 15u) {
#pragma unroll
                    for (int t = 0; t < 4; ++t) gv[t] = (m >> t) & 1u ? gv[t] : 0.f;
                }
                wp2(X[j], X[j + 1], gv, d, ts);
                if (ACTIVE) {
                    float R[5];
#pragma unroll
                    for (int t = 0; t < 5; ++t) R[t] = lerp<float>(G[j][t], G[j + 1][t], d[0]);
#pragma unroll
                    for (int t = 0; t < 4; ++t) y[t] = lerp<float>(R[t], R[t + 1], d[1]);
                } else {
                    load4<WSG>(ga + j * a.pg * 4, wsg, y);
                }
                if (CROP && m != 15u) {
#pragma unroll
                    for (int t = 0; t < 4; ++t) y[t] = (m >> t) & 1u ? y[t] : 0.f;
                }
            }
            __stcs((float4*)(o + j * orow), make_float4(y[0], y[1], y[2], y[3]));
        }
    }

    template <int WSX, int WSG, int WSV>
    TS_D void run_images2(unsigned char* smem, Ring& ring, unsigned char* dst, int npl, const PairCtx& pc0, float* ts) const {
        unsigned char* st = smem + (size_t)ring.s * a.stage_stride + GUARD;
        const unsigned sb = shared_addr(st);
        mbar_wait_parked(&wait_bar[ring.s], ring.phase);
        const int total = npl * a.img_pairs;
        if (tid < total && pc0.rows) pair2<WSX, WSG, WSV>(sb, dst, pc0, ts);      // the thread's first pair: context cached per unit
        for (int p = tid + nt; p < total; p += nt) {
            Pair q;
            if (!decode_pair(a, p, q)) continue;
            const PairCtx pc = pair_ctx<MODE, CROP>(a, ug, q, true);
            pair2<WSX, WSG, WSV>(sb, dst, pc, ts);
        }
        release(ring);
    }

    // ---------------------------------------------------------------------------------------------
    // 3-D: a thread owns its pair for the whole image; windows of the previous slab stay in registers
    struct Carry {
        float X[3][5];
        float G[(MODE == 2 && ACTIVE) ? 3 : 1][5];
    };

    // stage k of an image: combine the windows of slab k-1 (`prev`, registers) with this stage's (slab k), which are
    // loaded straight into `next`: the caller alternates two register sets, so nothing is copied from step to step
    template <int WSX, int WSG, int WSV>
    TS_D void step3(unsigned sb, unsigned char* dst_img, int k, const PairCtx& pc, const Carry& cy, Carry& nx, float* ts) const {
        if (pc.rows == 0) return;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        const int it = k - 1, orow = a.IG * 16;
        unsigned char* o = dst_img + pc.out_off + (long long)it * a.IB * orow;
        const bool slab_pass = MODE != 2 || !CROP || (it - a.lbA >= 0 && it - a.lbA < a.OA);
        const unsigned cm = (k >= 1 && slab_pass) ? pc.cmask : 0u;
        const unsigned xa = sb + pc.xo, ga = sb + pc.go, va = sb + pc.vo;
        const int pxb = a.px * 4, pgb = a.pg * 4;
        const bool gwin = MODE == 2 && ACTIVE && pc.cmask != 0u;
        float SL[2][5];
        load5<WSX>(xa, wsx, nx.X[0]); load5<WSX>(xa + pxb, wsx, nx.X[1]);
        if (gwin) { load5<WSG>(ga, wsg, nx.G[0]); load5<WSG>(ga + pgb, wsg, nx.G[1]); }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (j >= pc.rows) continue;
            if (j == 1) {
                load5<WSX>(xa + 2 * pxb, wsx, nx.X[2]);
                if (gwin) load5<WSG>(ga + 2 * pgb, wsg, nx.G[2]);
            }
            if (k < 1) continue;
            if (MODE != 2) {
                float P[5], y[4];
                // the slab lerp of row j + 1 is shared by both rows of the pair (same operations, same order: bit-exact)
                if (j == 0) {
#pragma unroll
                    for (int t = 0; t < 5; ++t) { SL[0][t] = lerp<float>(cy.X[0][t], nx.X[0][t], d[0]); SL[1][t] = lerp<float>(cy.X[1][t], nx.X[1][t], d[0]); }
                } else {
#pragma unroll
                    for (int t = 0; t < 5; ++t) { SL[0][t] = SL[1][t]; SL[1][t] = lerp<float>(cy.X[2][t], nx.X[2][t], d[0]); }
                }
#pragma unroll
                for (int t = 0; t < 5; ++t) P[t] = lerp<float>(SL[0][t], SL[1][t], d[1]);
#pragma unroll
                for (int t = 0; t < 4; ++t) y[t] = lerp<float>(P[t], P[t + 1], d[2]);
                __stcs((float4*)(o + j * orow), make_float4(y[0], y[1], y[2], y[3]));
            } else {
                const unsigned m = CROP ? (cm >> (4 * j)) & 15u : 15u;       // (no crop: k >= 1 and the row exists here)
                float y[4] = {0.f, 0.f, 0.f, 0.f};
                if (m) {
                    float gv[4];
                    load4<WSV>(va + j * a.OL * 4, wsv, gv);
                    if (CROP && m != 15u) {
#pragma unroll
                        for (int t = 0; t < 4; ++t) gv[t] = (m >> t) & 1u ? gv[t] : 0.f;
                    }
                    wp3(cy.X[j], nx.X[j], cy.X[j + 1], nx.X[j + 1], gv, d, ts);
                    if (ACTIVE) {
                        float P[5];
#pragma unroll
                        for (int t = 0; t < 5; ++t) P[t] = col3(cy.G[j][t], nx.G[j][t], cy.G[j + 1][t], nx.G[j + 1][t], d[0], d[1]);
#pragma unroll
                        for (int t = 0; t < 4; ++t) y[t] = lerp<float>(P[t], P[t + 1], d[2]);
                    } else {
                        load4<WSG>(ga + j * pgb, wsg, y);
                    }
                    if (CROP && m != 15u) {
#pragma unroll
                        for (int t = 0; t < 4; ++t) y[t] = (m >> t) & 1u ? y[t] : 0.f;
                    }
                }
                __stcs((float4*)(o + j * orow), make_float4(y[0], y[1], y[2], y[3]));
            }
        }
    }

    // ---------------------------------------------------------------------------------------------
    // 3-D fused with avg_pool3d (kernel = stride = (sA, 2, 2), ceil_mode).  Forward: the pair's 2 x 4 outputs of a slab step are
    // pooled into two values -- every window's elements added in (slab, row, column) order into ONE running sum, as ATen's
    // kernel; with sA = 2 the sum of an even slab step is carried in registers to the odd one -- and divided by the count.
    template <int WSX>
    TS_D void pool_step_fwd(unsigned sb, unsigned char* dst_img, int k, const PairCtx& pc, const Carry& cy, Carry& nx, float* run) const {
        if (pc.rows == 0) return;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        const unsigned xa = sb + pc.xo;
        const int pxb = a.px * 4;
        float y[2][4];
        int it;
        if constexpr (MODE == 0) {
            // the gather: output slab k is this stage's x slab (the ring's last stage only drains)
            if (k >= a.IA) return;
            it = k;
            load4<WSX>(xa, wsx, y[0]);
            if (pc.rows == 2) load4<WSX>(xa + pxb, wsx, y[1]);
        } else {
            load5<WSX>(xa, wsx, nx.X[0]); load5<WSX>(xa + pxb, wsx, nx.X[1]);
            if (pc.rows == 2) load5<WSX>(xa + 2 * pxb, wsx, nx.X[2]);
            if (k < 1) return;
            it = k - 1;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                if (j >= pc.rows) continue;
                float S0[5], S1[5], P[5];
#pragma unroll
                for (int t = 0; t < 5; ++t) { S0[t] = lerp<float>(cy.X[j][t], nx.X[j][t], d[0]); S1[t] = lerp<float>(cy.X[j + 1][t], nx.X[j + 1][t], d[0]); }
#pragma unroll
                for (int t = 0; t < 5; ++t) P[t] = lerp<float>(S0[t], S1[t], d[1]);
#pragma unroll
                for (int t = 0; t < 4; ++t) y[j][t] = lerp<float>(P[t], P[t + 1], d[2]);
            }
        }
        const bool two = pc.rows == 2, odd = a.sA == 2 && (it & 1);
        float s0 = odd ? __fadd_rn(run[0], y[0][0]) : y[0][0], s1 = odd ? __fadd_rn(run[1], y[0][2]) : y[0][2];
        s0 = __fadd_rn(s0, y[0][1]);
        s1 = __fadd_rn(s1, y[0][3]);
        if (two) {
            s0 = __fadd_rn(__fadd_rn(s0, y[1][0]), y[1][1]);
            s1 = __fadd_rn(__fadd_rn(s1, y[1][2]), y[1][3]);
        }
        if (a.sA == 2 && !odd && it != a.IA - 1) { run[0] = s0; run[1] = s1; return; }
        const float cnt = (float)((two ? 4 : 2) * (odd ? 2 : 1));
        const int pa = a.sA == 2 ? it >> 1 : it;
        __stcs((float2*)(dst_img + pc.out_off + (long long)pa * a.PH * a.PW * 4), make_float2(__fdiv_rn(s0, cnt), __fdiv_rn(s1, cnt)));
    }

    // Backward: step3's backward with the unshifted gradient read from the pooled tile (value x 1 / count of its window); the
    // grad tile that feeds grad_input was expanded by the fixer warp.  q: the pair (crops: element-wise pooled indices).
    template <int WSX, int WSG, int WSV>
    TS_D void pool_step_bwd(unsigned sb, unsigned char* dst_img, int k, const PairCtx& pc, const Pair& q, const Carry& cy, Carry& nx,
                            float* ts) const {
        if (pc.rows == 0) return;
        const float d[3] = {us.d[0], us.d[1], us.d[2]};
        const int it = k - 1, oa = it - a.lbA, orow = a.IG * 16;
        unsigned char* o = dst_img + pc.out_off + (long long)it * a.IB * orow;
        const bool slab_pass = !CROP || (oa >= 0 && oa < a.OA);
        const unsigned cm = (k >= 1 && slab_pass) ? pc.cmask : 0u;
        const unsigned xa = sb + pc.xo, ga = sb + pc.go, va = sb + pc.vo;
        const int pxb = a.px * 4, pgb = a.pg * 4;
        const bool gwin = ACTIVE && pc.cmask != 0u;
        const float fa = a.sA == 2 && (oa | 1) < a.OA ? 0.5f : 1.f;          // slabs in the window of output slab oa
        float pv[2] = {0.f, 0.f};
        load5<WSX>(xa, wsx, nx.X[0]); load5<WSX>(xa + pxb, wsx, nx.X[1]);
        if (gwin) { load5<WSG>(ga, wsg, nx.G[0]); load5<WSG>(ga + pgb, wsg, nx.G[1]); }
        if (!CROP && k >= 1) {
            // no crop: both rows of the pair lie in one pooled row, the group's 4 columns in 2 pooled columns
            const uint2 v = lds64(va);
            const float f = fa * (pc.rows == 2 ? 0.25f : 0.5f);
            pv[0] = __uint_as_float(v.x) * f; pv[1] = __uint_as_float(v.y) * f;
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            if (j >= pc.rows) continue;
            if (j == 1) {
                load5<WSX>(xa + 2 * pxb, wsx, nx.X[2]);
                if (gwin) load5<WSG>(ga + 2 * pgb, wsg, nx.G[2]);
            }
            if (k < 1) continue;
            const unsigned m = CROP ? (cm >> (4 * j)) & 15u : 15u;
            float y[4] = {0.f, 0.f, 0.f, 0.f};
            if (m) {
                float gv[4];
                if constexpr (CROP) {
                    const int pr = (q.r + j - a.lbB) >> 1;
                    const float f = fa * (2 * pr + 1 < a.OB ? 0.25f : 0.5f);
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const int oj = 4 * q.cg + t - a.lbL;
                        gv[t] = (m >> t) & 1u ? __uint_as_float(lds32(va + (unsigned)((pr * a.PW + (oj >> 1)) * 4))) * f : 0.f;
                    }
                } else {
                    gv[0] = gv[1] = pv[0]; gv[2] = gv[3] = pv[1];
                }
                wp3(cy.X[j], nx.X[j], cy.X[j + 1], nx.X[j + 1], gv, d, ts);
                if (ACTIVE) {
                    float P[5];
#pragma unroll
                    for (int t = 0; t < 5; ++t) P[t] = col3(cy.G[j][t], nx.G[j][t], cy.G[j + 1][t], nx.G[j + 1][t], d[0], d[1]);
#pragma unroll
                    for (int t = 0; t < 4; ++t) y[t] = lerp<float>(P[t], P[t + 1], d[2]);
                } else {
                    load4<WSG>(ga + j * pgb, wsg, y);
                }
                if (CROP && m != 15u) {
#pragma unroll
                    for (int t = 0; t < 4; ++t) y[t] = (m >> t) & 1u ? y[t] : 0.f;
                }
            }
            __stcs((float4*)(o + j * orow), make_float4(y[0], y[1], y[2], y[3]));
        }
    }

    template <int WSX, int WSG, int WSV>
    TS_D void run_images3_pool(unsigned char* smem, Ring& ring, unsigned char* dst_img, int npl, float* ts) const {
        Pair q;
        const bool valid = tid < npl * a.img_pairs && decode_pair(a, tid, q);
        if (!valid) { q.pl = 0; q.r = 0; q.cg = 0; }
        PairCtx pc = pair_ctx<MODE, CROP>(a, ug, q, valid);
        // the pooled tile of the unshifted gradient (crops: its origin, indexed element by element)
        if (MODE == 2) pc.vo = (unsigned)(a.off_v + q.pl * a.tile_v + (CROP ? 0 : ((q.r >> 1) * a.PW + 2 * q.cg) * 4));
        Carry ca, cb;
        if constexpr (MODE != 2) {
            float run[2] = {0.f, 0.f};
            for (int k = 0; k <= a.IA; ++k) {
                const unsigned sb = shared_addr(smem + (size_t)ring.s * a.stage_stride + GUARD);
                mbar_wait_parked(&wait_bar[ring.s], ring.phase);
                pool_step_fwd<WSX>(sb, dst_img, k, pc, ca, cb, run);
                if (MODE == 1) {
#pragma unroll
                    for (int j = 0; j < 3; ++j)
#pragma unroll
                        for (int t = 0; t < 5; ++t) ca.X[j][t] = cb.X[j][t];
                }
                release(ring);
            }
        } else {
            for (int k = 0; k <= a.IA; k += 2) {
                {
                    const unsigned sb = shared_addr(smem + (size_t)ring.s * a.stage_stride + GUARD);
                    mbar_wait_parked(&wait_bar[ring.s], ring.phase);
                    pool_step_bwd<WSX, WSG, WSV>(sb, dst_img, k, pc, q, cb, ca, ts);
                    release(ring);
                }
                if (k + 1 <= a.IA) {
                    const unsigned sb = shared_addr(smem + (size_t)ring.s * a.stage_stride + GUARD);
                    mbar_wait_parked(&wait_bar[ring.s], ring.phase);
                    pool_step_bwd<WSX, WSG, WSV>(sb, dst_img, k + 1, pc, q, ca, cb, ts);
                    release(ring);
                }
            }
        }
    }

    // The pair's context and its backward steps sit in loops of ONE trip on purpose: the compiler's schedule of the 3-D
    // kernels depends on that loop structure (straight-line code adds 36 bytes of spills per thread to the interpolating
    // backward and reorders both interpolating kernels).
    template <int WSX, int WSG, int WSV>
    TS_D void run_images3(unsigned char* smem, Ring& ring, unsigned char* dst_img, int npl, float* ts) const {
        if constexpr (POOL) {
            run_images3_pool<WSX, WSG, WSV>(smem, ring, dst_img, npl, ts);
            return;
        }
        PairCtx pc[1];
        Carry ca[1], cb[1];                    // the windows of two consecutive slabs, roles alternating from step to step
#pragma unroll
        for (int i = 0; i < 1; ++i) {
            Pair q;
            const bool valid = tid < npl * a.img_pairs && decode_pair(a, tid, q);
            if (!valid) { q.pl = 0; q.r = 0; q.cg = 0; }
            pc[i] = pair_ctx<MODE, CROP>(a, ug, q, valid);
        }
        if constexpr (MODE != 2) {
            // forward: four compile-time misalignment bodies; unrolling the slab loop by two on top of that spills, so the
            // new windows are copied into the carried set instead (15 moves per step)
            for (int k = 0; k <= a.IA; ++k) {
                const unsigned sb = shared_addr(smem + (size_t)ring.s * a.stage_stride + GUARD);
                mbar_wait_parked(&wait_bar[ring.s], ring.phase);
                step3<WSX, WSG, WSV>(sb, dst_img, k, pc[0], ca[0], cb[0], ts);
#pragma unroll
                for (int j = 0; j < 3; ++j)
#pragma unroll
                    for (int t = 0; t < 5; ++t) ca[0].X[j][t] = cb[0].X[j][t];
                release(ring);
            }
            return;
        }
        for (int k = 0; k <= a.IA; k += 2) {
            {
                const unsigned sb = shared_addr(smem + (size_t)ring.s * a.stage_stride + GUARD);
                mbar_wait_parked(&wait_bar[ring.s], ring.phase);
#pragma unroll
                for (int i = 0; i < 1; ++i) step3<WSX, WSG, WSV>(sb, dst_img, k, pc[i], cb[i], ca[i], ts);
                release(ring);
            }
            if (k + 1 <= a.IA) {
                const unsigned sb = shared_addr(smem + (size_t)ring.s * a.stage_stride + GUARD);
                mbar_wait_parked(&wait_bar[ring.s], ring.phase);
#pragma unroll
                for (int i = 0; i < 1; ++i) step3<WSX, WSG, WSV>(sb, dst_img, k + 1, pc[i], ca[i], cb[i], ts);
                release(ring);
            }
        }
    }

    template <int WSX, int WSG, int WSV>
    TS_D void run_images(unsigned char* smem, Ring& ring, unsigned char* dst, int npl, const PairCtx& pc0, float* ts) const {
        if constexpr (DIM == 2) run_images2<WSX, WSG, WSV>(smem, ring, dst, npl, pc0, ts);
        else run_images3<WSX, WSG, WSV>(smem, ring, dst, npl, ts);
    }

    // CLS 0..3: every window misalignment is a compile-time constant (x window: CLS words; grad_input window: the same
    // for the interpolating backward, 4 - CLS for the sparse gather; unshifted grad window aligned); CLS 4: run-time
    // misalignment (crops) or the element-wise routine (shift beyond the halo)
    template <int CLS>
    TS_D void run_unit(unsigned char* smem, Ring& ring, int c, int n0, int n1) {
        if (CLS == 4 && !ug.fits) {
            if (MODE != 2) slow_forward<DIM, MODE == 1, POOL>(a, c, n0, n1, us, tid, nt);
            else slow_backward<DIM, ACTIVE, POOL && MODE == 2>(a, c, n0, n1, us, tid, nt, acc);
            return;
        }
        const long long plane_bytes = a.out_plane_bytes;
        PairCtx pc0;
        pc0.rows = 0;
        if (DIM == 2) {
            Pair q;
            const bool valid = tid < a.pairs && decode_pair(a, tid, q);
            if (!valid) { q.pl = 0; q.r = 0; q.cg = 0; }
            pc0 = pair_ctx<MODE, CROP>(a, ug, q, valid);
        }
        for (int nb = n0; nb < n1; nb += a.np) {
            const int npl = n1 - nb < a.np ? n1 - nb : a.np;
            unsigned char* dst = (unsigned char*)a.out + ((long long)nb * a.g.C + c) * plane_bytes;
            float ts[3] = {0.f, 0.f, 0.f};
            if constexpr (CLS < 4) run_images<CLS, ACTIVE ? CLS : ((4 - CLS) & 3), 0>(smem, ring, dst, npl, pc0, ts);
            else run_images<-1, -1, -1>(smem, ring, dst, npl, pc0, ts);
#pragma unroll
            for (int k = 0; k < DIM; ++k) acc[k] += (double)ts[k];     // fp32 inside an image group, fp64 across
        }
    }

    template <int CLS>
    TS_D void run_class(unsigned char* smem, Ring& ring, const UnitOrder& uo, int& u, const UnitRange& ur) {
        const int N = (int)a.g.N;
        int k = CLS;
        while (u < ur.end && u < uo.cend[CLS]) {
            int chunk, c;
            uo.decode(u, k, c, chunk, a.unit_order);
            const int n0 = chunk * a.n_per_unit;
            const int n1 = n0 + a.n_per_unit < N ? n0 + a.n_per_unit : N;
            begin_unit(c);
            run_unit<CLS>(smem, ring, c, n0, n1);
            end_unit(c, chunk);
            u += ur.step;
        }
    }
};

template <int DIM, int MODE, bool ACTIVE, bool POOL, bool CROP = false>
__global__ void __launch_bounds__(MAXT, 1) k_halo(const __grid_constant__ HArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    uint64_t* full = (uint64_t*)(smem + (size_t)a.stages * a.stage_stride);
    uint64_t* empty = full + a.stages;
    uint64_t* ready = empty + a.stages;
    if (threadIdx.x == 0) {
        for (int s = 0; s < a.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], (unsigned)a.nw); mbar_init(&ready[s], (POOL && MODE == 2) ? (unsigned)a.nfix : 1u); }
        fence_barrier_init();
    }
    const int C = (int)a.g.C;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    UnitShift* tbl = (UnitShift*)(ready + a.stages);
    unsigned* lists = (unsigned*)(tbl + (a.table ? C : 0));
    int* cend = (int*)(lists + (a.need_fix ? 2 * FIXCAP : 0));       // [NCLS] units in classes 0..k
    int* coff = cend + NCLS;                                          // [NCLS + 1] channels in classes 0..k-1
    unsigned short* order = (unsigned short*)(coff + NCLS + 1);       // [C] channels sorted by class
    unsigned char* clsb = (unsigned char*)(order + (a.table ? C : 0)); // [C] class of a channel
    if (a.table)
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            const UnitShift us = compute_unit_shift(a, c);
            tbl[c] = us;
            clsb[c] = (unsigned char)classify(a, us);
        }
    __syncthreads();
    if (wid == 0) {
        if (a.table) {                       // counting sort by class: ballot compaction, channel order kept inside a class
            int base = 0;
            for (int k = 0; k < NCLS; ++k) {
                if (lane == 0) coff[k] = base;
                for (int c0 = 0; c0 < C; c0 += 32) {
                    const int c = c0 + lane;
                    const bool mine = c < C && clsb[c] == k;
                    const unsigned m = __ballot_sync(0xffffffffu, mine);
                    if (mine) order[base + __popc(m & ((1u << lane) - 1u))] = (unsigned short)c;
                    base += __popc(m);
                }
                if (lane == 0) cend[k] = base * a.chunks;
            }
            if (lane == 0) coff[NCLS] = base;
        } else if (lane == 0) {              // no table (C > TABLE_MAX_C): one class, run-time misalignment
            for (int k = 0; k < NCLS; ++k) { coff[k] = 0; cend[k] = k == NCLS - 1 ? a.units : 0; }
            coff[NCLS] = C;
        }
    }
    __syncthreads();
    const UnitOrder uo = {a.table ? order : nullptr, cend, coff, a.chunks, C};
    if (wid == a.nw) { producer<POOL && MODE == 2 && DIM == 3>(a, smem, full, empty, tbl, uo, lane); return; }
    if (wid > a.nw) {                                                         // launched only when the padding needs it
        // (the pooled-gradient expansion and its multi-warp fixer exist only in the POOL && MODE == 2 instantiations: the same
        // code merely PRESENT in the other kernels changed ptxas' schedule of their hot loops -- cfg4 forward 0.31 -> 0.37 ms)
        if constexpr (POOL && MODE == 2 && DIM == 3) fixer_pool3(a, smem, full, ready, lane, tbl, lists, uo);
        else if constexpr (POOL && MODE == 2) fixer_pool<true>(a, smem, full, ready, lane, wid - a.nw - 1, tbl, lists, uo);
        else fixer(a, smem, full, ready, lane, tbl, lists, uo);
        return;
    }
    Body<DIM, MODE, ACTIVE, POOL, CROP> body(a, threadIdx.x, a.nt, wid, lane, a.need_fix ? ready : full, empty, tbl);
    Ring ring = {0, 0u};
    const UnitRange ur = unit_range(a.units, a.unit_order);
    int u = ur.u;
    body.template run_class<0>(smem, ring, uo, u, ur);
    body.template run_class<1>(smem, ring, uo, u, ur);
    body.template run_class<2>(smem, ring, uo, u, ur);
    body.template run_class<3>(smem, ring, uo, u, ur);
    body.template run_class<4>(smem, ring, uo, u, ur);
}

int launch(void (*kernel)(HArgs), const HArgs& a, const HaloPlan& p, cudaStream_t s) {
    return launch_persistent(kernel, p.grid, (a.nw + 1 + (a.need_fix ? a.nfix : 0)) * 32, p.smem_bytes, s, false, a);
}

// The pointers and tensor maps of one launch; false: a map could not be encoded.
bool bind(HArgs& a, const void* x, const void* grad, void* out, const void* w, double* partials) {
    const Geo& g = a.g;
    a.x = (const float*)x; a.grad = (const float*)grad; a.out = (float*)out; a.w = (const float*)w; a.partials = partials;
    if (!make_tensor_map5(&a.map_x, x, 4, g.N, g.C, a.A, a.B, a.L, a.px, a.bpx, 1, 1)) return false;
    if (a.mode == 2 && a.pool_bwd) {
        if (!make_tensor_map5(&a.map_v, grad, 4, g.N, g.C, a.PA, a.PH, a.PW, a.PW, a.PH, 1, 1)) return false;
    } else if (a.mode == 2) {
        if (!make_tensor_map5(&a.map_g, grad, 4, g.N, g.C, a.OA, a.OB, a.OL, a.pg, a.bpg, 1, 1)) return false;
        if (a.dim == 3 && !make_tensor_map5(&a.map_v, grad, 4, g.N, g.C, a.OA, a.OB, a.OL, a.OL, a.OB, 1, 1)) return false;
    }
    return true;
}

}  // namespace

// ---- planning -----------------------------------------------------------------------------------
HaloPlan plan_halo(const Geo& g, int mode, int active, int dtype, bool dense_x, const void* x, const void* out, const void* grad,
                   int sm_count, bool forced, bool pool_bwd, int pool_sa) {
    HaloPlan p;
    memset(&p, 0, sizeof(p));
    p.ok = false;
    if (!tma_available() || !dense_x || dtype != TS_F32 || mode < 0 || mode > 2) return p;
    const int d = g.dim;
    if (d != 2 && d != 3) return p;
    const bool pool3 = d == 3 && (pool_sa == 1 || pool_sa == 2);
    if (mode == 0 && d != 2 && !pool3) return p;          // sparse forward: the pooled epilogues only; other 3-D gathers stay on ts_staged.cu
    if (g.N * g.C == 0 || g.in_plane == 0 || g.out_plane == 0) return p;
    for (int ax = 0; ax < d; ++ax)
        if (g.S[ax] < 2 || g.OS[ax] < 2) return p;        // a size-1 axis ignores its shift (shifts_kernels.h:40-50): other families
    const Levels lv(g);
    const int B = lv.B, L = lv.L, OB = lv.OB, OL = lv.OL;
    if (L % 4 || OL % 4) return p;
    if (pool_bwd && (mode != 2 || (d != 2 && !pool3) || OL % 8)) return p;      // pooled rows of a multiple of 16 bytes (TMA)
    if (((uintptr_t)x & 15) || ((uintptr_t)out & 15) || ((uintptr_t)grad & 15)) return p;
    if (g.N >= (1ll << 31) || g.C >= (1ll << 31)) return p;
    if (g.in_plane * 4 >= (1ll << 40) / (g.C > 0 ? g.C : 1)) return p;
    const Tuning& t = tuning();
    HArgs& a = p.a;
    a.g = g;
    a.mode = mode; a.active = active ? 1 : 0; a.dim = d;
    a.A = lv.A;    a.OA = lv.OA;    a.lbA = lv.lbA;
    a.B = B;       a.OB = OB;       a.lbB = lv.lbB;
    a.L = L;       a.OL = OL;       a.lbL = lv.lbL;
    const int halo = t.halo > 0 ? t.halo : 4;
    a.hr = halo;
    a.hc = (halo + 3) / 4 * 4;
    // row pitch = 4 (mod 8) words: the fixer warp walks DOWN the rows of a halo column (4-way bank conflicts instead of 32-way)
    a.px = L + 2 * a.hc;   a.bpx = B + 2 * a.hr;
    a.pg = OL + 2 * a.hc;  a.bpg = OB + 2 * a.hr;
    if (a.px % 8 == 0) a.px += 4;
    if (a.pg % 8 == 0) a.pg += 4;
    if (a.px > 256 || a.bpx > 256 || a.pg > 256 || a.bpg > 256) return p;           // TMA box extents
    a.PH = (OB + 1) / 2; a.PW = OL / 2;
    a.sA = pool3 ? pool_sa : 1;
    a.PA = pool3 ? (lv.OA + pool_sa - 1) / pool_sa : 1;
    a.pool_bwd = pool_bwd ? 1 : 0;
    a.need_fix = g.pad != TS_PAD_ZEROS || pool_bwd;
    const bool expand_warps = pool_bwd && d == 2;          // 3-D: the one fixer warp expands the pooled gradient
    a.nfix = expand_warps ? 4 : 1;
    a.tile_x = (int)round_up((long long)a.px * a.bpx * 4, 128);
    a.tile_g = mode == 2 ? (int)round_up((long long)a.pg * a.bpg * 4, 128) : 0;
    // the dense grad slab of the 3-D backward, or the pooled-gradient tile of the fused avg-pool backward
    a.tile_v = pool_bwd ? (int)round_up((long long)a.PH * a.PW * 4, 128) : (mode == 2 && d == 3) ? (int)round_up((long long)OL * OB * 4, 128) : 0;
    a.box_x = a.px * a.bpx * 4; a.box_g = a.pg * a.bpg * 4; a.box_v = pool_bwd ? a.PW * a.PH * 4 : OL * OB * 4;
    // (3-D pooled backward: two pooled tiles per image, the unshifted gradient's and the one expanded for grad_input)
    const long long per_image = (long long)a.tile_x + a.tile_g + a.tile_v * (pool_bwd && pool3 ? 2 : 1);
    a.IA = mode == 2 ? a.A : a.OA;
    const int IB = a.IB = mode == 2 ? B : OB, IG = a.IG = (mode == 2 ? L : OL) / 4;
    const int GP = a.GP = padded_groups(IG);
    a.RP = (IB + 1) / 2;
    const int img_pairs = a.img_pairs = a.RP * GP;
    const int max_nt = MAXT - 64 - (expand_warps ? 96 : 0);    // producer warp + fixer warp(s)
    const long long table_bytes = (g.C <= TABLE_MAX_C ? g.C * 36 : 0) + ((g.pad != TS_PAD_ZEROS || pool_bwd) ? 2 * FIXCAP * 4 : 0)      // + the fixer's cell lists
                                  + (2 * NCLS + 1) * 4 + (g.C <= TABLE_MAX_C ? g.C * 3 : 0) + 16;                             // + the class order
    const long long budget = SMEM_LIMIT - 1024 - table_bytes;
    long long np;
    if (d == 3) {
        if (img_pairs > max_nt) return p;                  // one (row pair, group) per thread for the whole image
        np = max_nt / img_pairs;
    } else {
        np = (48 * 1024) / per_image;                      // ~48 KB per stage
    }
    if (np < 1) np = 1;
    if (np > g.N) np = g.N;
    const long long tail = 4ll * (a.px > a.pg ? a.px : a.pg) + 256;       // a masked row may be read one row past the last tile
    auto stride_of = [&](long long n) { return round_up(n * per_image + GUARD + tail, 1024); };
    const int min_stages = d == 3 ? 3 : 2;
    while (np > 1 && budget / (stride_of(np) + 24) < min_stages + 1) --np;
    long long stages = budget / (stride_of(np) + 24);
    if (stages < min_stages) return p;
    const int want = t.halo_stages > 0 ? t.halo_stages : (d == 3 ? 6 : (mode == 2 ? 5 : 4));     // tools/knob_sweep.py cfg3ra / cfg4r
    if (stages > want) stages = want;
    if (np * per_image >= (1 << 20)) return p;             // mbarrier tx-count range
    const long long pairs = np * img_pairs;
    if (!forced && pairs < 128) return p;                  // tiny planes: too little work per stage hand-off
    if (np * g.C * (mode == 2 ? g.in_plane : g.out_plane) * 4 >= 0x7fffffffLL) return p;
    // consumer warps: 3-D needs one thread per pair; 2-D picks the count that fills the last pass best
    int warps;
    if (d == 3) {
        warps = (int)((pairs + 31) / 32);
    } else {
        auto eff = [&](int w) {
            const long long nt = 32ll * w, passes = (pairs + nt - 1) / nt;
            return (double)pairs / (double)(passes * nt);
        };
        warps = 8;
        for (int w = 8; w <= max_nt / 32; ++w)
            if (eff(w) > eff(warps) + 1e-9) warps = w;
    }
    if (t.halo_warps > 0 && d != 3) warps = t.halo_warps < max_nt / 32 ? t.halo_warps : max_nt / 32;
    if (warps < 1) warps = 1;
    const UnitPlan up = plan_units(np, t.chunk_planes > 0 ? t.chunk_planes : pick_unit_images(g.N, g.C, np, sm_count, mode == 2 ? 0.4 : 0.1),
                                   g.N, g.C, sm_count, warps);
    if (!up.ok) return p;
    a.np = (int)np; a.pairs = (int)pairs;
    a.off_g = a.np * a.tile_x;
    a.off_v = a.off_g + a.np * a.tile_g;
    a.stages = (int)stages; a.stage_stride = (int)stride_of(np); a.nw = warps; a.nt = warps * 32;
    a.n_per_unit = up.n_per_unit; a.units = up.units; a.chunks = up.chunks; a.unit_order = t.unit_order;
    a.table = g.C <= TABLE_MAX_C ? 1 : 0;
    a.out_plane_bytes = (mode == 2 ? g.in_plane : g.out_plane) * 4;
    a.d_GP = make_fastdiv((unsigned)GP);
    a.d_img = make_fastdiv((unsigned)img_pairs);
    a.d_C = make_fastdiv((unsigned)g.C);
    a.d_chunks = make_fastdiv((unsigned)a.chunks);
    a.d_PW = make_fastdiv((unsigned)(a.PW > 0 ? a.PW : 1));
    p.ok = true;
    p.grid = up.grid; p.slots = up.slots;
    p.smem_bytes = (size_t)(stages * stride_of(np) + 24 * stages + 64 + table_bytes);
    return p;
}

int halo_active_forward(const Geo& g, const HaloPlan& p, const void* x, const void* w, void* y, cudaStream_t s) {
    HArgs a = p.a;
    if (!bind(a, x, nullptr, y, w, nullptr)) return TS_ERR_UNSUPPORTED;
    return g.dim == 3 ? launch(k_halo<3, 1, true, false>, a, p, s) : launch(k_halo<2, 1, true, false>, a, p, s);
}

// 2-D forward (sparse or active) with the 2x2 / stride-2 / ceil_mode average pooling of modules/shifts.py:85-89 fused
// into the store: one read of x, one QUARTER-size write (pool == 0: the plain 2-D forward through the same kernels).
int halo_forward2d(const Geo& g, const HaloPlan& p, int active, int pool, const void* x, const void* w, void* y, cudaStream_t s) {
    if (g.dim != 2) return TS_ERR_UNSUPPORTED;
    HArgs a = p.a;
    a.pool = pool;
    if (pool) a.out_plane_bytes = (long long)a.PH * a.PW * 4;
    if (!bind(a, x, nullptr, y, w, nullptr)) return TS_ERR_UNSUPPORTED;
    if (active) return pool ? launch(k_halo<2, 1, true, true>, a, p, s) : launch(k_halo<2, 1, true, false>, a, p, s);
    return pool ? launch(k_halo<2, 0, false, true>, a, p, s) : launch(k_halo<2, 0, false, false>, a, p, s);
}

// 3-D forward (sparse or active) with avg_pool3d(kernel = stride = (sA, 2, 2), ceil_mode) fused into the store: one read of x,
// one pooled write.
int halo_forward3d_pool(const Geo& g, const HaloPlan& p, int active, const void* x, const void* w, void* y, cudaStream_t s) {
    if (g.dim != 3) return TS_ERR_UNSUPPORTED;
    HArgs a = p.a;
    a.pool = 1;
    a.out_plane_bytes = (long long)a.PA * a.PH * a.PW * 4;
    if (!bind(a, x, nullptr, y, w, nullptr)) return TS_ERR_UNSUPPORTED;
    return active ? launch(k_halo<3, 1, true, true>, a, p, s) : launch(k_halo<3, 0, false, true>, a, p, s);
}

int halo_backward(const Geo& g, const HaloPlan& p, int active, const void* grad, const void* x, const void* w, void* gi,
                  double* partials, cudaStream_t s) {
    HArgs a = p.a;
    if (!bind(a, x, grad, gi, w, partials)) return TS_ERR_UNSUPPORTED;
    bool crop = false;
    for (int ax = 0; ax < g.dim; ++ax) crop = crop || g.lb[ax] != 0 || g.OS[ax] != g.S[ax];
    if (a.pool_bwd && g.dim == 3) {
        if (active) return crop ? launch(k_halo<3, 2, true, true, true>, a, p, s) : launch(k_halo<3, 2, true, true, false>, a, p, s);
        return crop ? launch(k_halo<3, 2, false, true, true>, a, p, s) : launch(k_halo<3, 2, false, true, false>, a, p, s);
    }
    if (a.pool_bwd) {
        if (g.dim != 2) return TS_ERR_UNSUPPORTED;
        if (active) return crop ? launch(k_halo<2, 2, true, true, true>, a, p, s) : launch(k_halo<2, 2, true, true, false>, a, p, s);
        return crop ? launch(k_halo<2, 2, false, true, true>, a, p, s) : launch(k_halo<2, 2, false, true, false>, a, p, s);
    }
    switch (g.dim * 2 + (active ? 1 : 0) + (crop ? 8 : 0)) {
    case 4: return launch(k_halo<2, 2, false, false, false>, a, p, s);
    case 5: return launch(k_halo<2, 2, true, false, false>, a, p, s);
    case 6: return launch(k_halo<3, 2, false, false, false>, a, p, s);
    case 7: return launch(k_halo<3, 2, true, false, false>, a, p, s);
    case 12: return launch(k_halo<2, 2, false, false, true>, a, p, s);
    case 13: return launch(k_halo<2, 2, true, false, true>, a, p, s);
    case 14: return launch(k_halo<3, 2, false, false, true>, a, p, s);
    default: return launch(k_halo<3, 2, true, false, true>, a, p, s);
    }
}

}  // namespace ts

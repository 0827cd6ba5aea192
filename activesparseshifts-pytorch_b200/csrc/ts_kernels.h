// ts_kernels.h -- internal interface between the C ABI (ts_capi.cu) and the kernel families.
//
// A persistent family's plan (TmaPlan, StagedPlan, HaloPlan, FlatPlan) is the launch shape plus the argument block its
// kernels receive: the planner fills every field that does not depend on a pointer, the launcher adds the pointers,
// the weight kind, the quantized arguments and the tensor maps.
#pragma once
#include <cuda.h>

#include "ts_common.cuh"

namespace ts {

constexpr int SMEM_LIMIT = 232448;   // 227 KB opt-in dynamic shared memory per CTA on sm_100
constexpr int TABLE_MAX_C = 512;     // channels whose shift parameters a CTA tabulates in shared memory (TMA, staged, halo, flat)

template <int WK> struct WType;
template <> struct WType<WK_F32> { using type = float; };
template <> struct WType<WK_F64> { using type = double; };
template <> struct WType<WK_F16> { using type = __half; };
template <> struct WType<WK_BF16> { using type = __nv_bfloat16; };

template <int WK, int DIM>
TS_D void load_int_shifts(const void* __restrict__ w, int qkind, long long wzp, long long c, const Geo& g, int* sx) {
    if constexpr (WK == WK_QUANT) {
        load_qshifts<DIM>(w, qkind, wzp, c, g, sx);
    } else {
        using ST = typename WType<WK>::type;
        const ShiftParams<typename Elem<ST>::CT, DIM> p = load_params<ST, DIM>((const ST*)w, c, g, false, false);
#pragma unroll
        for (int a = 0; a < DIM; ++a) sx[a] = p.sx[a];
    }
}

// ---- planning helpers of the persistent families (TMA, staged, halo, flat) ----------------------
inline long long round_up(long long v, long long q) { return (v + q - 1) / q * q; }

// Padded row length of an item index space with `n` 16-byte groups per row: a multiple of 8 keeps every quarter-warp inside
// one row (conflict-free 128-bit shared-memory loads) -- used when it idles <= 15 % of the lanes.
inline int padded_groups(int n) { return n % 8 != 0 && (double)n / (double)((n + 7) / 8 * 8) >= 0.85 ? (n + 7) / 8 * 8 : n; }

// Extents per LEVEL (0 slab, 1 row, 2 column) of a geometry: input A, B, L, output OA, OB, OL and the crop origin
// lbA, lbB, lbL.  Absent levels have extent 1 and origin 0.
struct Levels {
    int A, B, L, OA, OB, OL, lbA, lbB, lbL;
    explicit Levels(const Geo& g) {
        const int d = g.dim;
        A = d == 3 ? g.S[0] : 1;        OA = d == 3 ? g.OS[0] : 1;      lbA = d == 3 ? g.lb[0] : 0;
        B = d >= 2 ? g.S[d - 2] : 1;    OB = d >= 2 ? g.OS[d - 2] : 1;  lbB = d >= 2 ? g.lb[d - 2] : 0;
        L = g.S[d - 1];                 OL = g.OS[d - 1];               lbL = g.lb[d - 1];
    }
};

// Work units of a persistent kernel: (channel, chunk of `n_per_unit` images of the batch), dealt to `grid` CTAs; each of the
// `warps` consumer warps writes one grad_weight partial per chunk (`slots`).  `npu` is the family's proposed images per unit,
// rounded here to a multiple of the `np` images of one stage; units = chunks * C.  ok = false: a count overflows 32 bits.
struct UnitPlan { bool ok; int n_per_unit, chunks, units, grid, slots; };
inline UnitPlan plan_units(long long np, long long npu, long long N, long long C, long long grid_max, int warps) {
    UnitPlan u = {false, 0, 0, 0, 0, 0};
    npu = (npu / np) * np;
    if (npu < np) npu = np;
    if (npu > N) npu = N;
    const long long chunks = (N + npu - 1) / npu;
    const long long units = chunks * C;
    if (units > 0x7fffffffLL || chunks * warps > 0x7fffffffLL) return u;
    u.ok = true;
    u.n_per_unit = (int)npu;
    u.chunks = (int)chunks;
    u.units = (int)units;
    u.grid = (int)(units < grid_max ? units : grid_max);
    u.slots = (int)(chunks * warps);
    return u;
}

// Images per work unit (a multiple of `np`, the images of one stage).  A unit has a fixed cost (parameter fetch, the
// pipeline restart of its first stage, for the backward the shuffle tree and the partial store: measured ~0.4 plane
// times in the 2-D backward, ~0.1 in the forward), the last round of units leaves CTAs idle: pick the size that
// minimises  rounds * (images + unit_cost)  -- large units for small per-GPU batches, where one-image units made the
// 32-image shard of the 8-GPU strong-scaling run 60 % slower than its HBM floor.
inline long long pick_unit_images(long long N, long long C, long long np, long long grid, double unit_cost) {
    long long best = np < N ? np : N;
    double best_cost = 1e300;
    const long long kmax = (N + np - 1) / np < 4096 ? (N + np - 1) / np : 4096;
    for (long long k = 1; k <= kmax; ++k) {
        const long long npu = k * np < N ? k * np : N;
        const long long chunks = (N + npu - 1) / npu, units = chunks * C, rounds = (units + grid - 1) / grid;
        const double cost = (double)rounds * ((double)npu + unit_cost);
        if (cost < best_cost * (1.0 - 1e-9)) { best_cost = cost; best = npu; }
    }
    return best;
}

// ---- generic family (ts_generic.cu) ----------------------------------------------------------
struct GenericBwdPlan { int threads, tiles, n_per_chunk, units; };
GenericBwdPlan plan_generic_backward(const Geo& g);

int generic_gather(const Geo& g, int wk, const void* x, void* y, unsigned long long fill, int esize, const void* w,
                   int qkind, long long wzp, cudaStream_t s);
int generic_active_forward(const Geo& g, int dtype, const void* x, const void* w, void* y, cudaStream_t s);
int generic_backward(const Geo& g, const GenericBwdPlan& p, int dtype, int active, const void* grad, const void* x, const void* w,
                     void* gi, double* partials, cudaStream_t s);

// Every backward runs in two passes.  Pass 1 (the family's *_backward launcher) writes grad_input and `slots` fp64
// partial sums of each of the C x dim grad_weight values to `partials`; pass 2 (this) reduces them into gw, in a fixed
// order.  peers != nullptr: the pass-2 kernel is the variant fused with the all-reduce over peer memory
// (ts_shift_backward_allreduce); slots may be 0 (a rank with an empty shard contributes zeros).
int reduce_partials(const Geo& g, int dtype, const double* partials, int slots, void* gw, const ts_peer_group* peers, cudaStream_t s);

// ---- channels-last gather (ts_nhwc.cu): input and output keep the channel axis innermost -------
int nhwc_gather(const Geo& g, const void* x, void* y, unsigned long long fill, int esize, const void* w, int qkind,
                long long wzp, int sm_count, int max_grid_x, int variant, int ring_rows, bool emulate, cudaStream_t s);

int nhwc_to_planar(const void* x, void* y, long long N, long long C, long long P, int esize, cudaStream_t s);

// ---- channels-last float forward / backward (ts_nhwc_float.cu): 2-D, fp32 / fp16 / bf16, dense NHWC, C % 32 == 0 ----
// TS_ERR_UNSUPPORTED (nothing launched) for what they do not serve.  partials: cl_backward_workspace_bytes(); *slots: the
// partial slots the backward filled.
int cl_forward(const Geo& g, int dtype, int active, const void* x, const void* w, void* y, int sm_count, cudaStream_t s);
size_t cl_backward_workspace_bytes(const Geo& g, int dtype, int sm_count);
int cl_backward(const Geo& g, int dtype, int active, const void* grad, const void* x, const void* w, void* gi, double* partials,
                size_t workspace_bytes, int sm_count, int* slots, cudaStream_t s);

// ---- staged family (ts_staged.cu): bulk-async shared-memory staging ---------------------------
struct Tuning {
    int stages;        // ring depth
    int stage_kb;      // target bytes per stage (KiB)
    int warps;         // consumer warps per CTA
    int ctas_per_sm;   // persistent CTAs per SM
    int chunk_planes;  // planes of one channel per work unit (0 = auto)
    int tma_stages;    // ring depth of the TMA-tensor kernels (0 = auto)
    int tma_warps;     // consumer warps of the TMA-tensor arithmetic kernels
    int use_tma;       // 0: the automatic path choice never picks the TMA-tensor family
    int tma_stage_kb;  // target bytes per stage of the TMA-tensor kernels (0 = auto)
    int nhwc_variant;  // channels-last gather: 0 auto, 1 direct (L1) kernel only, 2 ring (shared-memory) kernel only
    int nhwc_rows_warps; // consumer warps of the row-pipelined channels-last kernel (0 = auto)
    int nhwc_ring_rows;  // cap on the ring slots of the channels-last ring kernel (0 = as many as fit)
    int use_halo;      // 0: the automatic path choice never picks the halo family
    int halo;          // halo rows / columns of the halo family (0 = 4)
    int halo_stages;   // ring depth of the halo family (0 = auto)
    int halo_warps;    // consumer warps of the 2-D halo kernels (0 = auto)
    int unit_order;    // 1 (default): units dealt round-robin over (chunk, channel); 0: contiguous channel-major ranges per CTA
                       // (measured on B200: 4 % faster for 32-image shards, 5 % slower for cfg3 at N=256)
    int use_flat;      // 0: the automatic path choice never picks the flat zero-padding gather
    int flat_ctas, flat_stage_kb, flat_stages, flat_warps;   // flat gather: CTAs per SM (0 = 2), stage KiB (0 = 24), ring depth (0 = 4), consumer warps (0 = auto)
    int cl_ahead, cl_rows;   // channels-last float kernels: steps of copies in flight (0 = 2, at most 4), rows per step (0 = 2; 1, 2, 4, 8)
};
Tuning& tuning();

struct SArgs {
    Geo g;
    const unsigned char* x;
    const unsigned char* grad;
    unsigned char* out;
    const void* w;
    double* partials;
    long long wzp;
    unsigned long long fill;
    int qkind, wk, es, mode, active;
    int A, B, L, OA, OB, OL, lbA, lbB, lbL;   // sizes per level (0 slab, 1 row, 2 column); absent levels 1 / 0
    int IA, IB;                               // iteration space: output space (forward) / input space (backward)
    int VB, V;                                // bytes / elements per item
    int gpr, GP;                              // items per iteration-space row; padded row length of the index space
    int TA, tiles;                            // slabs per tile, tiles per image
    int xs, gvs, gis;                         // slab slots per image: x, grad at the output position, grad for grad_input (0: shares gvs)
    int slab_x, slab_g;                       // bytes of one slab of x / of grad
    int np, stages, stage_stride, nw, n_per_unit, units, chunks, unit_order;
    int off_gv, off_gi;                       // byte offsets of the grad regions inside a stage (after GUARD)
    int table;                                // per-channel shift parameters tabulated in shared memory (arithmetic kernels, C <= TABLE_MAX_C)
    int img_items;                            // TA * IB * GP
    long long img_stride;                     // output bytes between consecutive images of one channel
    FastDiv d_img, d_GP, d_IB;
};
struct StagedPlan {
    bool ok;           // staged path applicable
    int grid, slots;   // slots = partial slots (backward)
    size_t smem_bytes;
    SArgs a;
};
// mode: 0 sparse/quantized forward (esize = element bytes), 1 active forward, 2 backward
StagedPlan plan_staged(const Geo& g, int mode, int active, int esize, int dtype, bool dense_x, const void* x, const void* y_or_gi,
                       const void* grad, int sm_count);

int staged_gather(const Geo& g, const StagedPlan& p, int wk, const void* x, void* y, unsigned long long fill, int esize,
                  const void* w, int qkind, long long wzp, cudaStream_t s);
int staged_active_forward(const Geo& g, const StagedPlan& p, int dtype, const void* x, const void* w, void* y, cudaStream_t s);
int staged_backward(const Geo& g, const StagedPlan& p, int dtype, int active, const void* grad, const void* x, const void* w,
                    void* gi, double* partials, cudaStream_t s);

// ---- TMA-tensor family (ts_tma.cu): zeros padding done by the copy engine ----------------------
struct alignas(64) TArgs {
    CUtensorMap map_x;       // x,    box {(TG+1)*vec, xb, xa, 1, np}
    CUtensorMap map_gs;      // grad, box {(TG+1)*vec, TB, TA, 1, np}     (backward)
    CUtensorMap map_gb;      // grad, box {(TG+1)*vec, xb, xa, 1, np}     (active backward)
    Geo g;
    unsigned char* out;
    const void* w;
    double* partials;
    long long wzp;
    int qkind, wk, es, vec;  // vec = elements per 16-byte group
    int mode, active;
    int OA, OB, OGR;         // output slabs, rows, 16-byte groups per row
    int lbA, lbB, lbL;
    int TA, TB, TG;          // tile extents (slabs, rows, groups)
    int xa, xb;              // x box slabs / rows (TA or TA+1, TB or TB+1)
    int tiles_b, tiles_g, tiles;
    int np;                  // images per stage (1 unless a whole plane is one tile)
    int x_img_chunks;        // 16-byte groups of one image's x box
    int g_img_chunks;        // 16-byte groups of one image's small grad box
    int off_gv, off_g2;      // byte offsets of the grad boxes inside a stage
    int tx_bytes;            // bytes landing per stage
    int stage_stride, stages, nw, n_per_unit, units, chunks, unit_order;
    int GP, img_items;       // padded groups per row of the item index space; items per image = TA*TB*GP
    int img_stride16;        // output distance between consecutive images of one channel, in 16-byte units
    int R, nchunk;           // strip-mined arithmetic kernels: rows per strip, strips per tile column
    FastDiv d_img, d_GP, d_TB, d_tg, d_tb, d_TG, d_nchunk, d_TA, d_C, d_chunks;
    int table;               // per-channel shift table in shared memory (C <= TABLE_MAX_C): built once per CTA
};
struct TmaPlan {
    bool ok;
    int grid, slots;
    size_t smem_bytes;
    TArgs a;
};
// mode: 0 sparse/quantized forward, 1 active forward, 2 backward (active = interpolating backward)
TmaPlan plan_tma(const Geo& g, int mode, int active, int esize, int dtype, bool dense_x, unsigned long long fill, const void* x,
                 const void* out, const void* grad, int sm_count);
int tma_gather(const Geo& g, const TmaPlan& p, int wk, const void* x, void* y, int esize, const void* w, int qkind, long long wzp,
               cudaStream_t s);
// dtype: TS_F32, or (2-D, fp32 weights: g.wf32) TS_F16 / TS_BF16
int tma_active_forward(const Geo& g, const TmaPlan& p, int dtype, const void* x, const void* w, void* y, cudaStream_t s);
int tma_backward(const Geo& g, const TmaPlan& p, int dtype, int active, const void* grad, const void* x, const void* w, void* gi,
                 double* partials, cudaStream_t s);

// rank-5 tensor map over a dense [N][C][A][B][L] tensor, box {bl, bb, ba, 1, bn} (memoised per thread); `map` points to a
// CUtensorMap (128 bytes, 64-byte aligned)
bool tma_available();
bool make_tensor_map5(void* map, const void* base, int es, long long N, long long C, int A, int B, int L, int bl, int bb, int ba, int bn);

// ---- flat gather (ts_flat.cu): zeros padding, no crop -> a linear shifted copy of each dense slab + byte masks ----
struct FArgs {
    Geo g;
    const unsigned char* x;
    unsigned char* y;
    const void* w;
    long long wzp;
    long long planes;          // N * C
    unsigned fillw;            // pad value replicated to 32 bits
    int qkind, wk, es, dim;
    int B, Lb;                 // rows per plane, bytes per row
    int plane_bytes, ipp;      // bytes / 16-byte items of one plane
    int K, stages, stage_stride, nw;
    int nstages;               // ceil(planes / K)
    int table;                 // per-channel (row shift, column shift in bytes) table in shared memory
    FastDiv d_ipp, d_Lb, d_C;
};
struct FlatPlan {
    bool ok;
    int grid;
    size_t smem_bytes;
    FArgs a;
};
FlatPlan plan_flat(const Geo& g, int esize, bool dense_x, const void* x, const void* y, int sm_count, bool forced);
int flat_gather(const Geo& g, const FlatPlan& p, int wk, const void* x, void* y, unsigned long long fill, int esize, const void* w,
                int qkind, long long wzp, cudaStream_t s);

// ---- halo family (ts_halo.cu): whole slabs staged WITH a padded halo, every item is interior ----
struct alignas(64) HArgs {
    CUtensorMap map_x;       // x,    box {px, bpx, 1, 1, 1}
    CUtensorMap map_g;       // grad, box {pg, bpg, 1, 1, 1}
    CUtensorMap map_v;       // grad, box {OL, OB, 1, 1, 1}   (dense slab: unshifted grad of the 3-D backward)
                             // fused avg-pool backward: the POOLED grad, box {PW, PH, 1, 1, 1}
    Geo g;
    const float* x;
    const float* grad;
    float* out;
    const float* w;
    double* partials;
    int mode, active, dim;
    int A, B, L, OA, OB, OL, lbA, lbB, lbL;   // per level (0 slab, 1 row, 2 column); 2-D: A = OA = 1
    int IA, IB, IG, GP;                       // iteration space (output space forward, input space backward): slabs, rows, groups; padded groups
    int RP;                                   // row pairs per slab = ceil(IB / 2)
    int hr, hc;                               // halo rows / columns on each side of a staged slab
    int px, bpx, pg, bpg;                     // row pitch (elements) and rows of the x / grad tiles in shared memory
    int tile_x, tile_g, tile_v;               // bytes between consecutive tiles (128-byte multiples)
    int box_x, box_g, box_v;                  // bytes one TMA box delivers
    int off_g, off_v;                         // byte offsets of the grad tiles / dense grad tiles inside a stage (after GUARD)
    int stage_stride, stages, nw, nt, np;
    int img_pairs, pairs;                     // RP * GP, np * RP * GP
    int n_per_unit, units, chunks, unit_order;
    long long out_plane_bytes;                // bytes of one (n, c) plane of the OUTPUT (pooled plane for the fused avg-pool epilogue)
    int pool;                                 // forward only: 2x2 / stride 2 / ceil_mode average pooling fused into the store
    int need_fix;                             // padding != zeros: a fixer warp patches the halo of every stage
    int table;                                // per-channel shift table in shared memory (C <= TABLE_MAX_C)
    FastDiv d_GP, d_img, d_C, d_chunks, d_PW;
    int nfix;                                 // fixer warps (1; 4 when they also expand the pooled gradient)
    int pool_bwd, PH, PW;                     // backward fused with the adjoint of avg_pool2d(2, 2, ceil_mode): pooled rows / columns
    int sA, PA;                               // 3-D fused avg-pool (forward and backward): slab stride (1 or 2), pooled slabs; 2-D: 1, 1
};
struct HaloPlan {
    bool ok;
    int grid, slots;
    size_t smem_bytes;
    HArgs a;
};
// mode: 0 sparse forward (2-D only), 1 active forward, 2 backward (active = interpolating backward).  fp32, dims 2 and 3,
// every padding, border crops.
// pool_bwd (mode 2, 2-D): `grad` is the gradient of the 2x2 / stride-2 / ceil_mode average pooling of the shift's output;
// the kernel expands it while staging (ts_shift2d_avgpool2_backward); halo_backward then launches the pooled kernels.
// pool_sa (3-D, mode 0..2): the plan of the kernels fused with avg_pool3d(kernel = stride = (pool_sa, 2, 2), ceil_mode);
// 0: no 3-D pooling (a 3-D sparse forward is then declined: those gathers stay on the other families).
HaloPlan plan_halo(const Geo& g, int mode, int active, int dtype, bool dense_x, const void* x, const void* out, const void* grad,
                   int sm_count, bool forced, bool pool_bwd = false, int pool_sa = 0);
int halo_active_forward(const Geo& g, const HaloPlan& p, const void* x, const void* w, void* y, cudaStream_t s);
int halo_forward2d(const Geo& g, const HaloPlan& p, int active, int pool, const void* x, const void* w, void* y, cudaStream_t s);
// 3-D forward of a pool_sa plan: y_pooled dense [N, C, ceil(O0 / pool_sa), ceil(O1 / 2), O2 / 2]
int halo_forward3d_pool(const Geo& g, const HaloPlan& p, int active, const void* x, const void* w, void* y, cudaStream_t s);
int halo_backward(const Geo& g, const HaloPlan& p, int active, const void* grad, const void* x, const void* w, void* gi,
                  double* partials, cudaStream_t s);

}  // namespace ts

/*
 * torchshifts_b200.h -- C ABI of the B200-native (sm_100a) Sparse/Active Shift operator.
 *
 * This is the drop-in boundary for the hot path of DeadAt0m/ActiveSparseShifts-PyTorch: the
 * per-backend kernels behind torch.ops.torchshifts._shift{1,2,3}d_forward/_backward.  Every
 * entry point takes plain pointers, sizes and a CUDA stream handle (no torch types) and only
 * ENQUEUES work on that stream; it never synchronises, never allocates, never touches the host
 * copy of any tensor.  The caller owns every buffer.  Return value: 0 (TS_OK) or a ts_status
 * code; ts_error_string() describes it.  No exceptions cross this boundary.
 *
 * Reference interfaces replaced (paths relative to torchshifts/csrc/ in the reference):
 *   ts_cuda_version          <- shifts::cuda_version()                 torchshifts.cpp:25-31
 *   ts_check_borders         <- shifts::ops::check_borders()           ops/shifts.cpp:93-135
 *   ts_shift_forward         <- shiftnd_forward<nD,pad,active>()       ops/cuda/shifts_cuda.cu:202-266
 *                               (= ops/cpu/shifts_cpu.cpp:214-232, the oracle semantics)
 *   ts_shift_backward        <- shiftnd_backward<nD,pad,active>()      ops/cuda/shifts_cuda.cu:268-345
 *                               (= ops/cpu/shifts_cpu.cpp:235-255)
 *   ts_qshift_forward        <- qshiftnd<nD,pad>()                     ops/quantized/shifts_quantized.cpp:107-130
 *                               (the reference has no CUDA quantized kernel; this adds one)
 *
 * Semantics (identical to the reference CPU path, see DESIGN.md):
 *   - tensors are [N, C, S0(, S1(, S2))], last axis fastest; `x` may have arbitrary element
 *     strides, every output (y, grad_input, grad_weight) and `grad` is dense;
 *   - weights are [C, dim] dense, same dtype as x -- or fp32 for an fp16 / bf16 x when the dtype argument carries
 *     TS_WEIGHTS_F32 (mixed precision: grad_weight is then fp32 too); the integer/fractional split
 *     (round-half-even for the sparse shift, floor for the active shift; the backward variant of
 *     ops/cpu/shifts_cpu.cpp:242-244) happens inside the kernels;
 *   - padding modes 0 zeros, 1 border, 2 periodic, 3 reflect, 4 symmetric
 *     (ops/kernels/shifts_kernels.h:5-29);
 *   - lb/rb are the validated borders in input coordinates produced by ts_check_borders.
 */
#ifndef TORCHSHIFTS_B200_H
#define TORCHSHIFTS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TS_ABI_VERSION 2

typedef enum ts_status {
    TS_OK = 0,
    TS_ERR_INVALID_ARGUMENT = 1,   /* bad dim / padding / dtype / null pointer / negative size   */
    TS_ERR_UNSUPPORTED = 2,        /* valid request that this build has no kernel for             */
    TS_ERR_WORKSPACE = 3,          /* workspace pointer null, misaligned or too small             */
    TS_ERR_TOO_LARGE = 4,          /* a single (n,c) plane has >= 2^31 elements                   */
    TS_ERR_BORDERS = 5,            /* borders would give a negative output size (reference dies)  */
    TS_ERR_CUDA = 6,               /* a CUDA runtime call / launch failed: see ts_last_cuda_error */
    TS_ERR_NO_DEVICE = 7           /* no CUDA device: there is NO CPU fallback                    */
} ts_status;

typedef enum ts_dtype {            /* element type of x / y / grad / weights                      */
    TS_F32 = 0, TS_F64 = 1, TS_F16 = 2, TS_BF16 = 3
} ts_dtype;

/* Flag OR'd into the `dtype` argument of the float entry points (ts_shift_forward, ts_shift_backward,
 * ts_shift_backward_allreduce, ts_shift_backward_workspace_bytes, ts_shift_forward_nhwc, ts_shift_backward_nhwc,
 * ts_shift_backward_nhwc_workspace_bytes, ts_shift2d_avgpool2_forward / _backward): `weights` is fp32 [C, dim] and
 * grad_weight is written fp32, while x / y / grad / grad_input stay TS_F16 or TS_BF16 (mixed-precision training with fp32
 * master weights).  The weights are split in fp32, never rounded to 16 bits.  Only with TS_F16 or TS_BF16: any other
 * combination is TS_ERR_INVALID_ARGUMENT (the workspace queries return 0). */
#define TS_WEIGHTS_F32 0x100

typedef enum ts_padding {
    TS_PAD_ZEROS = 0, TS_PAD_BORDER = 1, TS_PAD_PERIODIC = 2, TS_PAD_REFLECT = 3, TS_PAD_SYMMETRIC = 4
} ts_padding;

typedef enum ts_qweight_kind {     /* storage of the raw integer shift weights (int_repr)         */
    TS_QW_U8 = 0, TS_QW_I8 = 1, TS_QW_I32 = 2
} ts_qweight_kind;

typedef enum ts_kernel_path {      /* which kernel family served the last call (diagnostics)      */
    TS_PATH_NONE = 0,
    TS_PATH_GENERIC = 1,           /* stride-generic one-element-per-thread kernels               */
    TS_PATH_STAGED = 2,            /* bulk-async (cp.async.bulk + mbarrier) shared-memory staged  */
    TS_PATH_TMA = 3,               /* TMA tensor copies: the copy engine applies shift + zero pad  */
    TS_PATH_NHWC = 4,              /* channels-last in, channels-last out (ts_qshift_forward_nhwc,
                                      ts_shift_forward_nhwc, ts_shift_backward_nhwc)                */
    TS_PATH_HALO = 5,              /* slabs staged with a padded halo (TMA tensor loads), all-interior
                                      arithmetic: fp32 active forward / backward, every padding, crops  */
    TS_PATH_FLAT = 6               /* zeros padding, no crop: linear shifted copy of each dense slab with
                                      byte masks (sparse / quantized forward, any row length)           */
} ts_kernel_path;

/* Geometry of one call.  Unused spatial axes: size 1, stride 0, lb 0, rb 1. */
typedef struct ts_geometry {
    int32_t dim;                   /* number of shifted axes: 1, 2 or 3                           */
    int32_t reserved;
    int64_t N, C;
    int64_t size[3];               /* input spatial sizes S0,S1,S2                                */
    int64_t x_stride[5];           /* input strides in ELEMENTS for (N, C, S0, S1, S2)            */
    int64_t lb[3], rb[3];          /* output window in input coordinates; output size rb-lb       */
} ts_geometry;

/* ---- library / diagnostics ------------------------------------------------------------------ */
int          ts_abi_version(void);
int          ts_cuda_version(void);            /* CUDART_VERSION this library was built with      */
const char*  ts_error_string(int status);
const char*  ts_last_cuda_error(void);         /* text of the last CUDA error seen by this thread */
int          ts_last_kernel_path(void);        /* ts_kernel_path of this thread's last launch     */
int          ts_set_kernel_path(int path);     /* 0 auto (default), 1 force generic, 2 force staged,
                                                  3 force TMA, 5 force halo, 6 force flat (calls fail with TS_ERR_UNSUPPORTED
                                                  when the forced family does not apply; the channels-last
                                                  float entry points always do); returns
                                                  the old value                                   */
uint64_t     ts_launch_count(void);            /* kernels launched by this library so far         */
int          ts_set_tuning(const char* spec);  /* "key=value,..." staged-path tuning knobs; see
                                                  DESIGN.md.  Returns TS_OK or INVALID_ARGUMENT   */

/* ---- host-side logic ------------------------------------------------------------------------ */
/* user_borders: dim*2 values (left_cut, right_cut per axis) or NULL.  Writes lb[3], rb[3].       */
int ts_check_borders(int dim, const int64_t* sizes, const int64_t* user_borders,
                     int64_t lb[3], int64_t rb[3]);

/* Pure host mirrors of the device index / weight arithmetic (used by the CPU-side tests to pin
 * the device code's formulas without a GPU). */
int     ts_debug_remap(int padding, int len, int idx);                 /* literal reference formula */
int     ts_debug_remap_reduced(int padding, int len, int pos, int64_t shift, int plus);
                                                                       /* division-free device form */
void    ts_debug_split_f32(int backward, int active, float w, int64_t* iw, float* dw);
void    ts_debug_split_f64(int backward, int active, double w, int64_t* iw, double* dw);

/* ---- device entry points (pointers are DEVICE pointers) ------------------------------------- */
int ts_shift_forward(const ts_geometry* g, int dtype, int padding, int active,
                     const void* x, const void* weights, void* y, void* stream);

/* Shift2d forward fused with the average pooling the reference module applies to a strided depth-wise-conv emulation
 * (modules/shifts.py:85-89, :153: avg_pool2d(kernel_size=stride, stride=stride, ceil_mode=True) after the shift and the
 * border crop), for stride 2: y_pooled is dense [N, C, ceil(O0/2), O1/2]; every window's elements are added in row-major
 * order and divided by their count (2 for the last row of an odd O0), like ATen's kernel.  One read of x, one
 * quarter-size write.  fp32, dim 2, dense x, O1 a multiple of 4: otherwise TS_ERR_UNSUPPORTED (callers then run
 * ts_shift_forward and pool separately).  Replaces the pair shiftnd_forward + at::avg_pool2d on that path. */
int ts_shift2d_avgpool2_forward(const ts_geometry* g, int dtype, int padding, int active,
                                const void* x, const void* weights, void* y_pooled, void* stream);

size_t ts_shift_backward_workspace_bytes(const ts_geometry* g, int dtype);

/* Backward of ts_shift2d_avgpool2_forward in ONE pass: grad_pooled is the gradient of the pooled output, dense
 * [N, C, ceil(O0/2), O1/2]; the adjoint of the pooling (ATen's avg_pool2d_backward: every element of a window receives
 * grad / count) is applied while the gradient is staged in shared memory, so the full-size gradient of the shift's output
 * is never written to or read from HBM (2.25 instead of 4.25 tensor passes for the layer's backward).  g describes the
 * SHIFT (x sizes, crop), exactly as for the forward; grad_input / grad_weight / workspace as for ts_shift_backward (the same
 * ts_shift_backward_workspace_bytes).  fp32, dim 2, dense x, O1 a multiple of 8, planes that fit a stage: otherwise
 * TS_ERR_UNSUPPORTED (callers then expand with avg_pool2d_backward and call ts_shift_backward).  Replaces the pair
 * at::avg_pool2d_backward + shiftnd_backward of modules/shifts.py:85-89 on that path. */
int ts_shift2d_avgpool2_backward(const ts_geometry* g, int dtype, int padding, int active,
                                 const void* grad_pooled, const void* x, const void* weights,
                                 void* grad_input, void* grad_weight,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* grad: dense [N,C,rb-lb]; grad_input: dense like x's logical shape; grad_weight: dense [C,dim]
 * in the weights' type (`dtype`, or fp32 under TS_WEIGHTS_F32), fully overwritten (deterministic two-pass reduction, no atomics).
 * workspace: >= ts_shift_backward_workspace_bytes(), 16-byte aligned. */
int ts_shift_backward(const ts_geometry* g, int dtype, int padding, int active,
                      const void* grad, const void* x, const void* weights,
                      void* grad_input, void* grad_weight,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Backward fused with the path's one collective: the deterministic pass-2 reduction of grad_weight
 * publishes this rank's C x dim result to every peer over NVLink peer memory and sums the `world`
 * contributions in rank order -- grad_weight leaves the call already all-reduced (sum), identical on
 * every rank, with no NCCL launch.  A contribution travels as one 64-bit word {call epoch : fp32 value}
 * written with a single 8-byte peer store; the receiver polls that word (no separate flag, no fence).
 *   bufs[p]   device pointer, valid on THIS device, to rank p's exchange buffer:
 *             2 (epoch parity) x world x capacity uint64 words, zero before the first call;
 *   state     THIS rank's private device words: 129 uint32, zero before the first call (per-CTA call
 *             counters; word 128 receives the epoch of a call that timed out).  The call counter lives on
 *             the device, so nothing call-specific crosses the ABI and the launch can be captured in a CUDA
 *             graph and replayed;
 *   timeout_ns  how long a rank waits for its peers before it records the failure and traps (0 = for ever).
 * Every rank must make the same sequence of calls with the same C x dim (replicated layers), one stream at
 * a time per peer group.  A rank whose shard is empty (N == 0) must still call: it contributes zeros.
 * dtype: TS_F32 / TS_F16 / TS_BF16 (contributions travel as fp32); capacity <= 4096. */
typedef struct ts_peer_group {
    int32_t  world, rank;          /* 1 <= world <= 8                                              */
    int32_t  capacity;             /* words per rank slot; C * dim must not exceed it              */
    int32_t  reserved;
    uint64_t timeout_ns;
    void*    bufs[8];
    void*    state;
} ts_peer_group;

int ts_shift_backward_allreduce(const ts_geometry* g, int dtype, int padding, int active,
                                const void* grad, const void* x, const void* weights,
                                void* grad_input, void* grad_weight,
                                void* workspace, size_t workspace_bytes,
                                const ts_peer_group* peers, void* stream);

/* Shift forward fused with the average pooling of a strided depth-wise-conv emulation (modules/shifts.py:85-89:
 * avg_poolNd(kernel_size=stride, stride=stride, ceil_mode=True) after the shift and the border crop), for the strides in
 * `stride` (g->dim entries): dim 2: (2, 2), the kernels of ts_shift2d_avgpool2_forward; dim 3: (1, 2, 2) or (2, 2, 2).
 * y_pooled is dense [N, C, ceil(O0/s0), ceil(O1/s1)(, ceil(O2/s2))]; every window's elements are added in (slab,) row,
 * column order into one fp32 sum and divided by their count, like ATen's kernels (bit-identical).  One read of x, one
 * pooled write.  fp32 (no TS_WEIGHTS_F32), dense x, input and output rows of a multiple of 4 elements, planes that fit a
 * stage; any other stride or shape: TS_ERR_UNSUPPORTED, nothing launched (callers then shift and pool separately).  A
 * stride entry below 1, a null pointer or a bad dtype: TS_ERR_INVALID_ARGUMENT. */
int ts_shift_avgpool_forward(const ts_geometry* g, int dtype, int padding, int active, const int32_t* stride,
                             const void* x, const void* weights, void* y_pooled, void* stream);

/* Workspace of ts_shift_avgpool_backward: enough for every stride and padding it serves on this geometry (16 when it
 * serves none). */
size_t ts_shift_avgpool_backward_workspace_bytes(const ts_geometry* g, int dtype);

/* Backward of ts_shift_avgpool_forward in ONE kernel plus the pass-2 reduction: grad_pooled is the gradient of the pooled
 * output; the adjoint of the pooling (every element of a window receives grad / count, as ATen's avg_poolNd_backward; the
 * count is a power of two, so this is exact) is applied while the gradient is staged in shared memory, so the full-size
 * gradient of the shift's output never exists in HBM.  grad_input / grad_weight as for ts_shift_backward; workspace: at least
 * ts_shift_avgpool_backward_workspace_bytes(), 16-byte aligned.  peers: NULL, or the peer group of an in-kernel grad_weight
 * exchange, with the rules of ts_shift_backward_allreduce.  Besides the forward's conditions, pooled rows of a multiple of
 * 16 bytes (O_last a multiple of 8); empty tensors: TS_ERR_UNSUPPORTED (callers take the two-step path, which zero-fills or
 * exchanges). */
int ts_shift_avgpool_backward(const ts_geometry* g, int dtype, int padding, int active, const int32_t* stride,
                              const void* grad_pooled, const void* x, const void* weights,
                              void* grad_input, void* grad_weight, void* workspace, size_t workspace_bytes,
                              const ts_peer_group* peers, void* stream);

/* Quantized forward on the raw integer representation.  elem_bytes: 1 (qint8/quint8) or
 * 4 (qint32).  zero_point: input zero point = pad value.  qweights: raw integer weights
 * [C,dim] of kind `qweight_kind`; effective shift = qweights - weight_zero_point. */
int ts_qshift_forward(const ts_geometry* g, int elem_bytes, int padding, int64_t zero_point,
                      const void* xq, const void* qweights, int qweight_kind,
                      int64_t weight_zero_point, void* yq, void* stream);

/* Channels-last variant of ts_qshift_forward      <- shift_forward_kernel_nhwdc_q, ops/kernels/shifts_kernels.h:574-624,
 * driven from ops/quantized/shifts_quantized.cpp:119-125 (the output takes the input's memory format).
 * xq is read through g->x_stride (channel stride 1 for a channels-last tensor); yq is written DENSE
 * channels-last: element (n, c, o0, o1, o2) lives at (((n*O0 + o0)*O1 + o1)*O2 + o2)*C + c.  One read and
 * one write of the tensor, no layout conversion on either side. */
int ts_qshift_forward_nhwc(const ts_geometry* g, int elem_bytes, int padding, int64_t zero_point,
                           const void* xq, const void* qweights, int qweight_kind,
                           int64_t weight_zero_point, void* yq, void* stream);

/* Channels-last float forward and backward: tensors keep the channel axis innermost, no layout pass on either side.
 * x dense channels-last (read through g->x_stride, channel stride 1); y dense [N, O0, O1(, O2), C];
 * grad dense [N, O0, O1(, O2), C]; grad_input dense [N, S0, S1(, S2), C]; grad_weight dense [C, dim] in dtype,
 * fully overwritten (deterministic two-pass reduction).  TS_ERR_UNSUPPORTED for what the kernels do not serve
 * (dim 3, fp64, C not a multiple of 32, rows too wide to stage, misaligned pointers, empty tensors, a forced kernel
 * family: see ts_set_kernel_path); callers then run the planar entry points and convert the layout.
 * peers: NULL, or the exchange of ts_shift_backward_allreduce (same rules).  workspace: 16-byte aligned, at least
 * ts_shift_backward_nhwc_workspace_bytes(). */
int    ts_shift_forward_nhwc(const ts_geometry* g, int dtype, int padding, int active,
                             const void* x, const void* weights, void* y, void* stream);
size_t ts_shift_backward_nhwc_workspace_bytes(const ts_geometry* g, int dtype);
int    ts_shift_backward_nhwc(const ts_geometry* g, int dtype, int padding, int active,
                              const void* grad, const void* x, const void* weights,
                              void* grad_input, void* grad_weight, void* workspace, size_t workspace_bytes,
                              const ts_peer_group* peers /* NULL: no exchange */, void* stream);

/* Layout adapter of the float path: x dense channels-last ([N, P, C] in memory, P = product of the spatial
 * sizes) -> y dense planar ([N, C, P]).  The reference hands channels-last float inputs to its nhwdc bodies
 * and returns planar tensors (ops/cpu/shifts_cpu.cpp:55-75, :221); here the planar bandwidth kernels serve
 * them after this one pass.  elem_bytes: 2, 4 or 8. */
int ts_nhwc_to_nchw(const void* x, void* y, int64_t N, int64_t C, int64_t P, int elem_bytes, void* stream);

/* Test aid (HOST pointers, no GPU work): walks every (block, thread) of the launch
 * ts_qshift_forward_nhwc would make on a device with `sm_count` SMs and runs the kernel's own per-thread
 * program on the host (barrier-separated phases in order, shared memory as a host buffer), so the
 * CPU-side tests can pin its index logic against the oracle.  Refuses tensors above 2^22 elements;
 * max_grid_x > 0 caps the grid to exercise the grid-stride loops; variant: 0 automatic choice, 1 the
 * direct (L1) kernel, 2 the ring (shared-memory) kernel or TS_ERR_UNSUPPORTED; ring_rows > 0 caps the
 * ring so small cases exercise its wrap-around and the global-memory fall-back. */
int ts_debug_nhwc_emulate(const ts_geometry* g, int elem_bytes, int padding, int64_t zero_point,
                          const void* xq_host, const void* qweights_host, int qweight_kind,
                          int64_t weight_zero_point, void* yq_host, int sm_count, int max_grid_x,
                          int variant, int ring_rows);

/* Test aid: no GPU work.  Runs the planar entry points' own route() for a call -- current forced path and tuning knobs,
 * this device's SM count, placeholder 256-byte-aligned pointers -- and writes what it chose:
 * out[0] path, then the plan's tiles_per_plane, tiles per level (a, b, g), images per stage, images per unit, units, grid,
 * stages, consumer warps, partial slots, table (0/1).  op: 0 sparse/quantized forward, 1 active forward, 2 backward.
 * dtype as for ts_shift_forward (TS_WEIGHTS_F32 allowed), or -1 with elem_bytes for the quantized forward (zero point 0).
 * n_out >= 13.  Fields a family does not have are 0 (the flat gather: images per stage counts (n, c) planes).
 * Returns the status the entry point's routing would return. */
int ts_debug_route(const ts_geometry* g, int op, int dtype, int elem_bytes, int padding, int active, int64_t* out, int n_out);

#ifdef __cplusplus
}
#endif
#endif /* TORCHSHIFTS_B200_H */

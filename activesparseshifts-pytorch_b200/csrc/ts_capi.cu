// ts_capi.cu -- the C ABI of include/torchshifts_b200.h: argument validation, host-side border
// logic, kernel-family routing, the backward's pass 2 and launch bookkeeping.  No torch types, no
// allocation, no synchronisation; every entry point only enqueues kernels on the caller's stream.
#include <atomic>
#include <mutex>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "ts_kernels.h"

namespace ts {

static std::atomic<unsigned long long> g_launches{0};
static std::atomic<int> g_forced_path{0};
static std::atomic<unsigned> g_tuning_epoch{0};     // bumped by ts_set_tuning: invalidates memoised plans
static thread_local int t_last_path = TS_PATH_NONE;
static thread_local char t_cuda_error[256] = "";

void note_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
void note_error(const char* text) { snprintf(t_cuda_error, sizeof(t_cuda_error), "%s", text); }

int check_launch() {
    const cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) return TS_OK;
    snprintf(t_cuda_error, sizeof(t_cuda_error), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
    return TS_ERR_CUDA;
}

bool ensure_dynamic_smem(const void* func, size_t bytes) {
    // The attribute belongs to the (function, device) pair of the PROCESS: the memo is shared by all threads (autograd runs
    // backward kernels on its own threads -- a per-thread memo let one thread lower the limit another thread relied on)
    // and the limit only ever grows.
    struct Slot { const void* func; int dev; size_t bytes; };
    static std::mutex mu;
    static Slot seen[256];
    static int used = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    std::lock_guard<std::mutex> lock(mu);
    int i = 0;
    for (; i < used; ++i)
        if (seen[i].func == func && seen[i].dev == dev) break;
    if (i < used && seen[i].bytes >= bytes) return true;
    if (cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return false;
    if (i == used) {
        if (used == 256) return true;         // table full: keep setting the attribute per launch for the rest
        ++used;
    }
    seen[i] = Slot{func, dev, bytes};
    return true;
}

static int cuda_fail(cudaError_t e) {
    snprintf(t_cuda_error, sizeof(t_cuda_error), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
    return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? TS_ERR_NO_DEVICE : TS_ERR_CUDA;
}

static int sm_count(int* out) {
    static std::atomic<int> cached[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return cuda_fail(e);
    if (dev >= 0 && dev < 64 && cached[dev].load() > 0) { *out = cached[dev].load(); return TS_OK; }
    int n = 0;
    e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return cuda_fail(e);
    if (dev >= 0 && dev < 64) cached[dev].store(n);
    *out = n;
    return TS_OK;
}

static int make_geo(const ts_geometry* in, int padding, Geo* g) {
    if (!in) return TS_ERR_INVALID_ARGUMENT;
    if (in->dim < 1 || in->dim > 3) return TS_ERR_INVALID_ARGUMENT;
    if (padding < 0 || padding > 4) return TS_ERR_INVALID_ARGUMENT;
    if (in->N < 0 || in->C < 0) return TS_ERR_INVALID_ARGUMENT;
    g->dim = in->dim;
    g->pad = padding;
    g->wf32 = 0;
    g->N = in->N;
    g->C = in->C;
    long long ip = 1, op = 1;
    for (int a = 0; a < 3; ++a) {
        const long long S = a < in->dim ? in->size[a] : 1;
        const long long lb = a < in->dim ? in->lb[a] : 0;
        const long long rb = a < in->dim ? in->rb[a] : 1;
        if (S < 0 || lb < 0 || rb > S || rb < lb) return TS_ERR_INVALID_ARGUMENT;
        if (S >= 0x7fffffffLL) return TS_ERR_TOO_LARGE;
        g->S[a] = (int)S;
        g->lb[a] = (int)lb;
        g->OS[a] = (int)(rb - lb);
        ip *= S;
        op *= (rb - lb);
        if (ip >= 0x7fffffffLL) return TS_ERR_TOO_LARGE;
    }
    for (int a = 0; a < 5; ++a) g->xs[a] = (a < 2 + in->dim) ? in->x_stride[a] : 0;
    g->in_plane = ip;
    g->out_plane = op;
    return TS_OK;
}

static bool x_is_dense(const Geo& g) {
    long long expect = 1;
    for (int a = g.dim - 1; a >= 0; --a) {
        if (g.S[a] != 1 && g.xs[2 + a] != expect) return false;
        expect *= g.S[a];
    }
    if (g.C != 1 && g.xs[1] != expect) return false;
    expect *= g.C;
    if (g.N != 1 && g.xs[0] != expect) return false;
    return true;
}

static int elem_size(int dtype) {
    switch (dtype) {
    case TS_F32: return 4;
    case TS_F64: return 8;
    case TS_F16: case TS_BF16: return 2;
    }
    return 0;
}

// The dtype argument of the float entry points: the element type, possibly OR'd with TS_WEIGHTS_F32 (fp16 / bf16 x with fp32
// weights and grad_weight; sets g->wf32).  -> the element type, or -1 for TS_WEIGHTS_F32 with any other element type.
static int weights_f32(int dtype, Geo* g) {
    if (!(dtype & TS_WEIGHTS_F32)) return dtype;
    dtype &= ~TS_WEIGHTS_F32;
    if (dtype != TS_F16 && dtype != TS_BF16) return -1;
    g->wf32 = 1;
    return dtype;
}

// grad_weight's type: the weights'
static int gw_dtype(const Geo& g, int dtype) { return g.wf32 ? TS_F32 : dtype; }

// Tuning knobs (ts_set_tuning): 0 = automatic, the planners pick per-mode defaults.
Tuning& tuning() {
    static Tuning t = [] {
        Tuning d;
        memset(&d, 0, sizeof(d));
        d.warps = 15;
        d.ctas_per_sm = 1;
        d.use_tma = d.use_halo = d.use_flat = 1;
        d.unit_order = 1;
        return d;
    }();
    return t;
}

// ---- kernel-family routing of the planar entry points -----------------------------------------
// One call as the planners see it.
struct Call {
    int mode;                   // 0 sparse / quantized forward, 1 active forward, 2 backward
    int active, esize, dtype;   // dtype -1: quantized (esize bytes per element)
    unsigned long long fill;    // quantized: the bit pattern of the zero point
    const void *x, *out, *grad; // out: y or grad_input; grad: null in a forward
};

struct Route {
    int path;                   // TS_PATH_* of the family that serves the call, with its plan
    TmaPlan tma;
    HaloPlan halo;
    FlatPlan flat;
    StagedPlan staged;
    GenericBwdPlan generic;
    int slots;                  // backward: partial slots pass 1 fills
};

// The families each operation tries, in order of preference.  3-D interpolating backward, automatic choice: the
// slab-streaming halo kernel (every slab staged once, windows of the previous slab in registers) beats the TMA family's
// tile kernel under zeros padding as well (cfg4: 0.50 against 0.55 ms).
static const int GATHER[] = {TS_PATH_TMA, TS_PATH_FLAT, TS_PATH_STAGED, TS_PATH_GENERIC};        // sparse and quantized forward
static const int ARITHMETIC[] = {TS_PATH_TMA, TS_PATH_HALO, TS_PATH_STAGED, TS_PATH_GENERIC};    // active forward, backward
static const int HALO_FIRST[] = {TS_PATH_HALO, TS_PATH_TMA, TS_PATH_STAGED, TS_PATH_GENERIC};

// Plans family `path` for `c`: false when it declines (the generic family never does).  forced: plan_halo / plan_flat take
// small planes too; pool: the pooled halo backward of ts_shift2d_avgpool2_backward.
static bool plan(int path, const Geo& g, const Call& c, bool dense_x, int sms, bool forced, bool pool, Route* r) {
    r->slots = 0;
    switch (path) {
    case TS_PATH_TMA:
        r->tma = plan_tma(g, c.mode, c.active, c.esize, c.dtype, dense_x, c.fill, c.x, c.out, c.grad, sms);
        r->slots = r->tma.slots;
        return r->tma.ok;
    case TS_PATH_HALO:
        r->halo = plan_halo(g, c.mode, c.active, c.dtype, dense_x, c.x, c.out, c.grad, sms, forced, pool);
        r->slots = r->halo.slots;
        return r->halo.ok;
    case TS_PATH_FLAT:
        r->flat = plan_flat(g, c.esize, dense_x, c.x, c.out, sms, forced);
        return r->flat.ok;
    case TS_PATH_STAGED:
        r->staged = plan_staged(g, c.mode, c.active, c.esize, c.dtype, dense_x, c.x, c.out, c.grad, sms);
        r->slots = r->staged.slots;
        return r->staged.ok;
    }
    if (c.mode == 2) {
        r->generic = plan_generic_backward(g);
        r->slots = r->generic.units;
    }
    return true;
}

// Automatic choice: the first family of the list whose use_* knob is on and whose plan is ok.  Under ts_set_kernel_path
// only the forced family is planned: TS_ERR_UNSUPPORTED when it is not in the list or declines.
static int route(const Geo& g, const Call& c, int sms, Route* r) {
    const int forced = g_forced_path.load();
    const int* list = c.mode == 0 ? GATHER : c.mode == 2 && c.active && g.dim == 3 && forced == TS_PATH_NONE ? HALO_FIRST : ARITHMETIC;
    const Tuning& t = tuning();
    const bool dense_x = x_is_dense(g);
    for (int i = 0; i < 4; ++i) {
        const int path = list[i];
        const bool on = path == TS_PATH_TMA ? t.use_tma : path == TS_PATH_HALO ? t.use_halo : path == TS_PATH_FLAT ? t.use_flat : true;
        if (forced == TS_PATH_NONE ? !on : path != forced) continue;
        if (plan(path, g, c, dense_x, sms, forced == path, false, r)) {
            r->path = path;
            return TS_OK;
        }
        if (forced != TS_PATH_NONE) break;
    }
    return TS_ERR_UNSUPPORTED;
}

}  // namespace ts

using namespace ts;

extern "C" {

int ts_abi_version(void) { return TS_ABI_VERSION; }
int ts_cuda_version(void) { return CUDART_VERSION; }

const char* ts_error_string(int status) {
    switch (status) {
    case TS_OK: return "ok";
    case TS_ERR_INVALID_ARGUMENT: return "invalid argument (dim must be 1..3, padding 0..4, sizes/borders consistent, pointers non-null)";
    case TS_ERR_UNSUPPORTED: return "unsupported request (no kernel for this element type / forced kernel path not applicable)";
    case TS_ERR_WORKSPACE: return "backward workspace missing, misaligned or smaller than ts_shift_backward_workspace_bytes()";
    case TS_ERR_TOO_LARGE: return "a single (n,c) plane must have fewer than 2^31 elements";
    case TS_ERR_BORDERS: return "borders produce a negative output dimension";
    case TS_ERR_CUDA: return "CUDA error (see ts_last_cuda_error())";
    case TS_ERR_NO_DEVICE: return "no CUDA device available: torchshifts-b200 has no CPU fallback";
    }
    return "unknown status";
}

const char* ts_last_cuda_error(void) { return t_cuda_error; }
int ts_last_kernel_path(void) { return t_last_path; }
int ts_set_kernel_path(int path) {
    if (path < 0 || path > 6 || path == TS_PATH_NHWC) return -1;
    return g_forced_path.exchange(path);
}
uint64_t ts_launch_count(void) { return (uint64_t)g_launches.load(); }

int ts_set_tuning(const char* spec) {
    if (!spec) return TS_ERR_INVALID_ARGUMENT;
    Tuning t = tuning();
    const char* p = spec;
    while (*p) {
        char key[32];
        int val = 0, n = 0;
        if (sscanf(p, " %31[a-z_]=%d%n", key, &val, &n) != 2) return TS_ERR_INVALID_ARGUMENT;
        if (!strcmp(key, "stages")) t.stages = val;
        else if (!strcmp(key, "stage_kb")) t.stage_kb = val;
        else if (!strcmp(key, "warps")) t.warps = val;
        else if (!strcmp(key, "ctas_per_sm")) t.ctas_per_sm = val;
        else if (!strcmp(key, "chunk_planes")) t.chunk_planes = val;
        else if (!strcmp(key, "tma_stages")) t.tma_stages = val;
        else if (!strcmp(key, "tma_warps")) t.tma_warps = val;
        else if (!strcmp(key, "use_tma")) t.use_tma = val != 0;
        else if (!strcmp(key, "tma_stage_kb")) t.tma_stage_kb = val;
        else if (!strcmp(key, "nhwc_variant")) t.nhwc_variant = val;
        else if (!strcmp(key, "nhwc_ring_rows")) t.nhwc_ring_rows = val;
        else if (!strcmp(key, "nhwc_rows_warps")) t.nhwc_rows_warps = val;
        else if (!strcmp(key, "use_halo")) t.use_halo = val != 0;
        else if (!strcmp(key, "halo")) t.halo = val;
        else if (!strcmp(key, "halo_stages")) t.halo_stages = val;
        else if (!strcmp(key, "halo_warps")) t.halo_warps = val;
        else if (!strcmp(key, "unit_order")) t.unit_order = val != 0;
        else if (!strcmp(key, "use_flat")) t.use_flat = val != 0;
        else if (!strcmp(key, "flat_ctas")) t.flat_ctas = val;
        else if (!strcmp(key, "flat_stage_kb")) t.flat_stage_kb = val;
        else if (!strcmp(key, "flat_stages")) t.flat_stages = val;
        else if (!strcmp(key, "flat_warps")) t.flat_warps = val;
        else if (!strcmp(key, "cl_ahead")) t.cl_ahead = val;
        else if (!strcmp(key, "cl_rows")) t.cl_rows = val;
        else return TS_ERR_INVALID_ARGUMENT;
        p += n;
        while (*p == ',' || *p == ' ') ++p;
    }
    if (t.stages < 0 || t.stages > 8 || t.stage_kb < 0 || t.stage_kb > 220 || t.warps < 1 || t.warps > 31 ||
        t.ctas_per_sm < 1 || t.ctas_per_sm > 8 || t.chunk_planes < 0 || t.tma_stages < 0 || t.tma_stages > 32 ||
        t.tma_warps < 0 || t.tma_warps > 31 || t.tma_stage_kb < 0 ||
        t.tma_stage_kb > 220 || t.nhwc_variant < 0 || t.nhwc_variant > 3 || t.nhwc_ring_rows < 0 || t.nhwc_rows_warps < 0 || t.nhwc_rows_warps > 12 || t.halo < 0 || t.halo > 16 ||
        t.halo_stages < 0 || t.halo_stages > 32 || t.halo_warps < 0 || t.halo_warps > 15 || t.flat_ctas < 0 || t.flat_ctas > 8 ||
        t.flat_stage_kb < 0 || t.flat_stage_kb > 100 || t.flat_stages < 0 || t.flat_stages > 16 || t.flat_warps < 0 || t.flat_warps > 15 ||
        t.cl_ahead < 0 || t.cl_ahead > 4 || (t.cl_rows != 0 && t.cl_rows != 1 && t.cl_rows != 2 && t.cl_rows != 4 && t.cl_rows != 8))
        return TS_ERR_INVALID_ARGUMENT;
    tuning() = t;
    g_tuning_epoch.fetch_add(1);
    return TS_OK;
}

// ---- host logic ------------------------------------------------------------------------------
int ts_check_borders(int dim, const int64_t* sizes, const int64_t* user, int64_t lb[3], int64_t rb[3]) {
    if (dim < 1 || dim > 3 || !sizes || !lb || !rb) return TS_ERR_INVALID_ARGUMENT;
    for (int a = 0; a < 3; ++a) { lb[a] = 0; rb[a] = a < dim ? sizes[a] : 1; }
    if (!user) return TS_OK;
    for (int a = 0; a < dim; ++a) {
        const int size = (int)sizes[a];
        int r = size - (int)user[2 * a + 1];
        int l = (int)user[2 * a];
        if (r - l < 1) r = l + 1;
        if (l == size) { l = size - 1; r = l + 1; }
        if (r == 0) { l = 0; r = 1; }
        if (l < 0) l = 0;
        if (r > size) r = size;
        if (r - l < 0) return TS_ERR_BORDERS;
        lb[a] = l;
        rb[a] = r;
    }
    return TS_OK;
}

int ts_debug_remap(int padding, int len, int idx) { return len == 1 ? 0 : remap_literal(idx, len, padding); }

int ts_debug_remap_reduced(int padding, int len, int pos, int64_t shift, int plus) {
    const int s = reduce_shift((long long)shift, len, padding);
    return axis_index(pos - s + plus, len, padding);
}

void ts_debug_split_f32(int backward, int active, float w, int64_t* iw, float* dw) {
    long long i; float d;
    if (backward) split_backward<float>(w, active != 0, i, d); else split_forward<float>(w, active != 0, i, d);
    *iw = i; *dw = d;
}
void ts_debug_split_f64(int backward, int active, double w, int64_t* iw, double* dw) {
    long long i; double d;
    if (backward) split_backward<double>(w, active != 0, i, d); else split_forward<double>(w, active != 0, i, d);
    *iw = i; *dw = d;
}

// ---- device entry points ---------------------------------------------------------------------
int ts_shift_forward(const ts_geometry* gin, int dtype, int padding, int active, const void* x, const void* weights,
                     void* y, void* stream) {
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    if ((dtype = weights_f32(dtype, &g)) < 0) return TS_ERR_INVALID_ARGUMENT;
    const int es = elem_size(dtype);
    if (!es) return TS_ERR_INVALID_ARGUMENT;
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    if (!x || !weights || !y) return TS_ERR_INVALID_ARGUMENT;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    Route r;
    if ((rc = route(g, Call{active ? 1 : 0, active, es, dtype, 0ull, x, y, nullptr}, sms, &r)) != TS_OK) return rc;
    t_last_path = r.path;
    cudaStream_t s = (cudaStream_t)stream;
    const int wk = g.wf32 ? WK_F32 : dtype;     // the weight kind of the gathers (the generic family reads g.wf32 itself)
    switch (r.path) {
    case TS_PATH_TMA:
        return active ? tma_active_forward(g, r.tma, dtype, x, weights, y, s) : tma_gather(g, r.tma, wk, x, y, es, weights, 0, 0, s);
    case TS_PATH_HALO: return halo_active_forward(g, r.halo, x, weights, y, s);
    case TS_PATH_FLAT: return flat_gather(g, r.flat, wk, x, y, 0ull, es, weights, 0, 0, s);
    case TS_PATH_STAGED:
        return active ? staged_active_forward(g, r.staged, dtype, x, weights, y, s)
                      : staged_gather(g, r.staged, wk, x, y, 0ull, es, weights, 0, 0, s);
    }
    return active ? generic_active_forward(g, dtype, x, weights, y, s) : generic_gather(g, dtype, x, y, 0ull, es, weights, 0, 0, s);
}

int ts_shift2d_avgpool2_forward(const ts_geometry* gin, int dtype, int padding, int active, const void* x, const void* weights,
                                void* y_pooled, void* stream) {
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    if ((dtype = weights_f32(dtype, &g)) < 0) return TS_ERR_INVALID_ARGUMENT;
    if (g.dim != 2 || dtype != TS_F32) return TS_ERR_UNSUPPORTED;
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    if (!x || !weights || !y_pooled) return TS_ERR_INVALID_ARGUMENT;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    const HaloPlan hp = plan_halo(g, active ? 1 : 0, active, dtype, x_is_dense(g), x, y_pooled, nullptr, sms, true);
    if (!hp.ok) return TS_ERR_UNSUPPORTED;
    t_last_path = TS_PATH_HALO;
    return halo_forward2d(g, hp, active, 1, x, weights, y_pooled, (cudaStream_t)stream);
}

size_t ts_shift_backward_workspace_bytes(const ts_geometry* gin, int dtype) {
    if (!gin) return 0;
    // memo of the last query of this thread: ts_shift_backward validates its workspace on every call
    static thread_local ts_geometry last_geo;
    static thread_local int last_dtype = -1;
    static thread_local unsigned last_epoch = 0;
    static thread_local size_t last_bytes = 0;
    const unsigned epoch = g_tuning_epoch.load();
    if (last_dtype == dtype && last_epoch == epoch && !memcmp(&last_geo, gin, sizeof(ts_geometry))) return last_bytes;
    Geo g;
    if (make_geo(gin, 0, &g) != TS_OK) return 0;
    const int et = weights_f32(dtype, &g);
    if (et < 0) return 0;
    size_t bytes = 16;
    if (g.N * g.C != 0) {
        int sms = 148;
        sm_count(&sms);
        // every plan the backward may pick: pointers are unknown here (assume dense, aligned x), the padding is zeros or
        // another one, the halo plans are forced and include the pooled kernel (ts_shift2d_avgpool2_backward shares this query)
        int slots = 0;
        for (int pad = 0; pad < 2; ++pad)
            for (int active = 0; active < 2; ++active)
                for (const int path : ARITHMETIC)
                    for (int pool = 0; pool < (path == TS_PATH_HALO ? 2 : 1); ++pool) {
                        Geo gp = g;
                        gp.pad = pad;
                        Route r;
                        if (plan(path, gp, Call{2, active, elem_size(et), et, 0ull, nullptr, nullptr, nullptr}, true, sms, true,
                                 pool != 0, &r) && r.slots > slots)
                            slots = r.slots;
                    }
        bytes = (size_t)slots * (size_t)(g.C * g.dim) * sizeof(double) + 16;
    }
    last_geo = *gin; last_dtype = dtype; last_epoch = epoch; last_bytes = bytes;
    return bytes;
}

static int backward_impl(const ts_geometry* gin, const int dtype_arg, int padding, int active, const void* grad, const void* x,
                         const void* weights, void* grad_input, void* grad_weight, void* workspace, size_t workspace_bytes,
                         const ts_peer_group* peers, void* stream) {
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    const int dtype = weights_f32(dtype_arg, &g);
    if (dtype < 0) return TS_ERR_INVALID_ARGUMENT;
    const int es = elem_size(dtype);
    if (!es) return TS_ERR_INVALID_ARGUMENT;
    cudaStream_t s = (cudaStream_t)stream;
    if (g.C * g.dim == 0) return TS_OK;
    if (!grad_weight) return TS_ERR_INVALID_ARGUMENT;
    if (g.N == 0 || g.in_plane == 0) {
        // an empty shard still takes part in the exchange: it contributes zeros
        if (peers) return reduce_partials(g, gw_dtype(g, dtype), nullptr, 0, grad_weight, peers, s);
        const cudaError_t e = cudaMemsetAsync(grad_weight, 0, (size_t)(g.C * g.dim) * elem_size(gw_dtype(g, dtype)), s);
        return e == cudaSuccess ? TS_OK : cuda_fail(e);
    }
    if (!grad || !x || !weights || !grad_input) return TS_ERR_INVALID_ARGUMENT;
    if (!workspace || ((uintptr_t)workspace & 15) || workspace_bytes < ts_shift_backward_workspace_bytes(gin, dtype_arg))
        return TS_ERR_WORKSPACE;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    Route r;
    if ((rc = route(g, Call{2, active, es, dtype, 0ull, x, grad_input, grad}, sms, &r)) != TS_OK) return rc;
    t_last_path = r.path;
    double* partials = (double*)workspace;
    switch (r.path) {
    case TS_PATH_TMA: rc = tma_backward(g, r.tma, dtype, active, grad, x, weights, grad_input, partials, s); break;
    case TS_PATH_HALO: rc = halo_backward(g, r.halo, active, grad, x, weights, grad_input, partials, s); break;
    case TS_PATH_STAGED: rc = staged_backward(g, r.staged, dtype, active, grad, x, weights, grad_input, partials, s); break;
    default: rc = generic_backward(g, r.generic, dtype, active, grad, x, weights, grad_input, partials, s); break;
    }
    return rc != TS_OK ? rc : reduce_partials(g, gw_dtype(g, dtype), partials, r.slots, grad_weight, peers, s);
}

int ts_shift2d_avgpool2_backward(const ts_geometry* gin, int dtype, int padding, int active, const void* grad_pooled, const void* x,
                                 const void* weights, void* grad_input, void* grad_weight, void* workspace, size_t workspace_bytes,
                                 void* stream) {
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    if (weights_f32(dtype, &g) < 0) return TS_ERR_INVALID_ARGUMENT;
    if (g.dim != 2 || dtype != TS_F32) return TS_ERR_UNSUPPORTED;      // (fp32 only: a flagged dtype lands here too)
    if (g.N * g.C == 0 || g.in_plane == 0 || g.out_plane == 0) return TS_ERR_UNSUPPORTED;     // (empty tensors: the two-step path)
    if (!grad_pooled || !x || !weights || !grad_input || !grad_weight) return TS_ERR_INVALID_ARGUMENT;
    if (!workspace || ((uintptr_t)workspace & 15) || workspace_bytes < ts_shift_backward_workspace_bytes(gin, dtype))
        return TS_ERR_WORKSPACE;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    const HaloPlan hp = plan_halo(g, 2, active, dtype, x_is_dense(g), x, grad_input, grad_pooled, sms, true, true);
    if (!hp.ok) return TS_ERR_UNSUPPORTED;
    t_last_path = TS_PATH_HALO;
    cudaStream_t s = (cudaStream_t)stream;
    rc = halo_backward(g, hp, active, grad_pooled, x, weights, grad_input, (double*)workspace, s);
    return rc != TS_OK ? rc : reduce_partials(g, dtype, (double*)workspace, hp.slots, grad_weight, nullptr, s);
}

int ts_shift_backward(const ts_geometry* gin, int dtype, int padding, int active, const void* grad, const void* x,
                      const void* weights, void* grad_input, void* grad_weight, void* workspace, size_t workspace_bytes,
                      void* stream) {
    return backward_impl(gin, dtype, padding, active, grad, x, weights, grad_input, grad_weight, workspace, workspace_bytes, nullptr,
                         stream);
}

// the peer group of a backward with the in-kernel grad_weight exchange (gin and peers non-null)
static int check_peers(const ts_geometry* gin, int dtype, const ts_peer_group* peers) {
    if (peers->world < 1 || peers->world > 8 || peers->rank < 0 || peers->rank >= peers->world || !peers->state)
        return TS_ERR_INVALID_ARGUMENT;
    if (dtype != TS_F32 && dtype != TS_F16 && dtype != TS_BF16) return TS_ERR_UNSUPPORTED;   // contributions travel as fp32
    if (gin->C * gin->dim > peers->capacity || peers->capacity > 4096 || gin->C == 0) return TS_ERR_INVALID_ARGUMENT;
    for (int p = 0; p < peers->world; ++p)
        if (!peers->bufs[p] || ((uintptr_t)peers->bufs[p] & 7)) return TS_ERR_INVALID_ARGUMENT;
    return TS_OK;
}

int ts_shift_backward_allreduce(const ts_geometry* gin, int dtype, int padding, int active, const void* grad, const void* x,
                                const void* weights, void* grad_input, void* grad_weight, void* workspace, size_t workspace_bytes,
                                const ts_peer_group* peers, void* stream) {
    if (!peers || !gin) return TS_ERR_INVALID_ARGUMENT;
    Geo flag;
    if (weights_f32(dtype, &flag) < 0) return TS_ERR_INVALID_ARGUMENT;
    const int rc = check_peers(gin, dtype & ~TS_WEIGHTS_F32, peers);
    if (rc != TS_OK) return rc;
    return backward_impl(gin, dtype, padding, active, grad, x, weights, grad_input, grad_weight, workspace, workspace_bytes, peers,
                         stream);
}

// The pooling of the fused avg-pool entry points: -> TS_OK and the slab stride (3-D; 1 for 2-D), TS_ERR_INVALID_ARGUMENT for a
// stride entry below 1, TS_ERR_UNSUPPORTED for a stride no kernel serves (2-D: (2, 2); 3-D: (1, 2, 2), (2, 2, 2)).
static int pool_stride(int dim, const int32_t* stride, int* sa) {
    for (int a = 0; a < dim; ++a)
        if (stride[a] < 1) return TS_ERR_INVALID_ARGUMENT;
    if (dim < 2 || stride[dim - 2] != 2 || stride[dim - 1] != 2) return TS_ERR_UNSUPPORTED;
    if (dim == 3 && stride[0] != 1 && stride[0] != 2) return TS_ERR_UNSUPPORTED;
    *sa = dim == 3 ? stride[0] : 1;
    return TS_OK;
}

// The halo plan of a fused avg-pool call (the kernels that serve it are forced: small planes too).
static HaloPlan pool_plan(const Geo& g, int mode, int active, int sa, const void* x, const void* out, const void* grad, int sms) {
    return plan_halo(g, mode, active, TS_F32, x_is_dense(g), x, out, grad, sms, true, mode == 2, g.dim == 3 ? sa : 0);
}

int ts_shift_avgpool_forward(const ts_geometry* gin, int dtype, int padding, int active, const int32_t* stride, const void* x,
                             const void* weights, void* y_pooled, void* stream) {
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    if ((dtype = weights_f32(dtype, &g)) < 0 || !elem_size(dtype) || !stride) return TS_ERR_INVALID_ARGUMENT;
    int sa = 1;
    if ((rc = pool_stride(g.dim, stride, &sa)) != TS_OK) return rc;
    if (dtype != TS_F32 || g.wf32) return TS_ERR_UNSUPPORTED;
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    if (!x || !weights || !y_pooled) return TS_ERR_INVALID_ARGUMENT;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    const int mode = active ? 1 : 0;
    const HaloPlan hp = pool_plan(g, mode, active, sa, x, y_pooled, nullptr, sms);
    if (!hp.ok) return TS_ERR_UNSUPPORTED;
    t_last_path = TS_PATH_HALO;
    cudaStream_t s = (cudaStream_t)stream;
    return g.dim == 3 ? halo_forward3d_pool(g, hp, active, x, weights, y_pooled, s) : halo_forward2d(g, hp, active, 1, x, weights, y_pooled, s);
}

size_t ts_shift_avgpool_backward_workspace_bytes(const ts_geometry* gin, int dtype) {
    Geo g;
    if (!gin || make_geo(gin, 0, &g) != TS_OK || weights_f32(dtype, &g) != TS_F32 || g.wf32) return 16;
    if (g.N * g.C == 0 || (g.dim != 2 && g.dim != 3)) return 16;
    int sms = 148;
    sm_count(&sms);
    // every plan the backward may pick: dense aligned x, zeros or another padding, sparse or active, every served stride
    int slots = 0;
    for (int pad = 0; pad < 2; ++pad)
        for (int active = 0; active < 2; ++active)
            for (int sa = 1; sa <= (g.dim == 3 ? 2 : 1); ++sa) {
                Geo gp = g;
                gp.pad = pad;
                const HaloPlan hp = pool_plan(gp, 2, active, sa, nullptr, nullptr, nullptr, sms);
                if (hp.ok && hp.slots > slots) slots = hp.slots;
            }
    return (size_t)slots * (size_t)(g.C * g.dim) * sizeof(double) + 16;
}

int ts_shift_avgpool_backward(const ts_geometry* gin, int dtype, int padding, int active, const int32_t* stride, const void* grad_pooled,
                              const void* x, const void* weights, void* grad_input, void* grad_weight, void* workspace,
                              size_t workspace_bytes, const ts_peer_group* peers, void* stream) {
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    const int et = weights_f32(dtype, &g);
    if (et < 0 || !elem_size(et) || !stride) return TS_ERR_INVALID_ARGUMENT;
    int sa = 1;
    if ((rc = pool_stride(g.dim, stride, &sa)) != TS_OK) return rc;
    if (peers && (rc = check_peers(gin, et, peers)) != TS_OK) return rc;
    if (et != TS_F32 || g.wf32) return TS_ERR_UNSUPPORTED;
    if (g.N * g.C == 0 || g.in_plane == 0 || g.out_plane == 0) return TS_ERR_UNSUPPORTED;     // (empty shards: the two-step path)
    if (!grad_pooled || !x || !weights || !grad_input || !grad_weight) return TS_ERR_INVALID_ARGUMENT;
    if (!workspace || ((uintptr_t)workspace & 15)) return TS_ERR_WORKSPACE;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    const HaloPlan hp = pool_plan(g, 2, active, sa, x, grad_input, grad_pooled, sms);
    if (!hp.ok) return TS_ERR_UNSUPPORTED;
    if (workspace_bytes < (size_t)hp.slots * (size_t)(g.C * g.dim) * sizeof(double)) return TS_ERR_WORKSPACE;
    t_last_path = TS_PATH_HALO;
    cudaStream_t s = (cudaStream_t)stream;
    rc = halo_backward(g, hp, active, grad_pooled, x, weights, grad_input, (double*)workspace, s);
    return rc != TS_OK ? rc : reduce_partials(g, TS_F32, (double*)workspace, hp.slots, grad_weight, peers, s);
}

int ts_shift_forward_nhwc(const ts_geometry* gin, int dtype, int padding, int active, const void* x, const void* weights, void* y,
                          void* stream) {
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    if ((dtype = weights_f32(dtype, &g)) < 0 || !elem_size(dtype)) return TS_ERR_INVALID_ARGUMENT;
    if (g_forced_path.load() != TS_PATH_NONE) return TS_ERR_UNSUPPORTED;      // a forced family: callers take the planar path
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_ERR_UNSUPPORTED;
    if (!x || !weights || !y) return TS_ERR_INVALID_ARGUMENT;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    rc = cl_forward(g, dtype, active, x, weights, y, sms, (cudaStream_t)stream);
    if (rc == TS_OK) t_last_path = TS_PATH_NHWC;
    return rc;
}

size_t ts_shift_backward_nhwc_workspace_bytes(const ts_geometry* gin, int dtype) {
    Geo g;
    if (make_geo(gin, 0, &g) != TS_OK || (dtype = weights_f32(dtype, &g)) < 0) return 0;
    int sms = 148;
    sm_count(&sms);
    return cl_backward_workspace_bytes(g, dtype, sms);
}

int ts_shift_backward_nhwc(const ts_geometry* gin, int dtype, int padding, int active, const void* grad, const void* x, const void* weights,
                           void* grad_input, void* grad_weight, void* workspace, size_t workspace_bytes, const ts_peer_group* peers,
                           void* stream) {
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    if ((dtype = weights_f32(dtype, &g)) < 0 || !elem_size(dtype)) return TS_ERR_INVALID_ARGUMENT;
    if (peers && (rc = check_peers(gin, dtype, peers)) != TS_OK) return rc;
    if (g_forced_path.load() != TS_PATH_NONE) return TS_ERR_UNSUPPORTED;
    if (g.N * g.C == 0 || g.in_plane == 0) return TS_ERR_UNSUPPORTED;        // empty shards: the planar path (zeros / exchange)
    if (!grad || !x || !weights || !grad_input || !grad_weight) return TS_ERR_INVALID_ARGUMENT;
    if (!workspace || ((uintptr_t)workspace & 15)) return TS_ERR_WORKSPACE;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    int slots = 0;
    rc = cl_backward(g, dtype, active, grad, x, weights, grad_input, (double*)workspace, workspace_bytes, sms, &slots, s);
    if (rc == TS_OK) rc = reduce_partials(g, gw_dtype(g, dtype), (double*)workspace, slots, grad_weight, peers, s);
    if (rc == TS_OK) t_last_path = TS_PATH_NHWC;
    return rc;
}

static int qshift_common(const ts_geometry* gin, int elem_bytes, int padding, int qweight_kind, Geo* g) {
    const int rc = make_geo(gin, padding, g);
    if (rc != TS_OK) return rc;
    if (elem_bytes != 1 && elem_bytes != 4) return TS_ERR_UNSUPPORTED;
    if (qweight_kind < TS_QW_U8 || qweight_kind > TS_QW_I32) return TS_ERR_INVALID_ARGUMENT;
    return TS_OK;
}

static unsigned long long qfill(int elem_bytes, int64_t zero_point) {
    return elem_bytes == 1 ? (unsigned long long)((unsigned)zero_point & 0xffu) : (unsigned long long)(uint32_t)(int32_t)zero_point;
}

int ts_qshift_forward(const ts_geometry* gin, int elem_bytes, int padding, int64_t zero_point, const void* xq,
                      const void* qweights, int qweight_kind, int64_t weight_zero_point, void* yq, void* stream) {
    Geo g;
    int rc = qshift_common(gin, elem_bytes, padding, qweight_kind, &g);
    if (rc != TS_OK) return rc;
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    if (!xq || !qweights || !yq) return TS_ERR_INVALID_ARGUMENT;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    const unsigned long long fill = qfill(elem_bytes, zero_point);
    Route r;
    if ((rc = route(g, Call{0, 0, elem_bytes, -1, fill, xq, yq, nullptr}, sms, &r)) != TS_OK) return rc;
    t_last_path = r.path;
    cudaStream_t s = (cudaStream_t)stream;
    switch (r.path) {
    case TS_PATH_TMA: return tma_gather(g, r.tma, WK_QUANT, xq, yq, elem_bytes, qweights, qweight_kind, weight_zero_point, s);
    case TS_PATH_FLAT: return flat_gather(g, r.flat, WK_QUANT, xq, yq, fill, elem_bytes, qweights, qweight_kind, weight_zero_point, s);
    case TS_PATH_STAGED:
        return staged_gather(g, r.staged, WK_QUANT, xq, yq, fill, elem_bytes, qweights, qweight_kind, weight_zero_point, s);
    }
    return generic_gather(g, WK_QUANT, xq, yq, fill, elem_bytes, qweights, qweight_kind, weight_zero_point, s);
}

int ts_qshift_forward_nhwc(const ts_geometry* gin, int elem_bytes, int padding, int64_t zero_point, const void* xq,
                           const void* qweights, int qweight_kind, int64_t weight_zero_point, void* yq, void* stream) {
    Geo g;
    int rc = qshift_common(gin, elem_bytes, padding, qweight_kind, &g);
    if (rc != TS_OK) return rc;
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    if (!xq || !qweights || !yq) return TS_ERR_INVALID_ARGUMENT;
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    t_last_path = TS_PATH_NHWC;
    return nhwc_gather(g, xq, yq, qfill(elem_bytes, zero_point), elem_bytes, qweights, qweight_kind, weight_zero_point, sms, 0,
                       tuning().nhwc_variant, tuning().nhwc_ring_rows, false, (cudaStream_t)stream);
}

int ts_nhwc_to_nchw(const void* x, void* y, int64_t N, int64_t C, int64_t P, int elem_bytes, void* stream) {
    if (N < 0 || C < 0 || P < 0) return TS_ERR_INVALID_ARGUMENT;
    if (N == 0 || C == 0 || P == 0) return TS_OK;
    if (!x || !y) return TS_ERR_INVALID_ARGUMENT;
    int sms = 0;
    const int rc = sm_count(&sms);      // fails loudly without a device
    if (rc != TS_OK) return rc;
    return nhwc_to_planar(x, y, N, C, P, elem_bytes, (cudaStream_t)stream);
}

int ts_debug_nhwc_emulate(const ts_geometry* gin, int elem_bytes, int padding, int64_t zero_point, const void* xq_host,
                          const void* qweights_host, int qweight_kind, int64_t weight_zero_point, void* yq_host, int sm_count_,
                          int max_grid_x, int variant, int ring_rows) {
    Geo g;
    const int rc = qshift_common(gin, elem_bytes, padding, qweight_kind, &g);
    if (rc != TS_OK) return rc;
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    if (!xq_host || !qweights_host || !yq_host || sm_count_ < 1 || variant < 0 || variant > 2 || ring_rows < 0)
        return TS_ERR_INVALID_ARGUMENT;
    if ((double)g.N * (double)g.C * (double)g.in_plane > 4194304.0) return TS_ERR_TOO_LARGE;   // a test aid, not a CPU path
    return nhwc_gather(g, xq_host, yq_host, qfill(elem_bytes, zero_point), elem_bytes, qweights_host, qweight_kind, weight_zero_point,
                       sm_count_, max_grid_x, variant, ring_rows, true, nullptr);
}

int ts_debug_route(const ts_geometry* gin, int op, int dtype, int elem_bytes, int padding, int active, int64_t* out, int n_out) {
    if (op < 0 || op > 2 || !out || n_out < 13) return TS_ERR_INVALID_ARGUMENT;
    Geo g;
    int rc = make_geo(gin, padding, &g);
    if (rc != TS_OK) return rc;
    int es = 0;
    if (dtype == -1) {
        if (op != 0) return TS_ERR_INVALID_ARGUMENT;
        if (elem_bytes != 1 && elem_bytes != 4) return TS_ERR_UNSUPPORTED;
        es = elem_bytes;
    } else if ((dtype = weights_f32(dtype, &g)) < 0 || !(es = elem_size(dtype))) {
        return TS_ERR_INVALID_ARGUMENT;
    }
    int sms = 0;
    if ((rc = sm_count(&sms)) != TS_OK) return rc;
    const Call c{op, op == 1 ? 1 : op == 2 ? (active != 0) : 0, es, dtype, 0ull, (const void*)256, (const void*)512,
                 op == 2 ? (const void*)768 : nullptr};
    Route r;
    if ((rc = route(g, c, sms, &r)) != TS_OK) return rc;
    int64_t v[13] = {r.path};
    switch (r.path) {
    case TS_PATH_TMA: {
        const TArgs& a = r.tma.a;
        const int64_t rest[12] = {a.tiles, a.tiles / (a.tiles_b * a.tiles_g), a.tiles_b, a.tiles_g,
                                  a.np, a.n_per_unit, a.units, r.tma.grid, a.stages, a.nw, r.slots, a.table};
        memcpy(v + 1, rest, sizeof(rest));
        break;
    }
    case TS_PATH_STAGED: {
        const SArgs& a = r.staged.a;
        const int64_t rest[12] = {a.tiles, a.tiles, 1, 1, a.np, a.n_per_unit, a.units, r.staged.grid, a.stages, a.nw, r.slots, a.table};
        memcpy(v + 1, rest, sizeof(rest));
        break;
    }
    case TS_PATH_HALO: {
        const HArgs& a = r.halo.a;
        const int64_t rest[12] = {1, 1, 1, 1, a.np, a.n_per_unit, a.units, r.halo.grid, a.stages, a.nw, r.slots, a.table};
        memcpy(v + 1, rest, sizeof(rest));
        break;
    }
    case TS_PATH_FLAT: {
        const FArgs& a = r.flat.a;        // units are stages of K (n, c) planes; the table flag selects the warp-per-plane variant
        const int64_t rest[12] = {1, 1, 1, 1, a.K, 0, a.nstages, r.flat.grid, a.stages, a.nw, 0, a.table};
        memcpy(v + 1, rest, sizeof(rest));
        break;
    }
    default:
        v[7] = op == 2 ? r.generic.units : 0;
        v[11] = r.slots;
    }
    for (int i = 0; i < n_out; ++i) out[i] = i < 13 ? v[i] : 0;
    return TS_OK;
}

}  // extern "C"

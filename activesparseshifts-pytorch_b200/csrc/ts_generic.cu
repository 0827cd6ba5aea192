// ts_generic.cu -- stride-generic kernels: every dim (1/2/3), padding mode, element type, border
// crop and input stride pattern.  One element per thread, block <-> (n,c) plane so the channel's
// shift parameters are block-uniform registers.  This is the coverage path (odd shapes, strided /
// channels-last inputs, volumes too large to stage); the bandwidth path is ts_staged.cu.
//
// Semantics: reference forward body  ops/kernels/shifts_kernels.h:156-220,
//            backward body           ops/kernels/shifts_kernels.h:222-327,
//            quantized body          ops/kernels/shifts_kernels.h:532-571.
// grad_weight is reduced deterministically: per-thread double accumulators -> fixed-shape block
// tree -> partials[unit][C*dim] (double) -> second pass in fixed order.  No atomics (the
// reference CUDA kernel issues up to 3 atomicAdds per element, cuda/shifts_cuda.cu:90-165).
#include "ts_kernels.h"

namespace ts {

namespace {

template <int DIM> TS_D void decode(int e, const int* sz, int* o) {
    if (DIM == 1) { o[0] = e; }
    else if (DIM == 2) { o[0] = e / sz[1]; o[1] = e - o[0] * sz[1]; }
    else { int t = e / sz[2]; o[2] = e - t * sz[2]; o[0] = t / sz[1]; o[1] = t - o[0] * sz[1]; }
}

// ------------------------------------------------------------------------------------------
// Sparse (integer) forward on raw element storage E; also the quantized forward.
template <typename E, int DIM, int WK>
__global__ void __launch_bounds__(256) k_gather_generic(Geo g, const E* __restrict__ x, E* __restrict__ y, E fill,
                                                        const void* __restrict__ w, int qkind, long long wzp) {
    const long long planes = g.N * g.C;
    for (long long p = blockIdx.x; p < planes; p += gridDim.x) {
        const long long n = p / g.C, c = p - n * g.C;
        int sx[DIM];
        load_int_shifts<WK, DIM>(w, qkind, wzp, c, g, sx);
        const E* xp = x + n * g.xs[0] + c * g.xs[1];
        E* yp = y + p * g.out_plane;
        for (int e = blockIdx.y * blockDim.x + threadIdx.x; e < (int)g.out_plane; e += gridDim.y * blockDim.x) {
            int o[3];
            decode<DIM>(e, g.OS, o);
            long long off = 0;
            bool ok = true;
#pragma unroll
            for (int a = 0; a < DIM; ++a) {
                const int t = axis_index(o[a] + g.lb[a] - sx[a], g.S[a], g.pad);
                ok = ok && (t >= 0);
                off += (long long)t * g.xs[2 + a];
            }
            yp[e] = ok ? xp[off] : fill;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Neighbour fetch (2^DIM values) with per-axis index pairs computed once.
template <typename ST, int DIM>
TS_D void fetch_neighbours(const ST* __restrict__ plane, const int* idx, const int* sizes, const long long* str, int pad,
                           typename Elem<ST>::CT* v) {
    using CT = typename Elem<ST>::CT;
    long long off[DIM][2];
    bool okk[DIM][2];
#pragma unroll
    for (int a = 0; a < DIM; ++a) {
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const int t = axis_index(idx[a] + b, sizes[a], pad);
            okk[a][b] = t >= 0;
            off[a][b] = (long long)t * str[a];
        }
    }
#pragma unroll
    for (int q = 0; q < (1 << DIM); ++q) {
        bool ok = true;
        long long o = 0;
#pragma unroll
        for (int a = 0; a < DIM; ++a) { ok = ok && okk[a][(q >> a) & 1]; o += off[a][(q >> a) & 1]; }
        v[q] = ok ? Elem<ST>::ld(plane[o]) : (CT)0;
    }
}

// Active (interpolating) forward.
template <typename ST, int DIM>
__global__ void __launch_bounds__(256) k_active_forward_generic(Geo g, const ST* __restrict__ x, const ST* __restrict__ w,
                                                                ST* __restrict__ y) {
    using CT = typename Elem<ST>::CT;
    const long long planes = g.N * g.C;
    for (long long p = blockIdx.x; p < planes; p += gridDim.x) {
        const long long n = p / g.C, c = p - n * g.C;
        const ShiftParams<CT, DIM> sp = load_params<ST, DIM>(w, c, g, true, false);
        const ST* xp = x + n * g.xs[0] + c * g.xs[1];
        ST* yp = y + p * g.out_plane;
        for (int e = blockIdx.y * blockDim.x + threadIdx.x; e < (int)g.out_plane; e += gridDim.y * blockDim.x) {
            int o[3], idx[DIM];
            decode<DIM>(e, g.OS, o);
#pragma unroll
            for (int a = 0; a < DIM; ++a) idx[a] = o[a] + g.lb[a] - sp.sx[a];
            CT v[8];
            fetch_neighbours<ST, DIM>(xp, idx, g.S, g.xs + 2, g.pad, v);
            yp[e] = Elem<ST>::st(interpolate<CT, DIM>(v, sp.d));
        }
    }
}

// ------------------------------------------------------------------------------------------
// Backward: block = (channel c, unit u); unit = (batch chunk, plane tile).
template <typename ST, int DIM, bool ACTIVE>
__global__ void __launch_bounds__(256) k_backward_generic(Geo g, const ST* __restrict__ grad, const ST* __restrict__ x,
                                                          const ST* __restrict__ w, ST* __restrict__ gi,
                                                          double* __restrict__ partials, int n_per_chunk, int tiles) {
    using CT = typename Elem<ST>::CT;
    const long long c = blockIdx.x;
    const int unit = blockIdx.y;
    const int chunk = unit / tiles, tile = unit - chunk * tiles;
    const ShiftParams<CT, DIM> sp = load_params<ST, DIM>(w, c, g, ACTIVE, true);
    long long gstr[3] = {(long long)g.OS[1] * g.OS[2], (long long)g.OS[2], 1};
    if (DIM == 1) gstr[0] = 1;
    if (DIM == 2) { gstr[0] = g.OS[1]; gstr[1] = 1; }
    double acc[DIM];
#pragma unroll
    for (int a = 0; a < DIM; ++a) acc[a] = 0.0;

    const long long n0 = (long long)chunk * n_per_chunk;
    const long long n1 = n0 + n_per_chunk < g.N ? n0 + n_per_chunk : g.N;
    for (long long n = n0; n < n1; ++n) {
        const long long p = n * g.C + c;
        const ST* xp = x + n * g.xs[0] + c * g.xs[1];
        const ST* gp = grad + p * g.out_plane;
        ST* gip = gi + p * g.in_plane;
        for (int e = tile * blockDim.x + threadIdx.x; e < (int)g.in_plane; e += tiles * blockDim.x) {
            int pos[3], o[3] = {0, 0, 0};
            decode<DIM>(e, g.S, pos);
            bool ok = true;
            long long goff = 0;
#pragma unroll
            for (int a = 0; a < DIM; ++a) {
                o[a] = pos[a] - g.lb[a];
                ok = ok && o[a] >= 0 && o[a] < g.OS[a];
                goff += (long long)o[a] * gstr[a];
            }
            CT r = (CT)0;
            if (ok) {
                const CT gv = Elem<ST>::ld(gp[goff]);
                int idx[DIM];
#pragma unroll
                for (int a = 0; a < DIM; ++a) idx[a] = pos[a] - sp.sx[a];
                CT v[8], wg[3];
                fetch_neighbours<ST, DIM>(xp, idx, g.S, g.xs + 2, g.pad, v);
                weight_partials<CT, DIM>(v, sp.d, wg);
#pragma unroll
                for (int a = 0; a < DIM; ++a) acc[a] += (double)Arith<CT>::mul(gv, wg[a]);
                if (ACTIVE) {
#pragma unroll
                    for (int a = 0; a < DIM; ++a) idx[a] = o[a] - sp.sg[a];
                    fetch_neighbours<ST, DIM>(gp, idx, g.OS, gstr, g.pad, v);
                    r = interpolate<CT, DIM>(v, sp.d);
                } else {
                    long long off = 0;
                    bool in = true;
#pragma unroll
                    for (int a = 0; a < DIM; ++a) {
                        const int t = axis_index(o[a] + sp.sg[a], g.OS[a], g.pad);
                        in = in && t >= 0;
                        off += (long long)t * gstr[a];
                    }
                    r = in ? Elem<ST>::ld(gp[off]) : (CT)0;
                }
            }
            gip[e] = Elem<ST>::st(r);
        }
    }

    // fixed-shape block reduction (deterministic): warp shuffles, then warp 0 over the warp sums
    __shared__ double red[DIM][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int a = 0; a < DIM; ++a) {
        double v = acc[a];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) red[a][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < DIM) {
        double s = 0.0;
        for (int k = 0; k < nwarps; ++k) s += red[threadIdx.x][k];
        partials[(long long)unit * (g.C * DIM) + c * DIM + threadIdx.x] = s;
    }
}

}  // namespace

// Second pass shared by both backward paths: one warp per (c, axis) output, lanes stride over
// the partial slots in a fixed order, shuffle tree, one rounding to the weight dtype.
template <typename ST>
__global__ void k_reduce_partials(const double* __restrict__ partials, int slots, int outputs, ST* __restrict__ gw) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    pdl_wait();             // the partials are the previous kernel's output
    if (warp >= outputs) return;
    double s = 0.0;
    for (int k = lane; k < slots; k += 32) s += partials[(long long)k * outputs + warp];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) gw[warp] = Elem<ST>::st((typename Elem<ST>::CT)s);
}

// ---- pass 2 fused with the all-reduce of grad_weight over NVLink peer memory -----------------------
// Same decomposition as k_reduce_partials (one warp per output, lanes stride over the partial slots,
// fixed shuffle tree -> the local value is bit-identical to the unfused pass 2); 32 outputs per CTA.
// Exchange = the "LL" scheme: a contribution travels as ONE 64-bit word {epoch : value}, written with a
// single 8-byte store (single-copy atomic) into slot [parity][sender][output] of EVERY peer's buffer,
// so there is no separate flag, no fence and no second NVLink round trip: lane p of the output's warp
// stores this rank's word to peer p and then polls peer p's word in this rank's own buffer until it
// carries the call's epoch.  The `world` values are summed in rank order -> identical on every rank.
//   * The epoch lives in DEVICE memory (`state[cta]`, bumped by the kernel): nothing call-specific is
//     passed from the host, so the launch can be captured in a CUDA graph and replayed.  Every rank makes
//     the same sequence of calls (replicated layers), so the per-CTA counters agree across ranks.
//   * Buffers are double-buffered by epoch parity: a rank can run at most one call ahead of the slowest
//     peer (it needs that peer's word of the call in between), so the word being polled is never the one
//     being overwritten.
//   * A peer that does not arrive within `timeout_ns` (0 = wait for ever, like a collective without a
//     watchdog) makes the kernel record the call's epoch in state[PEER_MAX_CTAS] and trap.
struct PeerArgs {
    int world, rank, capacity;
    unsigned long long timeout_ns;
    unsigned long long* bufs[8];
    unsigned* state;
};
constexpr int PEER_MAX_CTAS = 128;      // capacity 4096 outputs / 32 per CTA

TS_D unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

template <typename ST>
__global__ void __launch_bounds__(1024, 1) k_reduce_partials_allreduce(const double* __restrict__ partials, int slots, int outputs,
                                                                       ST* __restrict__ gw, const PeerArgs pa) {
    __shared__ unsigned s_epoch;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int o = blockIdx.x * 32 + wid;
    pdl_trigger();
    pdl_wait();             // the partials are the previous kernel's output
    if (threadIdx.x == 0) { const unsigned e = pa.state[blockIdx.x] + 1u; pa.state[blockIdx.x] = e; s_epoch = e; }
    __syncthreads();
    const unsigned epoch = s_epoch;
    if (o >= outputs) return;
    double s = 0.0;
    for (int k = lane; k < slots; k += 32) s += partials[(long long)k * outputs + o];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d);
    const float mine = __shfl_sync(0xffffffffu, (float)s, 0);
    const size_t half = (size_t)(epoch & 1u) * pa.world * pa.capacity;
    float v = 0.f;
    if (lane < pa.world) {
        const unsigned long long word = ((unsigned long long)epoch << 32) | (unsigned long long)__float_as_uint(mine);
        unsigned long long* remote = pa.bufs[lane] + half + (size_t)pa.rank * pa.capacity + o;
        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(remote), "l"(word) : "memory");
        const unsigned long long* local = pa.bufs[pa.rank] + half + (size_t)lane * pa.capacity + o;
        const unsigned long long t0 = pa.timeout_ns ? global_ns() : 0ull;
        unsigned spins = 0;
        for (;;) {
            unsigned long long got;
            asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(got) : "l"(local) : "memory");
            if ((unsigned)(got >> 32) == epoch) { v = __uint_as_float((unsigned)got); break; }
            if (pa.timeout_ns && (++spins & 1023u) == 0 && global_ns() - t0 > pa.timeout_ns) {
                pa.state[PEER_MAX_CTAS] = epoch;        // which call gave up (host-readable after the failure)
                __threadfence_system();
                __trap();
            }
        }
    }
    // sum in rank order (fixed): every rank computes the same bits
    float total = 0.f;
    for (int p = 0; p < pa.world; ++p) total += __shfl_sync(0xffffffffu, v, p);
    if (lane == 0) gw[o] = Elem<ST>::st(total);
}

template <typename ST>
static int launch_reduce_partials(const double* partials, int slots, int outputs, void* gw, const ts_peer_group* pg, cudaStream_t stream) {
    if (pg) {
        if constexpr (sizeof(ST) == 8) {
            return TS_ERR_UNSUPPORTED;
        } else {
            PeerArgs pa;
            pa.world = pg->world; pa.rank = pg->rank; pa.capacity = pg->capacity; pa.timeout_ns = pg->timeout_ns;
            for (int p = 0; p < 8; ++p) pa.bufs[p] = (unsigned long long*)pg->bufs[p];
            pa.state = (unsigned*)pg->state;
            if (outputs > 32 * PEER_MAX_CTAS || outputs > pg->capacity) return TS_ERR_INVALID_ARGUMENT;
            if (launch_pdl(k_reduce_partials_allreduce<ST>, dim3((outputs + 31) / 32), dim3(1024), 0, stream, partials, slots, outputs,
                           (ST*)gw, pa) != cudaSuccess) {
                (void)cudaGetLastError();
                k_reduce_partials_allreduce<ST><<<(outputs + 31) / 32, 1024, 0, stream>>>(partials, slots, outputs, (ST*)gw, pa);
            }
            note_launch();
            return check_launch();
        }
    }
    const int threads = 128;
    const int blocks = (outputs * 32 + threads - 1) / threads;
    if (launch_pdl(k_reduce_partials<ST>, dim3(blocks), dim3(threads), 0, stream, partials, slots, outputs, (ST*)gw) != cudaSuccess) {
        (void)cudaGetLastError();
        k_reduce_partials<ST><<<blocks, threads, 0, stream>>>(partials, slots, outputs, (ST*)gw);
    }
    note_launch();
    return check_launch();
}

int reduce_partials(const Geo& g, int dtype, const double* partials, int slots, void* gw, const ts_peer_group* peers, cudaStream_t s) {
    const int outputs = (int)(g.C * g.dim);
    switch (dtype) {
    case TS_F32: return launch_reduce_partials<float>(partials, slots, outputs, gw, peers, s);
    case TS_F64: return launch_reduce_partials<double>(partials, slots, outputs, gw, peers, s);
    case TS_F16: return launch_reduce_partials<__half>(partials, slots, outputs, gw, peers, s);
    default: return launch_reduce_partials<__nv_bfloat16>(partials, slots, outputs, gw, peers, s);
    }
}

// ------------------------------------------------------------------------------------------
// Host launchers.
static int pick_threads(long long plane) {
    int t = 32;
    while (t < 256 && t < plane) t <<= 1;
    return t;
}

static dim3 plane_grid(const Geo& g, long long plane, int threads) {
    long long tiles = (plane + (long long)threads * 4 - 1) / ((long long)threads * 4);
    if (tiles < 1) tiles = 1;
    if (tiles > 1024) tiles = 1024;
    long long planes = g.N * g.C;
    if (planes > 0x7fffffffLL) planes = 0x7fffffffLL;
    return dim3((unsigned)planes, (unsigned)tiles, 1);
}

template <typename E, int WK>
static int gather_dim(const Geo& g, const void* x, void* y, E fill, const void* w, int qkind, long long wzp, cudaStream_t s) {
    const int threads = pick_threads(g.out_plane);
    const dim3 grid = plane_grid(g, g.out_plane, threads);
    switch (g.dim) {
    case 1: k_gather_generic<E, 1, WK><<<grid, threads, 0, s>>>(g, (const E*)x, (E*)y, fill, w, qkind, wzp); break;
    case 2: k_gather_generic<E, 2, WK><<<grid, threads, 0, s>>>(g, (const E*)x, (E*)y, fill, w, qkind, wzp); break;
    default: k_gather_generic<E, 3, WK><<<grid, threads, 0, s>>>(g, (const E*)x, (E*)y, fill, w, qkind, wzp); break;
    }
    note_launch();
    return check_launch();
}

int generic_gather(const Geo& g, int wk, const void* x, void* y, unsigned long long fill, int esize, const void* w,
                   int qkind, long long wzp, cudaStream_t s) {
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    switch (wk) {
    case WK_F32: return gather_dim<uint32_t, WK_F32>(g, x, y, 0u, w, 0, 0, s);
    case WK_F64: return gather_dim<unsigned long long, WK_F64>(g, x, y, 0ull, w, 0, 0, s);
    case WK_F16: return gather_dim<uint16_t, WK_F16>(g, x, y, (uint16_t)0, w, 0, 0, s);
    case WK_BF16: return gather_dim<uint16_t, WK_BF16>(g, x, y, (uint16_t)0, w, 0, 0, s);
    case WK_QUANT:
        if (esize == 1) return gather_dim<uint8_t, WK_QUANT>(g, x, y, (uint8_t)fill, w, qkind, wzp, s);
        if (esize == 4) return gather_dim<uint32_t, WK_QUANT>(g, x, y, (uint32_t)fill, w, qkind, wzp, s);
        return TS_ERR_UNSUPPORTED;
    }
    return TS_ERR_INVALID_ARGUMENT;
}

template <typename ST>
static int active_fwd_t(const Geo& g, const void* x, const void* w, void* y, cudaStream_t s) {
    const int threads = pick_threads(g.out_plane);
    const dim3 grid = plane_grid(g, g.out_plane, threads);
    switch (g.dim) {
    case 1: k_active_forward_generic<ST, 1><<<grid, threads, 0, s>>>(g, (const ST*)x, (const ST*)w, (ST*)y); break;
    case 2: k_active_forward_generic<ST, 2><<<grid, threads, 0, s>>>(g, (const ST*)x, (const ST*)w, (ST*)y); break;
    default: k_active_forward_generic<ST, 3><<<grid, threads, 0, s>>>(g, (const ST*)x, (const ST*)w, (ST*)y); break;
    }
    note_launch();
    return check_launch();
}

int generic_active_forward(const Geo& g, int dtype, const void* x, const void* w, void* y, cudaStream_t s) {
    if (g.N * g.C == 0 || g.out_plane == 0) return TS_OK;
    switch (dtype) {
    case TS_F32: return active_fwd_t<float>(g, x, w, y, s);
    case TS_F64: return active_fwd_t<double>(g, x, w, y, s);
    case TS_F16: return active_fwd_t<__half>(g, x, w, y, s);
    case TS_BF16: return active_fwd_t<__nv_bfloat16>(g, x, w, y, s);
    }
    return TS_ERR_INVALID_ARGUMENT;
}

GenericBwdPlan plan_generic_backward(const Geo& g) {
    GenericBwdPlan p;
    p.threads = pick_threads(g.in_plane);
    long long tiles = (g.in_plane + 4095) / 4096;
    if (tiles < 1) tiles = 1;
    if (tiles > 64) tiles = 64;
    const long long C = g.C > 0 ? g.C : 1;
    long long chunks = (2048 + C * tiles - 1) / (C * tiles);
    if (chunks < 1) chunks = 1;
    if (chunks > g.N) chunks = g.N > 0 ? g.N : 1;
    long long npc = (g.N + chunks - 1) / chunks;
    if (npc < 1) npc = 1;
    chunks = (g.N + npc - 1) / npc;
    if (chunks < 1) chunks = 1;
    p.tiles = (int)tiles;
    p.n_per_chunk = (int)(npc > 0x7fffffffLL ? 0x7fffffffLL : npc);
    p.units = (int)(chunks * tiles);
    return p;
}

template <typename ST, bool ACTIVE>
static int bwd_dim(const Geo& g, const GenericBwdPlan& p, const void* grad, const void* x, const void* w, void* gi,
                   double* partials, cudaStream_t s) {
    const dim3 grid((unsigned)g.C, (unsigned)p.units, 1);
    switch (g.dim) {
    case 1: k_backward_generic<ST, 1, ACTIVE><<<grid, p.threads, 0, s>>>(g, (const ST*)grad, (const ST*)x, (const ST*)w, (ST*)gi, partials, p.n_per_chunk, p.tiles); break;
    case 2: k_backward_generic<ST, 2, ACTIVE><<<grid, p.threads, 0, s>>>(g, (const ST*)grad, (const ST*)x, (const ST*)w, (ST*)gi, partials, p.n_per_chunk, p.tiles); break;
    default: k_backward_generic<ST, 3, ACTIVE><<<grid, p.threads, 0, s>>>(g, (const ST*)grad, (const ST*)x, (const ST*)w, (ST*)gi, partials, p.n_per_chunk, p.tiles); break;
    }
    note_launch();
    return check_launch();
}

template <typename ST>
static int bwd_t(const Geo& g, const GenericBwdPlan& p, int active, const void* grad, const void* x, const void* w, void* gi,
                 double* partials, cudaStream_t s) {
    return active ? bwd_dim<ST, true>(g, p, grad, x, w, gi, partials, s) : bwd_dim<ST, false>(g, p, grad, x, w, gi, partials, s);
}

int generic_backward(const Geo& g, const GenericBwdPlan& p, int dtype, int active, const void* grad, const void* x, const void* w,
                     void* gi, double* partials, cudaStream_t s) {
    switch (dtype) {
    case TS_F32: return bwd_t<float>(g, p, active, grad, x, w, gi, partials, s);
    case TS_F64: return bwd_t<double>(g, p, active, grad, x, w, gi, partials, s);
    case TS_F16: return bwd_t<__half>(g, p, active, grad, x, w, gi, partials, s);
    case TS_BF16: return bwd_t<__nv_bfloat16>(g, p, active, grad, x, w, gi, partials, s);
    }
    return TS_ERR_INVALID_ARGUMENT;
}

}  // namespace ts

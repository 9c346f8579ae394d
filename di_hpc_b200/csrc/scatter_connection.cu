// scatter_connection.cu -- ScatterConnection (entity embeddings -> spatial map) and its backward gather, for sm_100a.
//
// Semantics: hpc_rll/origin/scatter_connection.py:25-64 run on the CPU, i.e. sequential in entity order m:
//   forward : out[b, n, y*W + x]  = ((0.f + x[b,m0,n]) + x[b,m1,n]) + ...   ("add", ascending m, fp32)
//                                 = x[b, m_last, n]                          ("cover": the last m at a cell wins)
//             cells no entity lands on are +0.f
//   backward: grad_x[b, m, n] = grad_out[b, n, y*W + x]   (the gather adjoint; overwritten "cover" entities included)
// An entity whose (y, x) lies outside [0,H) x [0,W) writes nothing and gets a zero gradient (DESIGN.md section 7).
// Replaces ScatterConnectionForward / ScatterConnectionBackward (/root/reference/src/torch_utils/network/
// scatter_connection.cu:8-76, kernels include/hpc/rll/cuda/torch_utils/network/scatter_connection_kernel.h:60-120),
// which memset the whole output, then scatter with float atomicAdd ("add") or racing plain stores ("cover").
//
// B200 design: no atomics, every output element written exactly once (zeros included), bit-identical run to run.
//   forward  one CTA per (batch b, 32 channels, range of <= 256 cells).  The tile lives in shared memory, zeroed there;
//            the CTA reads b's locations 256 at a time (the next round's in flight during this one), keeps the entities
//            of its cell range (ballot + prefix compaction, grouped by owning warp, m order inside a group), stages their
//            32-channel slices of x in shared memory with cp.async (all copies of a round in flight at once) and applies
//            them: warp w owns the cells with cell % 8 == w and applies exactly its group in m order, so each cell sees
//            its entities in sequence while all eight warps work.  The tile leaves as one cp.async.bulk store per channel row (the row's
//            cells are contiguous in (B,N,H,W)); per-thread streaming stores when H*W % 4 != 0 or `out` is misaligned.
//   backward two regimes, picked by bytes: the whole map B*N*H*W*4 against one 32-byte sector per gathered element
//            B*M*N*32.  Dense maps: one CTA per (b, 32 channels) bulk-copies its grad_out planes into shared memory and
//            gathers from there, writing grad_x rows coalesced.  Sparse maps: a warp per entity gathers straight from
//            global memory (one sector per element) -- the map is mostly never read.
#include <algorithm>

#include "common.cuh"

namespace hpcrll {

constexpr int kScThreads = 256;
constexpr int kScWarps = kScThreads / 32;
constexpr int kScChan = 32;       // channels per CTA: one per lane
constexpr int kScMaxCells = 256;  // cells per forward tile (33 KB of shared memory with 32 channels)
constexpr int kScSlabMax = 112 * 1024;  // shared-memory budget of one backward slab (32 channel planes)

// location (y, x) of entity r -> cell index, or -1 when outside the map
__device__ __forceinline__ int sc_cell(const int64_t* __restrict__ loc, int64_t r, int H, int W) {
    const int64_t y = __ldg(loc + 2 * r), x = __ldg(loc + 2 * r + 1);
    return (y >= 0 && y < H && x >= 0 && x < W) ? static_cast<int>(y) * W + static_cast<int>(x) : -1;
}

// 4-byte asynchronous copy global -> shared (no register round trip: every copy of a round is in flight at once)
__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Dynamic shared memory: the tile [kScChan][ct + 4] (channel rows of the cell range, 16-byte aligned rows), then the
// staged x slices [min(M, kScThreads)][kScChan] of one round's kept entities.
template <bool ADD, bool BULK>
__global__ void __launch_bounds__(kScThreads) scatter_conn_fwd_kernel(const float* __restrict__ x,
                                                                     const int64_t* __restrict__ loc,
                                                                     float* __restrict__ out, int M, int N, int H,
                                                                     int W, int ct, int ntiles, int nchunks) {
    extern __shared__ __align__(128) float sc_smem[];
    __shared__ int keep_m[kScThreads], keep_c[kScThreads];  // kept entities, grouped by owning warp, m order inside
    __shared__ int cnt[kScWarps * kScWarps];                // [owner][warp] kept counts -> their exclusive prefix
    __shared__ int ktotal;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int HW = H * W, pitch = ct + 4;
    int64_t blk = blockIdx.x;
    const int tile = static_cast<int>(blk % ntiles);
    blk /= ntiles;
    const int n0 = static_cast<int>(blk % nchunks) * kScChan;
    const int64_t b = blk / nchunks;
    const int c0 = tile * ct, cells = min(ct, HW - c0), nc = min(kScChan, N - n0);
    float* const sc_tile = sc_smem;
    float* const xs = sc_smem + kScChan * pitch;

    {
        float4* z = reinterpret_cast<float4*>(sc_tile);
        for (int i = tid; i < kScChan * pitch / 4; i += kScThreads) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const int64_t* lb = loc + 2 * b * M;
    const float* xb = x + b * M * N + n0 + lane;
    int64_t ly = -1, lx = -1;  // location of entity m0 + tid, loaded one round ahead
    if (tid < M) {
        ly = __ldg(lb + 2 * tid);
        lx = __ldg(lb + 2 * tid + 1);
    }
    __syncthreads();
    for (int m0 = 0; m0 < M; m0 += kScThreads) {
        // keep this round's entities that land in [c0, c0 + cells)
        const int m = m0 + tid;
        int c = -1;
        if (m < M && ly >= 0 && ly < H && lx >= 0 && lx < W) {
            c = static_cast<int>(ly) * W + static_cast<int>(lx) - c0;
            if (static_cast<unsigned>(c) >= static_cast<unsigned>(cells)) c = -1;
        }
        if (m + kScThreads < M) {
            ly = __ldg(lb + 2 * (m + kScThreads));
            lx = __ldg(lb + 2 * (m + kScThreads) + 1);
        }
        // compaction grouped by the warp that owns the cell (cell % 8), m order inside each group
        const int own = c >= 0 ? (c & (kScWarps - 1)) : -1;
        unsigned mine = 0;
#pragma unroll
        for (int o = 0; o < kScWarps; ++o) {
            const unsigned bo = __ballot_sync(0xffffffffu, own == o);
            if (own == o) mine = bo;
            if (lane == 0) cnt[o * kScWarps + warp] = __popc(bo);
        }
        __syncthreads();
        if (warp == 0) {  // exclusive prefix of the 64 counts, owner-major
            const int a0 = cnt[2 * lane], a1 = cnt[2 * lane + 1];
            int s = a0 + a1;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, s, d);
                if (lane >= d) s += t;
            }
            cnt[2 * lane] = s - a0 - a1;
            cnt[2 * lane + 1] = s - a1;
            if (lane == 31) ktotal = s;
        }
        __syncthreads();
        if (c >= 0) {
            const int pos = cnt[own * kScWarps + warp] + __popc(mine & ((1u << lane) - 1u));
            keep_m[pos] = m;
            keep_c[pos] = c;
        }
        __syncthreads();
        const int total = ktotal;
        for (int i = warp; i < total; i += kScWarps) {
            float* d = xs + i * kScChan + lane;
            if (lane < nc) cp_async4(d, xb + static_cast<int64_t>(keep_m[i]) * N);
            else *d = 0.f;
        }
        cp_async_wait_all();
        __syncthreads();
        // warp w applies, in m order, exactly the entities whose cell it owns
        const int e1 = warp == kScWarps - 1 ? total : cnt[(warp + 1) * kScWarps];
        for (int i = cnt[warp * kScWarps]; i < e1; ++i) {
            float* d = sc_tile + lane * pitch + keep_c[i];
            const float v = xs[i * kScChan + lane];
            *d = ADD ? *d + v : v;
        }
        __syncthreads();  // the kept lists, counts and staged slices are reused next round
    }

    float* dst = out + (b * N + n0) * static_cast<int64_t>(HW) + c0;
    if (BULK) {
        fence_proxy_async_smem();  // this thread's tile writes are visible to the bulk copy engine
        __syncthreads();
        if (tid < nc) {
            bulk_store_1d(dst + static_cast<int64_t>(tid) * HW, sc_tile + tid * pitch, static_cast<uint32_t>(cells) * 4u);
            bulk_commit_group();
            bulk_wait_group_read<0>();  // shared memory stays valid until the copy engine has read it
        }
    } else {
        for (int n = warp; n < nc; n += kScWarps)
            for (int cc = lane; cc < cells; cc += 32) st_stream(dst + static_cast<int64_t>(n) * HW + cc, sc_tile[n * pitch + cc]);
    }
}

// dense maps: grad_out[b, n0:n0+nc, :] is contiguous -> shared memory by bulk copies, gather from there
__global__ void __launch_bounds__(kScThreads) scatter_conn_bwd_slab_kernel(const float* __restrict__ g,
                                                                          const int64_t* __restrict__ loc,
                                                                          float* __restrict__ gx, int M, int N, int H,
                                                                          int W, int nchunks) {
    extern __shared__ __align__(128) float slab[];  // [nc][pitch]
    __shared__ __align__(8) uint64_t bar;
    __shared__ int cellbuf[kScThreads];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int HW = H * W, pitch = HW + 4;
    const int n0 = static_cast<int>(blockIdx.x % nchunks) * kScChan;
    const int64_t b = blockIdx.x / nchunks;
    const int nc = min(kScChan, N - n0);
    if (tid == 0) {
        mbar_init(&bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (tid == 0) {
        const float* src = g + (b * N + n0) * static_cast<int64_t>(HW);
        mbar_arrive_expect_tx(&bar, static_cast<uint32_t>(nc) * HW * 4u);
        for (int n = 0; n < nc; ++n)
            bulk_load_1d(slab + n * pitch, src + static_cast<int64_t>(n) * HW, static_cast<uint32_t>(HW) * 4u, &bar);
    }
    for (int m0 = 0; m0 < M; m0 += kScThreads) {
        // the cells of 256 entities at once (the first round's loads overlap the bulk copy)
        if (m0 + tid < M) cellbuf[tid] = sc_cell(loc, b * M + m0 + tid, H, W);
        if (m0 == 0) mbar_wait(&bar, 0);
        __syncthreads();
        const int mn = min(kScThreads, M - m0);
        float* dst = gx + (b * M + m0) * N + n0 + lane;
        for (int i = warp; i < mn; i += kScWarps) {
            const int c = cellbuf[i];
            if (lane < nc) dst[static_cast<int64_t>(i) * N] = c >= 0 ? slab[lane * pitch + c] : 0.f;
        }
        __syncthreads();  // cellbuf is refilled next round
    }
}

// sparse maps: a warp per entity, lanes along the channels, one 32-byte sector of grad_out per element
__global__ void __launch_bounds__(kScThreads) scatter_conn_bwd_gather_kernel(const float* __restrict__ g,
                                                                            const int64_t* __restrict__ loc,
                                                                            float* __restrict__ gx, int64_t rows,
                                                                            int M, int N, int H, int W) {
    const int lane = threadIdx.x & 31;
    const int64_t HW = static_cast<int64_t>(H) * W;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kScWarps;
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * kScWarps + (threadIdx.x >> 5); r < rows; r += stride) {
        const int c = sc_cell(loc, r, H, W);
        const float* src = g + (r / M) * N * HW + max(c, 0);
        float* dst = gx + r * N;
#pragma unroll 4
        for (int n = lane; n < N; n += 32) dst[n] = c >= 0 ? __ldg(src + n * HW) : 0.f;
    }
}

// cfg (HPC_RLL_CFG_SCATTER_CONNECTION / hpc_rll_debug_set_config): -1 automatic; otherwise bit 0 = forward with
// per-thread stores, bit 1 = backward by direct gather (a slab request the shapes cannot take runs the gather)
template <bool ADD, bool BULK>
static int launch_fwd(const float* x, const int64_t* loc, float* out, int64_t B, int M, int N, int H, int W,
                      cudaStream_t stream) {
    const int HW = H * W;
    const int ntiles = (HW + kScMaxCells - 1) / kScMaxCells;
    const int ct = ((HW + ntiles - 1) / ntiles + 3) & ~3;
    const int nchunks = (N + kScChan - 1) / kScChan;
    const int64_t blocks = B * ntiles * nchunks;
    HPC_REQUIRE(blocks <= INT32_MAX, "scatter_connection_forward: problem too large (%lld tiles)", (long long)blocks);
    const size_t smem = (static_cast<size_t>(kScChan) * (ct + 4) + static_cast<size_t>(std::min(M, kScThreads)) * kScChan) *
                        sizeof(float);
    static SmemOptIn opt;  // also selects the max-shared carveout: several CTAs per SM hide each other's latencies
    if (int rc = opt.ensure(scatter_conn_fwd_kernel<ADD, BULK>, static_cast<int>(smem))) return rc;
    scatter_conn_fwd_kernel<ADD, BULK><<<static_cast<unsigned>(blocks), kScThreads, smem, stream>>>(
        x, loc, out, M, N, H, W, ct, ntiles, nchunks);
    count_launch();
    HPC_LAUNCH_CHECK();
    return HPC_RLL_OK;
}

// every size fits an int and so does the cell index y*W + x (products of two sizes then fit an int64)
static bool sizes_fit(int64_t B, int64_t M, int64_t N, int64_t H, int64_t W) {
    return B <= INT32_MAX && M <= INT32_MAX && N <= INT32_MAX && H <= INT32_MAX && W <= INT32_MAX && H * W <= INT32_MAX;
}

static int scatter_forward(const float* x, const int64_t* loc, float* out, int64_t B, int64_t M, int64_t N, int64_t H,
                           int64_t W, int mode, cudaStream_t stream) {
    HPC_REQUIRE(B >= 0 && M >= 0 && N >= 0 && H >= 0 && W >= 0, "scatter_connection_forward: negative size");
    HPC_REQUIRE(mode == 0 || mode == 1, "scatter_connection_forward: mode must be 0 (cover) or 1 (add), got %d", mode);
    HPC_REQUIRE(sizes_fit(B, M, N, H, W), "scatter_connection_forward: sizes out of range");
    if (B == 0 || N == 0 || H * W == 0) return HPC_RLL_OK;
    HPC_REQUIRE(out && (M == 0 || (x && loc)), "scatter_connection_forward: null pointer");
    const int cfg = tuning_config(HPC_RLL_OP_SCATTER_CONNECTION);
    const bool bulk = (H * W) % 4 == 0 && aligned16(out) && !(cfg >= 0 && (cfg & 1));
    const int m = static_cast<int>(M), n = static_cast<int>(N), h = static_cast<int>(H), w = static_cast<int>(W);
    if (mode == 1)
        return bulk ? launch_fwd<true, true>(x, loc, out, B, m, n, h, w, stream)
                    : launch_fwd<true, false>(x, loc, out, B, m, n, h, w, stream);
    return bulk ? launch_fwd<false, true>(x, loc, out, B, m, n, h, w, stream)
                : launch_fwd<false, false>(x, loc, out, B, m, n, h, w, stream);
}

static int scatter_backward(const float* g, const int64_t* loc, float* gx, int64_t B, int64_t M, int64_t N, int64_t H,
                            int64_t W, cudaStream_t stream) {
    HPC_REQUIRE(B >= 0 && M >= 0 && N >= 0 && H >= 0 && W >= 0, "scatter_connection_backward: negative size");
    HPC_REQUIRE(sizes_fit(B, M, N, H, W), "scatter_connection_backward: sizes out of range");
    if (B == 0 || M == 0 || N == 0) return HPC_RLL_OK;
    const int64_t HW = H * W;
    HPC_REQUIRE(gx && loc && (HW == 0 || g), "scatter_connection_backward: null pointer");
    const int nchunks = static_cast<int>((N + kScChan - 1) / kScChan);
    const size_t slab = static_cast<size_t>(std::min<int64_t>(N, kScChan)) * (HW + 4) * sizeof(float);
    const bool slab_ok = HW > 0 && HW % 4 == 0 && aligned16(g) && slab <= kScSlabMax && B * nchunks <= INT32_MAX;
    const int cfg = tuning_config(HPC_RLL_OP_SCATTER_CONNECTION);
    const bool dense = HW * 4 <= M * 32;  // B*N*H*W*4 bytes of map against B*M*N 32-byte sectors
    const bool use_slab = slab_ok && (cfg >= 0 ? !(cfg & 2) : dense);
    const int m = static_cast<int>(M), n = static_cast<int>(N), h = static_cast<int>(H), w = static_cast<int>(W);
    if (use_slab) {
        static SmemOptIn opt;
        if (slab > 48 * 1024)
            if (int rc = opt.ensure(scatter_conn_bwd_slab_kernel, static_cast<int>(slab))) return rc;
        scatter_conn_bwd_slab_kernel<<<static_cast<unsigned>(B * nchunks), kScThreads, slab, stream>>>(g, loc, gx, m, n,
                                                                                                     h, w, nchunks);
    } else {
        const int64_t rows = B * M;
        const int64_t blocks = std::min<int64_t>((rows + kScWarps - 1) / kScWarps, static_cast<int64_t>(sm_count()) * 64);
        scatter_conn_bwd_gather_kernel<<<static_cast<unsigned>(blocks), kScThreads, 0, stream>>>(g, loc, gx, rows, m, n,
                                                                                               h, w);
    }
    count_launch();
    HPC_LAUNCH_CHECK();
    return HPC_RLL_OK;
}

}  // namespace hpcrll

extern "C" {

int hpc_rll_scatter_connection_forward(const float* x, const int64_t* location, float* out, int64_t B, int64_t M,
                                       int64_t N, int64_t H, int64_t W, int mode, void* stream) {
    HPC_NVTX("scatter_connection_forward");
    return hpcrll::scatter_forward(x, location, out, B, M, N, H, W, mode, hpcrll::as_stream(stream));
}

int hpc_rll_scatter_connection_backward(const float* grad_out, const int64_t* location, float* grad_x, int64_t B,
                                        int64_t M, int64_t N, int64_t H, int64_t W, void* stream) {
    HPC_NVTX("scatter_connection_backward");
    return hpcrll::scatter_backward(grad_out, location, grad_x, B, M, N, H, W, hpcrll::as_stream(stream));
}

}  // extern "C"

// Shared helpers for the sm_100a sub-LP engine: error plumbing, device buffers, the (row, scenario)
// thread mapping and the deterministic two-stage reductions used by every KKT / restart / merit kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/asm_b200.h"

namespace asmb {

// ---- error plumbing (no exception crosses the C ABI) ----------------------------------------------------
inline std::string &err_slot() {
    static thread_local std::string s;
    return s;
}
inline int fail(int code, const std::string &msg) {
    err_slot() = msg;
    return code;
}
#define ASM_CK(call)                                                                                      \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess) {                                                                         \
            char b__[512];                                                                                \
            snprintf(b__, sizeof b__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return ::asmb::fail(ASM_E_CUDA, b__);                                                         \
        }                                                                                                 \
    } while (0)
#define ASM_TRY(expr)                                                                                     \
    do {                                                                                                  \
        int r__ = (expr);                                                                                 \
        if (r__ != ASM_OK) return r__;                                                                    \
    } while (0)

// ---- device buffer ---------------------------------------------------------------------------------------
template <class T>
struct DBuf {
    T *p = nullptr;
    size_t n = 0;
    DBuf() = default;
    DBuf(const DBuf &) = delete;
    DBuf &operator=(const DBuf &) = delete;
    ~DBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    int alloc(size_t count) {
        release();
        n = count;
        if (count == 0) return ASM_OK;
        ASM_CK(cudaMalloc(&p, count * sizeof(T)));
        return ASM_OK;
    }
    int zero(cudaStream_t st) {
        if (n) ASM_CK(cudaMemsetAsync(p, 0, n * sizeof(T), st));
        return ASM_OK;
    }
    int upload(const T *host, size_t count, cudaStream_t st) {
        if (count) ASM_CK(cudaMemcpyAsync(p, host, count * sizeof(T), cudaMemcpyHostToDevice, st));
        return ASM_OK;
    }
};

// pinned host staging that grows on demand
struct Pinned {
    void *p = nullptr;
    size_t bytes = 0;
    ~Pinned() {
        if (p) cudaFreeHost(p);
    }
    int reserve(size_t b) {
        if (b <= bytes) return ASM_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        bytes = 0;
        ASM_CK(cudaHostAlloc(&p, b, cudaHostAllocDefault));
        bytes = b;
        return ASM_OK;
    }
};

// Host -> device copies of caller-owned arrays.  A Julia Vector{Float64} (or a numpy array) is pageable memory: an
// async copy from it is staged by the driver and is not asynchronous at all.  When the caller's pointer is pinned
// (cudaHostRegister / cudaHostAlloc) the copy goes straight from it; otherwise it goes through this handle's own ring
// of two pinned chunks, the memcpy into one chunk overlapping the DMA out of the other.
struct PinnedRing {
    static constexpr size_t kChunk = 8u << 20;
    Pinned buf[2];
    cudaEvent_t ev[2] = {nullptr, nullptr};
    bool used[2] = {false, false};
    int next = 0;
    ~PinnedRing() {
        for (auto &e : ev)
            if (e) cudaEventDestroy(e);
    }
    static bool is_pinned(const void *p) {
        cudaPointerAttributes at;
        const cudaError_t e = cudaPointerGetAttributes(&at, p);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
    }
    int h2d(void *dst, const void *src, size_t bytes, cudaStream_t st) {
        if (bytes == 0) return ASM_OK;
        if (is_pinned(src)) {
            ASM_CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
            return ASM_OK;
        }
        for (size_t off = 0; off < bytes; off += kChunk) {
            const size_t sz = std::min(kChunk, bytes - off);
            const int i = next;
            next ^= 1;
            ASM_TRY(buf[i].reserve(kChunk));
            if (!ev[i]) ASM_CK(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
            if (used[i]) ASM_CK(cudaEventSynchronize(ev[i]));   // the DMA out of this chunk has finished
            memcpy(buf[i].p, (const char *)src + off, sz);
            ASM_CK(cudaMemcpyAsync((char *)dst + off, buf[i].p, sz, cudaMemcpyHostToDevice, st));
            ASM_CK(cudaEventRecord(ev[i], st));
            used[i] = true;
        }
        return ASM_OK;
    }
};

// ---- launch geometry ---------------------------------------------------------------------------------------
// Device vectors of a batch are stored element-major: v[i * B + s] (scenario s fastest), so that the 32
// lanes of a warp hold 32 scenarios of the same row: index loads are warp-uniform, value loads and the
// x / y gathers are fully coalesced.  B is 1 (single LP) or a multiple of 32.
constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kSMs = 148;
constexpr int kMaxBlocksX = kSMs * 8;  // cap of gridDim.x for reduction kernels (fixed partial stride)

struct Geo {
    dim3 grid, block;
};
// geometry for a kernel whose work items are `count` rows (or columns) times B scenarios
inline Geo geo_for(int64_t count, int B) {
    Geo g;
    g.block = dim3(kThreads);
    if (B == 1) {
        int64_t nb = (count + kThreads - 1) / kThreads;
        if (nb < 1) nb = 1;
        if (nb > kMaxBlocksX) nb = kMaxBlocksX;
        g.grid = dim3((unsigned)nb);
    } else {
        int gy = B / 32;
        int64_t nb = (count + kWarps - 1) / kWarps;
        int64_t cap = (kMaxBlocksX * 2) / gy;
        if (cap < 1) cap = 1;
        if (cap > kMaxBlocksX) cap = kMaxBlocksX;
        if (nb < 1) nb = 1;
        if (nb > cap) nb = cap;
        g.grid = dim3((unsigned)nb, (unsigned)gy);
    }
    return g;
}

// iteration over the items of this thread: for (i = first; i < count; i += stride) with scenario s fixed
template <bool BATCH>
struct Map {
    int s;       // scenario of this thread
    int64_t first, stride;
    __device__ __forceinline__ Map() {
        if (BATCH) {
            s = blockIdx.y * 32 + (threadIdx.x & 31);
            first = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5);
            stride = (int64_t)gridDim.x * kWarps;
        } else {
            s = 0;
            first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
            stride = (int64_t)gridDim.x * blockDim.x;
        }
    }
};

// ---- deterministic block reduction -------------------------------------------------------------------------
// acc[q] of every thread is reduced over the threads that share a scenario and written to
// partials[((qbase + q) * kMaxBlocksX + blockIdx.x) * B + s].  Bit q of `maxmask` selects max instead of sum.
// A second-stage kernel (one block per scenario) adds the per-block partials in a fixed order, so results do
// not depend on scheduling.
template <bool BATCH, int NQ>
__device__ __forceinline__ void block_reduce_store(double (&acc)[NQ], unsigned maxmask, double *partials, int qbase,
                                                   int B) {
    __shared__ double sm[NQ][kWarps][BATCH ? 32 : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (BATCH) {
#pragma unroll
        for (int q = 0; q < NQ; ++q) sm[q][warp][lane] = acc[q];
        __syncthreads();
        if (warp == 0) {
            const int s = blockIdx.y * 32 + lane;
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                double v = sm[q][0][lane];
                for (int w = 1; w < kWarps; ++w) {
                    double u = sm[q][w][lane];
                    v = ((maxmask >> q) & 1u) ? fmax(v, u) : v + u;
                }
                partials[((size_t)(qbase + q) * kMaxBlocksX + blockIdx.x) * B + s] = v;
            }
        }
    } else {
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            double v = acc[q];
            for (int o = 16; o > 0; o >>= 1) {
                double u = __shfl_down_sync(0xffffffffu, v, o);
                v = ((maxmask >> q) & 1u) ? fmax(v, u) : v + u;
            }
            if (lane == 0) sm[q][warp][0] = v;
        }
        __syncthreads();
        if (threadIdx.x < NQ) {
            const int q = threadIdx.x;
            double v = sm[q][0][0];
            for (int w = 1; w < kWarps; ++w) {
                double u = sm[q][w][0];
                v = ((maxmask >> q) & 1u) ? fmax(v, u) : v + u;
            }
            partials[((size_t)(qbase + q) * kMaxBlocksX + blockIdx.x)] = v;
        }
    }
}

// second stage, called by all threads of a block that owns scenario s: returns the reduction of
// partials[q][0..nbx)[s] in a fixed tree order (blockDim.x must be kFinalThreads).
constexpr int kFinalThreads = 128;
__device__ __forceinline__ double final_reduce(const double *partials, int q, int nbx, int B, int s, bool is_max) {
    __shared__ double sm[kFinalThreads];
    double v = is_max ? -INFINITY : 0.0;
    for (int b = threadIdx.x; b < nbx; b += kFinalThreads) {
        double u = partials[((size_t)q * kMaxBlocksX + b) * B + s];
        v = is_max ? fmax(v, u) : v + u;
    }
    __syncthreads();  // protect sm from the previous call
    sm[threadIdx.x] = v;
    __syncthreads();
    for (int o = kFinalThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            double u = sm[threadIdx.x + o];
            sm[threadIdx.x] = is_max ? fmax(sm[threadIdx.x], u) : sm[threadIdx.x] + u;
        }
        __syncthreads();
    }
    return sm[0];
}

// host (scenario-major, h[s * len + i], S scenarios) <-> device (element-major, d[i * B + s]) layout change,
// tiled through shared memory so both sides are coalesced.  grid (ceil(len/32), B/32), block (32, 8).
// Padding scenarios (s >= S) replicate scenario 0; S == 1 broadcasts one vector to the whole batch.
__global__ void k_layout_in(const double *__restrict__ src, double *__restrict__ dst, int64_t len, int S, int B) {
    __shared__ double tile[32][33];
    const int64_t i0 = (int64_t)blockIdx.x * 32;
    const int s0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int s = s0 + r;
        const int64_t i = i0 + threadIdx.x;
        if (i < len && s < B) tile[r][threadIdx.x] = src[(int64_t)(s < S ? s : 0) * len + i];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int64_t i = i0 + r;
        const int s = s0 + threadIdx.x;
        if (i < len && s < B) dst[i * B + s] = tile[threadIdx.x][r];
    }
}
__global__ void k_layout_out(const double *__restrict__ src, double *__restrict__ dst, int64_t len, int S, int B) {
    __shared__ double tile[32][33];
    const int64_t i0 = (int64_t)blockIdx.x * 32;
    const int s0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int64_t i = i0 + r;
        const int s = s0 + threadIdx.x;
        if (i < len && s < B) tile[r][threadIdx.x] = src[i * B + s];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int s = s0 + r;
        const int64_t i = i0 + threadIdx.x;
        if (i < len && s < S) dst[(int64_t)s * len + i] = tile[threadIdx.x][r];
    }
}

// k_layout_in for k lanes of a batch: host [k][len] (entry j in the order of `lanes`) -> device d[i * B + lanes[j]],
// tiled like k_layout_in so that the staging reads coalesce.  grid (ceil(len/32), ceil(k/32)), block (32, 8).
// The other lanes are not touched.
__global__ void k_lanes_in(const double *__restrict__ src, double *__restrict__ dst, const int *__restrict__ lanes,
                           int64_t len, int k, int B) {
    __shared__ double tile[32][33];
    const int64_t i0 = (int64_t)blockIdx.x * 32;
    const int j0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int j = j0 + r;
        const int64_t i = i0 + threadIdx.x;
        if (i < len && j < k) tile[r][threadIdx.x] = src[(int64_t)j * len + i];
    }
    __syncthreads();
    const int j = j0 + threadIdx.x;
    const int s = j < k ? lanes[j] : 0;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int64_t i = i0 + r;
        if (i < len && j < k) dst[i * B + s] = tile[threadIdx.x][r];
    }
}

// 1, or a multiple of 32; batches beyond 32 round up to 64 so that the two-scenarios-per-lane kernels apply
inline int pad_batch(int b) { return b <= 1 ? 1 : (b <= 32 ? 32 : ((b + 63) / 64) * 64); }

}  // namespace asmb

// Persistent, on-chip-resident PDHG loop: one *group* of G thread blocks owns one LP of the batch for its
// whole solve.
//
// Why: a sub-LP of the SLP path (reference MOI.optimize!(qp.model), /root/reference/src/algorithms/
// subproblem.jl:490) needs 10^4..10^6 PDHG iterations of two dependent SpMVs each.  One LP is at most
// ~37 MB per iteration (SURVEY.md App. D), so a launch-per-half-iteration design is bound by launch latency
// (~7 us per kernel) and not by HBM.  Here the scaled matrix K (sliced-ELL, rows sorted by length inside a
// block) and K' live in the shared memory of the G blocks for the whole solve (MATS) or stream from L2 in
// sliced-ELL order (large LPs), the iterate pieces (x, y, anchors, bounds) are always in shared memory; only the
// two exchange vectors (xbar, y) go through L2: after each barrier a block copies the entries its rows (columns)
// touch -- its *halo*, a sorted index list fixed by the pattern -- into shared memory with near-coalesced loads
// and gathers from there (an SM sustains only ~0.5 scattered global loads per cycle, but ~8 shared ones).
// A block owns a contiguous range of rows and of columns; a warp owns 32-slot slices.  Blocks of a group meet at
// two barriers per iteration:
//   CLUSTER mode  G <= 16 : the group is a thread-block cluster, barrier = barrier.cluster (hardware); when the push
//                           lists fit (PUSH) the exchange does not touch L2 at all: the block that computes an
//                           entry of xbar (y) stores it straight into the halo buffers of the blocks that need it,
//                           through distributed shared memory, and the cluster barrier publishes the stores
//   GRID mode     G  > 16 : cooperative launch, barrier = one global counter per group
// Groups pull LPs of the batch from an atomic queue, so every LP stops at its own convergence.
// The iteration's arithmetic and the check decision (KKT, restart, primal weight: pdhg_decide) are the ones of
// pdhg.cuh; every block of the group takes the decision redundantly and bit-identically from the same ordered
// partial sums.
#pragma once
#include <cooperative_groups.h>

#include "pdhg.cuh"

namespace asmb {

constexpr int kGThreads = 1024;
constexpr int kGWarps = kGThreads / 32;
constexpr int kMaxClusterG = 16;
constexpr int kMaxSteps = 256;  // check_every is capped to this in the group engine

struct GroupCta {
    int r0, nR, nSR, sellR_base, sellR_cnt, ptrR_base, slotR_base, haloR_base, haloR_cnt;
    int c0, nC, nSC, sellC_base, sellC_cnt, ptrC_base, slotC_base, haloC_base, haloC_cnt;
    int pushR_base, pushR_cnt, pushC_base, pushC_cnt;  // consumers of this block's y (rows) and xbar (columns)
};

// shared-memory carve (element counts are the maxima over the blocks of the group)
struct GroupSmem {
    int maxSellR, maxSellC, maxRpad, maxCpad, maxNSR, maxNSC, maxHaloR, maxHaloC;
    int mats;  // 1: matrix values in shared memory, 0: streamed from L2
    int push, maxPushR, maxPushC;  // 1: exchange through distributed shared memory (cluster, mats only)
    size_t bytes() const {
        size_t b = 0;
        if (mats) b += sizeof(double) * ((size_t)maxSellR + maxSellC);
        // iterates (y, anchor | x, anchor) always; the per-slot constants (rl, ru | c, lb, ub) only next to the
        // matrix values -- in streaming mode they are re-read from L2 together with the halo
        b += sizeof(double) * ((mats ? 4 : 2) * (size_t)maxRpad + (mats ? 5 : 2) * (size_t)maxCpad);
        b += sizeof(double) * ((size_t)maxHaloR + maxHaloC);
        b += sizeof(double) * (size_t)(16 * kGWarps);  // reduction scratch
        b += sizeof(int) * ((size_t)maxHaloR + maxHaloC + maxRpad + maxCpad + maxNSR + 1 + maxNSC + 1);
        b += sizeof(unsigned short) * ((size_t)maxSellR + maxSellC);
        b += (size_t)maxRpad + maxCpad;  // tail bytes
        if (push) b += sizeof(int) * ((size_t)maxRpad + 1 + maxCpad + 1 + maxPushR + maxPushC + 4);
        return b + 64;
    }
};

struct GroupPlan {
    int G = 0;
    bool cluster = true;
    GroupSmem sm{};
    std::vector<GroupCta> cta;
    DBuf<GroupCta> d_cta;
    DBuf<int> sellR_src, sellR_idx, ptrR, slotR, haloR, sellC_src, sellC_idx, ptrC, slotC, haloC;
    DBuf<unsigned char> tailR, tailC;
    DBuf<int> pushR_ptr, pushR_dst, pushC_ptr, pushC_dst;  // per slot: (consumer rank << 16 | halo position) lists
    int totSellR = 0, totSellC = 0;
    DBuf<double> gA, gAT;  // per resident group: matrix values in sliced-ELL order (streamed when !mats)
    DBuf<double> gconst;   // per resident group and block: rl, ru, c, lb, ub by slot (when !mats)
    // per-launch workspace
    int n_groups = 0, max_groups = 0;
    DBuf<double> gx, gx2, gxp, grc, gy, gyp, gray, part;
    DBuf<unsigned> bar;
    DBuf<int> queue, slot;
};

// ---- host: partition + sliced-ELL layout -----------------------------------------------------------------------
// `ptr`/`idx` is CSR (for the row side) or CSC (for the column side) of the pattern; `count` rows (columns),
// gathered indices range over `other`.  Per block: a contiguous range, its halo (sorted distinct gathered
// indices), and a sliced-ELL layout over *slots*: a row longer than kSlotCap is cut into pieces that sit in
// consecutive lanes of one slice (the head lane owns the row, a segmented warp reduction adds the pieces), so
// no lane walks more than ~kSlotCap entries.  Rows are ordered by (pieces, length) so slices are nearly
// rectangular.  Every element stores the source position in the value array (-1 = padding) and the halo
// position of the gathered index.
constexpr int kSlotCap = 8;
struct SellSide {
    std::vector<int> first, cnt, nslice, base, ecnt, ptr_base, slot_base, halo_base, halo_cnt;
    std::vector<int> src, idx, ptr, slot, halo;
    std::vector<unsigned char> tail;  // per slot: lanes that follow in the same row group
};
inline void build_sell_side(int count, int other, const int *ptr, const int *idx, const int *srcmap, int G, SellSide &o) {
    o = SellSide();
    std::vector<int> pos(other, -1);
    std::vector<long long> pre(count + 1, 0);
    for (int i = 0; i < count; ++i) pre[i + 1] = pre[i] + (ptr[i + 1] - ptr[i]) + 2;
    int start = 0;
    for (int c = 0; c < G; ++c) {
        int end;
        if (c == G - 1) {
            end = count;
        } else {
            const long long target = pre[count] * (c + 1) / G;
            end = (int)(std::lower_bound(pre.begin(), pre.end(), target) - pre.begin());
            end = std::max(start, std::min(end, count));
        }
        const int nloc = end - start;
        std::vector<int> hl;
        for (int k = ptr[start]; k < ptr[end]; ++k)
            if (pos[idx[k]] < 0) {
                pos[idx[k]] = 0;
                hl.push_back(idx[k]);
            }
        std::sort(hl.begin(), hl.end());
        for (size_t t = 0; t < hl.size(); ++t) pos[hl[t]] = (int)t;
        o.halo_base.push_back((int)o.halo.size());
        o.halo_cnt.push_back((int)hl.size());
        o.halo.insert(o.halo.end(), hl.begin(), hl.end());
        auto pieces = [&](int i) {
            const int L = ptr[i + 1] - ptr[i];
            return std::max(1, std::min(32, (L + kSlotCap - 1) / kSlotCap));
        };
        std::vector<int> order(nloc);
        for (int i = 0; i < nloc; ++i) order[i] = start + i;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
            const int pa = pieces(a), pb = pieces(b);
            if (pa != pb) return pa > pb;
            return (ptr[a + 1] - ptr[a]) > (ptr[b + 1] - ptr[b]);
        });
        // pack whole rows into 32-lane slices
        struct Lane {
            int row, k0, k1, tail;
            bool head;
        };
        std::vector<std::vector<Lane>> slices;
        std::vector<Lane> cur;
        for (int i : order) {
            const int pc = pieces(i), L = ptr[i + 1] - ptr[i];
            const int plen = (L + pc - 1) / pc;
            if ((int)cur.size() + pc > 32) {
                slices.push_back(cur);
                cur.clear();
            }
            for (int q = 0; q < pc; ++q) {
                Lane ln;
                ln.row = i;
                ln.k0 = ptr[i] + std::min(L, q * plen);
                ln.k1 = ptr[i] + std::min(L, (q + 1) * plen);
                ln.tail = pc - 1 - q;
                ln.head = q == 0;
                cur.push_back(ln);
            }
        }
        if (!cur.empty()) slices.push_back(cur);
        const int ns = (int)slices.size();
        o.first.push_back(start);
        o.cnt.push_back(nloc);
        o.nslice.push_back(ns);
        o.base.push_back((int)o.src.size());
        o.ptr_base.push_back((int)o.ptr.size());
        o.slot_base.push_back((int)o.slot.size());
        int cols = 0;
        o.ptr.push_back(0);
        for (int q = 0; q < ns; ++q) {
            int len = 0;
            for (const Lane &ln : slices[q]) len = std::max(len, ln.k1 - ln.k0);
            const size_t at = o.src.size();
            o.src.resize(at + (size_t)len * 32, -1);
            o.idx.resize(at + (size_t)len * 32, 0);
            for (int lane = 0; lane < 32; ++lane) {
                if (lane < (int)slices[q].size()) {
                    const Lane &ln = slices[q][lane];
                    for (int k = ln.k0; k < ln.k1; ++k) {
                        o.src[at + (size_t)(k - ln.k0) * 32 + lane] = srcmap ? srcmap[k] : k;
                        o.idx[at + (size_t)(k - ln.k0) * 32 + lane] = pos[idx[k]];
                    }
                    o.slot.push_back(ln.head ? ln.row : -1);
                    o.tail.push_back((unsigned char)ln.tail);
                } else {
                    o.slot.push_back(-1);
                    o.tail.push_back(0);
                }
            }
            cols += len;
            o.ptr.push_back(cols);
        }
        o.ecnt.push_back(cols * 32);
        for (int t : hl) pos[t] = -1;
        start = end;
    }
}

// ---- device ---------------------------------------------------------------------------------------------------
struct GroupArgs {
    LpView v;
    const GroupCta *cta;
    const int *sellR_src, *sellR_idx, *ptrR, *slotR, *haloR, *sellC_src, *sellC_idx, *ptrC, *slotC, *haloC;
    const unsigned char *tailR, *tailC;
    const int *pushR_ptr, *pushR_dst, *pushC_ptr, *pushC_dst;
    double *gA, *gAT;  // [groups][totSellR], [groups][totSellC]
    double *gconst;    // [groups][G][2 maxRpad + 3 maxCpad]
    int totSellR, totSellC;
    double *gx, *gx2, *gxp, *grc, *gy, *gyp, *gray, *part;
    unsigned *bar;
    int *queue, *slot;
    int G, Buser;
    long long max_iter, budget;  // per-LP iteration limit; iterations one launch may add to an LP
    int steps;
    GroupSmem sm;
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

template <bool CLUSTER>
__device__ __forceinline__ void group_sync(unsigned *bar, unsigned &epoch, int G) {
    if (CLUSTER) {
        // one fence per block (not per warp): the block barrier orders every thread's stores before thread 0's fence
        __syncthreads();
        if (threadIdx.x == 0) __threadfence();
        asm volatile("barrier.cluster.arrive.relaxed.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    } else {
        __syncthreads();
        if (threadIdx.x == 0) {
            epoch += (unsigned)G;
            __threadfence();
            atomicAdd(bar, 1u);
            while ((int)(ld_acquire_u32(bar) - epoch) < 0) {
            }
            __threadfence();
        }
        __syncthreads();
    }
}

// exchange vectors are written by other blocks of the group between barriers: read them through L2
__device__ __forceinline__ double ldx(const double *p) { return __ldcg(p); }

// sum / max of `NQ` per-thread values over the block -> out[q] (thread 0 only has the result)
template <int NQ>
__device__ __forceinline__ void block_reduce(double (&acc)[NQ], unsigned maxmask, double *scratch, double *out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        double v = acc[q];
        for (int o = 16; o > 0; o >>= 1) {
            const double u = __shfl_down_sync(0xffffffffu, v, o);
            v = ((maxmask >> q) & 1u) ? fmax(v, u) : v + u;
        }
        if (lane == 0) scratch[q * kGWarps + warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < NQ) {
        const int q = threadIdx.x;
        double v = scratch[q * kGWarps];
        for (int w = 1; w < kGWarps; ++w) {
            const double u = scratch[q * kGWarps + w];
            v = ((maxmask >> q) & 1u) ? fmax(v, u) : v + u;
        }
        out[q] = v;
    }
    __syncthreads();
}

// halo copy: shared[t] = vec[list[t]] (list sorted => neighbouring lanes hit neighbouring sectors)
__device__ __forceinline__ void halo_fetch(double *__restrict__ dst, const double *__restrict__ vec,
                                           const int *__restrict__ list, int cnt) {
    for (int t = threadIdx.x; t < cnt; t += kGThreads) dst[t] = __ldcg(vec + list[t]);
    __syncthreads();
}

// one sliced-ELL row (column) of this lane: sum_k val[k] * halo[idx[k]]
// segmented suffix sum over the lanes of one row group: the head lane (largest tail) ends with the row total
__device__ __forceinline__ double seg_reduce(double v, int tail) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double u = __shfl_down_sync(0xffffffffu, v, o);
        if (tail >= o) v += u;
    }
    return v;
}
template <bool MATS>
__device__ __forceinline__ double sell_dot(const double *__restrict__ sval, const double *__restrict__ gval,
                                           const unsigned short *__restrict__ idx, const double *__restrict__ halo,
                                           int p0, int len, int tail, bool split) {
    double acc = 0.0;
#pragma unroll 8
    for (int k = 0; k < len; ++k) {
        const double a = MATS ? sval[p0 + k * 32] : __ldcg(gval + p0 + k * 32);
        acc += a * halo[idx[p0 + k * 32]];
    }
    return split ? seg_reduce(acc, tail) : acc;
}

// store `val` into the halo buffer of every block of the cluster that gathers this entry
__device__ __forceinline__ void push_halo(double *halo_local, const int *__restrict__ ptr, const int *__restrict__ dst,
                                          int sl, double val, int my_rank) {
    namespace cg = cooperative_groups;
    cg::cluster_group cl = cg::this_cluster();
    if (my_rank < 0) {   // one-block group: every consumer is this block
        for (int k = ptr[sl]; k < ptr[sl + 1]; ++k) halo_local[dst[k] & 0xffff] = val;
        return;
    }
    for (int k = ptr[sl]; k < ptr[sl + 1]; ++k) {
        const int t = dst[k];
        cl.map_shared_rank(halo_local, t >> 16)[t & 0xffff] = val;
    }
}
// barrier that publishes (distributed-)shared-memory stores; a one-block group only needs the block barrier
__device__ __forceinline__ void cluster_sync_dsm(int G) {
    if (G == 1)
        __syncthreads();
    else
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <bool CLUSTER, bool MATS, bool PUSH = false>
__global__ void __launch_bounds__(kGThreads, 1) k_pdhg_group(const GroupArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const LpView &v = a.v;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = a.G;
    const int rank = blockIdx.x % G, grp = blockIdx.x / G;
    const int B = v.B, n = v.n, m = v.m;
    const GroupCta d = a.cta[rank];
    // ---- carve shared memory
    double *a_val = reinterpret_cast<double *>(smem_raw);
    double *t_val = a_val + (MATS ? a.sm.maxSellR : 0);
    double *sy = t_val + (MATS ? a.sm.maxSellC : 0);
    double *sya = sy + a.sm.maxRpad;
    double *sx = sya + a.sm.maxRpad;
    double *sxa = sx + a.sm.maxCpad;
    double *cst = MATS ? sxa + a.sm.maxCpad
                       : a.gconst + ((size_t)(blockIdx.x / a.G) * a.G + blockIdx.x % a.G) * (2 * (size_t)a.sm.maxRpad + 3 * (size_t)a.sm.maxCpad);
    double *srl = cst;
    double *sru = srl + a.sm.maxRpad;
    double *scc = sru + a.sm.maxRpad;
    double *slb = scc + a.sm.maxCpad;
    double *sub = slb + a.sm.maxCpad;
    double *hx = MATS ? sub + a.sm.maxCpad : sxa + a.sm.maxCpad;  // halo of the row side: entries of xbar
    double *hy = hx + a.sm.maxHaloR;       // halo of the column side: entries of y
    double *scratch = hy + a.sm.maxHaloC;
    int *listR = reinterpret_cast<int *>(scratch + 16 * kGWarps);
    int *listC = listR + a.sm.maxHaloR;
    int *rmap = listC + a.sm.maxHaloC;
    int *cmap = rmap + a.sm.maxRpad;
    int *ptrR = cmap + a.sm.maxCpad;
    int *ptrC = ptrR + a.sm.maxNSR + 1;
    unsigned short *a_idx = reinterpret_cast<unsigned short *>(ptrC + a.sm.maxNSC + 1);
    unsigned short *t_idx = a_idx + a.sm.maxSellR;
    unsigned char *tailR = reinterpret_cast<unsigned char *>(t_idx + a.sm.maxSellC);
    unsigned char *tailC = tailR + a.sm.maxRpad;
    // push lists (PUSH only), 4-byte aligned after the tail bytes
    int *spushR_ptr = reinterpret_cast<int *>(reinterpret_cast<size_t>(tailC + a.sm.maxCpad + 3) & ~(size_t)3);
    int *spushC_ptr = spushR_ptr + a.sm.maxRpad + 1;
    int *spushR_dst = spushC_ptr + a.sm.maxCpad + 1;
    int *spushC_dst = spushR_dst + a.sm.maxPushR;
    __shared__ ScenState st;
    __shared__ double wtab[kMaxSteps];
    __shared__ DevParams P;
    __shared__ double qred[Q_COUNT];
    __shared__ int s_cur;

    // ---- pattern (shared by every LP of the batch): staged once
    for (int i = tid; i < d.sellR_cnt; i += kGThreads) a_idx[i] = (unsigned short)a.sellR_idx[d.sellR_base + i];
    for (int i = tid; i < d.sellC_cnt; i += kGThreads) t_idx[i] = (unsigned short)a.sellC_idx[d.sellC_base + i];
    for (int i = tid; i < d.haloR_cnt; i += kGThreads) listR[i] = a.haloR[d.haloR_base + i];
    for (int i = tid; i < d.haloC_cnt; i += kGThreads) listC[i] = a.haloC[d.haloC_base + i];
    for (int i = tid; i < d.nSR * 32; i += kGThreads) {
        rmap[i] = a.slotR[d.slotR_base + i];
        tailR[i] = a.tailR[d.slotR_base + i];
    }
    for (int i = tid; i < d.nSC * 32; i += kGThreads) {
        cmap[i] = a.slotC[d.slotC_base + i];
        tailC[i] = a.tailC[d.slotC_base + i];
    }
    if (PUSH) {
        for (int i = tid; i <= d.nSR * 32; i += kGThreads) spushR_ptr[i] = a.pushR_ptr[d.slotR_base + rank + i];
        for (int i = tid; i <= d.nSC * 32; i += kGThreads) spushC_ptr[i] = a.pushC_ptr[d.slotC_base + rank + i];
        for (int i = tid; i < d.pushR_cnt; i += kGThreads) spushR_dst[i] = a.pushR_dst[d.pushR_base + i];
        for (int i = tid; i < d.pushC_cnt; i += kGThreads) spushC_dst[i] = a.pushC_dst[d.pushC_base + i];
    }
    for (int i = tid; i <= d.nSR; i += kGThreads) ptrR[i] = a.ptrR[d.ptrR_base + i];
    for (int i = tid; i <= d.nSC; i += kGThreads) ptrC[i] = a.ptrC[d.ptrC_base + i];
    if (tid == 0) P = *v.prm;
    __syncthreads();

    double *gx = a.gx + (size_t)grp * n, *gx2 = a.gx2 + (size_t)grp * n, *gxp = a.gxp + (size_t)grp * n,
           *grc = a.grc + (size_t)grp * n;
    double *gy = a.gy + (size_t)grp * m, *gyp = a.gyp + (size_t)grp * m, *gray = a.gray + (size_t)grp * m;
    double *gA = a.gA + (size_t)grp * a.totSellR + d.sellR_base;    // this block's slice
    double *gAT = a.gAT + (size_t)grp * a.totSellC + d.sellC_base;
    double *part = a.part + (size_t)grp * G * Q_COUNT;
    unsigned *bar = a.bar + grp;
    unsigned epoch = 0;

    for (;;) {
        // ---- next LP of the batch
        if (rank == 0 && tid == 0) a.slot[grp] = atomicAdd(a.queue, 1);
        group_sync<CLUSTER>(bar, epoch, G);
        if (tid == 0) s_cur = __ldcg(a.slot + grp);
        __syncthreads();
        const int s = s_cur;
        if (s >= a.Buser) break;
        if (tid == 0) st = v.state[s];
        __syncthreads();
        if (st.status >= 0) continue;  // already finished (hybrid hand-over from the streaming engine): uniform in the group
        // ---- stage the values of this LP
        for (int i = tid; i < d.sellR_cnt; i += kGThreads) {
            const int src = a.sellR_src[d.sellR_base + i];
            const double val = src >= 0 ? v.A[(size_t)src * B + s] : 0.0;
            if (MATS)
                a_val[i] = val;
            else
                gA[i] = val;
        }
        for (int i = tid; i < d.sellC_cnt; i += kGThreads) {
            const int src = a.sellC_src[d.sellC_base + i];
            const double val = src >= 0 ? v.AT[(size_t)src * B + s] : 0.0;
            if (MATS)
                t_val[i] = val;
            else
                gAT[i] = val;
        }
        for (int sl = tid; sl < d.nSR * 32; sl += kGThreads) {
            const int gi = rmap[sl];
            double y0 = 0.0, ya0 = 0.0, l = -INFINITY, u = INFINITY;
            if (gi >= 0) {
                const size_t e = (size_t)gi * B + s;
                y0 = v.y[e];
                ya0 = v.ya[e];
                l = v.rls[e];
                u = v.rus[e];
                gy[gi] = y0;
            }
            sy[sl] = y0;
            sya[sl] = ya0;
            srl[sl] = l;
            sru[sl] = u;
        }
        for (int sl = tid; sl < d.nSC * 32; sl += kGThreads) {
            const int gj = cmap[sl];
            double x0 = 0.0, xa0 = 0.0, c = 0.0, l = 0.0, u = 0.0;
            if (gj >= 0) {
                const size_t e = (size_t)gj * B + s;
                x0 = v.x[e];
                xa0 = v.xa[e];
                c = v.cs[e];
                l = v.lbs[e];
                u = v.ubs[e];
            }
            sx[sl] = x0;
            sxa[sl] = xa0;
            scc[sl] = c;
            slb[sl] = l;
            sub[sl] = u;
        }
        group_sync<CLUSTER>(bar, epoch, G);
        if (PUSH) {   // the halos are kept current by the pushes from here on
            halo_fetch(hy, gy, listC, d.haloC_cnt);
            cluster_sync_dsm(G);
        }

        const bool live0 = true;
        long long it = st.total;
        const long long it_stop = it + a.budget;
        bool done = false;
        while (!done && it < a.max_iter && it < it_stop) {
            // step sizes and Halpern weights of this block of iterations (they only change at its last check)
            const double tau = st.eta / st.omega, sigma = st.eta * st.omega, isig = 1.0 / sigma;
            if (tid < a.steps) {
                wtab[tid] = pdhg_halpern_weight(st.k0 + tid + 1);
            }
            __syncthreads();
            for (int j = 0; j < a.steps && !done; ++j) {
                const bool check = (j == 0 || j == a.steps - 1);
                const double w = wtab[j];
                if (!check) {
                    // ------------------------------ primal half
                    if (!PUSH) halo_fetch(hy, gy, listC, d.haloC_cnt);
                    for (int q = warp; q < d.nSC; q += kGWarps) {
                        const int sl = q * 32 + lane;
                        const int p0 = ptrC[q] * 32 + lane, len = ptrC[q + 1] - ptrC[q];
                        const int tl = tailC[sl];
                        const double acc = sell_dot<MATS>(t_val, gAT, t_idx, hy, p0, len, tl, __any_sync(0xffffffffu, tl));
                        const int gj = cmap[sl];
                        const double xv = sx[sl];
                        const double xpv = pdhg_primal_step(xv, scc[sl] - acc, tau, slb[sl], sub[sl]);
                        const double xb = pdhg_reflect(xpv, xv);
                        if (gj >= 0) {
                            if (PUSH)
                                push_halo(hx, spushC_ptr, spushC_dst, sl, xb, G == 1 ? -1 : rank);
                            else
                                gx[gj] = xb;
                        }
                        sx[sl] = pdhg_halpern(w, xb, sxa[sl]);
                    }
                    if (PUSH)
                        cluster_sync_dsm(G);
                    else
                        group_sync<CLUSTER>(bar, epoch, G);
                    // ------------------------------ dual half
                    if (!PUSH) halo_fetch(hx, gx, listR, d.haloR_cnt);
                    for (int q = warp; q < d.nSR; q += kGWarps) {
                        const int sl = q * 32 + lane;
                        const int p0 = ptrR[q] * 32 + lane, len = ptrR[q + 1] - ptrR[q];
                        const int tl = tailR[sl];
                        const double acc = sell_dot<MATS>(a_val, gA, a_idx, hx, p0, len, tl, __any_sync(0xffffffffu, tl));
                        const int gi = rmap[sl];
                        const double yv = sy[sl];
                        const double ypv = pdhg_dual_step(acc, yv, sigma, isig, srl[sl], sru[sl]);
                        const double yn = pdhg_halpern(w, pdhg_reflect(ypv, yv), sya[sl]);
                        sy[sl] = yn;
                        if (gi >= 0) {
                            if (PUSH)
                                push_halo(hy, spushR_ptr, spushR_dst, sl, yn, G == 1 ? -1 : rank);
                            else
                                gy[gi] = yn;
                        }
                    }
                    if (PUSH)
                        cluster_sync_dsm(G);
                    else
                        group_sync<CLUSTER>(bar, epoch, G);
                    continue;
                }
                // ================================== check iteration ==========================================
                // (second operand of the two-vector products is gathered straight from L2: rare, so slow is fine)
                double acc[Q_COUNT];
#pragma unroll
                for (int i = 0; i < Q_COUNT; ++i) acc[i] = 0.0;
                if (!PUSH) halo_fetch(hy, gy, listC, d.haloC_cnt);
                for (int q = warp; q < d.nSC; q += kGWarps) {
                    const int sl = q * 32 + lane;
                    const int p0 = ptrC[q] * 32 + lane, len = ptrC[q + 1] - ptrC[q];
                    const int tl = tailC[sl];
                    const double s1 = sell_dot<MATS>(t_val, gAT, t_idx, hy, p0, len, tl, true);
                    const int gj = cmap[sl];
                    if (gj < 0) continue;
                    const double cj = scc[sl], xv = sx[sl];
                    const double xpv = pdhg_primal_step(xv, cj - s1, tau, slb[sl], sub[sl]);
                    const double xb = pdhg_reflect(xpv, xv);
                    gx[gj] = xb;
                    if (PUSH) push_halo(hx, spushC_ptr, spushC_dst, sl, xb, G == 1 ? -1 : rank);
                    gx2[gj] = xv;
                    gxp[gj] = xpv;
                    pdhg_col_terms(xpv, xv, sxa[sl], cj, acc[Q_DX2], acc[Q_DXA2], acc[Q_POBJ]);
                }
                group_sync<CLUSTER>(bar, epoch, G);
                if (PUSH) cluster_sync_dsm(G);
                const double inv_sb = 1.0 / st.sb, inv_sc = 1.0 / st.sc;
                if (!PUSH) halo_fetch(hx, gx, listR, d.haloR_cnt);
                for (int q = warp; q < d.nSR; q += kGWarps) {
                    const int sl = q * 32 + lane;
                    const int p0 = ptrR[q] * 32 + lane, len = ptrR[q + 1] - ptrR[q];
                    double s1 = 0.0, s2 = 0.0;
                    for (int k = 0; k < len; ++k) {
                        const double av = MATS ? a_val[p0 + k * 32] : __ldcg(gA + p0 + k * 32);
                        const int hp = a_idx[p0 + k * 32];
                        s1 += av * hx[hp];
                        s2 += av * __ldcg(gx2 + listR[hp]);
                    }
                    s1 = seg_reduce(s1, tailR[sl]);
                    s2 = seg_reduce(s2, tailR[sl]);
                    const int gi = rmap[sl];
                    if (gi < 0) continue;
                    const double yv = sy[sl];
                    const double l = srl[sl], u = sru[sl];
                    const double ypv = pdhg_dual_step(s1, yv, sigma, isig, l, u);
                    gyp[gi] = ypv;
                    const double dri = v.dr[(size_t)gi * B + s];
                    pdhg_row_terms(ypv, yv, sya[sl], s1, s2, l, u, inv_sb, dri, acc[Q_DY2], acc[Q_DYADX], acc[Q_DYA2],
                                   acc[Q_PRES2], acc[Q_DOBJ_ROW]);
                    const double dd = pdhg_ray(ypv - yv, l, u);
                    gray[gi] = dd;
                    pdhg_ray_row_terms(dd, l, u, dri, acc[Q_RAY_ROW], acc[Q_RAY_MAX]);
                }
                group_sync<CLUSTER>(bar, epoch, G);
                halo_fetch(hy, gyp, listC, d.haloC_cnt);
                for (int q = warp; q < d.nSC; q += kGWarps) {
                    const int sl = q * 32 + lane;
                    const int p0 = ptrC[q] * 32 + lane, len = ptrC[q + 1] - ptrC[q];
                    double s1 = 0.0, s2 = 0.0;
                    for (int k = 0; k < len; ++k) {
                        const double tv = MATS ? t_val[p0 + k * 32] : __ldcg(gAT + p0 + k * 32);
                        const int hp = t_idx[p0 + k * 32];
                        s1 += tv * hy[hp];
                        s2 += tv * __ldcg(gray + listC[hp]);
                    }
                    s1 = seg_reduce(s1, tailC[sl]);
                    s2 = seg_reduce(s2, tailC[sl]);
                    const int gj = cmap[sl];
                    if (gj < 0) continue;
                    const double rc = scc[sl] - s1;
                    grc[gj] = rc;
                    const double xpv = gxp[gj], l = slb[sl], u = sub[sl];
                    const double dcj = v.dc[(size_t)gj * B + s];
                    pdhg_rc_terms(rc, xpv, l, u, inv_sc, dcj, acc[Q_DRES2], acc[Q_DOBJ_COL]);
                    pdhg_ray_col_terms(s2, l, u, dcj, acc[Q_RAY_COL], acc[Q_KTY_MAX]);
                }
                block_reduce<Q_COUNT>(acc, kQMax, scratch, part + (size_t)rank * Q_COUNT);
                group_sync<CLUSTER>(bar, epoch, G);
                if (tid < Q_COUNT) {
                    const bool is_max = (kQMax >> tid) & 1u;
                    double t = __ldcg(part + tid);
                    for (int r = 1; r < G; ++r) {
                        const double u = __ldcg(part + (size_t)r * Q_COUNT + tid);
                        t = is_max ? fmax(t, u) : t + u;
                    }
                    qred[tid] = t;
                }
                __syncthreads();
                if (tid == 0) pdhg_decide(st, P, qred, j, a.steps, s == 0 && blockIdx.x == 0 ? "pdhg-g" : nullptr);
                __syncthreads();
                const int flag = st.restart_flag;
                // ------------------------------ apply: restart / freeze, or finish the Halpern step
                for (int sl = tid; sl < d.nSC * 32; sl += kGThreads) {
                    const int gj = cmap[sl];
                    if (gj < 0) continue;
                    const double xpv = gxp[gj];
                    if (flag) {
                        sx[sl] = xpv;
                        sxa[sl] = xpv;
                    } else {
                        sx[sl] = pdhg_halpern(w, pdhg_reflect(xpv, sx[sl]), sxa[sl]);
                    }
                }
                for (int sl = tid; sl < d.nSR * 32; sl += kGThreads) {
                    const int gi = rmap[sl];
                    if (gi < 0) continue;
                    const double ypv = gyp[gi];
                    double yn;
                    if (flag) {
                        yn = ypv;
                        sya[sl] = ypv;
                    } else {
                        yn = pdhg_halpern(w, pdhg_reflect(ypv, sy[sl]), sya[sl]);
                    }
                    sy[sl] = yn;
                    gy[gi] = yn;
                    if (PUSH) push_halo(hy, spushR_ptr, spushR_dst, sl, yn, G == 1 ? -1 : rank);
                }
                if (st.status >= 0) done = true;
                group_sync<CLUSTER>(bar, epoch, G);
                if (PUSH) cluster_sync_dsm(G);
            }
            it += a.steps;
        }
        // ---- hand the last checked point to k_finalize (element-major arrays of the solver)
        for (int sl = tid; sl < d.nSC * 32; sl += kGThreads) {
            const int gj = cmap[sl];
            if (gj < 0) continue;
            const size_t e = (size_t)gj * B + s;
            if (live0) {
                v.xp[e] = gxp[gj];
                v.gyp[e] = grc[gj];
            }
            v.x[e] = sx[sl];
            v.xa[e] = sxa[sl];
        }
        for (int sl = tid; sl < d.nSR * 32; sl += kGThreads) {
            const int gi = rmap[sl];
            if (gi < 0) continue;
            const size_t e = (size_t)gi * B + s;
            if (live0) v.yp[e] = gyp[gi];
            v.y[e] = sy[sl];
            v.ya[e] = sya[sl];
        }
        if (rank == 0 && tid == 0) v.state[s] = st;
        __syncthreads();
    }
}

}  // namespace asmb

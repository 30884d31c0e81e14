// Host-side symbolic analysis of the quasi-definite KKT matrix of the barrier engine (ipm.cuh)
//
//        M = [ -(Dx + d)    K'     ]      nodes 0..n-1   : columns of the LP (primal step)
//            [    K      (Ew + d)  ]      nodes n..n+m-1 : rows of the LP    (dual step)
//
// The sparsity pattern of the Jacobian is fixed for the life of a handle (the reference uploads j_str once,
// /root/reference/src/model.jl:10, and only pushes values per iteration, src/algorithms/subproblem.jl:438-457),
// so everything that depends on the pattern alone is done here once, on the host, in plain C++:
//   * a fill-reducing ordering (exact minimum degree on the explicit elimination graph),
//   * the pattern of L in  P M P' = L D L'  (any symmetric permutation of a quasi-definite matrix has such a
//     factorisation with D diagonal -- no numerical pivoting, hence a schedule that is identical for every LP of
//     a batch and every iteration),
//   * a level schedule (column j only needs columns of lower levels; levels grow strictly along the
//     elimination tree),
//   * for every entry of L and every pivot the products  W[i,k] * W[j,k] / d[k]  that update it ("terms";
//     W = L D), grouped by the LEVEL OF THE SOURCE COLUMN k: step l of the numerical factorisation applies the
//     updates of the columns of level l to all their targets (fan-out), one "chunk" = the terms of one target
//     in that step, summed in ascending k by one thread -- no atomics, bit-reproducible, and the critical path
//     of a step is the longest chunk (one term near the root of the tree, where a fan-in dot product would be
//     hundreds of terms long).  Nine chunks in ten are a single term: those are stored first in every step so
//     that the kernel can keep four of them in flight per warp,
//   * the same chunked fan-out lists for the forward substitution; the backward substitution needs no chunks
//     (the rows of a column are its ancestors, which sit on distinct levels),
//   * optionally (sn > 1) SUPERNODES: chains c_0 -> c_1 -> ... of at most sn columns along the elimination tree whose
//     patterns nest exactly (pattern(c_i) = {c_i+1} + pattern(c_i+1)), the separators of the network.  All columns
//     of a supernode share one step; the updates inside a supernode (its dense diagonal block and the rows below
//     it, "panel") are taken out of the term lists and done by a dense panel kernel at the start of the step, the
//     updates that leave it stay in the lists -- now one chunk of up to sn terms per target and step instead of
//     sn single-term read-modify-writes on sn steps.  A 1354-bus KKT matrix goes from 310 levels to 49 steps and
//     from 2.47 M to 0.47 M target updates per factorisation.
// No CUDA in this header: it is also compiled into the host-only self test (asm_kkt_selftest).
#pragma once
#include <stdint.h>
#include <stdlib.h>
#include <algorithm>
#include <atomic>
#include <functional>
#include <memory>
#include <thread>
#include <queue>
#include <utility>
#include <vector>

#ifdef KKT_PROFILE
#include <chrono>
#include <cstdio>
#define KKT_PHASE(name)                                                                                           \
    do {                                                                                                          \
        const auto now__ = std::chrono::steady_clock::now();                                                      \
        fprintf(stderr, "[kkt] %-28s %8.3f s\n", name, std::chrono::duration<double>(now__ - t_phase__).count()); \
        t_phase__ = now__;                                                                                        \
    } while (0)
#else
#define KKT_PHASE(name) ((void)0)
#endif

namespace asmb {

struct KktTerm {
    int a, b, k, t;  // target t -= W[a] * W[b] * invd[k];  t < nnzL: entry of L, else pivot t - nnzL (see kLastBit)
};
struct KktFwdItem {
    int pos, src, k, dst;  // v[dst] -= W[pos] * v[src] * invd[k]   (src, dst: node ids; k: permuted column of src)
};
struct KktBwdItem {
    int pos, src, dst, k;  // v[dst] -= invd[k] * W[pos] * v[src]   (k: permuted column of dst)
};
struct KktRange {
    int begin, end;
};
constexpr int kLastBit = 1 << 30;  // in KktTerm::t of the first term of a chunk: last update of this pivot -> invert it
constexpr int kSnMax = 16;         // widest supernode
constexpr int kSnSmall = 4;        // panels up to this width are factorised by one warp per task, wider ones by a block
constexpr int kPanelRows = 32;     // rows of a narrow panel one task (warp) solves
constexpr int kPanelRowsWide = 16; // rows of a wide panel one task (block) solves
struct KktPanel {                  // a supernode of 2..kSnMax columns c_0 < c_1 < ... (permuted numbering)
    int w, nr;                     // columns; rows below the diagonal block (= pattern of the last column)
    int off;                       // first of its w (w + 1) / 2 slots in the buffer of factorised diagonal blocks
    int col[kSnMax];
    int node[kSnMax];              // perm[col[i]]: where the right-hand side entry of column i lives
    int lp[kSnMax];                // Lp[c_i]: entry (c_j, c_i), j > i, is lp[i] + j-i-1; entry (row t below, c_i) is lp[i] + w-1-i + t
};
struct KktPanelTask {
    int panel, r0;                 // rows [r0, r0 + kPanelRows(Wide)) of the panel
};

// f(i) for every i in [0, n) on the host's cores, in dynamically claimed chunks.  Everything built with it writes to
// positions that are fixed beforehand, so the result does not depend on the number of threads (ASM_HOST_THREADS caps it)
template <class F>
inline void kkt_parallel_for(int n, int chunk, F f) {
    unsigned nt = std::thread::hardware_concurrency();
    if (const char *e = getenv("ASM_HOST_THREADS")) nt = (unsigned)atoi(e);
    nt = std::max(1u, std::min(nt, 16u));
    if (nt == 1 || n <= chunk) {
        for (int i = 0; i < n; ++i) f(i);
        return;
    }
    std::atomic<int> next(0);
    auto worker = [&]() {
        for (;;) {
            const int b = next.fetch_add(chunk);
            if (b >= n) break;
            const int e = std::min(n, b + chunk);
            for (int i = b; i < e; ++i) f(i);
        }
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) {
        try {
            th.emplace_back(worker);
        } catch (...) {   // no more threads to be had: the ones we have (at least this one) do the work
            break;
        }
    }
    worker();
    for (std::thread &x : th) x.join();
}

// widest supernode, the one parameter of the schedule: ASM_IPM_SUPERNODE, default kSnMax; 1 = no supernodes, one step
// per level of the elimination tree
inline int kkt_supernode_width() {
    const char *e = getenv("ASM_IPM_SUPERNODE");
    if (e) return std::max(1, std::min(atoi(e), kSnMax));
    return kSnMax;
}

struct KktSymbolic {
    int n = 0, m = 0, N = 0;
    int64_t nnzL = 0, nterms = 0;
    int n_levels = 0;
    std::vector<int> perm, inv;  // perm[k] = node eliminated k-th; inv[node] = k
    std::vector<int> Lp, Li;     // columns of L (permuted numbering), rows ascending
    std::vector<int> kmap;       // CSR entry of K -> entry of L
    std::vector<int> level;      // per permuted column
    // factorisation: terms grouped by step (= level of the source column).  Inside a step the chunks that consist of
    // a single term come first -- terms [fs_beg[l], fs_end[l]), one independent update each, which the kernel
    // software-pipelines four at a time -- followed by the multi-term chunks fmchunk[fmstep[l] .. fmstep[l+1]) =
    // (begin, end) ranges of terms with a common target, summed in ascending k
    std::vector<KktTerm> terms;
    std::vector<int> fs_beg, fs_end, fmstep;
    std::vector<KktRange> fmchunk;
    int64_t n_fchunks = 0, n_wchunks = 0;
    // distinct f64 operands a step has to read / targets it has to read and write, summed over the steps: the traffic a
    // batch whose working set exceeds L2 cannot avoid (nothing survives in cache from one level to the next)
    int64_t f_distinct_reads = 0, f_targets = 0, w_distinct_reads = 0, w_targets = 0, b_distinct_reads = 0, b_targets = 0;
    int longest_chunk = 0;
    // forward substitution, same layout
    std::vector<KktFwdItem> fwd;
    std::vector<int> ws_beg, ws_end, wmstep;
    std::vector<KktRange> wmchunk;
    // backward substitution: items of step l = entries whose row has level l (walked downwards); with supernodes a
    // column can have several rows on one step, hence the same singles / chunks layout
    std::vector<KktBwdItem> bwd;
    std::vector<int> bs_beg, bs_end, bmstep;
    std::vector<KktRange> bmchunk;
    // supernodes (empty when built with sn <= 1): panels sorted by step, pstep[l] .. pstep[l+1]; the row tasks of the
    // factorisation likewise in ptstep
    int sn_width = 1;
    std::vector<int> snid;         // per permuted column
    std::vector<KktPanel> panels;
    std::vector<int> pstep, ptstep;
    std::vector<int> ptwide, pwide;   // per step: how many of its tasks / panels are wider than kSnSmall (they come first)
    std::vector<KktPanelTask> ptasks;
    int64_t n_intra = 0;           // update terms that the panels absorb
    int64_t panel_slots = 0;       // size of the buffer of factorised diagonal blocks (entries per LP)

    // K: m x n CSR pattern (0-based).  Returns 0, or -1 when an index is out of range / the term count overflows.
    int build(int n_, int m_, const int *row_ptr, const int *col_idx, int sn) {
        sn_width = std::max(1, std::min(sn, kSnMax));
        n_intra = 0;
        n = n_;
        m = m_;
        N = n + m;
#ifdef KKT_PROFILE
        auto t_phase__ = std::chrono::steady_clock::now();
#endif
        std::vector<std::vector<int>> adj(N);
        for (int i = 0; i < m; ++i)
            for (int q = row_ptr[i]; q < row_ptr[i + 1]; ++q) {
                const int j = col_idx[q];
                if (j < 0 || j >= n) return -1;
                adj[j].push_back(n + i);
                adj[n + i].push_back(j);
            }
        for (auto &a : adj) {
            std::sort(a.begin(), a.end());
            a.erase(std::unique(a.begin(), a.end()), a.end());
        }
        // ---- minimum degree, explicit fill, ties by node id (deterministic)
        typedef std::pair<int, int> DN;
        std::priority_queue<DN, std::vector<DN>, std::greater<DN>> heap;
        std::vector<char> gone(N, 0);
        for (int v = 0; v < N; ++v) heap.push(DN((int)adj[v].size(), v));
        perm.assign(N, -1);
        inv.assign(N, -1);
        std::vector<std::vector<int>> colpat(N);
        std::vector<int> merged;
        for (int k = 0; k < N; ++k) {
            int v = -1;
            while (true) {
                const DN top = heap.top();
                heap.pop();
                if (!gone[top.second] && (int)adj[top.second].size() == top.first) {
                    v = top.second;
                    break;
                }
            }
            gone[v] = 1;
            perm[k] = v;
            inv[v] = k;
            std::vector<int> S;
            S.swap(adj[v]);
            for (int u : S) {
                const std::vector<int> &a = adj[u];
                merged.clear();
                merged.reserve(a.size() + S.size());
                size_t ia = 0, is = 0;
                while (ia < a.size() || is < S.size()) {
                    int x;
                    if (is >= S.size() || (ia < a.size() && a[ia] < S[is]))
                        x = a[ia++];
                    else if (ia >= a.size() || S[is] < a[ia])
                        x = S[is++];
                    else {
                        x = a[ia++];
                        ++is;
                    }
                    if (x != u && x != v) merged.push_back(x);
                }
                if (merged.size() != a.size()) heap.push(DN((int)merged.size(), u));
                adj[u].assign(merged.begin(), merged.end());
            }
            colpat[v].swap(S);
        }
        adj.clear();
        adj.shrink_to_fit();
        KKT_PHASE("minimum degree");
        // ---- pattern of L in the permuted numbering
        Lp.assign(N + 1, 0);
        for (int k = 0; k < N; ++k) Lp[k + 1] = Lp[k] + (int)colpat[perm[k]].size();
        nnzL = Lp[N];
        Li.resize(nnzL);
        for (int k = 0; k < N; ++k) {
            std::vector<int> &S = colpat[perm[k]];
            int *dst = Li.data() + Lp[k];
            for (size_t t = 0; t < S.size(); ++t) dst[t] = inv[S[t]];
            std::sort(dst, dst + S.size());
            std::vector<int>().swap(S);
        }
        colpat.clear();
        auto find_entry = [&](int col, int row) -> int {
            const int *b = Li.data() + Lp[col], *e = Li.data() + Lp[col + 1];
            const int *p = std::lower_bound(b, e, row);
            return (p != e && *p == row) ? (int)(p - Li.data()) : -1;
        };
        kmap.assign(row_ptr[m], -1);
        for (int i = 0; i < m; ++i)
            for (int q = row_ptr[i]; q < row_ptr[i + 1]; ++q) {
                const int a = inv[col_idx[q]], b = inv[n + i];
                kmap[q] = find_entry(std::min(a, b), std::max(a, b));
                if (kmap[q] < 0) return -1;
            }
        // ---- levels
        level.assign(N, 0);
        for (int k = 0; k < N; ++k)
            for (int p = Lp[k]; p < Lp[k + 1]; ++p) level[Li[p]] = std::max(level[Li[p]], level[k] + 1);
        snid.resize(N);
        for (int k = 0; k < N; ++k) snid[k] = k;
        panels.clear();
        if (sn_width > 1) supernodes();
        n_levels = 0;
        for (int k = 0; k < N; ++k) n_levels = std::max(n_levels, level[k] + 1);
        KKT_PHASE("pattern, levels, supernodes");
        if (panels.empty()) {
            pstep.assign(n_levels + 1, 0);
            ptstep.assign(n_levels + 1, 0);
            ptwide.assign(n_levels, 0);
            pwide.assign(n_levels, 0);
            ptasks.clear();
        }
        // ---- terms, target-major first (column k updates entry (r_a, r_b) and pivot r_b for every pair of its rows
        //      r_a >= r_b), then a stable counting sort by the level of k: (level, target, k) order
        const int64_t n_targets = nnzL + N;
        // rows of L: (column k, position of the entry) of row j, k ascending
        std::vector<int> rptr(N + 1, 0), rcol(nnzL), rpos(nnzL);
        {
            for (int64_t p = 0; p < nnzL; ++p) ++rptr[Li[p] + 1];
            for (int k = 0; k < N; ++k) rptr[k + 1] += rptr[k];
            std::vector<int> pos(rptr.begin(), rptr.end() - 1);
            for (int k = 0; k < N; ++k)
                for (int p = Lp[k]; p < Lp[k + 1]; ++p) {
                    rcol[pos[Li[p]]] = k;
                    rpos[pos[Li[p]]++] = p;
                }
        }
        {
            // The targets in column j (its entries and its pivot) get their terms from the columns k of row j: entry
            // (j, k) at position pb pairs with every entry (i, k) below it.  Sizes are known without searching (one
            // term per such pair), so every column writes its own slice of the target-major list, in parallel.
            std::vector<int64_t> eoff(N + 1, 0), poff(N + 1, 0);
            for (int j = 0; j < N; ++j) {
                int64_t ce = 0, cp = 0;
                for (int q = rptr[j]; q < rptr[j + 1]; ++q) {
                    const int k = rcol[q];
                    if (snid[j] == snid[k]) {   // target column in the supernode of k: the panel kernel's work
                        n_intra += Lp[k + 1] - rpos[q];
                        continue;
                    }
                    ce += Lp[k + 1] - rpos[q] - 1;
                    ++cp;
                }
                eoff[j + 1] = eoff[j] + ce;
                poff[j + 1] = poff[j] + cp;
            }
            nterms = eoff[N] + poff[N];
            if (nterms > 0x3fffffffLL || n_targets >= kLastBit) return -1;
            std::unique_ptr<KktTerm[]> tm_buf(new KktTerm[std::max<int64_t>(nterms, 1)]);   // no zero fill: every slot is written below
            KktTerm *const tm = tm_buf.get();
            const int64_t pbase = eoff[N];
            kkt_parallel_for(N, 64, [&](int jj) {
                const int j = N - 1 - jj;   // the heavy columns (root of the tree) first
                static thread_local std::vector<KktTerm> tmp;
                static thread_local std::vector<int> cnt;
                const int c0 = Lp[j], nc = Lp[j + 1] - Lp[j];
                tmp.clear();
                cnt.assign(nc + 1, 0);
                int64_t pp = pbase + poff[j];
                for (int q = rptr[j]; q < rptr[j + 1]; ++q) {
                    const int k = rcol[q], pb = rpos[q];
                    if (snid[j] == snid[k]) continue;
                    tm[pp++] = KktTerm{pb, pb, k, (int)(nnzL + j)};
                    int ptr = c0;
                    for (int pa = pb + 1; pa < Lp[k + 1]; ++pa) {
                        const int i = Li[pa];
                        while (Li[ptr] < i) ++ptr;   // (i, j) exists: fill of column k
                        tmp.push_back(KktTerm{pa, pb, k, ptr});
                        ++cnt[ptr - c0 + 1];
                    }
                }
                for (int t = 0; t < nc; ++t) cnt[t + 1] += cnt[t];
                KktTerm *out = tm + eoff[j];
                for (const KktTerm &u : tmp) out[cnt[u.t - c0]++] = u;   // stable: (target, k) order
            });
            // stable counting sort by the level of k with per-slice histograms: (level, target, k) order
            const int nsl = 64;
            std::vector<int64_t> hist((size_t)nsl * n_levels, 0);
            auto slice = [&](int t) { return nterms * t / nsl; };
            kkt_parallel_for(nsl, 1, [&](int t) {
                int64_t *h = hist.data() + (size_t)t * n_levels;
                for (int64_t q = slice(t); q < slice(t + 1); ++q) ++h[level[tm[q].k]];
            });
            int64_t run = 0;
            for (int l = 0; l < n_levels; ++l)
                for (int t = 0; t < nsl; ++t) {
                    const int64_t c = hist[(size_t)t * n_levels + l];
                    hist[(size_t)t * n_levels + l] = run;
                    run += c;
                }
            terms.resize(nterms);
            kkt_parallel_for(nsl, 1, [&](int t) {
                int64_t *h = hist.data() + (size_t)t * n_levels;
                for (int64_t q = slice(t); q < slice(t + 1); ++q) terms[h[level[tm[q].k]]++] = tm[q];
            });
        }
        KKT_PHASE("terms");
        n_fchunks = regroup(terms, [&](const KktTerm &u) { return level[u.k]; }, [](const KktTerm &u) { return u.t; },
                            fs_beg, fs_end, fmstep, fmchunk);
        KKT_PHASE("regroup terms");
        {   // the last chunk of every pivot inverts it
            std::vector<int> last(N, -1);
            for (size_t q = 0; q < terms.size(); ++q)
                if (terms[q].t >= nnzL) last[terms[q].t - nnzL] = (int)q;   // terms of a chunk are contiguous: its first
            for (int l = 0; l < n_levels; ++l) {                             // term carries the flag
                for (int q = fs_beg[l]; q < fs_end[l]; ++q)
                    if (terms[q].t >= nnzL && last[terms[q].t - nnzL] == q) terms[q].t |= kLastBit;
                for (int c = fmstep[l]; c < fmstep[l + 1]; ++c) {
                    const int t = terms[fmchunk[c].begin].t;
                    if (t >= nnzL && last[t - nnzL] >= fmchunk[c].begin && last[t - nnzL] < fmchunk[c].end)
                        terms[fmchunk[c].begin].t |= kLastBit;
                }
            }
        }
        // ---- forward substitution: row-major items (target i, sources ascending), then by level of the source
        {
            std::vector<KktFwdItem> rl(nnzL);
            for (int j = 0; j < N; ++j)
                for (int q = rptr[j]; q < rptr[j + 1]; ++q) rl[q] = KktFwdItem{rpos[q], perm[rcol[q]], rcol[q], perm[j]};
            std::vector<int64_t> lpos(n_levels + 1, 0);
            int64_t kept = 0;
            for (const KktFwdItem &u : rl)
                if (snid[inv[u.dst]] != snid[u.k]) ++lpos[level[u.k] + 1], ++kept;
            for (int l = 0; l < n_levels; ++l) lpos[l + 1] += lpos[l];
            fwd.resize(kept);
            for (const KktFwdItem &u : rl)
                if (snid[inv[u.dst]] != snid[u.k]) fwd[lpos[level[u.k]]++] = u;
        }
        n_wchunks = regroup(fwd, [&](const KktFwdItem &u) { return level[u.k]; }, [](const KktFwdItem &u) { return u.dst; },
                            ws_beg, ws_end, wmstep, wmchunk);
        // ---- backward substitution: entry (i, j) is applied when x_i is final, i.e. at the level of its row
        {   // items of one (step, column) are contiguous: k ascending, p ascending
            std::vector<int64_t> bstep(n_levels + 1, 0);
            for (int k = 0; k < N; ++k)
                for (int p = Lp[k]; p < Lp[k + 1]; ++p)
                    if (snid[Li[p]] != snid[k]) ++bstep[level[Li[p]] + 1];
            for (int l = 0; l < n_levels; ++l) bstep[l + 1] += bstep[l];
            bwd.resize(bstep[n_levels]);
            std::vector<int64_t> pos(bstep.begin(), bstep.end() - 1);
            for (int k = 0; k < N; ++k)
                for (int p = Lp[k]; p < Lp[k + 1]; ++p)
                    if (snid[Li[p]] != snid[k]) bwd[pos[level[Li[p]]]++] = KktBwdItem{p, perm[Li[p]], perm[k], k};
        }
        regroup(bwd, [&](const KktBwdItem &u) { return level[inv[u.src]]; }, [](const KktBwdItem &u) { return u.dst; },
                bs_beg, bs_end, bmstep, bmchunk);
        KKT_PHASE("substitution lists");
        {   // compulsory traffic per step (see f_distinct_reads)
            std::vector<int> stampW(nnzL + 1, -1), stampD(N, -1), stampV(N, -1), stampT(nnzL + N + 1, -1);
            size_t q = 0;
            for (int l = 0; l < n_levels; ++l)
                for (; q < terms.size() && level[terms[q].k] == l; ++q) {
                    const KktTerm &u = terms[q];
                    const int t = u.t & ~kLastBit;
                    if (stampW[u.a] != l) { stampW[u.a] = l; ++f_distinct_reads; }
                    if (stampW[u.b] != l) { stampW[u.b] = l; ++f_distinct_reads; }
                    if (stampD[u.k] != l) { stampD[u.k] = l; ++f_distinct_reads; }
                    if (stampT[t] != l) { stampT[t] = l; ++f_targets; }
                }
            std::fill(stampD.begin(), stampD.end(), -1);
            std::vector<int> stampDst(N, -1);
            q = 0;
            for (int l = 0; l < n_levels; ++l)
                for (; q < fwd.size() && level[fwd[q].k] == l; ++q) {
                    const KktFwdItem &u = fwd[q];
                    ++w_distinct_reads;                                   // W[pos]: every entry of L exactly once
                    if (stampV[u.src] != l) { stampV[u.src] = l; w_distinct_reads += 2; }   // v[src], 1/d[k]
                    if (stampDst[u.dst] != l) { stampDst[u.dst] = l; ++w_targets; }
                }
            std::fill(stampV.begin(), stampV.end(), -1);
            std::fill(stampDst.begin(), stampDst.end(), -1);
            q = 0;
            for (int l = 0; l < n_levels; ++l)
                for (; q < bwd.size() && level[inv[bwd[q].src]] == l; ++q) {
                    const KktBwdItem &u = bwd[q];
                    ++b_distinct_reads;
                    if (stampV[u.src] != l) { stampV[u.src] = l; ++b_distinct_reads; }
                    if (stampDst[u.dst] != l) { stampDst[u.dst] = l; b_distinct_reads += 1; ++b_targets; }   // 1/d[dst]
                }
            // panels: every entry of a panel is read and written once by the factorisation (the diagonal block once
            // more per row task) and read once by each substitution; the right-hand side entries are targets
            for (const KktPanel &P : panels) {
                const int64_t tri = (int64_t)P.w * (P.w - 1) / 2;
                const bool wide = P.w > kSnSmall;
                const int64_t tasks = wide ? (P.nr + kPanelRowsWide - 1) / kPanelRowsWide : std::max(1, (P.nr + kPanelRows - 1) / kPanelRows);
                f_targets += tri + P.w + (int64_t)P.nr * (P.w - 1);
                f_distinct_reads += (wide ? tasks * tri : (tasks - 1) * (tri + P.w)) + P.nr;
                w_distinct_reads += tri + P.w;
                w_targets += P.w;
                b_distinct_reads += tri + P.w;
                b_targets += P.w;
            }
        }
        KKT_PHASE("traffic statistics");
        return 0;
    }

    // Supernodes and their steps.  Column c and its parent p (the first row of c) are merged when the pattern of c is
    // {p} + pattern(p) -- equal counts suffice, pattern(c) \ {p} is always contained in pattern(p).  A supernode
    // starts when every update from outside to any of its columns has been applied: step(S) = 1 + max step over the
    // supernodes with an entry in a row of S.  Processing the supernodes by their LAST column is a topological
    // order (an outside updater of c_j lies, with its whole chain, strictly below c_j in the elimination tree).
    // Overwrites level[] with the step of the column's supernode.
    void supernodes() {
        auto cnt = [&](int c) { return Lp[c + 1] - Lp[c]; };
        std::fill(snid.begin(), snid.end(), -1);
        std::vector<std::vector<int>> mem;
        for (int c = 0; c < N; ++c) {
            if (snid[c] >= 0) continue;
            const int id = (int)mem.size();
            mem.emplace_back();
            int cur = c;
            snid[c] = id;
            mem[id].push_back(c);
            while ((int)mem[id].size() < sn_width && cnt(cur) > 0) {
                const int p = Li[Lp[cur]];
                if (cnt(p) + 1 != cnt(cur) || snid[p] >= 0) break;
                snid[p] = id;
                mem[id].push_back(p);
                cur = p;
            }
        }
        const int nsn = (int)mem.size();
        std::vector<int> ord(nsn), step(nsn, 0);
        for (int i = 0; i < nsn; ++i) ord[i] = i;
        std::sort(ord.begin(), ord.end(), [&](int a, int b) { return mem[a].back() < mem[b].back(); });
        for (int o = 0; o < nsn; ++o) {
            const int sid = ord[o];
            for (int c : mem[sid])
                for (int p = Lp[c]; p < Lp[c + 1]; ++p) {
                    const int r = snid[Li[p]];
                    if (r != sid) step[r] = std::max(step[r], step[sid] + 1);
                }
        }
        int nsteps = 0;
        for (int c = 0; c < N; ++c) {
            level[c] = step[snid[c]];
            nsteps = std::max(nsteps, level[c] + 1);
        }
        // panels of the supernodes with more than one column, by step
        pstep.assign(nsteps + 1, 0);
        ptstep.assign(nsteps + 1, 0);
        for (int sid = 0; sid < nsn; ++sid)
            if (mem[sid].size() > 1) ++pstep[step[sid] + 1];
        for (int l = 0; l < nsteps; ++l) pstep[l + 1] += pstep[l];
        panels.resize(pstep[nsteps]);
        std::vector<int> pos(pstep.begin(), pstep.end() - 1);
        for (int wide = 1; wide >= 0; --wide)   // the wide panels of a step first
            for (int sid = 0; sid < nsn; ++sid) {
                if (mem[sid].size() < 2 || ((int)mem[sid].size() > kSnSmall) != (wide == 1)) continue;
                KktPanel P = {};
                P.w = (int)mem[sid].size();
                P.nr = cnt(mem[sid].back());
                for (int i = 0; i < P.w; ++i) {
                    P.col[i] = mem[sid][i];
                    P.node[i] = perm[mem[sid][i]];
                    P.lp[i] = Lp[mem[sid][i]];
                }
                panels[pos[step[sid]]++] = P;
            }
        ptasks.clear();
        ptwide.assign(nsteps, 0);
        pwide.assign(nsteps, 0);
        panel_slots = 0;
        for (int l = 0; l < nsteps; ++l) {
            for (int q = pstep[l]; q < pstep[l + 1]; ++q) {
                panels[q].off = (int)panel_slots;
                panel_slots += panels[q].w * (panels[q].w + 1) / 2;
                if (panels[q].w > kSnSmall) ++pwide[l];
                // narrow panels: every task redoes the small diagonal block, the first one stores it (a panel without
                // rows still needs that); wide panels: the block is factorised by k_sn_diag, tasks are rows only
                const bool wide = panels[q].w > kSnSmall;
                const int rows = wide ? kPanelRowsWide : kPanelRows;
                for (int r0 = 0; r0 < std::max(panels[q].nr, wide ? 0 : 1); r0 += rows) {
                    ptasks.push_back(KktPanelTask{q, r0});
                    if (wide) ++ptwide[l];
                }
            }
            ptstep[l + 1] = (int)ptasks.size();
        }
    }

    // chunk = maximal run of items with the same (step, target).  Reorders the items of every step (singles first) and
    // fills the step tables; returns the number of chunks
    template <class T, class FL, class FT>
    int64_t regroup(std::vector<T> &items, FL lvl, FT tgt, std::vector<int> &sbeg, std::vector<int> &send,
                    std::vector<int> &mstep, std::vector<KktRange> &mchunk) {
        sbeg.assign(n_levels, 0);
        send.assign(n_levels, 0);
        mstep.assign(n_levels + 1, 0);
        mchunk.clear();
        // the items of a step stay in the step's range: the steps are independent of each other
        std::vector<size_t> lo(n_levels + 1, 0);
        {
            size_t q = 0;
            for (int l = 0; l < n_levels; ++l) {
                lo[l] = q;
                while (q < items.size() && lvl(items[q]) == l) ++q;
            }
            lo[n_levels] = q;
        }
        std::vector<std::vector<KktRange>> mc(n_levels);
        std::vector<int64_t> nch(n_levels, 0);
        std::vector<int> longest(n_levels, 0);
        kkt_parallel_for(n_levels, 1, [&](int l) {
            const size_t q0 = lo[l], q = lo[l + 1];
            static thread_local std::vector<T> in;   // the step's items in their old order; rewritten in place
            in.assign(items.begin() + q0, items.begin() + q);
            const size_t cnt = q - q0;
            size_t w = q0;
            // pass 1: singles
            for (size_t a = 0; a < cnt;) {
                size_t b = a + 1;
                while (b < cnt && tgt(in[b]) == tgt(in[a])) ++b;
                if (b - a == 1) items[w++] = in[a];
                a = b;
            }
            sbeg[l] = (int)q0;
            send[l] = (int)w;
            // pass 2: multi-item chunks
            for (size_t a = 0; a < cnt;) {
                size_t b = a + 1;
                while (b < cnt && tgt(in[b]) == tgt(in[a])) ++b;
                ++nch[l];
                if (b - a > 1) {
                    mc[l].push_back(KktRange{(int)w, (int)(w + (b - a))});
                    std::copy(in.begin() + a, in.begin() + b, items.begin() + w);
                    w += b - a;
                    longest[l] = std::max(longest[l], (int)(b - a));
                }
                a = b;
            }
        });
        int64_t n_chunks = 0;
        for (int l = 0; l < n_levels; ++l) {
            mchunk.insert(mchunk.end(), mc[l].begin(), mc[l].end());
            mstep[l + 1] = (int)mchunk.size();
            n_chunks += nch[l];
            longest_chunk = std::max(longest_chunk, longest[l]);
        }
        return n_chunks;
    }

    // ---- host reference of the device numerics (same lists, same order): used by the CPU self test ------------
    // W: nnzL values (in: assembled lower triangle, out: L D), diag: N assembled pivots (permuted; out: D),
    // invd: N out
    void factor_host(std::vector<double> &W, std::vector<double> &diag, std::vector<double> &invd) const {
        invd.resize(N);
        for (int j = 0; j < N; ++j) invd[j] = 1.0 / diag[j];
        auto apply = [&](int q0, int q1) {
            int t = terms[q0].t;
            const bool last = t & kLastBit;
            t &= ~kLastBit;
            double acc = 0.0;
            for (int q = q0; q < q1; ++q) acc += W[terms[q].a] * W[terms[q].b] * invd[terms[q].k];
            if (t >= nnzL) {
                diag[t - nnzL] -= acc;
                if (last) invd[t - nnzL] = 1.0 / diag[t - nnzL];
            } else {
                W[t] -= acc;
            }
        };
        for (int l = 0; l < n_levels; ++l) {
            for (int q = pstep[l]; q < pstep[l + 1]; ++q) {   // k_sn_factor: diagonal block (right-looking), then the rows
                const KktPanel &P = panels[q];
                const int w = P.w;
                auto S = [&](int j, int i) -> double & { return W[P.lp[i] + j - i - 1]; };
                for (int i = 0; i < w; ++i) {
                    const double iv = 1.0 / diag[P.col[i]];
                    invd[P.col[i]] = iv;
                    for (int k = i + 1; k < w; ++k) {
                        const double f = S(k, i) * iv;
                        diag[P.col[k]] -= S(k, i) * f;
                        for (int j = k + 1; j < w; ++j) S(j, k) -= S(j, i) * f;
                    }
                }
                for (int t = 0; t < P.nr; ++t) {
                    double y[kSnMax];
                    for (int i = 0; i < w; ++i) {
                        double &e = W[P.lp[i] + w - 1 - i + t];
                        double acc = e;
                        for (int k = 0; k < i; ++k) acc -= y[k] * S(i, k);
                        e = acc;
                        y[i] = acc * invd[P.col[i]];
                    }
                }
            }
            for (int q = fs_beg[l]; q < fs_end[l]; ++q) apply(q, q + 1);
            for (int c = fmstep[l]; c < fmstep[l + 1]; ++c) apply(fmchunk[c].begin, fmchunk[c].end);
        }
    }
    // v (indexed by node id): right-hand side in, solution out
    void solve_host(const std::vector<double> &W, const std::vector<double> &invd, std::vector<double> &v) const {
        auto apply = [&](int q0, int q1) {
            double acc = 0.0;
            for (int q = q0; q < q1; ++q) acc += W[fwd[q].pos] * v[fwd[q].src] * invd[fwd[q].k];
            v[fwd[q0].dst] -= acc;
        };
        auto applyb = [&](int q0, int q1) {
            double acc = 0.0;
            for (int q = q0; q < q1; ++q) acc += invd[bwd[q].k] * W[bwd[q].pos] * v[bwd[q].src];
            v[bwd[q0].dst] -= acc;
        };
        for (int l = 0; l < n_levels; ++l) {
            for (int q = pstep[l]; q < pstep[l + 1]; ++q) {   // k_sn_solve<true>
                const KktPanel &P = panels[q];
                for (int j = 1; j < P.w; ++j) {
                    double acc = v[perm[P.col[j]]];
                    for (int i = 0; i < j; ++i) acc -= W[P.lp[i] + j - i - 1] * invd[P.col[i]] * v[perm[P.col[i]]];
                    v[perm[P.col[j]]] = acc;
                }
            }
            for (int q = ws_beg[l]; q < ws_end[l]; ++q) apply(q, q + 1);
            for (int c = wmstep[l]; c < wmstep[l + 1]; ++c) apply(wmchunk[c].begin, wmchunk[c].end);
        }
        for (int k = 0; k < N; ++k) v[perm[k]] *= invd[k];
        for (int l = n_levels - 1; l >= 0; --l) {
            for (int q = pstep[l]; q < pstep[l + 1]; ++q) {   // k_sn_solve<false>
                const KktPanel &P = panels[q];
                for (int i = P.w - 2; i >= 0; --i) {
                    double acc = v[perm[P.col[i]]];
                    for (int j = i + 1; j < P.w; ++j) acc -= W[P.lp[i] + j - i - 1] * invd[P.col[i]] * v[perm[P.col[j]]];
                    v[perm[P.col[i]]] = acc;
                }
            }
            for (int q = bs_beg[l]; q < bs_end[l]; ++q) applyb(q, q + 1);
            for (int c = bmstep[l]; c < bmstep[l + 1]; ++c) applyb(bmchunk[c].begin, bmchunk[c].end);
        }
    }
};

}  // namespace asmb

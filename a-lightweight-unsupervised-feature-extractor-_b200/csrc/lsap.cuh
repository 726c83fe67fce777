// Rectangular linear-sum assignment on the GPU: shortest augmenting paths with float64 duals,
// one problem per group of cooperating threads (device functions).
//
// Follows the algorithm behind scipy.optimize.linear_sum_assignment, which the reference calls
// at model/utils/costTool/hung.py:28 (Crouse 2016, no initialisation phase), step for step:
// the same descending initial column list, the same swap-removal of scanned columns, the same
// tie rule (first minimum in list order unless a later minimum is an unassigned column) and the
// same expression ((minv + c) - u[i]) - v[j] for the reduced cost, so the result -- including
// which optimum is returned under ties -- is the one scipy returns.  What is parallel is the
// scan of the remaining columns inside one Dijkstra step: each thread owns list positions
// tid, tid+nt, ...; the (value, tie rule) argmin is an associative reduction over them.
#pragma once
#include "common.cuh"

namespace b200 {
namespace lsap {

constexpr int kMaxThreads = 256;
// Widest problem of the single-warp solver; wider ones use the multi-warp register solver.  One warp wins up to 128
// columns and loses from 256 on (the 64 / 128 / 256 / 512-column timings in the comment of solve_block).
constexpr int kWarpSolverMaxCols = 128;

struct Work {              // all arrays in shared memory, sized for R rows / Cc columns
    double* u;             // [R]
    double* v;             // [Cc]
    double* dist;          // [Cc]
    int* pred;             // [Cc]
    int* c4r;              // [R]
    int* r4c;              // [Cc]
    int* todo;             // [Cc]
    int* seen_rows;        // [R]   rows scanned in the current search (SR)
    int* seen_cols;        // [Cc]  columns scanned in the current search (SC)
    double* red_val;       // [kMaxThreads / 32] cross-warp reduction scratch
    int* red_it;           // [kMaxThreads / 32]
    int* red_un;           // [kMaxThreads / 32]
    int* flag;             // [1]
};

__host__ __device__ inline size_t work_bytes(int R, int Cc) {
    const size_t d = (size_t)R + 2 * (size_t)Cc + kMaxThreads / 32;
    const size_t i = 2 * (size_t)R + 4 * (size_t)Cc + 2 * (kMaxThreads / 32) + 2;
    return d * 8 + ((i * 4 + 7) & ~(size_t)7);
}

__device__ __forceinline__ Work carve(unsigned char* base, int R, int Cc) {
    Work w;
    double* d = reinterpret_cast<double*>(base);
    w.u = d; d += R;
    w.v = d; d += Cc;
    w.dist = d; d += Cc;
    w.red_val = d; d += kMaxThreads / 32;
    int* p = reinterpret_cast<int*>(d);
    w.pred = p; p += Cc;
    w.c4r = p; p += R;
    w.r4c = p; p += Cc;
    w.todo = p; p += Cc;
    w.seen_rows = p; p += R;
    w.seen_cols = p; p += Cc;
    w.red_it = p; p += kMaxThreads / 32;
    w.red_un = p; p += kMaxThreads / 32;
    w.flag = p;
    return w;
}

// Barrier among the `nt` cooperating threads (named barrier 1 when they span several warps).
__device__ __forceinline__ void group_sync(int nt) {
    if (nt <= 32) __syncwarp();
    else asm volatile("bar.sync 1, %0;" ::"r"(nt) : "memory");
}

struct Cand {
    double val;
    int it;      // position in the todo list
    int un;      // 1 if that column is unassigned
};

// scipy's selection rule as an associative combine.
__device__ __forceinline__ Cand better(const Cand& a, const Cand& b) {
    if (a.it < 0) return b;
    if (b.it < 0) return a;
    if (a.val < b.val) return a;
    if (b.val < a.val) return b;
    if (a.un != b.un) return a.un ? a : b;
    if (a.un) return a.it > b.it ? a : b;      // last unassigned minimum in list order
    return a.it < b.it ? a : b;                // else the first minimum
}

__device__ __forceinline__ Cand warp_best(Cand c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Cand d;
        d.val = __shfl_xor_sync(0xffffffffu, c.val, o);
        d.it = __shfl_xor_sync(0xffffffffu, c.it, o);
        d.un = __shfl_xor_sync(0xffffffffu, c.un, o);
        c = better(c, d);
    }
    return c;
}

// Solves the R x Cc problem (R <= Cc) whose row i is cost[i * ld + 0..Cc).  `tid` in [0, nt),
// nt a multiple of 32 (<= kMaxThreads); all nt threads must call.  On return w.c4r / w.r4c hold
// the assignment.  Returns B200_OK, B200_ENUMERIC or B200_EINFEASIBLE (same on every thread).
__device__ inline int solve(const float* cost, int R, int Cc, int ld, const Work& w, int tid, int nt,
                         bool checked = false) {
    const double kInf = __longlong_as_double(0x7ff0000000000000LL);
    // NaN / -inf check (scipy: "matrix contains invalid numeric entries").
    if (tid == 0) *w.flag = 0;
    group_sync(nt);
    int bad = 0;
    if (!checked)
        for (int i = 0; i < R; ++i)
            for (int j = tid; j < Cc; j += nt) {
                const float c = cost[(size_t)i * ld + j];
                if (c != c || c == -__int_as_float(0x7f800000)) bad = 1;
            }
    if (bad) *w.flag = 1;
    for (int i = tid; i < R; i += nt) { w.u[i] = 0.0; w.c4r[i] = -1; }
    for (int j = tid; j < Cc; j += nt) { w.v[j] = 0.0; w.r4c[j] = -1; w.pred[j] = -1; }
    group_sync(nt);
    if (*w.flag) return B200_ENUMERIC;

    for (int cur = 0; cur < R; ++cur) {
        for (int t = tid; t < Cc; t += nt) {
            w.todo[t] = Cc - 1 - t;
            w.dist[t] = kInf;
        }
        group_sync(nt);
        int i = cur, n_todo = Cc, n_sr = 0, n_sc = 0, sink = -1;
        double minv = 0.0;
        while (sink < 0) {
            if (tid == 0) w.seen_rows[n_sr] = i;
            ++n_sr;
            const double ui = w.u[i];
            const float* crow = cost + (size_t)i * ld;
            Cand best;
            best.val = kInf; best.it = -1; best.un = 0;
            for (int it = tid; it < n_todo; it += nt) {
                const int j = w.todo[it];
                const double r = ((minv + (double)crow[j]) - ui) - w.v[j];
                double d = w.dist[j];
                if (r < d) {
                    d = r;
                    w.dist[j] = r;
                    w.pred[j] = i;
                }
                const int un = w.r4c[j] < 0;
                if (best.it < 0 || d < best.val || (d == best.val && un)) {
                    best.val = d; best.it = it; best.un = un;
                }
            }
            best = warp_best(best);
            if (nt > 32) {
                const int wid = tid >> 5;
                if ((tid & 31) == 0) { w.red_val[wid] = best.val; w.red_it[wid] = best.it; w.red_un[wid] = best.un; }
                group_sync(nt);
                Cand c;
                c.val = kInf; c.it = -1; c.un = 0;
                if ((tid & 31) < (nt >> 5)) {
                    c.val = w.red_val[tid & 31]; c.it = w.red_it[tid & 31]; c.un = w.red_un[tid & 31];
                }
                best = warp_best(c);
            }
            minv = best.val;
            if (best.it < 0 || minv == kInf) return B200_EINFEASIBLE;      // uniform across the group
            const int j = w.todo[best.it];
            const int rj = w.r4c[j];
            group_sync(nt);                    // everyone has read todo[best.it] / red_* before they change
            if (tid == 0) {
                w.seen_cols[n_sc] = j;
                w.todo[best.it] = w.todo[n_todo - 1];
            }
            ++n_sc;
            --n_todo;
            if (rj < 0) sink = j; else i = rj;
            group_sync(nt);
        }
        // dual update (scipy: u[cur] += minv; u[i] += minv - dist[c4r[i]]; v[j] -= minv - dist[j])
        for (int s = tid; s < n_sr; s += nt) {
            const int r = w.seen_rows[s];
            if (r == cur) w.u[r] += minv;
            else w.u[r] += minv - w.dist[w.c4r[r]];
        }
        for (int s = tid; s < n_sc; s += nt) {
            const int j = w.seen_cols[s];
            w.v[j] -= minv - w.dist[j];
        }
        group_sync(nt);
        if (tid == 0) {                       // augment along the predecessor chain
            int j = sink;
            for (;;) {
                const int r = w.pred[j];
                w.r4c[j] = r;
                const int prev = w.c4r[r];
                w.c4r[r] = j;
                j = prev;
                if (r == cur) break;
            }
        }
        group_sync(nt);
    }
    return B200_OK;
}


// ---- rows whose search is known in advance ---------------------------------------------------------------
// The search for row `cur` starts with minv = 0 and u[cur] = 0, so its first Dijkstra step sees the reduced
// costs c[cur][j] - v[j].  Column duals only ever decrease (v[j] -= minv - dist[j] with minv >= dist[j]), and
// only for columns scanned by a search of length > 1.  Hence, if the row's smallest entry is attained by ONE
// column fj, that column is still unassigned and v[fj] == 0 (and no v[j] > 0 has ever appeared, which rounding
// could produce in principle), every other reduced cost is strictly larger, the step selects fj whatever the
// tie rule says, fj is the sink, and the search degenerates to: u[cur] = c[cur][fj], col4row[cur] = fj,
// row4col[fj] = cur, v untouched (minv - dist[fj] == 0).  solve_block computes (fj, unique?) for all rows in
// parallel while it validates the matrix; the solvers take the shortcut when its premises hold and run the
// full search otherwise, so the result is still scipy's, step for step.  In a tracker's steady state (one
// clearly best detection per track) almost every row takes it.
__device__ __forceinline__ double first_step_dual(float c) { return 0.0 + (((0.0 + (double)c) - 0.0) - 0.0); }

// Applies the rule to a run of consecutive rows, 32 at a time (one warp; lane l looks at row cur + l): a lane's
// row qualifies if its column is free, unmoved, and not claimed by an earlier lane of the batch (then the rows
// before it only take other free columns and leave every v alone, so applying them together equals applying
// them in order).  The batch is applied up to the first row that does not qualify; returns that row (or R).
// r4c_s / v_s / u_s / c4r_s are the shared-memory copies of row4col, v, u, col4row.
__device__ inline int known_first_step_run(int cur, int R, const int* first_col, const float* first_val, int* r4c_s,
                                           const double* v_s, double* u_s, int* c4r_s, int lane) {
    const unsigned kFull = 0xffffffffu;
    while (cur < R) {
        const int row = cur + lane;
        const int fj = row < R ? first_col[row] : -1;
        bool ok = fj >= 0;
        if (ok) ok = r4c_s[fj] < 0 && v_s[fj] == 0.0;
        const unsigned same = __match_any_sync(kFull, fj);
        ok = ok && (__ffs(same) - 1 == lane);
        const unsigned bad = ~__ballot_sync(kFull, ok);
        const int lead = bad ? __ffs(bad) - 1 : 32;
        if (lane < lead) {
            r4c_s[fj] = row;
            c4r_s[row] = fj;
            u_s[row] = first_step_dual(first_val[row]);
        }
        __syncwarp();
        cur += lead;
        if (lead < 32) break;
    }
    return cur < R ? cur : R;
}

// ---- single-warp solver: all per-column state in registers -------------------------------------
// Same algorithm and tie rule as solve(), for Cc <= 32 * CPL columns.  Lane l owns columns
// l, l+32, ...; for each it keeps dist, v, pred, r4c and the column's POSITION in scipy's
// "remaining" list (-1 once scanned), so the swap-removal of a scanned column is a register update
// (the column sitting at the last position moves to the freed position) and no list lives in
// memory.  The argmin of a Dijkstra step is three warp-wide integer min reductions (redux.sync):
// the distance mapped to an order-preserving 64-bit key (high word, then low word), then -- only
// when several lanes tie -- a key encoding scipy's tie rule.  u and col4row live in shared memory.
// No block barriers: the calling warp runs alone.  The caller has rejected NaN / -inf entries.
// On return c4r_s[R] / r4c_s[Cc] (shared memory) hold the assignment.
__device__ __forceinline__ unsigned long long dist_key(double d) {
    const long long b = __double_as_longlong(d + 0.0);          // +0.0 folds -0.0 into +0.0
    return (unsigned long long)(b ^ ((b >> 63) | (long long)0x8000000000000000LL));
}
__device__ __forceinline__ double key_dist(unsigned long long k) {
    const long long b = (k >> 63) ? (long long)(k ^ 0x8000000000000000ULL) : (long long)~k;
    return __longlong_as_double(b);
}
// scipy's tie rule among equal distances as a min-key: an unassigned column beats an assigned one;
// among unassigned the LAST list position wins, among assigned the FIRST.
__device__ __forceinline__ unsigned tie_key(int it, bool un) { return un ? (0xFFFFu - (unsigned)it) : (0x10000u | (unsigned)it); }

template <int CPL>
__device__ inline int solve_warp(const float* cost, int R, int Cc, int ld, double* u_s, int* c4r_s, int* r4c_s,
                                 double* v_s, const int* first_col, const float* first_val) {
    const unsigned kFull = 0xffffffffu;
    const double kInf = __longlong_as_double(0x7ff0000000000000LL);
    const int lane = threadIdx.x & 31;
    double v[CPL], dist[CPL];
    int pred[CPL], r4c[CPL], pos[CPL];
#pragma unroll
    for (int q = 0; q < CPL; ++q) { v[q] = 0.0; r4c[q] = -1; pred[q] = -1; }
    for (int i = lane; i < R; i += 32) { u_s[i] = 0.0; c4r_s[i] = -1; }
    for (int j = lane; j < Cc; j += 32) { r4c_s[j] = -1; v_s[j] = 0.0; }
    __syncwarp();
    bool v_positive = false;                             // some v[j] > 0 appeared: no more shortcuts
    for (int cur = 0; cur < R; ++cur) {
        if (!v_positive) {                               // run of rows whose first step is known (see above)
            cur = known_first_step_run(cur, R, first_col, first_val, r4c_s, v_s, u_s, c4r_s, lane);
            if (cur >= R) break;
#pragma unroll
            for (int q = 0; q < CPL; ++q)
                if (lane + 32 * q < Cc) r4c[q] = r4c_s[lane + 32 * q];
        }
#pragma unroll
        for (int q = 0; q < CPL; ++q) {
            const int j = lane + 32 * q;
            pos[q] = j < Cc ? Cc - 1 - j : -1;          // remaining[it] = Cc - 1 - it
            dist[q] = kInf;
        }
        unsigned scanned = 0;                            // bit q: own column q scanned in this search
        int i = cur, n_todo = Cc, sink = -1;
        double minv = 0.0;
        while (sink < 0) {
            const double ui = u_s[i];
            const float* crow = cost + (size_t)i * ld;
            unsigned long long bk = ~0ull;
            unsigned bt = 0xffffffffu;
            int bq = 0;
#pragma unroll
            for (int q = 0; q < CPL; ++q) {
                if (pos[q] >= 0) {
                    const double r = ((minv + (double)crow[lane + 32 * q]) - ui) - v[q];
                    if (r < dist[q]) { dist[q] = r; pred[q] = i; }
                    const unsigned long long k = dist_key(dist[q]);
                    const unsigned t = tie_key(pos[q], r4c[q] < 0);
                    if (k < bk || (k == bk && t < bt)) { bk = k; bt = t; bq = q; }
                }
            }
            const unsigned hi = (unsigned)(bk >> 32), lo = (unsigned)bk;
            const unsigned mh = __reduce_min_sync(kFull, hi);
            const unsigned ml = __reduce_min_sync(kFull, hi == mh ? lo : 0xffffffffu);
            bool cand = hi == mh && lo == ml && bt != 0xffffffffu;
            unsigned who = __ballot_sync(kFull, cand);
            if (__popc(who) > 1) {
                const unsigned mt = __reduce_min_sync(kFull, cand ? bt : 0xffffffffu);
                cand = cand && bt == mt;
                who = __ballot_sync(kFull, cand);
            }
            minv = key_dist(((unsigned long long)mh << 32) | ml);
            if (who == 0 || minv == kInf) return B200_EINFEASIBLE;
            const int wl = __ffs(who) - 1;
            int packed = 0, rj = 0;
            if (lane == wl) {
#pragma unroll
                for (int q = 0; q < CPL; ++q)
                    if (q == bq) { rj = r4c[q]; packed = (q << 16) | pos[q]; pos[q] = -1; scanned |= 1u << q; }
            }
            packed = __shfl_sync(kFull, packed, wl);
            rj = __shfl_sync(kFull, rj, wl);
            const int j = wl + 32 * (packed >> 16), freed = packed & 0xffff;
            --n_todo;                                    // swap-removal: the last list entry fills the gap
#pragma unroll
            for (int q = 0; q < CPL; ++q)
                if (pos[q] == n_todo) pos[q] = freed;
            if (rj < 0) sink = j; else i = rj;
        }
        // dual update: u[cur] += minv; for every scanned column j with a row: u[r4c[j]] += minv - dist[j];
        // v[j] -= minv - dist[j]  (the sink column has dist == minv, so it does not move)
        if (lane == 0) u_s[cur] += minv;
        bool vp = false;
#pragma unroll
        for (int q = 0; q < CPL; ++q)
            if (scanned & (1u << q)) {
                const double delta = minv - dist[q];
                if (r4c[q] >= 0) u_s[r4c[q]] += delta;
                v[q] -= delta;
                v_s[lane + 32 * q] = v[q];
                vp = vp || v[q] > 0.0;
            }
        v_positive = v_positive || __any_sync(kFull, vp);
        // augment along the predecessor chain; only lane 0 touches col4row
        int j = sink;
        for (;;) {
            int pi = 0;
#pragma unroll
            for (int q = 0; q < CPL; ++q)
                if (q == (j >> 5)) pi = pred[q];
            pi = __shfl_sync(kFull, pi, j & 31);
            if (lane == (j & 31)) {
#pragma unroll
                for (int q = 0; q < CPL; ++q)
                    if (q == (j >> 5)) r4c[q] = pi;
                r4c_s[j] = pi;
            }
            int prev = 0;
            if (lane == 0) { prev = c4r_s[pi]; c4r_s[pi] = j; }
            j = __shfl_sync(kFull, prev, 0);
            if (pi == cur) break;
        }
        __syncwarp();                                    // u_s / v_s / r4c_s updates visible before the next search
    }
    __syncwarp();
    return B200_OK;
}

// ---- multi-warp register solver: wide problems ---------------------------------------------------------
// The same search with the columns spread over nt = 32 * W threads (W <= 8), CPL columns each, all
// per-column state but the predecessor in registers.  A Dijkstra step is: local best -> warp redux (as in
// solve_warp) -> the W per-warp candidates go to a double-buffered shared-memory slot -> ONE named barrier ->
// every thread combines the W candidates with the same (distance, tie-key) order and applies the removal to
// its own registers.  The augmentation walks pred / col4row / row4col in shared memory on thread 0 while the
// other threads apply the dual update; one more barrier ends the search.  Exactness argument as above: the
// combine is the associative (min distance, then scipy's tie rule) order.
template <int CPL>
__device__ inline int solve_regs(const float* cost, int R, int Cc, int ld, const Work& w, int tid, int nt) {
    __shared__ __align__(16) unsigned slot[2][kMaxThreads / 32][8];
    const unsigned kFull = 0xffffffffu;
    const double kInf = __longlong_as_double(0x7ff0000000000000LL);
    const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
    double v[CPL], dist[CPL];
    int r4c[CPL], pos[CPL];
#pragma unroll
    for (int q = 0; q < CPL; ++q) { v[q] = 0.0; r4c[q] = -1; }
    const int* first_col = w.seen_rows;                   // filled by solve_block
    const float* first_val = reinterpret_cast<const float*>(w.dist);
    for (int i = tid; i < R; i += nt) { w.u[i] = 0.0; w.c4r[i] = -1; }
    for (int j = tid; j < Cc; j += nt) { w.r4c[j] = -1; w.pred[j] = -1; w.v[j] = 0.0; }
    if (tid == 0) w.red_un[0] = 0;                        // "some v[j] > 0 appeared"
    group_sync(nt);
    int par = 0;
    for (int cur = 0;; ++cur) {
        if (wid == 0) {                                   // run of rows with a known first step (see above)
            int c = cur;
            if (!w.red_un[0]) c = known_first_step_run(cur, R, first_col, first_val, w.r4c, w.v, w.u, w.c4r, lane);
            if (lane == 0) *w.flag = c;
        }
        group_sync(nt);
        cur = *w.flag;
        if (cur >= R) break;
#pragma unroll
        for (int q = 0; q < CPL; ++q) {
            const int j = tid + nt * q;
            pos[q] = j < Cc ? Cc - 1 - j : -1;
            dist[q] = kInf;
            if (j < Cc) r4c[q] = w.r4c[j];
        }
        if (cur + 1 < R && tid * 32 < Cc)                // the matrix may sit in L2: pull the next first row closer
            asm volatile("prefetch.L1 [%0];" ::"l"(cost + (size_t)(cur + 1) * ld + tid * 32));
        unsigned scanned = 0;
        int i = cur, n_todo = Cc, sink = -1;
        double minv = 0.0;
        while (sink < 0) {
            const double ui = w.u[i];
            const float* crow = cost + (size_t)i * ld;
            unsigned long long bk = ~0ull;
            unsigned bt = 0xffffffffu;
            int bq = 0;
#pragma unroll
            for (int q = 0; q < CPL; ++q) {
                if (pos[q] >= 0) {
                    const int j = tid + nt * q;
                    const double r = ((minv + (double)crow[j]) - ui) - v[q];
                    if (r < dist[q]) { dist[q] = r; w.pred[j] = i; }
                    const unsigned long long k = dist_key(dist[q]);
                    const unsigned t = tie_key(pos[q], r4c[q] < 0);
                    if (k < bk || (k == bk && t < bt)) { bk = k; bt = t; bq = q; }
                }
            }
            const unsigned hi = (unsigned)(bk >> 32), lo = (unsigned)bk;
            const unsigned mh = __reduce_min_sync(kFull, hi);
            const unsigned ml = __reduce_min_sync(kFull, hi == mh ? lo : 0xffffffffu);
            bool cand = hi == mh && lo == ml && bt != 0xffffffffu;
            unsigned who = __ballot_sync(kFull, cand);
            if (__popc(who) > 1) {
                const unsigned mt = __reduce_min_sync(kFull, cand ? bt : 0xffffffffu);
                cand = cand && bt == mt;
                who = __ballot_sync(kFull, cand);
            }
            if (lane == (who ? __ffs(who) - 1 : 0)) {      // this warp's candidate (or "none")
                int pj = 0, pp = 0, pr = 0;
#pragma unroll
                for (int q = 0; q < CPL; ++q)
                    if (q == bq) { pj = tid + nt * q; pp = pos[q]; pr = r4c[q]; }
                uint4* sl = reinterpret_cast<uint4*>(slot[par][wid]);
                sl[0] = make_uint4(who ? mh : 0xffffffffu, who ? ml : 0xffffffffu, who ? bt : 0xffffffffu, (unsigned)pj);
                sl[1] = make_uint4((unsigned)pp, (unsigned)pr, 0u, 0u);
            }
            group_sync(nt);
            unsigned gh = 0xffffffffu, gl = 0xffffffffu, gt = 0xffffffffu;
            int gw = 0, j = 0;
            for (int ww = 0; ww < nw; ++ww) {
                const uint4 c = reinterpret_cast<const uint4*>(slot[par][ww])[0];
                if (c.x < gh || (c.x == gh && (c.y < gl || (c.y == gl && c.z < gt)))) {
                    gh = c.x; gl = c.y; gt = c.z; j = (int)c.w; gw = ww;
                }
            }
            minv = key_dist(((unsigned long long)gh << 32) | gl);
            if (gt == 0xffffffffu || minv == kInf) return B200_EINFEASIBLE;      // uniform across the group
            const uint4 c1 = reinterpret_cast<const uint4*>(slot[par][gw])[1];
            const int freed = (int)c1.x, rj = (int)c1.y;
            par ^= 1;
            --n_todo;
#pragma unroll
            for (int q = 0; q < CPL; ++q) {
                if (tid + nt * q == j) { pos[q] = -1; scanned |= 1u << q; }
                else if (pos[q] == n_todo) pos[q] = freed;
            }
            if (rj < 0) sink = j; else i = rj;
        }
        if (tid == 0) {                                   // augment along the predecessor chain
            w.u[cur] += minv;
            int j = sink;
            for (;;) {
                const int r = w.pred[j];
                w.r4c[j] = r;
                const int prev = w.c4r[r];
                w.c4r[r] = j;
                j = prev;
                if (r == cur) break;
            }
        }
#pragma unroll
        for (int q = 0; q < CPL; ++q)
            if (scanned & (1u << q)) {
                const double delta = minv - dist[q];
                if (r4c[q] >= 0) w.u[r4c[q]] += delta;
                v[q] -= delta;
                w.v[tid + nt * q] = v[q];
                if (v[q] > 0.0) w.red_un[0] = 1;
            }
        group_sync(nt);
    }
    return B200_OK;
}

// One pass over the matrix for solve_block: NaN / -inf check, optional copy to shared memory, and for every row
// the column of its unique minimum (or -1).  A warp takes RB rows at a time and issues all their loads (LPR per
// lane and row, 16 in flight) before touching any: the pass is a few global round trips per warp instead of
// one per row.  NaN is detected through the row sum (a NaN makes it NaN; +inf with -inf does too, and -inf is
// invalid anyway), -inf through the minimum.  Returns 1 on an invalid entry (this thread's view).
template <int LPR>
__device__ __forceinline__ int row_minima_pass(const float* cost, int R, int Cc, int ld, float* stage_or_null,
                                               int* first_col, float* first_val) {
    constexpr int RB = LPR >= 16 ? 1 : 16 / LPR;
    const unsigned kFull = 0xffffffffu;
    const float kPosInf = __int_as_float(0x7f800000);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int bad = 0;
    for (int i0 = wid * RB; i0 < R; i0 += nw * RB) {
        float c[RB][LPR];
#pragma unroll
        for (int rb = 0; rb < RB; ++rb)
#pragma unroll
            for (int k = 0; k < LPR; ++k) {
                const int i = i0 + rb, j = lane + 32 * k;
                c[rb][k] = (i < R && j < Cc) ? cost[(size_t)i * ld + j] : kPosInf;
            }
#pragma unroll
        for (int rb = 0; rb < RB; ++rb) {
            const int i = i0 + rb;
            if (i >= R) break;                                    // uniform across the warp
            float m = kPosInf, sum = 0.0f;
#pragma unroll
            for (int k = 0; k < LPR; ++k) {
                m = fminf(m, c[rb][k]);                           // fminf ignores NaN; the sum catches it
                sum += c[rb][k];
                if (stage_or_null && lane + 32 * k < Cc) stage_or_null[i * Cc + lane + 32 * k] = c[rb][k];
            }
            if (sum != sum || m == -kPosInf) bad = 1;
            const unsigned bits = (unsigned)__float_as_int(m + 0.0f);                      // -0.0 ties with +0.0
            const unsigned key = bits ^ ((unsigned)((int)bits >> 31) | 0x80000000u);      // order-preserving
            const unsigned kmin = __reduce_min_sync(kFull, key);
            const float wm = __int_as_float((int)(kmin ^ ((kmin >> 31) ? 0x80000000u : 0xffffffffu)));
            int cnt = 0, kk = 0;
#pragma unroll
            for (int k = 0; k < LPR; ++k)
                if (c[rb][k] == wm) { ++cnt; kk = k; }
            const int total = __reduce_add_sync(kFull, cnt);
            if (total == 1 && wm < kPosInf) {
                if (cnt == 1) {
                    float val = 0.0f;
#pragma unroll
                    for (int k = 0; k < LPR; ++k)
                        if (k == kk) val = c[rb][k];
                    first_col[i] = lane + 32 * kk;
                    first_val[i] = val;
                }
            } else if (lane == 0) {
                first_col[i] = -1;
            }
        }
    }
    return bad;
}

// Block-level driver shared by the operator kernel and the tracker: validates the matrix, optionally
// stages it in shared memory and finds every row's unique minimum (all warps, a row each), then runs the
// single-warp solver (Cc <= 128), the multi-warp register solver (up to 4 columns per thread) or, beyond
// that, the shared-memory one.  Measured on B200 (association step, one stream): 64 columns 135 us (warp) vs
// 149 us (multi-warp); 128: 213 vs 220; 256: 752 vs 392; 512: 1 387 (shared-memory solver) vs 897.  Every thread of the CTA must call; the
// status is returned on every thread and w.c4r / w.r4c hold the assignment.
// pre_col / pre_val (optional, R entries in global memory): the producer of the matrix already knows every
// row's unique minimum (column, or -1) and has checked the row (-2 = NaN / -inf): when the matrix is not to be
// staged, the pass over it is skipped altogether.
__device__ __noinline__ inline int solve_block(const float* cost, int R, int Cc, int ld, const Work& w, float* stage_or_null,
                                  const int* pre_col = nullptr, const float* pre_val = nullptr) {
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31;
    int bad = 0;
    const float kNegInf = -__int_as_float(0x7f800000);
    int* first_col = w.seen_rows;                         // [R] column of the row's unique minimum, or -1
    float* first_val = reinterpret_cast<float*>(w.dist);  // [R] that minimum
    const int lpr = (pre_col && !stage_or_null) ? 0 : (Cc + 31) / 32;
    if (lpr == 0) {
        for (int i = tid; i < R; i += nthr) {
            const int fc = pre_col[i];
            if (fc == -2) bad = 1;
            first_col[i] = fc;
            first_val[i] = pre_val[i];
        }
    } else
    bad = lpr <= 1    ? row_minima_pass<1>(cost, R, Cc, ld, stage_or_null, first_col, first_val)
          : lpr <= 2  ? row_minima_pass<2>(cost, R, Cc, ld, stage_or_null, first_col, first_val)
          : lpr <= 4  ? row_minima_pass<4>(cost, R, Cc, ld, stage_or_null, first_col, first_val)
          : lpr <= 8  ? row_minima_pass<8>(cost, R, Cc, ld, stage_or_null, first_col, first_val)
          : lpr <= 16 ? row_minima_pass<16>(cost, R, Cc, ld, stage_or_null, first_col, first_val)
                      : -1;
    if (bad < 0) {                                        // more than 512 columns: plain loop, a row per warp
        bad = 0;
        for (int i = tid >> 5; i < R; i += nthr >> 5) {
            const float* row = cost + (size_t)i * ld;
            float m = __int_as_float(0x7f800000);
            int mj = -1, cnt = 0;
#pragma unroll 4
            for (int j = lane; j < Cc; j += 32) {
                const float c = row[j];
                if (c != c || c == kNegInf) bad = 1;
                if (stage_or_null) stage_or_null[i * Cc + j] = c;
                if (c < m) { m = c; mj = j; cnt = 1; }
                else if (c == m) ++cnt;
            }
            const unsigned bits = (unsigned)__float_as_int(m + 0.0f);                      // -0.0 ties with +0.0
            const unsigned key = bits ^ ((unsigned)((int)bits >> 31) | 0x80000000u);      // order-preserving
            const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
            const unsigned eq = __ballot_sync(0xffffffffu, key == kmin && mj >= 0);
            if (eq && lane == __ffs(eq) - 1) {
                const bool unique = __popc(eq) == 1 && cnt == 1 && m < __int_as_float(0x7f800000);
                first_col[i] = unique ? mj : -1;
                first_val[i] = m;
            }
            if (!eq && lane == 0) first_col[i] = -1;
        }
    }
    bad = __syncthreads_or(bad);
    if (bad) return B200_ENUMERIC;
    if (stage_or_null) { cost = stage_or_null; ld = Cc; }
    __shared__ int s_status;
    const int nt = nthr < kMaxThreads ? (nthr & ~31) : kMaxThreads;
    if (Cc <= kWarpSolverMaxCols) {
        if (tid < 32) {
            const int rc = Cc <= 64 ? solve_warp<2>(cost, R, Cc, ld, w.u, w.c4r, w.r4c, w.v, first_col, first_val)
                                    : solve_warp<4>(cost, R, Cc, ld, w.u, w.c4r, w.r4c, w.v, first_col, first_val);
            if (tid == 0) s_status = rc;
        }
    } else if (tid < nt) {
        const int per = (Cc + nt - 1) / nt;
        const int rc = per <= 1   ? solve_regs<1>(cost, R, Cc, ld, w, tid, nt)
                       : per <= 2 ? solve_regs<2>(cost, R, Cc, ld, w, tid, nt)
                       : per <= 4 ? solve_regs<4>(cost, R, Cc, ld, w, tid, nt)
                                  : solve(cost, R, Cc, ld, w, tid, nt, true);
        if (tid == 0) s_status = rc;
    }
    __syncthreads();
    return s_status;
}

}  // namespace lsap
}  // namespace b200

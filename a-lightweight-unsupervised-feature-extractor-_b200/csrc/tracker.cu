// GPU-resident multi-stream tracker: Tracking.update (model/mainTracking.py:450-610) as six
// kernels per frame-step, batched over independent streams (one CTA, or one grid slice, each).
//
//   begin   (CTA / stream)  :467-487  empty-frame shortcut, predict_all, main/ReID row split,
//                                     detection prep (unit embeddings, z, float32 boxes), gate prep
//   cost1   (grid)          :496-511  Mahalanobis gate first, then bank top-k appearance + box + conf terms
//                                     for the surviving pairs, written once as C and C^T
//   assign<1> (CTA / stream):514-538  LSAP + cost_max filter, match bookkeeping, mark_missed
//   cost2   (grid)          :552-558  ReID-only appearance cost for long-lost rows x leftover dets
//   assign<2> (CTA / stream):560-610  LSAP, match bookkeeping, mark_missed, births, purge, result table
//   update  (grid)          :375-448  Kalman update, posterior gate, EMA, bank push for every match of the step
//
// State never leaves the device.  Tracks live in fixed physical slots (banks are never moved);
// `order` lists the live slots by ascending track id, which is the row order the reference uses
// (sorted(rows_main), :486-487) because ids are handed out monotonically (:371-372).
#include <stdlib.h>
#include <string.h>

#include <new>

#include <cuda_fp16.h>

#include "assoc_cost.cuh"
#include "kalman.cuh"
#include "lsap.cuh"

namespace b200 {
namespace trk {

// Programmatic dependent launch (used for small stream counts, see b200_tracker_step): let the next kernel of
// the step become resident while this one runs, then wait until the previous kernel has completed and its
// writes are visible.  Both instructions are no-ops for a kernel launched without the attribute.
#define TRK_PDL_PROLOGUE()                                        \
    do {                                                          \
        asm volatile("griddepcontrol.launch_dependents;");        \
        asm volatile("griddepcontrol.wait;" ::: "memory");        \
    } while (0)

constexpr int kThreads = 256;
constexpr int kHdr = 8;                 // ints per stream in hdr / cnt
enum { H_NLIVE = 0, H_NEXT = 1, H_NFREE = 2 };
enum { C_M1 = 0, C_M2 = 1, C_NU = 2, C_MODE = 3, C_NMATCH = 4, C_NUT = 5, C_STATUS = 6 };
enum { MODE_SKIP = 0, MODE_EMPTY = 1, MODE_NORMAL = 2, MODE_FAILED = 3 };   // FAILED: scipy would have raised in stage 1
enum { R_NMATCH = 0, R_NUT = 1, R_NUD = 2, R_NLIVE = 3, R_NEXT = 4, R_STATUS = 5, R_M1 = 6, R_M2 = 7, R_HDR = 8 };

struct Dev {
    int S, MT, MD, HIST, res_stride;
    // persistent state
    double *kf_x, *kf_P, *last_bbox, *last_conf, *last_cost;
    uint8_t* kf_stage;
    float *ema, *bank;
    int *bank_len, *bank_head, *tid, *miss, *age, *last_frame, *order, *free_list, *hdr;
    // per-step scratch
    float *det_unit, *det_z, *det_boxf, *det_conff, *prev_boxf, *prev_conff, *C1, *C1T, *C2, *C2T;
    double* gate_SI;
    int* row_fc;                     // stage 1, written by the cost kernel: column of each row's unique minimum (-1: none, -2: NaN / -inf in the row)
    float* row_fv;                   //          that minimum
    int *rows_main, *rows_reid, *cnt, *ud1, *det_used, *m_row, *m_det, *tmp;
    int* born;                       // [S, MD] detection index of each birth of the step, in order
    int2 *work1, *work2;             // (stream, row * 64 + detection tile) items of the two cost launches
    int* wcount;                     // [3] items queued for this step: cost1, cost2, updates
    int *upd_slot, *upd_det;         // update queue: global slot / detection index of every match
    float* upd_cost;                 //               its (float32) cost, negative-zero-safe flag in upd_flag
    uint8_t* upd_flag;               //               1 = matched in the ReID-only stage
    // configuration
    cost::PairWeights pw;
    double maha_thr, cost_max, conf_update_min, cost_update_max, reid_only_cost_max, init_conf_min;
    float ema_a, ema_b;
    int topk, max_age, lost_reid_after;
    // this step's inputs / output
    const int* n_det;
    const double *boxes, *confs;
    const float* embs;
    const int* frame_id;
    int* result;
};

__device__ __forceinline__ int* res_matches(const Dev& d, int* res) { return res + R_HDR; }
__device__ __forceinline__ int* res_ut(const Dev& d, int* res) { return res + R_HDR + 2 * d.MD; }
__device__ __forceinline__ int* res_ud(const Dev& d, int* res) { return res + R_HDR + 2 * d.MD + d.MT; }

// Ordered stream compaction over [0, n): emit(position, i) for every i with pred(i), ascending.
// All threads of the CTA must call; returns the count.  scratch: kThreads / 32 ints of smem.
template <typename Pred, typename Emit>
__device__ inline int block_compact(int n, Pred pred, Emit emit, int* scratch) {
    int base = 0;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        const bool p = i < n && pred(i);
        const unsigned m = __ballot_sync(0xffffffffu, p);
        if (lane == 0) scratch[w] = __popc(m);
        __syncthreads();
        int off = 0, tot = 0;
        for (int k = 0; k < nw; ++k) {
            const int c = scratch[k];
            if (k < w) off += c;
            tot += c;
        }
        if (p) emit(base + off + __popc(m & ((1u << lane) - 1u)), i);
        base += tot;
        __syncthreads();
    }
    return base;
}

__device__ __forceinline__ void load_kf(const Dev& d, size_t slot, double* x, double* P) {
    const double2* px = reinterpret_cast<const double2*>(d.kf_x + slot * 8);
    const double2* pP = reinterpret_cast<const double2*>(d.kf_P + slot * 64);
#pragma unroll
    for (int k = 0; k < 4; ++k) { const double2 v = px[k]; x[2 * k] = v.x; x[2 * k + 1] = v.y; }
#pragma unroll
    for (int k = 0; k < 32; ++k) { const double2 v = pP[k]; P[2 * k] = v.x; P[2 * k + 1] = v.y; }
}
__device__ __forceinline__ void store_kf(const Dev& d, size_t slot, const double* x, const double* P) {
    double2* px = reinterpret_cast<double2*>(d.kf_x + slot * 8);
    double2* pP = reinterpret_cast<double2*>(d.kf_P + slot * 64);
#pragma unroll
    for (int k = 0; k < 4; ++k) px[k] = make_double2(x[2 * k], x[2 * k + 1]);
#pragma unroll
    for (int k = 0; k < 32; ++k) pP[k] = make_double2(P[2 * k], P[2 * k + 1]);
}

// purge_dead (:357-360): drop slots with miss > max_age from `order`, return them to the free list.
__device__ inline void purge(const Dev& d, int s, int nl, int* scratch) {
    int* order = d.order + (size_t)s * d.MT;
    int* tmp = d.tmp + (size_t)s * d.MT;
    int* fl = d.free_list + (size_t)s * d.MT;
    int* hdr = d.hdr + s * kHdr;
    const size_t sb = (size_t)s * d.MT;
    for (int i = threadIdx.x; i < nl; i += blockDim.x) tmp[i] = order[i];
    __syncthreads();
    const int nfree = hdr[H_NFREE];
    const int keep = block_compact(nl, [&](int i) { return d.miss[sb + tmp[i]] <= d.max_age; },
                                   [&](int pos, int i) { order[pos] = tmp[i]; }, scratch);
    const int dead = block_compact(nl, [&](int i) { return d.miss[sb + tmp[i]] > d.max_age; },
                                   [&](int pos, int i) { fl[nfree + pos] = tmp[i]; }, scratch);
    if (threadIdx.x == 0) { hdr[H_NLIVE] = keep; hdr[H_NFREE] = nfree + dead; }
    __syncthreads();
}

// The header of a stream's row of the result table.
__device__ __forceinline__ void put_result_header(int* res, int nmatch, int nut, int nud, int nlive, int next, int status,
                                                  int m1, int m2) {
    res[R_NMATCH] = nmatch; res[R_NUT] = nut; res[R_NUD] = nud; res[R_NLIVE] = nlive;
    res[R_NEXT] = next; res[R_STATUS] = status; res[R_M1] = m1; res[R_M2] = m2;
}

// Start of a stream's step in the first kernel of every schedule: an idle stream (n < 0) and an empty frame (n == 0) are
// the whole step.  Returns true when stream s is done for this step.  All threads of the CTA call; only the CTA with
// `writer` set touches the stream's state and result row.
__device__ __forceinline__ bool step_prologue(const Dev& d, int s, int n, int nl, bool writer, int* scratch) {
    const int* hdr = d.hdr + s * kHdr;
    int* cnt = d.cnt + s * kHdr;
    int* res = d.result + (size_t)s * d.res_stride;
    if (n < 0) {                                   // stream idle this step
        if (writer && threadIdx.x == 0) {
            cnt[C_MODE] = MODE_SKIP;
            put_result_header(res, 0, 0, 0, nl, hdr[H_NEXT], 0, 0, 0);
        }
        return true;
    }
    if (n > 0) return false;
    if (!writer) return true;
    // :467-471 -- every track missed, NO predict
    const size_t sb = (size_t)s * d.MT;
    const int* order = d.order + sb;
    int* ut = res_ut(d, res);
    for (int p = threadIdx.x; p < nl; p += blockDim.x) {
        const size_t slot = sb + order[p];
        d.miss[slot] += 1;
        ut[p] = d.tid[slot];
    }
    __syncthreads();
    purge(d, s, nl, scratch);
    if (threadIdx.x == 0) {
        cnt[C_MODE] = MODE_EMPTY;
        put_result_header(res, 0, nl, 0, hdr[H_NLIVE], hdr[H_NEXT], 0, 0, 0);
    }
    return true;
}

// Queues one work item per (row, 64-detection tile) of this stream for the persistent cost kernel.
__device__ inline void enqueue_cost_work(int2* work, int* counter, int s, int M, int N, int* scratch) {
    const int tiles = (N + cost::kTileN - 1) / cost::kTileN, total = M * tiles;
    if (total <= 0) return;                       // uniform across the CTA
    __syncthreads();
    if (threadIdx.x == 0) scratch[0] = atomicAdd(counter, total);
    __syncthreads();
    const int base = scratch[0];
    for (int i = threadIdx.x; i < total; i += blockDim.x) work[base + i] = make_int2(s, (i / tiles) * 64 + i % tiles);
}

// ---- detections: unit embeddings (:167-168), z (KalmanFilter.py:5-16), float32 boxes/confs (all threads of a CTA) ----
// part / nparts: the CTAs of one stream share the work (front_kernel); 0 / 1 = the whole stream.
__device__ inline void prep_detections(const Dev& d, int s, int n, int part = 0, int nparts = 1) {
    const size_t db = (size_t)s * d.MD;
    const int tid = threadIdx.x;
    const int nw = blockDim.x >> 5, nt = blockDim.x;
    for (int j = part * nw + (tid >> 5); j < n; j += nparts * nw) {
        const float4 v = reinterpret_cast<const float4*>(d.embs + (db + j) * cost::kD)[tid & 31];
        reinterpret_cast<float4*>(d.det_unit + (db + j) * cost::kD)[tid & 31] = cost::unit_row(v);
    }
    for (int j = part * nt + tid; j < n; j += nparts * nt) {
        double b[4];
        float z[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { b[k] = d.boxes[(db + j) * 4 + k]; d.det_boxf[(db + j) * 4 + k] = (float)b[k]; }
        kf::box_to_z(b, z);
#pragma unroll
        for (int k = 0; k < 4; ++k) d.det_z[(db + j) * 4 + k] = z[k];
        d.det_conff[db + j] = (float)d.confs[db + j];
        d.det_used[db + j] = 0;
    }
}

// predict_all (:340-345) for one track + the per-track inputs of the stage-1 cost (by slot): predicted box and
// confidence as float32, inverse innovation covariance for the gate.
__device__ inline void predict_slot(const Dev& d, size_t slot) {
    const float q[8] = {1.f, 1.f, 1.f, 1.f, 100.f, 100.f, 100.f, 100.f};    // KalmanFilter.py:91-95
    const float rdiag[4] = {1.f, 1.f, 1.f, 1.f};                           // KalmanFilter.py:98-99
    double x[8], P[64], b[4];
    load_kf(d, slot, x, P);
    const int st = d.kf_stage[slot];
    kf::predict(x, P, st, q);
    store_kf(d, slot, x, P);
    kf::x_to_box(x, b);
#pragma unroll
    for (int k = 0; k < 4; ++k) { d.last_bbox[slot * 4 + k] = b[k]; d.prev_boxf[slot * 4 + k] = (float)b[k]; }
    d.prev_conff[slot] = (float)d.last_conf[slot];
    kf::Gate g;
    kf::gate_prepare(x, P, st, rdiag, &g);
#pragma unroll
    for (int k = 0; k < 16; ++k) d.gate_SI[slot * 16 + k] = g.SI[k];
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) begin_kernel(Dev d) {
    __shared__ int scratch[kThreads / 32];
    const int s = blockIdx.x, tid = threadIdx.x;
    int* cnt = d.cnt + s * kHdr;
    const size_t sb = (size_t)s * d.MT;
    const int n = d.n_det[s], nl = d.hdr[s * kHdr + H_NLIVE];
    int* order = d.order + sb;
    if (blockIdx.y == 1) {                         // second CTA of the stream: detection prep only
        if (n <= 0) return;
        prep_detections(d, s, n);
        return;
    }
    if (s == 0 && tid == 0) d.wcount[2] = 0;       // last step's update_kernel is done; nothing queued yet
    if (step_prologue(d, s, n, nl, true, scratch)) return;
    // ---- predict_all (:340-345) + per-track inputs of the stage-1 cost (by slot): predicted box and
    // confidence as float32, inverse innovation covariance for the gate -------------------------------
    for (int p = tid; p < nl; p += blockDim.x) predict_slot(d, sb + order[p]);
    // ---- rows_main / rows_reid in ascending track-id order (:478-487) -----------------------------
    int* rm = d.rows_main + sb;
    int* rr = d.rows_reid + sb;
    const int M1 = block_compact(nl, [&](int i) { return d.miss[sb + order[i]] <= d.lost_reid_after; },
                                 [&](int pos, int i) { rm[pos] = order[i]; }, scratch);
    const int M2 = block_compact(nl, [&](int i) { return d.miss[sb + order[i]] > d.lost_reid_after; },
                                 [&](int pos, int i) { rr[pos] = order[i]; }, scratch);
    if (tid == 0) {
        cnt[C_M1] = M1; cnt[C_M2] = M2; cnt[C_NU] = 0; cnt[C_MODE] = MODE_NORMAL;
        cnt[C_NMATCH] = 0; cnt[C_NUT] = 0; cnt[C_STATUS] = 0;
    }
    enqueue_cost_work(d.work1, d.wcount + 0, s, M1, 1, scratch);      // one item per row (all detections)
}

// ------------------------------------------------------------------------------------------------
// ReID-only stage (:552-558): rows_reid x leftover detections, appearance cost only, dense tiles (bank and
// 64 detection rows staged in shared memory, see assoc_cost.cuh).  Persistent CTAs over queued work items.
// One (long-lost row r, tile of 64 leftover detections starting at j0) item of stream s; every thread of a
// cost::kThreads-wide CTA must call.  smem: cost::smem_bytes(HIST) bytes; s_idx: cost::kTileN ints of shared memory.
__device__ inline void cost2_item(const Dev& d, int s, int r, int j0, float* smem, int* s_idx) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int N = d.cnt[s * kHdr + C_NU];
    const size_t sb = (size_t)s * d.MT, db = (size_t)s * d.MD;
    const size_t slot = sb + d.rows_reid[sb + r];
    int T = d.bank_len[slot];
    const float* rows = d.bank + slot * d.HIST * cost::kD;
    if (T <= 0) { rows = d.ema + slot * cost::kD; T = 1; }        // :180-182 fallback to the EMA
    if (tid < cost::kTileN) {                                      // leftover detections are gathered through ud1
        const int j = j0 + tid;
        s_idx[tid] = j < N ? d.ud1[db + j] : 0;
    }
    __syncthreads();
    const int tc = cost::bank_cap(T);
    float* sBank = smem;
    float* sDet = sBank + tc * cost::kD;
    float* sSim = sDet + cost::kTileN * cost::kDetStride;
    for (int t = warp; t < tc; t += cost::kThreads / 32) {
        float4 v = make_float4(0, 0, 0, 0);
        if (t < T) v = cost::unit_row(reinterpret_cast<const float4*>(rows + (size_t)t * cost::kD)[lane]);
        reinterpret_cast<float4*>(sBank + t * cost::kD)[lane] = v;
    }
    for (int j = warp; j < cost::kTileN; j += cost::kThreads / 32) {
        float4 v = make_float4(0, 0, 0, 0);
        if (j0 + j < N) v = reinterpret_cast<const float4*>(d.det_unit + (db + s_idx[j]) * cost::kD)[lane];
        reinterpret_cast<float4*>(sDet + j * cost::kDetStride)[lane] = v;
    }
    __syncthreads();
    const float c_app = cost::sims_and_topk(sBank, sDet, sSim, tc, T, d.topk, true);   // ends with a barrier
    const int j = j0 + tid;
    if (tid < cost::kTileN && j < N) {
        d.C2[(sb + r) * d.MD + j] = c_app;
        d.C2T[(db + j) * d.MT + r] = c_app;
    }
}

__global__ void __launch_bounds__(cost::kThreads) cost2_kernel(Dev d) {
    TRK_PDL_PROLOGUE();
    extern __shared__ __align__(16) float smem[];
    __shared__ int s_idx[cost::kTileN];
    const int total = d.wcount[1];
    for (int wi = blockIdx.x; wi < total; wi += gridDim.x) {        // uniform trip count per CTA
        const int2 item = d.work2[wi];
        cost2_item(d, item.x, item.y >> 6, (item.y & 63) * cost::kTileN, smem, s_idx);
    }
}

// Per-row summary of a stage-1 cost row for the assignment kernel's known-first-step rule (lsap.cuh): each lane
// feeds the entries it wrote; finish() leaves the column of the row's unique minimum (-1 if the minimum is tied
// or +inf, -2 if the row holds a NaN or -inf, which scipy rejects) and its value.
struct RowMin {
    float m = __builtin_huge_valf(), first = 0.0f;
    int mj = -1, cnt = 0, bad = 0;
    __device__ __forceinline__ void see(float c, int j) {
        if (c != c || c == -__builtin_huge_valf()) bad = 1;
        if (c < m) { m = c; mj = j; cnt = 1; first = c; }
        else if (c == m) ++cnt;
    }
    __device__ __forceinline__ void finish(int* fc, float* fv, int lane) const {
        const unsigned kFull = 0xffffffffu;
        const unsigned bits = (unsigned)__float_as_int(m + 0.0f);                      // -0.0 ties with +0.0
        const unsigned key = bits ^ ((unsigned)((int)bits >> 31) | 0x80000000u);
        const unsigned kmin = __reduce_min_sync(kFull, key);
        const unsigned eq = __ballot_sync(kFull, key == kmin && mj >= 0);
        const bool any_bad = __any_sync(kFull, bad);
        const int total = __reduce_add_sync(kFull, (key == kmin && mj >= 0) ? cnt : 0);
        if (any_bad) { if (lane == 0) *fc = -2; return; }
        if (eq && lane == __ffs(eq) - 1) {
            *fc = (total == 1 && m < __builtin_huge_valf()) ? mj : -1;
            *fv = first;
        }
        if (!eq && lane == 0) *fc = -1;
    }
};

// ---- stage-1 cost, gate first -----------------------------------------------------------------------
// apply_kalman_gating (:306-338) overwrites every pair with d2 > maha_thr by 1e9 AFTER the reference has
// computed its full cost (:496-511).  The result does not depend on the order, and in steady state ~98 %
// of the pairs are gated (SURVEY.md section 7), so this kernel evaluates the gate for all pairs first and
// runs the bank contraction + top-k only for the pairs that survive.  One warp owns one track row:
//   lane = detection (chunks of 32): d2 and, for survivors, the box/conf terms; ballot -> survivors;
//   per survivor: lanes split the 128 dimensions (one coalesced 512 B read per bank row, eight rows in
//   flight), a shuffle reduction gives <bank_t, det>, lane t keeps the similarity of row t, then k rounds
//   of warp-max give the top-k mean.  No shared memory and few registers, so every row of a 64-stream
//   group is resident at once and the kernel can share SMs with ROI Align.  Four warps per CTA: with two or one,
//   neither the six-kernel chain alone nor the overlapped step changed (profiles/r02_chain_cta_sweep.txt, builds
//   c1w2 / c1w1).
constexpr int kCost1Warps = 4;

__device__ __forceinline__ unsigned fkey(float f) {                 // order-preserving float -> uint
    const unsigned b = __float_as_uint(f);
    return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}

__global__ void __launch_bounds__(kCost1Warps * 32) cost1_sparse_kernel(Dev d) {
    TRK_PDL_PROLOGUE();
    const int total = d.wcount[0];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float kNegInf = -__int_as_float(0x7f800000);
    for (int wi = blockIdx.x * kCost1Warps + warp; wi < total; wi += gridDim.x * kCost1Warps) {
        const int2 item = d.work1[wi];
        const int s = item.x, r = item.y >> 6;
        const int N = d.n_det[s];
        const size_t sb = (size_t)s * d.MT, db = (size_t)s * d.MD;
        const size_t slot = sb + d.rows_main[sb + r];
        int T = d.bank_len[slot];
        const float* rows = d.bank + slot * d.HIST * cost::kD;
        if (T <= 0) { rows = d.ema + slot * cost::kD; T = 1; }        // :180-182 fallback to the EMA
        const int kk = min(d.topk, T);
        double SI[16], xs[4];                                         // per-row gate inputs
#pragma unroll
        for (int k = 0; k < 16; ++k) SI[k] = d.gate_SI[slot * 16 + k];
#pragma unroll
        for (int k = 0; k < 4; ++k) xs[k] = d.kf_x[slot * 8 + k];
        const int stage = d.kf_stage[slot];
        float pb[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) pb[k] = d.prev_boxf[slot * 4 + k];
        const float pconf = d.prev_conff[slot];
        float inv0 = 0.0f, inv1 = 0.0f;           // 1 / (|bank_t| + 1e-12) of rows lane and lane + 32 (:188-189)
        bool have_norm = false;
        RowMin rmin;
        for (int j0 = 0; j0 < N; j0 += 32) {
            const int j = j0 + lane;
            bool alive = false;
            if (j < N) alive = !(kf::gate_d2(SI, xs, stage, d.det_z + (db + j) * 4) > d.maha_thr);   // :335
            unsigned todo = __ballot_sync(0xffffffffu, alive);
            float c_app = 0.0f;
            while (todo) {
                const int jl = __ffs(todo) - 1;
                todo &= todo - 1;
                const float4 dv = reinterpret_cast<const float4*>(d.det_unit + (db + j0 + jl) * cost::kD)[lane];
                float s0 = kNegInf, s1 = kNegInf;                    // similarities of bank rows lane, lane + 32
                for (int t0 = 0; t0 < T; t0 += 8) {
                    float4 bv[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u)
                        if (t0 + u < T) bv[u] = reinterpret_cast<const float4*>(rows + (size_t)(t0 + u) * cost::kD)[lane];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int t = t0 + u;
                        if (t >= T) break;                          // uniform
                        float p = bv[u].x * dv.x;
                        p = fmaf(bv[u].y, dv.y, p); p = fmaf(bv[u].z, dv.z, p); p = fmaf(bv[u].w, dv.w, p);
                        p = warp_sum(p);
                        if (!have_norm) {
                            float q = bv[u].x * bv[u].x;
                            q = fmaf(bv[u].y, bv[u].y, q); q = fmaf(bv[u].z, bv[u].z, q); q = fmaf(bv[u].w, bv[u].w, q);
                            q = warp_sum(q);
                            const float iv = __fdiv_rn(1.0f, __fadd_rn(sqrtf(q), 1e-12f));
                            if (lane == (t & 31)) { if (t < 32) inv0 = iv; else inv1 = iv; }
                        }
                        if (lane == (t & 31)) { if (t < 32) s0 = p; else s1 = p; }
                    }
                }
                have_norm = true;
                if (lane < T) s0 *= inv0;
                if (lane + 32 < T) s1 *= inv1;
                float sum = 0.0f;                                   // top-k mean, largest first (:196-202)
                for (int q = 0; q < kk; ++q) {
                    const float mine = fmaxf(s0, s1);
                    const unsigned m = __reduce_max_sync(0xffffffffu, fkey(mine));
                    const unsigned who = __ballot_sync(0xffffffffu, fkey(mine) == m);
                    if (lane == __ffs(who) - 1) {
                        if (s0 >= s1) s0 = kNegInf; else s1 = kNegInf;
                    }
                    const unsigned bits = m ^ ((m >> 31) ? 0x80000000u : 0xffffffffu);
                    sum = __fadd_rn(sum, __uint_as_float(bits));
                }
                const float ca = __fsub_rn(1.0f, __fdiv_rn(sum, (float)kk));
                if (lane == jl) c_app = ca;
            }
            if (j < N) {
                float total_c = 1e9f;
                if (alive)
                    total_c = cost::pair_cost(pb, d.det_boxf + (db + j) * 4, pconf, d.det_conff[db + j], d.pw, c_app).total;
                d.C1[(sb + r) * d.MD + j] = total_c;
                d.C1T[(db + j) * d.MT + r] = total_c;
                rmin.see(total_c, j);
            }
        }
        rmin.finish(d.row_fc + sb + r, d.row_fv + sb + r, lane);
    }
}

// Sum over lanes of 32 per-lane partials at once: after the call lane t holds the full sum of
// partial[t] in p[0].  31 shuffles instead of 32 x 5 (each stage sends the half the partner lane owns).
__device__ __forceinline__ void transpose_reduce32(float (&p)[32]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const bool up = lane & o;
#pragma unroll
        for (int i = 0; i < o; ++i) {
            const float keep = up ? p[i + o] : p[i], send = up ? p[i] : p[i + o];
            p[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
}

// Stage-1 cost for hist_max <= 32 (the shipped 30): same algorithm as cost1_sparse_kernel, but the row's
// whole bank is read once into registers (one global round trip, reused by every surviving detection) and
// the 32 dot products of a detection are reduced together (transpose_reduce32).
// One track row of the stage-1 cost (one warp): gate for every detection, contraction for the survivors, C / C^T / row
// summary written.  FLY = false: the detection-side inputs (z, float32 boxes / confidences, unit embeddings) were
// prepared by begin_kernel; FLY = true (front_kernel): they are derived here from the caller's arrays with the same
// functions, value for value.
template <bool FLY>
__device__ __forceinline__ void cost1_row32(const Dev& d, int s, int r, size_t slot, int N, int lane) {
    const float kNegInf = -__int_as_float(0x7f800000);
    const size_t sb = (size_t)s * d.MT, db = (size_t)s * d.MD;
    int T = d.bank_len[slot];
    const float* rows = d.bank + slot * d.HIST * cost::kD;
    if (T <= 0) { rows = d.ema + slot * cost::kD; T = 1; }        // :180-182 fallback to the EMA
    const int kk = min(d.topk, T);
    double SI[16], xs[4];
#pragma unroll
    for (int k = 0; k < 16; ++k) SI[k] = d.gate_SI[slot * 16 + k];
#pragma unroll
    for (int k = 0; k < 4; ++k) xs[k] = d.kf_x[slot * 8 + k];
    const int stage = d.kf_stage[slot];
    float pb[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) pb[k] = d.prev_boxf[slot * 4 + k];
    const float pconf = d.prev_conff[slot];
    float4 bv[32];
    float inv = 0.0f;                          // 1 / (|bank_lane| + 1e-12), :188-189
    bool have_bank = false;
    RowMin rmin;
    for (int j0 = 0; j0 < N; j0 += 32) {
        const int j = j0 + lane;
        bool alive = false;
        float zl[4], bf[4];
        float cf = 0.0f;
        if (j < N) {
            if (FLY) {
                double b[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) { b[k] = d.boxes[(db + j) * 4 + k]; bf[k] = (float)b[k]; }
                kf::box_to_z(b, zl);
                cf = (float)d.confs[db + j];
                alive = !(kf::gate_d2(SI, xs, stage, zl) > d.maha_thr);                     // :335
            } else {
                alive = !(kf::gate_d2(SI, xs, stage, d.det_z + (db + j) * 4) > d.maha_thr);   // :335
            }
        }
        unsigned todo = __ballot_sync(0xffffffffu, alive);
        float c_app = 0.0f;
        // the first survivor's embedding is requested together with the bank, not after the bank's norms have been
        // computed: one dependent global round trip per row less
        float4 dv_first = make_float4(0, 0, 0, 0);
        if (todo) {
            const int jf = __ffs(todo) - 1;
            if (FLY) dv_first = reinterpret_cast<const float4*>(d.embs + (db + j0 + jf) * cost::kD)[lane];
            else dv_first = reinterpret_cast<const float4*>(d.det_unit + (db + j0 + jf) * cost::kD)[lane];
        }
        if (todo && !have_bank) {
            float q[32];
#pragma unroll
            for (int t = 0; t < 32; ++t)
                bv[t] = t < T ? reinterpret_cast<const float4*>(rows + (size_t)t * cost::kD)[lane] : make_float4(0, 0, 0, 0);
#pragma unroll
            for (int t = 0; t < 32; ++t) {
                float a = bv[t].x * bv[t].x;
                a = fmaf(bv[t].y, bv[t].y, a); a = fmaf(bv[t].z, bv[t].z, a); a = fmaf(bv[t].w, bv[t].w, a);
                q[t] = a;
            }
            transpose_reduce32(q);
            inv = __fdiv_rn(1.0f, __fadd_rn(sqrtf(q[0]), 1e-12f));
            have_bank = true;
        }
        bool first = true;
        while (todo) {
            const int jl = __ffs(todo) - 1;
            todo &= todo - 1;
            float4 dv = dv_first;
            if (!first) {
                if (FLY) dv = reinterpret_cast<const float4*>(d.embs + (db + j0 + jl) * cost::kD)[lane];
                else dv = reinterpret_cast<const float4*>(d.det_unit + (db + j0 + jl) * cost::kD)[lane];
            }
            first = false;
            if (FLY) dv = cost::unit_row(dv);
            float p[32];
#pragma unroll
            for (int t = 0; t < 32; ++t) {
                float a = bv[t].x * dv.x;
                a = fmaf(bv[t].y, dv.y, a); a = fmaf(bv[t].z, dv.z, a); a = fmaf(bv[t].w, dv.w, a);
                p[t] = a;
            }
            transpose_reduce32(p);
            float sim = lane < T ? p[0] * inv : kNegInf;        // <bank_lane, det> of unit vectors
            float sum = 0.0f;                                   // top-k mean, largest first (:196-202)
            for (int q = 0; q < kk; ++q) {
                const unsigned m = __reduce_max_sync(0xffffffffu, fkey(sim));
                const unsigned who = __ballot_sync(0xffffffffu, fkey(sim) == m);
                if (lane == __ffs(who) - 1) sim = kNegInf;
                const unsigned bits = m ^ ((m >> 31) ? 0x80000000u : 0xffffffffu);
                sum = __fadd_rn(sum, __uint_as_float(bits));
            }
            const float ca = __fsub_rn(1.0f, __fdiv_rn(sum, (float)kk));
            if (lane == jl) c_app = ca;
        }
        if (j < N) {
            float total_c = 1e9f;
            if (alive) {
                if (FLY) total_c = cost::pair_cost(pb, bf, pconf, cf, d.pw, c_app).total;
                else total_c = cost::pair_cost(pb, d.det_boxf + (db + j) * 4, pconf, d.det_conff[db + j], d.pw, c_app).total;
            }
            d.C1[(sb + r) * d.MD + j] = total_c;
            d.C1T[(db + j) * d.MT + r] = total_c;
            rmin.see(total_c, j);
        }
    }
    rmin.finish(d.row_fc + sb + r, d.row_fv + sb + r, lane);
}

__global__ void __launch_bounds__(kCost1Warps * 32, 2) cost1_sparse32_kernel(Dev d) {
    TRK_PDL_PROLOGUE();
    const int total = d.wcount[0];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int wi = blockIdx.x * kCost1Warps + warp; wi < total; wi += gridDim.x * kCost1Warps) {
        const int2 item = d.work1[wi];
        const int s = item.x, r = item.y >> 6;
        const size_t sb = (size_t)s * d.MT;
        cost1_row32<false>(d, s, r, sb + d.rows_main[sb + r], d.n_det[s], lane);
    }
}

// update_matched (:375-448), part 1, inside the assignment kernel: the bookkeeping that later steps of the same
// frame depend on (:403-415: last box / conf / frame, age, miss reset, match cost), and one queue entry per
// match for update_kernel, which does the arithmetic (Kalman update, posterior gate, EMA, bank push).
// queue_base >= 0: the entries go to upd_*[queue_base ..] (the fused path keeps one queue per stream); < 0: they are
// appended to the step's global queue (update_kernel).
__device__ inline void note_matches(const Dev& d, int s, int nm, const int* rows, const float* C, int ldc,
                                    const int* m_col, int reid_stage, int* scratch, int queue_base = -1) {
    if (nm <= 0) return;                                          // uniform across the CTA
    const size_t sb = (size_t)s * d.MT, db = (size_t)s * d.MD;
    const int frame = d.frame_id[s];
    int base = queue_base;
    if (queue_base < 0) {
        __syncthreads();
        if (threadIdx.x == 0) scratch[0] = atomicAdd(d.wcount + 2, nm);
        __syncthreads();
        base = scratch[0];
    }
    for (int qd = threadIdx.x; qd < nm; qd += blockDim.x) {
        const int r = d.m_row[sb + qd], j = d.m_det[sb + qd];
        const size_t slot = sb + rows[r];
        const float c = C[(size_t)r * ldc + m_col[qd]];
#pragma unroll
        for (int k = 0; k < 4; ++k) d.last_bbox[slot * 4 + k] = d.boxes[(db + j) * 4 + k];
        d.last_conf[slot] = d.confs[db + j];
        d.last_frame[slot] = frame;
        d.age[slot] += 1;
        d.miss[slot] = 0;
        d.last_cost[slot] = (double)c;
        d.upd_slot[base + qd] = (int)slot;
        d.upd_det[base + qd] = (int)(db + j);
        d.upd_cost[base + qd] = c;
        d.upd_flag[base + qd] = (uint8_t)reid_stage;
    }
}

// update_matched, part 2: every match of every stream, both stages (they touch disjoint tracks).  A warp takes
// four queue entries: eight lanes per match run the Kalman update (:400, kf::update_rows_t) and the posterior
// gate (:424-426), then the warp applies the EMA and pushes the bank rows of those four matches (:429-448).
constexpr int kUpdWarps = 4;

// Queue entries first .. first + total - 1, four per warp and pass; `wq` = index of this warp among the `nwq` warps that
// share the range; scratch: 4 x 96 doubles of shared memory private to the warp.
__device__ __forceinline__ void update_entries(const Dev& d, int first, int total, int wq, int nwq, double* scratch) {
    const int lane = threadIdx.x & 31, sub = lane & 7, grp = lane >> 3;
    double* sP = scratch + (size_t)grp * 96;
    double* sK = sP + 64;
    const float rdiag[4] = {1.f, 1.f, 1.f, 1.f};                           // KalmanFilter.py:98-99
    for (int w0 = wq * 4; w0 < total; w0 += nwq * 4) {
        const int idx = first + w0 + grp;
        const bool on = w0 + grp < total;
        size_t slot = 0, det = 0;
        int st = -1, reid = 0;
        double c = 0.0, conf = 0.0;
        if (on) {
            slot = (size_t)d.upd_slot[idx];
            det = (size_t)d.upd_det[idx];
            c = (double)d.upd_cost[idx];
            reid = d.upd_flag[idx];
            st = d.kf_stage[slot];
            conf = d.confs[det];
        }
        const float* z = d.det_z + det * 4;
        const double cmax = reid ? d.reid_only_cost_max : d.cost_update_max;   // :563 / :530
        int app = on && !(conf < d.conf_update_min) && !(c > cmax);             // :418-421
        const int nst = st < 2 ? st + 1 : 2;
        // Inputs of the EMA / bank push of this warp's four matches: they do not depend on the Kalman result (only whether
        // they are USED does, through the posterior gate), so they are requested now and arrive during the float64 work.
        float4 e[4], o[4];
        size_t slots[4];
        int len[4], head[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const bool on_u = __shfl_sync(0xffffffffu, (int)on, u * 8) != 0;
            const unsigned long long sl = __shfl_sync(0xffffffffu, (unsigned long long)slot, u * 8);
            const unsigned long long dt = __shfl_sync(0xffffffffu, (unsigned long long)det, u * 8);
            slots[u] = (size_t)sl;
            if (on_u) {
                e[u] = reinterpret_cast<const float4*>(d.det_unit + (size_t)dt * cost::kD)[lane];
                o[u] = reinterpret_cast<const float4*>(d.ema + slots[u] * cost::kD)[lane];
                len[u] = d.bank_len[slots[u]];
                head[u] = d.bank_head[slots[u]];
            }
        }
        double d2 = 0.0;
#pragma unroll
        for (int v = 0; v < 6; ++v) {               // arithmetic variant x (stage 1: posterior gate, stage 2: none)
            const bool mine = on && st == (v >> 1) && reid == (v & 1);
            const unsigned mask = __ballot_sync(0xffffffffu, mine);
            if (mine) {
                double* gx = d.kf_x + slot * 8;
                double* gP = d.kf_P + slot * 64;
                const bool want = !(v & 1);          // uniform over the lanes of `mask`
                if ((v >> 1) == 0) d2 = kf::update_rows_t<float, float>(gx, gP, z, rdiag, sP, sK, sub, mask, nst, want);
                else if ((v >> 1) == 1) d2 = kf::update_rows_t<float, double>(gx, gP, z, rdiag, sP, sK, sub, mask, nst, want);
                else d2 = kf::update_rows_t<double, double>(gx, gP, z, rdiag, sP, sK, sub, mask, nst, want);
            }
        }
        if (on && sub == 0) d.kf_stage[slot] = (uint8_t)nst;
        if (app && !reid && d2 > d.maha_thr) app = 0;                           // :424-426
        // EMA + bank push for this warp's four matches
        bool go[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) go[u] = __shfl_sync(0xffffffffu, app, u * 8) != 0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (!go[u]) continue;
            float4 f;
            f.x = __fadd_rn(__fmul_rn(d.ema_a, o[u].x), __fmul_rn(d.ema_b, e[u].x));
            f.y = __fadd_rn(__fmul_rn(d.ema_a, o[u].y), __fmul_rn(d.ema_b, e[u].y));
            f.z = __fadd_rn(__fmul_rn(d.ema_a, o[u].z), __fmul_rn(d.ema_b, e[u].z));
            f.w = __fadd_rn(__fmul_rn(d.ema_a, o[u].w), __fmul_rn(d.ema_b, e[u].w));
            reinterpret_cast<float4*>(d.ema + slots[u] * cost::kD)[lane] = cost::unit_row(f);
            int pos;
            if (len[u] < d.HIST) { pos = head[u] + len[u]; if (pos >= d.HIST) pos -= d.HIST; ++len[u]; }
            else { pos = head[u]; head[u] = head[u] + 1 == d.HIST ? 0 : head[u] + 1; }
            reinterpret_cast<float4*>(d.bank + (slots[u] * d.HIST + pos) * cost::kD)[lane] = e[u];
            __syncwarp();
            if (lane == 0) { d.bank_len[slots[u]] = len[u]; d.bank_head[slots[u]] = head[u]; }
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kUpdWarps * 32) update_kernel(Dev d) {
    TRK_PDL_PROLOGUE();
    __shared__ double scratch[kUpdWarps * 4 * 96];
    const int warp = threadIdx.x >> 5;
    update_entries(d, 0, d.wcount[2], blockIdx.x * kUpdWarps + warp, gridDim.x * kUpdWarps, scratch + (size_t)warp * 4 * 96);
}

// create_new_tracks (:362-373) for the detections listed in born[0..want) (already filtered by init_conf_min, in
// order): free slots, Kalman initial state, creat_item (:98-139), ids next_id, next_id + 1, ...  All threads of the
// CTA must call; returns the number of tracks created (fewer than `want` only when the handle is full, which is
// reported as B200_ECAPACITY in the stream's status).
__device__ inline int spawn_tracks(const Dev& d, int s, const int* born, int want) {
    const int tid = threadIdx.x;
    int* hdr = d.hdr + s * kHdr;
    int* cnt = d.cnt + s * kHdr;
    const size_t sb = (size_t)s * d.MT, db = (size_t)s * d.MD;
    const int nl = hdr[H_NLIVE], nfree = hdr[H_NFREE], next_id = hdr[H_NEXT];
    int* order = d.order + sb;
    const int* fl = d.free_list + sb;
    const int nb = min(want, nfree);
    const int frame = d.frame_id[s];
    __syncthreads();
    for (int b = tid; b < nb; b += blockDim.x) {
        const int j = born[b], sl = fl[nfree - 1 - b];
        const size_t slot = sb + sl;
        double x[8], P[64], box[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { box[k] = d.boxes[(db + j) * 4 + k]; d.last_bbox[slot * 4 + k] = box[k]; }
        kf::init_state(box, x, P);
        store_kf(d, slot, x, P);
        d.kf_stage[slot] = 0;
        d.last_conf[slot] = d.confs[db + j];
        d.last_cost[slot] = __longlong_as_double(0x7ff8000000000000LL);      // None
        d.last_frame[slot] = frame;
        d.tid[slot] = next_id + b;
        d.miss[slot] = 0;
        d.age[slot] = 1;
        d.bank_len[slot] = 1;
        d.bank_head[slot] = 0;
        order[nl + b] = sl;
    }
    for (int i = tid; i < nb * (cost::kD / 4); i += blockDim.x) {              // creat_item :98-139
        const int b = i / (cost::kD / 4), k = i % (cost::kD / 4);
        const size_t slot = sb + fl[nfree - 1 - b];
        const float4 e = reinterpret_cast<const float4*>(d.det_unit + (db + born[b]) * cost::kD)[k];
        reinterpret_cast<float4*>(d.ema + slot * cost::kD)[k] = e;
        reinterpret_cast<float4*>(d.bank + slot * d.HIST * cost::kD)[k] = e;
    }
    __syncthreads();
    if (tid == 0) {
        hdr[H_NLIVE] = nl + nb;
        hdr[H_NFREE] = nfree - nb;
        hdr[H_NEXT] = next_id + nb;
        if (want > nb && cnt[C_STATUS] == 0) cnt[C_STATUS] = B200_ECAPACITY;
    }
    __syncthreads();
    return nb;
}

// hungarian_assign (hung.py:5-45) for this stream's matrix; fills m_row/m_det, marks misses.
// Returns the number of matches; *n_unmatched_rows is the count appended to the unmatched list.
// Returns true when stream s has nothing more to do in this step (idle / empty frame / the assignment failed / stage 2
// done).  FUSED (back_kernel): both stages, the ReID cost and the updates of a stream run in ONE CTA, so nothing is queued
// for other kernels and the matches go to the stream's own update queue.
// INLINE: the caller computes the ReID cost itself between the stages (back_kernel) instead of queueing it for
// cost2_kernel; OWNQ: the matches go to the stream's own update queue instead of the step's global one.
template <int STAGE, bool INLINE, bool OWNQ>
__device__ inline bool assign_body(const Dev& d, int s, unsigned char* smem_raw, int smem_matrix_floats) {
    __shared__ int scratch[kThreads / 32];
    __shared__ int s_rc;
    const int tid = threadIdx.x;
    int* cnt = d.cnt + s * kHdr;
    // both cost launches of this step are done: clear their queues for the next step
    if (!INLINE && STAGE == 2 && s == 0 && tid == 0) { d.wcount[0] = 0; d.wcount[1] = 0; }
    int* hdr = d.hdr + s * kHdr;
    int* res = d.result + (size_t)s * d.res_stride;
    if (STAGE == 2 && cnt[C_MODE] == MODE_FAILED) {
        // Stage 1 hit a NaN / infeasible matrix: the reference raises inside hungarian_assign (hung.py:28) before
        // any mark_missed / update_matched / birth / purge, so the stream's state stays "predict only".
        if (tid == 0) put_result_header(res, 0, 0, 0, hdr[H_NLIVE], hdr[H_NEXT], cnt[C_STATUS], cnt[C_M1], cnt[C_M2]);
        return true;
    }
    if (cnt[C_MODE] != MODE_NORMAL) return true;
    const size_t sb = (size_t)s * d.MT, db = (size_t)s * d.MD;
    const int M = STAGE == 1 ? cnt[C_M1] : cnt[C_M2];
    const int N = STAGE == 1 ? d.n_det[s] : cnt[C_NU];
    const int* rows = (STAGE == 1 ? d.rows_main : d.rows_reid) + sb;
    const float* C = (STAGE == 1 ? d.C1 : d.C2) + sb * d.MD;
    const float* CT = (STAGE == 1 ? d.C1T : d.C2T) + db * d.MT;
    const double cmax = STAGE == 1 ? d.cost_max : d.reid_only_cost_max;
    const int match0 = STAGE == 1 ? 0 : cnt[C_NMATCH], ut0 = STAGE == 1 ? 0 : cnt[C_NUT];
    int* out_m = res_matches(d, res);
    int* out_ut = res_ut(d, res);
    int* m_col = d.tmp + sb;                        // column (local det index) of each match
    int n_match = 0, n_ut = 0, n_left = N;
    bool failed = false;                            // uniform across the CTA

    if (M > 0 && N > 0) {
        const bool tall = M > N;
        const int R = tall ? N : M, Cc = tall ? M : N;
        const float* costp = tall ? CT : C;
        const int ld = tall ? d.MT : d.MD;
        const lsap::Work w = lsap::carve(smem_raw, R, Cc);
        float* stage = (size_t)R * Cc <= (size_t)smem_matrix_floats
                           ? reinterpret_cast<float*>(smem_raw + lsap::work_bytes(R, Cc)) : nullptr;
        // stage 1, rows = tracks: the cost kernel has already summarised every row (RowMin)
        const bool pre = STAGE == 1 && !tall;
        const int rc = lsap::solve_block(costp, R, Cc, ld, w, stage, pre ? d.row_fc + sb : nullptr,
                                         pre ? d.row_fv + sb : nullptr);
        if (tid == 0) s_rc = rc;
        __syncthreads();
        if (s_rc != B200_OK) {                      // NaN / infeasible: scipy would raise
            failed = true;
            if (tid == 0) { cnt[C_STATUS] = s_rc; if (STAGE == 1) cnt[C_MODE] = MODE_FAILED; }
        } else {
            const int* col = tall ? w.r4c : w.c4r;  // assigned column of row r (-1: unassigned)
            auto is_match = [&](int r) {
                const int j = col[r];
                return j >= 0 && (double)C[(size_t)r * d.MD + j] <= cmax;      // hung.py:35-40
            };
            n_match = block_compact(M, is_match, [&](int pos, int r) {
                const int jl = col[r], j = STAGE == 1 ? jl : d.ud1[db + jl];
                d.m_row[sb + pos] = r;
                d.m_det[sb + pos] = j;
                m_col[pos] = jl;
                d.det_used[db + j] = 1;
                out_m[2 * (match0 + pos)] = d.tid[sb + rows[r]];
                out_m[2 * (match0 + pos) + 1] = j;
            }, scratch);
            n_ut = block_compact(M, [&](int r) { return !is_match(r); }, [&](int pos, int r) {
                const size_t slot = sb + rows[r];
                d.miss[slot] += 1;                                              // mark_missed :347-355
                out_ut[ut0 + pos] = d.tid[slot];
            }, scratch);
            __syncthreads();
            note_matches(d, s, n_match, rows, C, d.MD, m_col, STAGE == 2, scratch, OWNQ ? (int)sb + match0 : -1);
        }
    } else if (M > 0) {                             // no detections left for these rows: all missed
        for (int r = tid; r < M; r += blockDim.x) {
            const size_t slot = sb + rows[r];
            d.miss[slot] += 1;
            out_ut[ut0 + r] = d.tid[slot];
        }
        n_ut = M;
        __syncthreads();
    }

    if (STAGE == 1) {
        if (failed) {                               // nothing else happens to this stream in this step
            if (tid == 0) { cnt[C_NU] = 0; cnt[C_NMATCH] = 0; cnt[C_NUT] = 0; }
            return true;
        }
        // leftover detections, ascending (hung.py:43)
        n_left = block_compact(N, [&](int j) { return d.det_used[db + j] == 0; },
                               [&](int pos, int j) { d.ud1[db + pos] = j; }, scratch);
        if (tid == 0) { cnt[C_NU] = n_left; cnt[C_NMATCH] = n_match; cnt[C_NUT] = n_ut; }
        if (!INLINE) enqueue_cost_work(d.work2, d.wcount + 1, s, n_left > 0 ? cnt[C_M2] : 0, n_left, scratch);
        __syncthreads();
        return false;
    }

    if (failed) {
        // The ReID-stage assignment raised (:560): stage 1's updates and misses stand, no births, no purge.
        if (tid == 0)
            put_result_header(res, match0, ut0, 0, hdr[H_NLIVE], hdr[H_NEXT], cnt[C_STATUS], cnt[C_M1], cnt[C_M2]);
        return true;
    }
    // ---- stage 2 tail: leftover dets, births (:362-373), purge (:357-360), result table ------------
    int* out_ud = res_ud(d, res);
    n_left = block_compact(N, [&](int jl) { return d.det_used[db + d.ud1[db + jl]] == 0; },
                           [&](int pos, int jl) { out_ud[pos] = d.ud1[db + jl]; }, scratch);
    int* born = d.born + db;                        // det index of each birth, in order
    const int want = block_compact(n_left, [&](int k) { return !(d.confs[db + out_ud[k]] < d.init_conf_min); },
                                   [&](int pos, int k) { born[pos] = out_ud[k]; }, scratch);
    const int nl = hdr[H_NLIVE];
    const int nb = spawn_tracks(d, s, born, want);
    purge(d, s, nl + nb, scratch);
    if (tid == 0)
        put_result_header(res, match0 + n_match, ut0 + n_ut, n_left, hdr[H_NLIVE], hdr[H_NEXT], cnt[C_STATUS], cnt[C_M1],
                          cnt[C_M2]);
    return true;
}

template <int STAGE>
__global__ void __launch_bounds__(kThreads) assign_kernel(Dev d, int smem_matrix_floats) {
    TRK_PDL_PROLOGUE();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    assign_body<STAGE, false, false>(d, blockIdx.x, smem_raw, smem_matrix_floats);
}

// ---- fused step for tracking-sized streams (max_tracks <= 512, max_dets <= 256, hist_max <= 32): two launches ------
// front_kernel (grid G x S, 128 threads): what begin_kernel and the stage-1 cost kernel do, without a kernel boundary
// between them.  Every CTA of a stream derives the stream's row split itself (a block compaction over <= 512 miss
// counters: cheaper than a dependent launch), predicts the tracks whose rows it owns (thread per track) and then runs
// those rows' stage-1 cost, one warp per row, deriving the detection-side inputs (z, float32 box / confidence, unit
// embedding of the few surviving detections) on the fly with the same functions begin_kernel uses.  The CTAs of a stream
// share the detection prep the back kernel needs.
// back_kernel (one CTA of 256 threads per stream): stage-1 assignment and bookkeeping, the ReID-only cost of the
// stream's long-lost rows (usually none), stage-2 assignment, births, purge, result table, and finally the Kalman / EMA
// / bank updates of the stream's own matches.  Streams are independent, so nothing inside waits for another CTA.
// Four warps per front CTA: two or one do not shorten the overlapped 64-stream step (profiles/r02_footprint_sweep.txt,
// builds fw2 / fw1).
constexpr int kFrontWarps = 4;

__global__ void __launch_bounds__(kFrontWarps * 32, 2) front_kernel(Dev d) {
    extern __shared__ __align__(16) int s_rows[];              // rows_main [MT] | rows_reid [MT]
    __shared__ int scratch[kThreads / 32];
    const int s = blockIdx.y, g = blockIdx.x, G = gridDim.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int* cnt = d.cnt + s * kHdr;
    const size_t sb = (size_t)s * d.MT;
    const int n = d.n_det[s], nl = d.hdr[s * kHdr + H_NLIVE];
    const int* order = d.order + sb;
    if (s == 0 && g == 0 && tid == 0) d.wcount[2] = 0;     // three-launch chain: last step's update_kernel is done
    if (step_prologue(d, s, n, nl, g == 0, scratch)) return;
    // ---- rows_main / rows_reid in ascending track-id order (:478-487), in every CTA of the stream ----
    int* rm = s_rows;
    int* rr = s_rows + d.MT;
    const int M1 = block_compact(nl, [&](int i) { return d.miss[sb + order[i]] <= d.lost_reid_after; },
                                 [&](int pos, int i) { rm[pos] = order[i]; }, scratch);
    const int M2 = block_compact(nl, [&](int i) { return d.miss[sb + order[i]] > d.lost_reid_after; },
                                 [&](int pos, int i) { rr[pos] = order[i]; }, scratch);
    if (g == 0) {
        for (int i = tid; i < M1; i += blockDim.x) d.rows_main[sb + i] = rm[i];
        for (int i = tid; i < M2; i += blockDim.x) d.rows_reid[sb + i] = rr[i];
        if (tid == 0) {
            cnt[C_M1] = M1; cnt[C_M2] = M2; cnt[C_NU] = 0; cnt[C_MODE] = MODE_NORMAL;
            cnt[C_NMATCH] = 0; cnt[C_NUT] = 0; cnt[C_STATUS] = 0;
        }
    }
    prep_detections(d, s, n, g, G);
    // ---- predict_all (:340-345): thread per track, the tracks of the rows this CTA owns (r = g, g + G, ...) ----
    const int own1 = M1 > g ? (M1 - g + G - 1) / G : 0, own2 = M2 > g ? (M2 - g + G - 1) / G : 0;
    for (int i = tid; i < own1 + own2; i += blockDim.x)
        predict_slot(d, sb + (i < own1 ? rm[g + i * G] : rr[g + (i - own1) * G]));
    __syncthreads();
    // ---- stage-1 cost of the owned rows, one warp per row ----
    for (int i = warp; i < own1; i += kFrontWarps) {
        const int r = g + i * G;
        cost1_row32<true>(d, s, r, sb + rm[r], n, lane);
    }
}

// Launched as thread-block clusters of kBackCluster CTAs per stream when the handle has few streams (latency mode): CTA 0
// of the cluster runs the serial part (assignments, births, purge, result table) while the others wait at the cluster
// barrier, then all CTAs of the cluster share the stream's Kalman / EMA / bank updates -- 12.5 -> 6 us for 64 matches,
// 23 -> 6 us for 128 (profiles/r02_fused_timeline.txt).  Without the cluster attribute the cluster is the CTA itself.
// Clusters of 2 and of 8 CTAs were measured against 4 and neither was faster (commit 7145e8b; no profile recorded).
constexpr int kBackCluster = 4;

__device__ __forceinline__ unsigned cluster_ctarank() {
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ unsigned cluster_nctarank() {
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {       // release / acquire at cluster scope: CTA 0's global writes are visible
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// UPDATES = false (three-launch chain of stream groups): the same kernel without the update phase -- its matches go to
// the step's global queue and update_kernel, spread over the whole GPU, does the arithmetic; at ~80 registers the CTA then
// fits beside resident ROI Align CTAs, which the 238-register form does not.
template <bool UPDATES>
__global__ void __launch_bounds__(kThreads, UPDATES ? 1 : 2) back_kernel(Dev d, int smem_matrix_floats) {
    TRK_PDL_PROLOGUE();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_idx[cost::kTileN];
    const unsigned rank = cluster_ctarank(), nrank = cluster_nctarank();
    const int s = blockIdx.x / nrank, tid = threadIdx.x;
    const int* cnt = d.cnt + s * kHdr;
    if (rank == 0) {
        if (!assign_body<1, true, UPDATES>(d, s, smem_raw, smem_matrix_floats)) {
            // ReID-only cost (:552-558) of this stream's long-lost rows against the leftover detections
            const int M2 = cnt[C_M2], NU = cnt[C_NU];
            if (M2 > 0 && NU > 0) {
                const int tiles = (NU + cost::kTileN - 1) / cost::kTileN;
                for (int it = 0; it < M2 * tiles; ++it)
                    cost2_item(d, s, it / tiles, (it % tiles) * cost::kTileN, reinterpret_cast<float*>(smem_raw), s_idx);
            }
            __syncthreads();
        }
        assign_body<2, true, UPDATES>(d, s, smem_raw, smem_matrix_floats);
        __syncthreads();
    }
    if (!UPDATES) return;
    if (nrank > 1) cluster_sync_all();
    if (cnt[C_MODE] != MODE_NORMAL) return;        // idle, empty or failed in stage 1: nothing was matched
    // ---- update_matched, arithmetic half, for this stream's own queue (stage 1 then stage 2 entries) ----
    const int total = d.result[(size_t)s * d.res_stride + R_NMATCH];
    const int warp = tid >> 5;
    update_entries(d, (int)((size_t)s * d.MT), total, (int)rank * (kThreads / 32) + warp, (int)nrank * (kThreads / 32),
                   reinterpret_cast<double*>(smem_raw) + (size_t)warp * 4 * 96);
}


// ---- the pieces of Tracking.update as separate operations on one stream of a handle (mainTracking.py:340-448) ----
// One CTA each; they exist so that a caller that drives the association step by step, like the reference's own
// methods allow, finds the same methods on the device state.  The fused step (b200_tracker_step) does not use them.
__device__ inline int find_slot(const Dev& d, int s, int nl, int track_id) {       // live slot of a track id, -1 if none
    const size_t sb = (size_t)s * d.MT;
    int lo = 0, hi = nl - 1;                                                         // `order` is ascending in track id
    while (lo <= hi) {
        const int mid = (lo + hi) >> 1, sl = d.order[sb + mid], t = d.tid[sb + sl];
        if (t == track_id) return sl;
        if (t < track_id) lo = mid + 1; else hi = mid - 1;
    }
    return -1;
}

__global__ void __launch_bounds__(kThreads) op_predict_kernel(Dev d, int s) {        // predict_all :340-345
    const size_t sb = (size_t)s * d.MT;
    const int nl = d.hdr[s * kHdr + H_NLIVE];
    for (int p = threadIdx.x; p < nl; p += blockDim.x) predict_slot(d, sb + d.order[sb + p]);
}

__global__ void __launch_bounds__(kThreads) op_mark_missed_kernel(Dev d, int s, const int* tids, int n) {   // :347-355
    const size_t sb = (size_t)s * d.MT;
    const int nl = d.hdr[s * kHdr + H_NLIVE];
    if (threadIdx.x == 0)                       // serial: the reference increments once per list entry, duplicates included
        for (int i = 0; i < n; ++i) {
            const int sl = find_slot(d, s, nl, tids[i]);
            if (sl >= 0) d.miss[sb + sl] += 1;   // unknown ids are skipped (:350-351)
        }
}

__global__ void __launch_bounds__(kThreads) op_purge_kernel(Dev d, int s) {          // purge_dead :357-360
    __shared__ int scratch[kThreads / 32];
    purge(d, s, d.hdr[s * kHdr + H_NLIVE], scratch);
}

// create_new_tracks (:362-373): det_ids in the caller's order, filtered by init_conf_min; d.boxes / confs / embs hold the
// frame's detections of stream s.  out[0] = tracks created, out[1] = status.
__global__ void __launch_bounds__(kThreads) op_create_kernel(Dev d, int s, const int* det_ids, int n_ids, int n_det, int* out) {
    __shared__ int scratch[kThreads / 32];
    const size_t db = (size_t)s * d.MD;
    if (threadIdx.x == 0) d.cnt[s * kHdr + C_STATUS] = 0;
    prep_detections(d, s, n_det);
    __syncthreads();
    int* born = d.born + db;
    const int want = block_compact(n_ids, [&](int k) { return !(d.confs[db + det_ids[k]] < d.init_conf_min); },
                                   [&](int pos, int k) { born[pos] = det_ids[k]; }, scratch);
    const int nb = spawn_tracks(d, s, born, want);
    if (threadIdx.x == 0) { out[0] = nb; out[1] = d.cnt[s * kHdr + C_STATUS]; }
}

// update_matched (:375-448), bookkeeping half: (track id, detection, cost) triples -> the update queue of update_kernel.
// out[1] = B200_EINVAL if a track id is not live (the reference raises KeyError at :390).
__global__ void __launch_bounds__(kThreads) op_queue_matches_kernel(Dev d, int s, const int* tids, const int* dets,
                                                                     const float* costs, int n, int n_det, int* out) {
    const size_t sb = (size_t)s * d.MT, db = (size_t)s * d.MD;
    const int nl = d.hdr[s * kHdr + H_NLIVE], frame = d.frame_id[s];
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    prep_detections(d, s, n_det);
    __syncthreads();
    for (int q = threadIdx.x; q < n; q += blockDim.x)
        if (find_slot(d, s, nl, tids[q]) < 0 || dets[q] < 0 || dets[q] >= n_det) bad = 1;
    __syncthreads();
    if (bad) {
        if (threadIdx.x == 0) { out[1] = B200_EINVAL; d.wcount[2] = 0; }
        return;
    }
    for (int q = threadIdx.x; q < n; q += blockDim.x) {
        const size_t slot = sb + find_slot(d, s, nl, tids[q]);
        const int j = dets[q];
#pragma unroll
        for (int k = 0; k < 4; ++k) d.last_bbox[slot * 4 + k] = d.boxes[(db + j) * 4 + k];
        d.last_conf[slot] = d.confs[db + j];
        d.last_frame[slot] = frame;
        d.age[slot] += 1;
        d.miss[slot] = 0;
        d.last_cost[slot] = (double)costs[q];
        d.upd_slot[q] = (int)slot;
        d.upd_det[q] = (int)(db + j);
        d.upd_cost[q] = costs[q];
        d.upd_flag[q] = 0;
    }
    if (threadIdx.x == 0) { out[1] = 0; d.wcount[2] = n; }
}

// ---- state images (b200_tracker_state): export / import of any set of streams ------------------------------------------
// One warp per (image row, track): a full 64-stream group of 256 tracks is 16 384 warps.  About 94 % of the bytes are the
// history bank (hist_max x 512 B per track), moved one 512-byte row per warp instruction in 16-byte vectors with
// kRowsInFlight rows of loads issued before their stores.
constexpr int kStateWarps = 8;
constexpr int kRowsInFlight = 6;

// Moves one track between slot `slot` of the handle and track `it` (row * cap + position) of an image.  EXPORT: slot ->
// image, the bank ring unrolled oldest row first and rows past bank_len zeroed (what b200_tracker_export writes); import:
// image -> slot, every bank row in order (the slot's ring then starts at row 0).
template <bool EXPORT>
__device__ __forceinline__ void copy_track(const Dev& d, const b200_tracker_state& im, size_t slot, size_t it, int lane) {
    auto mv = [&](auto* s_side, auto* i_side) { if (EXPORT) *i_side = *s_side; else *s_side = *i_side; };
    const int H = d.HIST;
    const int len = EXPORT ? d.bank_len[slot] : H, head = EXPORT ? d.bank_head[slot] : 0;
    float4* sb = reinterpret_cast<float4*>(d.bank) + slot * H * 32 + lane;
    float4* ib = reinterpret_cast<float4*>(im.bank) + it * H * 32 + lane;
    for (int j0 = 0; j0 < H; j0 += kRowsInFlight) {
        float4 v[kRowsInFlight];
#pragma unroll
        for (int u = 0; u < kRowsInFlight; ++u) {
            const int j = j0 + u;
            const int sr = head + j < H ? head + j : head + j - H;        // slot row of image row j
            v[u] = j < len ? (EXPORT ? sb[(size_t)sr * 32] : ib[(size_t)j * 32]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < kRowsInFlight; ++u)
            if (j0 + u < H) (EXPORT ? ib : sb)[(size_t)(j0 + u) * 32] = v[u];
    }
    // P and ema: 512 B each, one vector per lane; x (64 B) and last_bbox (32 B): lanes 0-5; the scalars: lanes 8-14
    mv(reinterpret_cast<float4*>(d.kf_P) + slot * 32 + lane, reinterpret_cast<float4*>(im.P) + it * 32 + lane);
    mv(reinterpret_cast<float4*>(d.ema) + slot * 32 + lane, reinterpret_cast<float4*>(im.ema) + it * 32 + lane);
    if (lane < 4) mv(reinterpret_cast<float4*>(d.kf_x) + slot * 4 + lane, reinterpret_cast<float4*>(im.x) + it * 4 + lane);
    else if (lane < 6) mv(reinterpret_cast<float4*>(d.last_bbox) + slot * 2 + lane - 4,
                          reinterpret_cast<float4*>(im.last_bbox) + it * 2 + lane - 4);
    switch (lane) {
        case 8: mv(d.tid + slot, im.ids + it); break;
        case 9: mv(d.kf_stage + slot, im.stage + it); break;
        case 10: mv(d.bank_len + slot, im.bank_len + it); break;
        case 11: mv(d.miss + slot, im.miss + it); break;
        case 12: mv(d.age + slot, im.age + it); break;
        case 13: mv(d.last_conf + slot, im.last_conf + it); break;
        case 14: mv(d.last_cost + slot, im.last_cost + it); break;
        default: break;
    }
}

__device__ __forceinline__ int image_stream(const int* streams, int s0, int r) { return streams ? streams[r] : s0 + r; }

// grid (ceil(cap / kStateWarps), n_rows).  Row r is stream streams[r] (streams == nullptr: s0 + r); b200_tracker_export
// runs it as a one-row image over its staging buffer.
__global__ void __launch_bounds__(kStateWarps * 32) export_state_kernel(Dev d, b200_tracker_state im, const int* streams,
                                                                         int s0, int* status) {
    const int r = blockIdx.y;
    const int s = image_stream(streams, s0, r);
    const bool in_range = s >= 0 && s < d.S;
    const int nl = in_range ? d.hdr[s * kHdr + H_NLIVE] : 0;
    const bool ok = in_range && nl <= im.cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (status) status[r] = !in_range ? B200_EINVAL : ok ? B200_OK : B200_ECAPACITY;
        if (ok) { im.n_live[r] = nl; im.next_id[r] = d.hdr[s * kHdr + H_NEXT]; }
    }
    const int p = blockIdx.x * kStateWarps + (threadIdx.x >> 5);
    if (!ok || p >= nl) return;
    const size_t sb = (size_t)s * d.MT;
    copy_track<true>(d, im, sb + d.order[sb + p], (size_t)r * im.cap + p, threadIdx.x & 31);
}

// The slot layout an import leaves in stream s (all threads of the CTA): tracks in slots 0..n-1 in id order, their bank
// rings at row 0, free list MT-1 ... n, header counts.
__device__ void finish_import(const Dev& d, int s, int n, int next_id) {
    const size_t sb = (size_t)s * d.MT;
    for (int i = threadIdx.x; i < d.MT; i += blockDim.x) {
        if (i < n) { d.order[sb + i] = i; d.bank_head[sb + i] = 0; d.last_frame[sb + i] = 0; }
        if (i < d.MT - n) d.free_list[sb + i] = d.MT - 1 - i;
    }
    if (threadIdx.x == 0) {
        d.hdr[s * kHdr + H_NLIVE] = n;
        d.hdr[s * kHdr + H_NEXT] = next_id;
        d.hdr[s * kHdr + H_NFREE] = d.MT - n;
    }
}

// One CTA per image row, ahead of import_state_kernel: validates the row (every index it reads is checked first) and, if it
// passes, rebuilds the stream's header, order and free list.  imp_row[s] = r names the row import_state_kernel copies into
// stream s (-1: none); only entries of streams named by this image are read, and each is written here first.  Streams as
// in export_state_kernel; b200_tracker_import runs both kernels on a one-row image of its host arrays.
__global__ void __launch_bounds__(kThreads) import_check_kernel(Dev d, b200_tracker_state im, const int* streams, int s0,
                                                                 int* imp_row, int* status) {
    const int r = blockIdx.x;
    const int s = image_stream(streams, s0, r);
    if (s < 0 || s >= d.S) {
        if (status && threadIdx.x == 0) status[r] = B200_EINVAL;
        return;
    }
    bool dup = false;                                // another row naming the same stream: neither is applied
    if (streams)
        for (int q = threadIdx.x; q < im.n_rows; q += blockDim.x) dup |= q != r && streams[q] == s;
    const int n = im.n_live[r], next_id = im.next_id[r];
    int st = __syncthreads_or(dup) || n < 0 ? B200_EINVAL
             : n > (im.cap < d.MT ? im.cap : d.MT) ? B200_ECAPACITY : B200_OK;
    if (st == B200_OK) {
        const size_t rb = (size_t)r * im.cap;
        bool bad = false;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const int id = im.ids[rb + i], bl = im.bank_len[rb + i];
            bad |= id < 0 || id >= next_id || (i > 0 && im.ids[rb + i - 1] >= id) || bl < 0 || bl > d.HIST ||
                   im.stage[rb + i] > 2;
        }
        if (__syncthreads_or(bad)) st = B200_EINVAL;
    }
    if (st == B200_OK) finish_import(d, s, n, next_id);
    if (threadIdx.x == 0) {
        imp_row[s] = st == B200_OK ? r : -1;
        if (status) status[r] = st;
    }
}

// grid (ceil(cap / kStateWarps), n_rows): copies the rows import_check_kernel accepted into slots 0..n-1 of their streams.
__global__ void __launch_bounds__(kStateWarps * 32) import_state_kernel(Dev d, b200_tracker_state im, const int* streams,
                                                                         int s0, const int* imp_row) {
    const int r = blockIdx.y;
    const int s = image_stream(streams, s0, r);
    if (s < 0 || s >= d.S || imp_row[s] != r) return;
    const int p = blockIdx.x * kStateWarps + (threadIdx.x >> 5);
    if (p >= im.n_live[r]) return;
    copy_track<false>(d, im, (size_t)s * d.MT + p, (size_t)r * im.cap + p, threadIdx.x & 31);
}

__global__ void reset_kernel(Dev d) {
    const int s = blockIdx.x;
    for (int i = threadIdx.x; i < d.MT; i += blockDim.x) d.free_list[(size_t)s * d.MT + i] = d.MT - 1 - i;
    if (threadIdx.x == 0) {
        d.hdr[s * kHdr + H_NLIVE] = 0;
        d.hdr[s * kHdr + H_NEXT] = 0;
        d.hdr[s * kHdr + H_NFREE] = d.MT;
        if (s == 0) { d.wcount[0] = 0; d.wcount[1] = 0; d.wcount[2] = 0; }
    }
}

// ---- b200_tracker_step_packed: detections in the detector's / encoder's layout -> the step's padded per-stream layout ----
// pack_kernel (one CTA per stream) selects the stream's detections in input order with block_compact, widens them into the
// handle's packed-input block, writes n_det and sets every track_of_det entry to -1; b200_tracker_step runs on that block;
// finish_kernel (one CTA per stream) reports overflowing streams and writes the track id of every match of the result table
// to the input row of its (stream, det_idx).  Each pack CTA walks all K stream indices (one ballot round per 1 024 rows), so
// the CTA is as wide as possible: the walk is a chain of dependent rounds, not a bandwidth cost.
struct Packed {
    int S, MD, K, box_stride, conf_stride, det_half, emb_half;
    const void *boxes, *confs, *embs;
    const int *stream_index, *active;
    // the handle's packed-input block
    int* n_det;
    double *p_boxes, *p_confs;
    float* p_embs;
    int* inv;                         // [S, MD] input row k of det_idx j of stream s
    int* over;                        // [S] 1 = the stream had more than MD detections and was not stepped
    int* track_of_det;                // [K] or null
};

constexpr int kPackThreads = 1024;

__device__ __forceinline__ int stream_of(const Packed& p, int k) { return p.stream_index ? p.stream_index[k] : 0; }

__device__ __forceinline__ double widen(const void* base, size_t i, int half) {      // exact: f16 -> f32 -> f64
    return half ? (double)__half2float(static_cast<const __half*>(base)[i]) : (double)static_cast<const float*>(base)[i];
}

__global__ void __launch_bounds__(kPackThreads) pack_kernel(Packed p) {
    __shared__ int scratch[kPackThreads / 32];
    const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t db = (size_t)s * p.MD;
    if (p.track_of_det)                              // finish_kernel overwrites the matched entries after the step
        for (int k = s * kPackThreads + threadIdx.x; k < p.K; k += p.S * kPackThreads) p.track_of_det[k] = -1;
    const bool on = p.active == nullptr || p.active[s] != 0;
    int n = 0;
    if (on)
        n = block_compact(p.K, [&](int k) { return stream_of(p, k) == s; }, [&](int j, int k) {
            if (j >= p.MD) return;
            p.inv[db + j] = k;
#pragma unroll
            for (int c = 0; c < 4; ++c) p.p_boxes[(db + j) * 4 + c] = widen(p.boxes, (size_t)k * p.box_stride + c, p.det_half);
            p.p_confs[db + j] = widen(p.confs, (size_t)k * p.conf_stride, p.det_half);
        }, scratch);
    const bool over = n > p.MD;
    if (threadIdx.x == 0) { p.n_det[s] = on && !over ? n : -1; p.over[s] = over ? 1 : 0; }
    if (!on || over) return;                         // uniform across the CTA
    __syncthreads();                                 // inv[] of this stream is complete
    for (int j = warp; j < n; j += kPackThreads / 32) {   // one warp per embedding row, four elements per lane
        const size_t k = (size_t)p.inv[db + j];
        float4 v;
        if (p.emb_half) {
            const uint2 raw = reinterpret_cast<const uint2*>(static_cast<const __half*>(p.embs) + k * cost::kD)[lane];
            const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
            const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
            v = make_float4(a.x, a.y, b.x, b.y);
        } else {
            v = reinterpret_cast<const float4*>(static_cast<const float*>(p.embs) + k * cost::kD)[lane];
        }
        reinterpret_cast<float4*>(p.p_embs + (db + j) * cost::kD)[lane] = v;
    }
}

__global__ void __launch_bounds__(kThreads) finish_kernel(Packed p, int* result, int res_stride) {
    const int s = blockIdx.x;
    int* res = result + (size_t)s * res_stride;
    if (threadIdx.x == 0 && p.over[s]) res[R_STATUS] = B200_ECAPACITY;
    if (p.track_of_det == nullptr) return;
    // the matched rows (an idle, overflowing or failed stream has none in its row); every other entry is pack_kernel's -1
    const int nm = res[R_NMATCH];
    const int* m = res + R_HDR;
    for (int i = threadIdx.x; i < nm; i += blockDim.x) p.track_of_det[p.inv[(size_t)s * p.MD + m[2 * i + 1]]] = m[2 * i];
}

// ---- host-side buffer layouts ----------------------------------------------------------------------------------------
// Lays buffers out one after another at 256-byte aligned offsets from `base`.  With base = nullptr it only measures: the
// fields receive offsets and `off` ends as the size of the layout.
struct Carver {
    char* base = nullptr;
    size_t off = 0;
    static size_t aligned(size_t n) { return (n + 255) & ~(size_t)255; }
    template <typename T> void take(T*& field, size_t n) {
        off = aligned(off);
        field = reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(base) + off);
        off += n * sizeof(T);
    }
};

// One step's inputs in the padded per-stream layout b200_tracker_step reads.
struct StepInputs {
    int* n_det;
    int* frame;
    double* boxes;
    double* confs;
    float* embs;
};

// The inputs of S streams of MD detections as one contiguous range, so that a host step uploads them with a single copy.
inline void take_inputs(Carver& c, StepInputs& in, size_t S, size_t MD) {
    c.take(in.n_det, S);
    c.take(in.frame, S);
    c.take(in.boxes, S * MD * 4);
    c.take(in.confs, S * MD);
    c.take(in.embs, S * MD * 128);
}

// One slot of the host-step ring, pinned or device (the two sides share the layout): the step's inputs, then its result
// table.
struct Slot {
    StepInputs in;
    size_t in_bytes;                  // the inputs: one range from the slot's base
    int* result;
    size_t bytes;                     // the whole slot
    Slot(void* base, const Dev& d) {
        Carver c{static_cast<char*>(base)};
        take_inputs(c, in, d.S, d.MD);
        in_bytes = c.off;
        c.take(result, (size_t)d.S * d.res_stride);
        bytes = Carver::aligned(c.off);
    }
};

}  // namespace trk
}  // namespace b200

using namespace b200;

struct b200_tracker {
    trk::Dev d;
    void* arena = nullptr;          // one device allocation holding state + scratch + inputs + result
    static constexpr int kRing = 4;  // host staging slots: step_host_async may run this many steps ahead of their results
    void* pinned = nullptr;         // host staging: kRing x trk::Slot
    size_t res_bytes = 0, slot_bytes = 0;
    cudaEvent_t done[kRing] = {};   // result of the step staged in slot i is on the host
    // Device side of the ring (inputs then result per slot, same layout as a pinned slot) and two private streams: the
    // upload of step k+1 and the download of step k's result run beside the kernels of step k instead of in line with
    // them (a DMA queued between kernels costs ~20 us of engine hand-over each: 292 -> 120 us per pipelined 64-stream step).
    void* ring_dev = nullptr;
    cudaStream_t up_stream = nullptr, down_stream = nullptr;
    cudaEvent_t up[kRing] = {}, ran[kRing] = {};
    long long ticket_of[kRing] = {-1, -1, -1, -1};
    long long next_ticket = 0;
    trk::StepInputs in = {};        // inputs of the step-by-step operations
    int* dev_result = nullptr;
    // input block of b200_tracker_step_packed (its frame ids are the caller's), separate from `in` and the ring so that a
    // packed step queued on one stream never races with a host step or a step-by-step operation queued on another
    trk::StepInputs pk = {};
    int* pk_inv = nullptr; int* pk_over = nullptr;
    int* imp_row = nullptr;         // [S] import_check_kernel: the image row accepted for each stream
    int cost_grid = 0, cost1_grid = 0, upd_grid = 0;   // persistent CTAs of the cost kernels (resident CTAs per SM x SMs)
    size_t assign_smem = 0;
    int smem_matrix_floats = 0;
    // tracking-sized streams: 2 = front_kernel + back_kernel (a few streams, latency mode), 3 = front_kernel + back_kernel
    // without updates + update_kernel (stream groups), 6 = the six-kernel chain (any size)
    int chain = 6;
    int front_resident = 0;             // CTAs of front_kernel the device holds at once
    size_t front_smem = 0, back_smem = 0;
};

extern "C" int b200_tracker_create(b200_tracker** out, int n_streams, int max_tracks, int max_dets,
                                   const b200_tracker_conf* conf) {
    B200_REQUIRE(out && conf, "tracker_create: null pointer");
    B200_REQUIRE(n_streams >= 1 && n_streams <= 65535, "tracker_create: n_streams %d out of range", n_streams);
    B200_REQUIRE(max_tracks >= 1 && max_tracks <= 4096 && max_dets >= 1 && max_dets <= 4096 && n_streams * (long long)max_tracks < (1 << 25),
                 "tracker_create: capacities out of range (tracks %d, dets %d)", max_tracks, max_dets);
    B200_REQUIRE(conf->hist_max >= 1 && conf->hist_max <= cost::kMaxBank, "tracker_create: hist_max %d outside [1,%d]",
                 conf->hist_max, cost::kMaxBank);
    B200_REQUIRE(conf->emb_top_k >= 1, "tracker_create: emb_top_k must be >= 1");
    b200_tracker* t = new (std::nothrow) b200_tracker();
    B200_REQUIRE(t, "tracker_create: out of host memory");
    trk::Dev& d = t->d;
    memset(&d, 0, sizeof(d));
    const size_t S = n_streams, MT = max_tracks, MD = max_dets, H = conf->hist_max;
    d.S = n_streams; d.MT = max_tracks; d.MD = max_dets; d.HIST = conf->hist_max;
    d.res_stride = trk::R_HDR + 2 * max_dets + max_tracks + max_dets;
    const size_t tiles_max = (MD + cost::kTileN - 1) / cost::kTileN;
    auto carve_arena = [&](trk::Carver& c) {
        c.take(d.kf_x, S * MT * 8); c.take(d.kf_P, S * MT * 64); c.take(d.last_bbox, S * MT * 4);
        c.take(d.last_conf, S * MT); c.take(d.last_cost, S * MT); c.take(d.kf_stage, S * MT);
        c.take(d.ema, S * MT * 128); c.take(d.bank, S * MT * H * 128);
        c.take(d.bank_len, S * MT); c.take(d.bank_head, S * MT); c.take(d.tid, S * MT); c.take(d.miss, S * MT);
        c.take(d.age, S * MT); c.take(d.last_frame, S * MT); c.take(d.order, S * MT); c.take(d.free_list, S * MT);
        c.take(d.hdr, S * trk::kHdr);
        c.take(d.det_unit, S * MD * 128); c.take(d.det_z, S * MD * 4); c.take(d.det_boxf, S * MD * 4);
        c.take(d.det_conff, S * MD); c.take(d.prev_boxf, S * MT * 4); c.take(d.prev_conff, S * MT);
        c.take(d.C1, S * MT * MD); c.take(d.C1T, S * MT * MD); c.take(d.C2, S * MT * MD);
        c.take(d.C2T, S * MT * MD); c.take(d.gate_SI, S * MT * 16);
        c.take(d.row_fc, S * MT); c.take(d.row_fv, S * MT);
        c.take(d.rows_main, S * MT); c.take(d.rows_reid, S * MT); c.take(d.cnt, S * trk::kHdr);
        c.take(d.ud1, S * MD); c.take(d.det_used, S * MD); c.take(d.m_row, S * MT); c.take(d.m_det, S * MT);
        c.take(d.tmp, S * MT); c.take(d.born, S * MD);
        c.take(d.work1, S * MT * tiles_max); c.take(d.work2, S * MT * tiles_max); c.take(d.wcount, 4);
        c.take(d.upd_slot, S * MT); c.take(d.upd_det, S * MT); c.take(d.upd_cost, S * MT); c.take(d.upd_flag, S * MT);
        trk::take_inputs(c, t->in, S, MD);
        c.take(t->dev_result, S * (size_t)d.res_stride);
        trk::take_inputs(c, t->pk, S, MD);
        c.take(t->pk_inv, S * MD); c.take(t->pk_over, S);
        c.take(t->imp_row, S);
    };
    trk::Carver size;
    carve_arena(size);
    cudaError_t e = cudaMalloc(&t->arena, size.off);
    if (e != cudaSuccess) {
        delete t;
        return fail(B200_ECUDA, "tracker_create: cudaMalloc(%zu bytes): %s", size.off, cudaGetErrorString(e));
    }
    trk::Carver c{static_cast<char*>(t->arena)};
    carve_arena(c);
    cudaMemset(t->arena, 0, c.off);
    t->res_bytes = S * (size_t)d.res_stride * sizeof(int);
    t->slot_bytes = trk::Slot(nullptr, d).bytes;
    e = cudaMallocHost(&t->pinned, t->slot_bytes * b200_tracker::kRing);
    if (e == cudaSuccess) e = cudaMalloc(&t->ring_dev, t->slot_bytes * b200_tracker::kRing);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&t->up_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&t->down_stream, cudaStreamNonBlocking);
    for (int i = 0; e == cudaSuccess && i < b200_tracker::kRing; ++i) {
        e = cudaEventCreateWithFlags(&t->done[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->up[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&t->ran[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
        b200_tracker_destroy(t);
        return fail(B200_ECUDA, "tracker_create: host ring / streams: %s", cudaGetErrorString(e));
    }
    d.pw = cost::PairWeights{(float)conf->w_app, (float)conf->w_bbox, (float)conf->w_conf, (float)conf->alpha,
                             (float)conf->beta, 1e-6f};
    d.maha_thr = conf->maha_thr; d.cost_max = conf->cost_max; d.conf_update_min = conf->conf_update_min;
    d.cost_update_max = conf->cost_update_max; d.reid_only_cost_max = conf->reid_only_cost_max;
    d.init_conf_min = conf->init_conf_min;
    d.ema_a = (float)conf->ema_alpha;
    d.ema_b = (float)(1.0 - conf->ema_alpha);
    d.topk = conf->emb_top_k; d.max_age = conf->max_age; d.lost_reid_after = conf->lost_reid_after;
    // shared memory of the assignment kernels: LSAP work arrays + the matrix when it fits
    const int Rm = max_tracks < max_dets ? max_tracks : max_dets, Cm = max_tracks < max_dets ? max_dets : max_tracks;
    const size_t wb = lsap::work_bytes(Rm, Cm), budget = 200 * 1024;
    if (wb > budget) {
        b200_tracker_destroy(t);
        return fail(B200_EINVAL, "tracker_create: %d x %d exceeds the assignment kernel's shared memory", max_tracks, max_dets);
    }
    size_t mat = (size_t)Rm * Cm * sizeof(float);
    if (wb + mat > budget) mat = budget - wb;
    // Small problems (the tracking shapes) keep the shared-memory footprint of the assignment kernels modest
    // so that they can share an SM with resident ROI Align CTAs.
    // (A frame's actual matrix is live tracks x detections, not the capacities; one that does not fit is read from global.)
    if (max_tracks <= 1024 && max_dets <= 256 && mat > 32 * 1024) mat = 32 * 1024;
    t->smem_matrix_floats = (int)(mat / sizeof(float));
    t->assign_smem = wb + mat;
    // The opt-in belongs to the kernel function (per device), not to this handle: always the full budget, so
    // handles of different capacities can be stepped in any order.
    cudaFuncSetAttribute(trk::assign_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget);
    cudaFuncSetAttribute(trk::assign_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget);
    cudaFuncSetAttribute(trk::cost2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cost::smem_bytes(cost::kMaxBank));
    trk::reset_kernel<<<n_streams, 128>>>(d);
    e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        b200_tracker_destroy(t);
        return fail(B200_ECUDA, "tracker_create: %s", cudaGetErrorString(e));
    }
    g_launches.fetch_add(1);
    {
        int per_sm = 1, sms = kSMs, devid = 0;
        cudaGetDevice(&devid);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, devid);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trk::cost2_kernel, cost::kThreads,
                                                      cost::smem_bytes(d.HIST));
        t->cost_grid = sms * (per_sm > 0 ? per_sm : 1);
        per_sm = 1;
        if (d.HIST <= 32)
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trk::cost1_sparse32_kernel, trk::kCost1Warps * 32, 0);
        else
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trk::cost1_sparse_kernel, trk::kCost1Warps * 32, 0);
        t->cost1_grid = sms * (per_sm > 0 ? per_sm : 1);
        t->upd_grid = sms * 2;
        // Fewer, fatter launches for tracking-sized streams.  Two launches for a handful of streams (latency mode: one
        // stream 43.5 -> 35.8 us per frame).  With a stream group the chain shares the GPU with ROI Align of the next frame,
        // where every kernel boundary costs 25-40 us of waiting for SM slots and a CTA that needs a whole SM (back_kernel
        // with the updates: 238 registers x 256 threads) waits longest (two launches: chain alone 68 -> 59 us but the
        // overlapped step 232 -> 273 us), so groups use three launches: front, back without updates (80 registers), and
        // the update kernel spread over the GPU.  B200TRACK_CHAIN=2|3|6 forces a path (tests, experiments).
        const bool fits = max_tracks <= 512 && max_dets <= 256 && d.HIST <= 32;
        t->chain = !fits ? 6 : n_streams <= 8 ? 2 : 3;
        if (const char* e = getenv("B200TRACK_CHAIN")) {
            const int want = atoi(e);
            if (want == 6 || (fits && (want == 2 || want == 3))) t->chain = want;
        }
        if (t->chain != 6) {
            t->front_smem = sizeof(int) * 2 * (size_t)max_tracks;
            size_t bs = t->assign_smem;
            if (cost::smem_bytes(d.HIST) > bs) bs = cost::smem_bytes(d.HIST);
            if (sizeof(double) * (trk::kThreads / 32) * 4 * 96 > bs) bs = sizeof(double) * (trk::kThreads / 32) * 4 * 96;
            t->back_smem = bs;
            cudaFuncSetAttribute(trk::back_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget);
            cudaFuncSetAttribute(trk::back_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget);
            per_sm = 1;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trk::front_kernel, trk::kFrontWarps * 32, t->front_smem);
            t->front_resident = sms * (per_sm > 0 ? per_sm : 1);
        }
    }
    *out = t;
    return B200_OK;
}

extern "C" void b200_tracker_destroy(b200_tracker* t) {
    if (!t) return;
    if (t->up_stream) { cudaStreamSynchronize(t->up_stream); cudaStreamDestroy(t->up_stream); }
    if (t->down_stream) { cudaStreamSynchronize(t->down_stream); cudaStreamDestroy(t->down_stream); }
    for (int i = 0; i < b200_tracker::kRing; ++i) {
        if (t->done[i]) cudaEventDestroy(t->done[i]);
        if (t->up[i]) cudaEventDestroy(t->up[i]);
        if (t->ran[i]) cudaEventDestroy(t->ran[i]);
    }
    cudaFreeHost(t->pinned);
    cudaFree(t->ring_dev);
    cudaFree(t->arena);
    delete t;
}

extern "C" int b200_tracker_reset(b200_tracker* t, void* stream) {
    B200_REQUIRE(t, "tracker_reset: null handle");
    trk::reset_kernel<<<t->d.S, 128, 0, as_stream(stream)>>>(t->d);
    return check_launch("reset_kernel");
}

extern "C" int b200_tracker_result_stride(const b200_tracker* t) { return t ? t->d.res_stride : 0; }

extern "C" int b200_tracker_live_counts(b200_tracker* t, int32_t* n_live_host, int32_t* next_id_host, void* stream) {
    B200_REQUIRE(t, "tracker_live_counts: null handle");
    cudaStream_t st = as_stream(stream);
    const int S = t->d.S;
    int* h = static_cast<int*>(malloc(sizeof(int) * trk::kHdr * (size_t)S));
    B200_REQUIRE(h, "tracker_live_counts: out of host memory");
    cudaError_t e = cudaMemcpyAsync(h, t->d.hdr, sizeof(int) * trk::kHdr * (size_t)S, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        free(h);
        return fail(B200_ECUDA, "tracker_live_counts: %s", cudaGetErrorString(e));
    }
    for (int s = 0; s < S; ++s) {
        if (n_live_host) n_live_host[s] = h[s * trk::kHdr + trk::H_NLIVE];
        if (next_id_host) next_id_host[s] = h[s * trk::kHdr + trk::H_NEXT];
    }
    free(h);
    return B200_OK;
}

extern "C" int b200_tracker_step(b200_tracker* t, const int32_t* n_det, const double* boxes, const double* confs,
                                 const float* embs, const int32_t* frame_id, int32_t* result, void* stream) {
    B200_REQUIRE(t && n_det && boxes && confs && embs && frame_id && result, "tracker_step: null pointer");
    cudaStream_t st = as_stream(stream);
    trk::Dev d = t->d;
    d.n_det = n_det; d.boxes = boxes; d.confs = confs; d.embs = embs; d.frame_id = frame_id; d.result = result;
    const size_t csm = cost::smem_bytes(d.HIST);
    const int cost_grid = t->cost_grid;
    int rc;
    if (t->chain != 6) {
        // CTAs per stream of the front kernel: fill the device once, never more than one CTA per four rows
        int G = t->front_resident / d.S;
        const int gmax = (d.MT + 3) / 4;
        G = G < 1 ? 1 : G > gmax ? gmax : G;
        trk::front_kernel<<<dim3(G, d.S), trk::kFrontWarps * 32, t->front_smem, st>>>(d);
        if ((rc = check_launch("trk front_kernel"))) return rc;
        if (t->chain == 3) {
            trk::back_kernel<false><<<d.S, trk::kThreads, t->assign_smem > cost::smem_bytes(d.HIST) ? t->assign_smem
                                                                                                    : cost::smem_bytes(d.HIST), st>>>(
                d, t->smem_matrix_floats);
            if ((rc = check_launch("trk back_kernel<false>"))) return rc;
            trk::update_kernel<<<t->upd_grid, trk::kUpdWarps * 32, 0, st>>>(d);
            return check_launch("trk update_kernel");
        }
        // few streams: a cluster of CTAs per stream shares the updates, and the kernel is resident when the front one ends
        const bool few = d.S <= 8;
        const int cl = few ? trk::kBackCluster : 1;
        launch_ex(trk::back_kernel<true>, dim3(d.S * cl), dim3(trk::kThreads), t->back_smem, st, few, few ? cl : 0, d,
                  t->smem_matrix_floats);
        return check_launch("trk back_kernel");
    }
    trk::begin_kernel<<<dim3(d.S, 2), trk::kThreads, 0, st>>>(d);
    rc = check_launch("trk begin_kernel");
    if (rc) return rc;
    // With a handful of streams the step is a chain of short, latency-bound kernels: launch the dependent ones
    // with programmatic stream serialisation so that each is resident (and past its launch latency) by the
    // time its predecessor finishes.  With many streams the chain shares the GPU with ROI Align of the next
    // frame and early-resident CTAs would only take SM slots away from it.
    const bool pdl = d.S <= 8;
    const dim3 c1_grid(t->cost1_grid), c1_block(trk::kCost1Warps * 32);
    if (d.HIST <= 32) launch_ex(trk::cost1_sparse32_kernel, c1_grid, c1_block, 0, st, pdl, 0, d);
    else launch_ex(trk::cost1_sparse_kernel, c1_grid, c1_block, 0, st, pdl, 0, d);
    if ((rc = check_launch("trk cost1_sparse_kernel"))) return rc;
    launch_ex(trk::assign_kernel<1>, dim3(d.S), dim3(trk::kThreads), t->assign_smem, st, pdl, 0, d, t->smem_matrix_floats);
    if ((rc = check_launch("trk assign_kernel<1>"))) return rc;
    launch_ex(trk::cost2_kernel, dim3(cost_grid), dim3(cost::kThreads), csm, st, pdl, 0, d);
    if ((rc = check_launch("trk cost2_kernel"))) return rc;
    launch_ex(trk::assign_kernel<2>, dim3(d.S), dim3(trk::kThreads), t->assign_smem, st, pdl, 0, d, t->smem_matrix_floats);
    if ((rc = check_launch("trk assign_kernel<2>"))) return rc;
    launch_ex(trk::update_kernel, dim3(t->upd_grid), dim3(trk::kUpdWarps * 32), 0, st, pdl, 0, d);
    if ((rc = check_launch("trk update_kernel"))) return rc;
    return B200_OK;
}

extern "C" int b200_tracker_step_packed(b200_tracker* t, int64_t K, const void* boxes, int box_stride, const void* confs,
                                        int conf_stride, int det_dtype, const void* embs, int emb_dtype,
                                        const int32_t* stream_index, const int32_t* active, const int32_t* frame_id,
                                        int32_t* result, int32_t* track_of_det, void* stream) {
    B200_REQUIRE(t, "tracker_step_packed: null handle");
    B200_REQUIRE(K >= 0 && K <= 0x7fffffff, "tracker_step_packed: K = %lld out of range", (long long)K);
    B200_REQUIRE(box_stride >= 4, "tracker_step_packed: box_stride %d < 4", box_stride);
    B200_REQUIRE(conf_stride >= 1, "tracker_step_packed: conf_stride %d < 1", conf_stride);
    B200_REQUIRE(det_dtype == B200_DTYPE_F32 || det_dtype == B200_DTYPE_F16, "tracker_step_packed: unknown det_dtype %d", det_dtype);
    B200_REQUIRE(emb_dtype == B200_DTYPE_F32 || emb_dtype == B200_DTYPE_F16, "tracker_step_packed: unknown emb_dtype %d", emb_dtype);
    B200_REQUIRE(frame_id, "tracker_step_packed: null frame_id");
    B200_REQUIRE(result, "tracker_step_packed: null result");
    if (K > 0) {
        B200_REQUIRE(boxes, "tracker_step_packed: null boxes");
        B200_REQUIRE(confs, "tracker_step_packed: null confs");
        B200_REQUIRE(embs, "tracker_step_packed: null embs");
        B200_REQUIRE(reinterpret_cast<uintptr_t>(embs) % (emb_dtype == B200_DTYPE_F32 ? 16 : 8) == 0,
                     "tracker_step_packed: embs must be %d-byte aligned", emb_dtype == B200_DTYPE_F32 ? 16 : 8);
    }
    cudaStream_t st = as_stream(stream);
    trk::Packed p;
    p.S = t->d.S; p.MD = t->d.MD; p.K = (int)K; p.box_stride = box_stride; p.conf_stride = conf_stride;
    p.det_half = det_dtype == B200_DTYPE_F16; p.emb_half = emb_dtype == B200_DTYPE_F16;
    p.boxes = boxes; p.confs = confs; p.embs = embs; p.stream_index = stream_index; p.active = active;
    const trk::StepInputs& in = t->pk;
    p.n_det = in.n_det; p.p_boxes = in.boxes; p.p_confs = in.confs; p.p_embs = in.embs;
    p.inv = t->pk_inv; p.over = t->pk_over; p.track_of_det = track_of_det;
    trk::pack_kernel<<<p.S, trk::kPackThreads, 0, st>>>(p);
    int rc = check_launch("trk pack_kernel");
    if (rc) return rc;
    if ((rc = b200_tracker_step(t, in.n_det, in.boxes, in.confs, in.embs, frame_id, result, stream))) return rc;
    trk::finish_kernel<<<p.S, trk::kThreads, 0, st>>>(p, result, t->d.res_stride);
    return check_launch("trk finish_kernel");
}

// Host-buffer step, asynchronous: stages the detections in the next slot of a pinned ring, uploads them into the slot's
// device block on the handle's upload stream, runs the step's kernels on `stream` (which waits for that upload), downloads
// the result table on the handle's download stream, records the slot's event and returns a ticket.
// b200_tracker_step_result waits for that event only.  Up to kRing steps may be in flight; taking a slot whose result was
// never collected first waits for it (its result is then lost to the caller).
// direct = the caller's arrays are page-locked and stay untouched until the result is collected: they are read by DMA
// straight from where they are (no staging memcpy, which at 64 streams x 64 detections is 2.3 MB = most of the host time).
namespace {
// inline_dma (the synchronous b200_tracker_step_host): nothing can overlap anyway, so the copies go on the caller's stream
// as well and the cross-stream event hops are saved.
int step_host_submit(b200_tracker* t, const int32_t* n_det_host, const double* boxes_host, const double* confs_host,
                     const float* embs_host, const int32_t* frame_id_host, int64_t* ticket, void* stream, bool direct,
                     bool inline_dma = false) {
    B200_REQUIRE(t && n_det_host && frame_id_host && ticket, "tracker_step_host_async: null pointer");
    cudaStream_t st = as_stream(stream);
    const trk::Dev& d = t->d;
    const int slot = (int)(t->next_ticket % b200_tracker::kRing);
    if (t->ticket_of[slot] >= 0) B200_CUDA(cudaEventSynchronize(t->done[slot]));      // the DMA that last used this slot
    char* pin = static_cast<char*>(t->pinned) + (size_t)slot * t->slot_bytes;
    char* dslot = static_cast<char*>(t->ring_dev) + (size_t)slot * t->slot_bytes;
    const trk::Slot hs(pin, d), ds(dslot, d);
    const trk::StepInputs& h = hs.in;
    const trk::StepInputs& dv = ds.in;
    bool dense = true;                               // every stream full: three large copies instead of 3 S small ones
    int n_max = 0;
    for (int s = 0; s < d.S; ++s) {
        const int n = n_det_host[s];
        B200_REQUIRE(n <= d.MD, "tracker_step_host: stream %d has %d detections, capacity %d", s, n, d.MD);
        h.n_det[s] = n;
        h.frame[s] = frame_id_host[s];
        if (n != d.MD) dense = false;
        if (n > n_max) n_max = n;
        if (n > 0) B200_REQUIRE(boxes_host && confs_host && embs_host, "tracker_step_host: null detection arrays");
    }
    cudaStream_t up = inline_dma ? st : t->up_stream, down = inline_dma ? st : t->down_stream;
    if (direct) {
        const void* arrs[3] = {boxes_host, confs_host, embs_host};
        for (int k = 0; k < 3 && n_max > 0; ++k) {
            cudaPointerAttributes pa = {};
            const cudaError_t e = cudaPointerGetAttributes(&pa, arrs[k]);
            if (e != cudaSuccess) cudaGetLastError();
            B200_REQUIRE(e == cudaSuccess && pa.type == cudaMemoryTypeHost,
                         "tracker_step_pinned_async: the detection arrays must be page-locked host memory "
                         "(cudaHostAlloc / cudaHostRegister / torch pin_memory)");
        }
        // the two small per-stream vectors go through the ring slot (the caller may reuse them at once)
        B200_CUDA(cudaMemcpyAsync(dv.n_det, h.n_det, sizeof(int) * d.S, cudaMemcpyHostToDevice, up));
        B200_CUDA(cudaMemcpyAsync(dv.frame, h.frame, sizeof(int) * d.S, cudaMemcpyHostToDevice, up));
        if (n_max > 0) {
            B200_CUDA(cudaMemcpyAsync(dv.boxes, boxes_host, sizeof(double) * 4 * (size_t)d.S * d.MD, cudaMemcpyHostToDevice, up));
            B200_CUDA(cudaMemcpyAsync(dv.confs, confs_host, sizeof(double) * (size_t)d.S * d.MD, cudaMemcpyHostToDevice, up));
            B200_CUDA(cudaMemcpyAsync(dv.embs, embs_host, sizeof(float) * 128 * (size_t)d.S * d.MD, cudaMemcpyHostToDevice, up));
        }
    } else {
        if (dense) {
            memcpy(h.boxes, boxes_host, sizeof(double) * 4 * (size_t)d.S * d.MD);
            memcpy(h.confs, confs_host, sizeof(double) * (size_t)d.S * d.MD);
            memcpy(h.embs, embs_host, sizeof(float) * 128 * (size_t)d.S * d.MD);
        } else {
            for (int s = 0; s < d.S; ++s) {
                const int n = n_det_host[s];
                if (n <= 0) continue;
                memcpy(h.boxes + (size_t)s * d.MD * 4, boxes_host + (size_t)s * d.MD * 4, sizeof(double) * 4 * n);
                memcpy(h.confs + (size_t)s * d.MD, confs_host + (size_t)s * d.MD, sizeof(double) * n);
                memcpy(h.embs + (size_t)s * d.MD * 128, embs_host + (size_t)s * d.MD * 128, sizeof(float) * 128 * n);
            }
        }
        B200_CUDA(cudaMemcpyAsync(dslot, pin, hs.in_bytes, cudaMemcpyHostToDevice, up));
    }
    if (!inline_dma) {
        B200_CUDA(cudaEventRecord(t->up[slot], up));
        B200_CUDA(cudaStreamWaitEvent(st, t->up[slot], 0));        // the caller's stream runs the kernels
    }
    const int rc = b200_tracker_step(t, dv.n_det, dv.boxes, dv.confs, dv.embs, dv.frame, ds.result, stream);
    if (rc) return rc;
    if (!inline_dma) {
        B200_CUDA(cudaEventRecord(t->ran[slot], st));
        B200_CUDA(cudaStreamWaitEvent(down, t->ran[slot], 0));
    }
    B200_CUDA(cudaMemcpyAsync(hs.result, ds.result, t->res_bytes, cudaMemcpyDeviceToHost, down));
    B200_CUDA(cudaEventRecord(t->done[slot], down));
    t->ticket_of[slot] = t->next_ticket;
    *ticket = t->next_ticket++;
    return B200_OK;
}
}  // namespace

extern "C" int b200_tracker_step_host_async(b200_tracker* t, const int32_t* n_det_host, const double* boxes_host,
                                            const double* confs_host, const float* embs_host,
                                            const int32_t* frame_id_host, int64_t* ticket, void* stream) {
    return step_host_submit(t, n_det_host, boxes_host, confs_host, embs_host, frame_id_host, ticket, stream, false);
}

extern "C" int b200_tracker_step_pinned_async(b200_tracker* t, const int32_t* n_det_host, const double* boxes_pinned,
                                              const double* confs_pinned, const float* embs_pinned,
                                              const int32_t* frame_id_host, int64_t* ticket, void* stream) {
    return step_host_submit(t, n_det_host, boxes_pinned, confs_pinned, embs_pinned, frame_id_host, ticket, stream, true);
}

extern "C" int b200_tracker_step_result(b200_tracker* t, int64_t ticket, int32_t* result_host) {
    B200_REQUIRE(t && result_host, "tracker_step_result: null pointer");
    const int slot = (int)(ticket % b200_tracker::kRing);
    B200_REQUIRE(ticket >= 0 && t->ticket_of[slot] == ticket, "tracker_step_result: ticket %lld is not in flight (at most %d steps may be pending)",
                 (long long)ticket, b200_tracker::kRing);
    B200_CUDA(cudaEventSynchronize(t->done[slot]));
    const trk::Slot hs(static_cast<char*>(t->pinned) + (size_t)slot * t->slot_bytes, t->d);
    memcpy(result_host, hs.result, t->res_bytes);
    t->ticket_of[slot] = -1;
    return B200_OK;
}

extern "C" int b200_tracker_step_host(b200_tracker* t, const int32_t* n_det_host, const double* boxes_host,
                                      const double* confs_host, const float* embs_host, const int32_t* frame_id_host,
                                      int32_t* result_host, void* stream) {
    B200_REQUIRE(result_host, "tracker_step_host: null pointer");
    int64_t ticket = -1;
    const int rc = step_host_submit(t, n_det_host, boxes_host, confs_host, embs_host, frame_id_host, &ticket, stream, false, true);
    if (rc) return rc;
    return b200_tracker_step_result(t, ticket, result_host);
}

// ---- step-by-step operations (host arrays in, synchronous) ----------------------------------------------------------
namespace {

// Uploads one stream's detections of a frame into the handle's input block (stream s's slices) and points a Dev copy at it.
int stage_stream_inputs(b200_tracker* t, int s, int n_det, const double* boxes_host, const double* confs_host,
                        const float* embs_host, int frame_id, cudaStream_t st, trk::Dev* d) {
    *d = t->d;
    B200_REQUIRE(n_det >= 0 && n_det <= d->MD, "tracker op: %d detections, capacity %d", n_det, d->MD);
    const size_t MD = d->MD;
    const trk::StepInputs& in = t->in;
    if (n_det > 0) {
        B200_REQUIRE(boxes_host && confs_host && embs_host, "tracker op: null detection arrays");
        B200_CUDA(cudaMemcpyAsync(in.boxes + (size_t)s * MD * 4, boxes_host, sizeof(double) * 4 * n_det, cudaMemcpyHostToDevice, st));
        B200_CUDA(cudaMemcpyAsync(in.confs + (size_t)s * MD, confs_host, sizeof(double) * n_det, cudaMemcpyHostToDevice, st));
        B200_CUDA(cudaMemcpyAsync(in.embs + (size_t)s * MD * 128, embs_host, sizeof(float) * 128 * n_det, cudaMemcpyHostToDevice, st));
    }
    B200_CUDA(cudaMemcpyAsync(in.frame + s, &frame_id, sizeof(int), cudaMemcpyHostToDevice, st));
    d->n_det = in.n_det; d->boxes = in.boxes; d->confs = in.confs; d->embs = in.embs; d->frame_id = in.frame;
    d->result = t->dev_result;
    return B200_OK;
}

int upload_ints(const int32_t* host, int n, int** dev, cudaStream_t st) {
    *dev = nullptr;
    if (n <= 0) return B200_OK;
    B200_CUDA(cudaMallocAsync(reinterpret_cast<void**>(dev), sizeof(int) * (size_t)n, st));
    B200_CUDA(cudaMemcpyAsync(*dev, host, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));
    return B200_OK;
}

}  // namespace

#define B200_STREAM_ARG(fn)                                                                                  \
    B200_REQUIRE(t, fn ": null handle");                                                                     \
    B200_REQUIRE(stream_idx >= 0 && stream_idx < t->d.S, fn ": stream %d out of range", stream_idx);         \
    cudaStream_t st = as_stream(stream)

extern "C" int b200_tracker_predict_all(b200_tracker* t, int stream_idx, void* stream) {
    B200_STREAM_ARG("tracker_predict_all");
    trk::op_predict_kernel<<<1, trk::kThreads, 0, st>>>(t->d, stream_idx);
    int rc = check_launch("trk op_predict_kernel");
    if (rc) return rc;
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

extern "C" int b200_tracker_mark_missed(b200_tracker* t, int stream_idx, const int32_t* track_ids_host, int n, void* stream) {
    B200_STREAM_ARG("tracker_mark_missed");
    B200_REQUIRE(n >= 0 && (n == 0 || track_ids_host), "tracker_mark_missed: bad id list");
    if (n == 0) return B200_OK;
    int* ids = nullptr;
    int rc = upload_ints(track_ids_host, n, &ids, st);
    if (rc) return rc;
    trk::op_mark_missed_kernel<<<1, trk::kThreads, 0, st>>>(t->d, stream_idx, ids, n);
    rc = check_launch("trk op_mark_missed_kernel");
    cudaFreeAsync(ids, st);
    if (rc) return rc;
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

extern "C" int b200_tracker_purge_dead(b200_tracker* t, int stream_idx, void* stream) {
    B200_STREAM_ARG("tracker_purge_dead");
    trk::op_purge_kernel<<<1, trk::kThreads, 0, st>>>(t->d, stream_idx);
    int rc = check_launch("trk op_purge_kernel");
    if (rc) return rc;
    B200_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

extern "C" int b200_tracker_create_tracks(b200_tracker* t, int stream_idx, const int32_t* det_ids_host, int n_ids,
                                          const double* boxes_host, const double* confs_host, const float* embs_host,
                                          int n_det, int frame_id, void* stream) {
    B200_STREAM_ARG("tracker_create_tracks");
    B200_REQUIRE(n_ids >= 0 && (n_ids == 0 || det_ids_host), "tracker_create_tracks: bad id list");
    for (int i = 0; i < n_ids; ++i)
        B200_REQUIRE(det_ids_host[i] >= 0 && det_ids_host[i] < n_det, "tracker_create_tracks: detection index %d out of range", det_ids_host[i]);
    if (n_ids == 0) return 0;
    B200_REQUIRE(n_ids <= t->d.MD, "tracker_create_tracks: %d ids, capacity %d", n_ids, t->d.MD);
    trk::Dev d;
    int rc = stage_stream_inputs(t, stream_idx, n_det, boxes_host, confs_host, embs_host, frame_id, st, &d);
    if (rc) return rc;
    int* ids = nullptr;
    if ((rc = upload_ints(det_ids_host, n_ids + 2, &ids, st))) return rc;     // two extra ints: the kernel's output
    trk::op_create_kernel<<<1, trk::kThreads, 0, st>>>(d, stream_idx, ids, n_ids, n_det, ids + n_ids);
    rc = check_launch("trk op_create_kernel");
    int out[2] = {0, 0};
    if (rc == B200_OK && cudaMemcpyAsync(out, ids + n_ids, sizeof(out), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = B200_ECUDA;
    if (rc == B200_OK && cudaStreamSynchronize(st) != cudaSuccess) rc = B200_ECUDA;
    cudaFreeAsync(ids, st);
    if (rc) return rc == B200_ECUDA ? fail(B200_ECUDA, "tracker_create_tracks: %s", cudaGetErrorString(cudaGetLastError())) : rc;
    if (out[1] == B200_ECAPACITY) return fail(B200_ECAPACITY, "tracker_create_tracks: the handle is full (max_tracks %d)", t->d.MT);
    return out[0];
}

extern "C" int b200_tracker_update_matched(b200_tracker* t, int stream_idx, const int32_t* match_tid_host,
                                           const int32_t* match_det_host, const float* match_cost_host, int n_matches,
                                           const double* boxes_host, const double* confs_host, const float* embs_host,
                                           int n_det, int frame_id, double ema_alpha, double conf_update_min,
                                           double cost_update_max, double maha_thr, void* stream) {
    B200_STREAM_ARG("tracker_update_matched");
    B200_REQUIRE(n_matches >= 0 && n_matches <= t->d.MT, "tracker_update_matched: %d matches, capacity %d", n_matches, t->d.MT);
    if (n_matches == 0) return B200_OK;
    B200_REQUIRE(match_tid_host && match_det_host && match_cost_host, "tracker_update_matched: null match arrays");
    trk::Dev d;
    int rc = stage_stream_inputs(t, stream_idx, n_det, boxes_host, confs_host, embs_host, frame_id, st, &d);
    if (rc) return rc;
    d.ema_a = (float)ema_alpha;
    d.ema_b = (float)(1.0 - ema_alpha);
    d.conf_update_min = conf_update_min; d.cost_update_max = cost_update_max; d.maha_thr = maha_thr;
    int* buf = nullptr;                              // tids | dets | costs | out[2]
    const size_t n = (size_t)n_matches;
    B200_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&buf), sizeof(int) * (3 * n + 2), st));
    cudaMemcpyAsync(buf, match_tid_host, sizeof(int) * n, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(buf + n, match_det_host, sizeof(int) * n, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(buf + 2 * n, match_cost_host, sizeof(float) * n, cudaMemcpyHostToDevice, st);
    trk::op_queue_matches_kernel<<<1, trk::kThreads, 0, st>>>(d, stream_idx, buf, buf + n, reinterpret_cast<const float*>(buf + 2 * n),
                                                              n_matches, n_det, buf + 3 * n);
    rc = check_launch("trk op_queue_matches_kernel");
    if (rc == B200_OK) {
        trk::update_kernel<<<t->upd_grid, trk::kUpdWarps * 32, 0, st>>>(d);
        rc = check_launch("trk update_kernel");
    }
    int out[2] = {0, 0};
    if (rc == B200_OK && cudaMemcpyAsync(out, buf + 3 * n, sizeof(out), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = B200_ECUDA;
    if (rc == B200_OK && cudaStreamSynchronize(st) != cudaSuccess) rc = B200_ECUDA;
    cudaFreeAsync(buf, st);
    if (rc) return rc == B200_ECUDA ? fail(B200_ECUDA, "tracker_update_matched: %s", cudaGetErrorString(cudaGetLastError())) : rc;
    if (out[1]) return fail(B200_EINVAL, "tracker_update_matched: a match names a track id that is not live or a detection index out of range");
    return B200_OK;
}

namespace {

// Host-side argument checks shared by the two image entry points: the image's own first, then against the handle.
int check_image(const b200_tracker* t, const int32_t* streams, const b200_tracker_state* im, const char* fn) {
    B200_REQUIRE(im, "%s: null image", fn);
    B200_REQUIRE(im->cap >= 1, "%s: image cap %d must be >= 1", fn, im->cap);
    B200_REQUIRE(im->n_rows >= 0 && im->n_rows <= 65535, "%s: image n_rows %d outside [0, 65535]", fn, im->n_rows);
    if (im->n_rows > 0) {
        B200_REQUIRE(im->n_live && im->next_id && im->ids && im->x && im->P && im->stage && im->ema && im->bank &&
                     im->bank_len && im->miss && im->age && im->last_bbox && im->last_conf && im->last_cost,
                     "%s: null image field", fn);
        const uintptr_t vec = reinterpret_cast<uintptr_t>(im->x) | reinterpret_cast<uintptr_t>(im->P) |
                              reinterpret_cast<uintptr_t>(im->ema) | reinterpret_cast<uintptr_t>(im->bank) |
                              reinterpret_cast<uintptr_t>(im->last_bbox);
        B200_REQUIRE((vec & 15) == 0, "%s: image x / P / ema / bank / last_bbox must be 16-byte aligned", fn);
    }
    B200_REQUIRE(t, "%s: null handle", fn);
    B200_REQUIRE(im->hist_max == t->d.HIST, "%s: image hist_max %d, handle hist_max %d", fn, im->hist_max, t->d.HIST);
    B200_REQUIRE(streams || im->n_rows == t->d.S, "%s: streams == NULL needs n_rows == n_streams (%d, %d)", fn,
                 im->n_rows, t->d.S);
    return B200_OK;
}

dim3 image_grid(const b200_tracker_state& im) {
    return dim3((unsigned)((im.cap + trk::kStateWarps - 1) / trk::kStateWarps), (unsigned)im.n_rows);
}

// The staging buffer of b200_tracker_export / b200_tracker_import, allocated in stream order on `st`: a one-row image of
// `cap` slots.  n_live, next_id and the row's status share the first range.
cudaError_t alloc_row_image(b200_tracker_state& s, size_t cap, int hist_max, cudaStream_t st, char*& buf) {
    const size_t H = hist_max;
    s.n_rows = 1; s.cap = (int)cap; s.hist_max = hist_max;
    auto carve = [&](trk::Carver& c) {
        c.take(s.n_live, 3); s.next_id = s.n_live + 1;
        c.take(s.ids, cap); c.take(s.x, cap * 8); c.take(s.P, cap * 64); c.take(s.stage, cap); c.take(s.ema, cap * 128);
        c.take(s.bank, cap * H * 128); c.take(s.bank_len, cap); c.take(s.miss, cap); c.take(s.age, cap);
        c.take(s.last_bbox, cap * 4); c.take(s.last_conf, cap); c.take(s.last_cost, cap);
    };
    trk::Carver size;
    carve(size);
    const cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&buf), size.off, st);
    trk::Carver c{buf};
    carve(c);
    return e;
}

}  // namespace

extern "C" int b200_tracker_export_device(b200_tracker* t, const int32_t* streams, const b200_tracker_state* img,
                                          int32_t* status, void* stream) {
    int rc = check_image(t, streams, img, "tracker_export_device");
    if (rc || img->n_rows == 0) return rc;
    trk::export_state_kernel<<<image_grid(*img), trk::kStateWarps * 32, 0, as_stream(stream)>>>(t->d, *img, streams, 0, status);
    return check_launch("trk export_state_kernel");
}

extern "C" int b200_tracker_import_device(b200_tracker* t, const int32_t* streams, const b200_tracker_state* img,
                                          int32_t* status, void* stream) {
    int rc = check_image(t, streams, img, "tracker_import_device");
    if (rc || img->n_rows == 0) return rc;
    cudaStream_t st = as_stream(stream);
    trk::import_check_kernel<<<img->n_rows, trk::kThreads, 0, st>>>(t->d, *img, streams, 0, t->imp_row, status);
    if ((rc = check_launch("trk import_check_kernel"))) return rc;
    trk::import_state_kernel<<<image_grid(*img), trk::kStateWarps * 32, 0, st>>>(t->d, *img, streams, 0, t->imp_row);
    return check_launch("trk import_state_kernel");
}

extern "C" int b200_tracker_export(b200_tracker* t, int stream_idx, int32_t* ids, double* x, double* P, uint8_t* stage,
                                   float* ema, float* bank, int32_t* bank_len, int32_t* miss, int32_t* age,
                                   double* last_bbox, double* last_conf, double* last_cost, int32_t* next_id,
                                   void* stream) {
    B200_REQUIRE(t, "tracker_export: null handle");
    const trk::Dev& d = t->d;
    B200_REQUIRE(stream_idx >= 0 && stream_idx < d.S, "tracker_export: stream %d out of range", stream_idx);
    cudaStream_t st = as_stream(stream);
    const size_t H = d.HIST;
    b200_tracker_state s{};
    char* buf = nullptr;
    B200_CUDA(alloc_row_image(s, d.MT, d.HIST, st, buf));
    trk::export_state_kernel<<<image_grid(s), trk::kStateWarps * 32, 0, st>>>(d, s, nullptr, stream_idx, nullptr);
    int rc = check_launch("trk export_state_kernel");
    if (rc) return rc;
    int hdr[2];
    B200_CUDA(cudaMemcpyAsync(hdr, s.n_live, sizeof(hdr), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    const size_t n = hdr[0];
#define PULL(dst, src, per) if (dst && n) B200_CUDA(cudaMemcpyAsync(dst, src, sizeof(*src) * (per) * n, cudaMemcpyDeviceToHost, st))
    PULL(ids, s.ids, 1); PULL(x, s.x, 8); PULL(P, s.P, 64); PULL(stage, s.stage, 1); PULL(ema, s.ema, 128);
    PULL(bank, s.bank, H * 128); PULL(bank_len, s.bank_len, 1); PULL(miss, s.miss, 1); PULL(age, s.age, 1);
    PULL(last_bbox, s.last_bbox, 4); PULL(last_conf, s.last_conf, 1); PULL(last_cost, s.last_cost, 1);
#undef PULL
    if (next_id) *next_id = hdr[1];
    B200_CUDA(cudaStreamSynchronize(st));
    B200_CUDA(cudaFreeAsync(buf, st));
    return (int)n;
}

extern "C" int b200_tracker_import(b200_tracker* t, int stream_idx, int n, const int32_t* ids, const double* x,
                                   const double* P, const uint8_t* stage, const float* ema, const float* bank,
                                   const int32_t* bank_len, const int32_t* miss, const int32_t* age,
                                   const double* last_bbox, const double* last_conf, const double* last_cost,
                                   int32_t next_id, void* stream) {
    B200_REQUIRE(t, "tracker_import: null handle");
    const trk::Dev& d = t->d;
    B200_REQUIRE(stream_idx >= 0 && stream_idx < d.S, "tracker_import: stream %d out of range", stream_idx);
    B200_REQUIRE(n >= 0 && n <= d.MT, "tracker_import: %d tracks exceed max_tracks %d", n, d.MT);
    B200_REQUIRE(n == 0 || (ids && x && P && stage && ema && bank && bank_len && miss && age && last_bbox && last_conf &&
                            last_cost), "tracker_import: null array");
    cudaStream_t st = as_stream(stream);
    const size_t H = d.HIST;
    b200_tracker_state s{};
    char* buf = nullptr;
    B200_CUDA(alloc_row_image(s, n > 0 ? n : 1, d.HIST, st, buf));
    const int hdr[2] = {n, next_id};
    cudaError_t e = cudaMemcpyAsync(s.n_live, hdr, sizeof(hdr), cudaMemcpyHostToDevice, st);
    auto push = [&](auto* dst, const auto* src, size_t per) {
        if (e == cudaSuccess && n > 0) e = cudaMemcpyAsync(dst, src, sizeof(*dst) * per * n, cudaMemcpyHostToDevice, st);
    };
    push(s.ids, ids, 1); push(s.x, x, 8); push(s.P, P, 64); push(s.stage, stage, 1); push(s.ema, ema, 128);
    push(s.bank, bank, H * 128); push(s.bank_len, bank_len, 1); push(s.miss, miss, 1); push(s.age, age, 1);
    push(s.last_bbox, last_bbox, 4); push(s.last_conf, last_conf, 1); push(s.last_cost, last_cost, 1);
    B200_CUDA(e);
    int* status = s.n_live + 2;
    trk::import_check_kernel<<<1, trk::kThreads, 0, st>>>(d, s, nullptr, stream_idx, t->imp_row, status);
    int rc = check_launch("trk import_check_kernel");
    if (rc) return rc;
    trk::import_state_kernel<<<image_grid(s), trk::kStateWarps * 32, 0, st>>>(d, s, nullptr, stream_idx, t->imp_row);
    if ((rc = check_launch("trk import_state_kernel"))) return rc;
    int row_status = B200_OK;
    B200_CUDA(cudaMemcpyAsync(&row_status, status, sizeof(row_status), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));          // the host arrays may be released after return
    B200_CUDA(cudaFreeAsync(buf, st));
    // n fits the image and max_tracks (checked above), so the only status left is B200_EINVAL: the stream is untouched.
    B200_REQUIRE(row_status == B200_OK, "tracker_import: stream %d: malformed state (ids not ascending or outside "
                 "[0, next_id), bank_len outside [0, hist_max] or stage > 2)", stream_idx);
    return B200_OK;
}

// Dense appearance cost on the 5th-generation tensor cores (tcgen05 + TMEM), for launches large enough to be a real
// GEMM (BASELINE config 4: 512 tracks x 30 bank rows x 128 against 512 detections = 2.0 GFLOP).
//
// Replaces the contraction of Tracking.build_C_app_topk (model/mainTracking.py:141-211: one [T,128] @ [128,N] matmul +
// topk + mean per track, in a Python loop) behind b200_app_cost_topk_f32 and the tracker's ReID-only stage.
//
//   sims[(track, t), det] = <bank_t / |bank_t|, det / |det|>          one [M*32, 128] x [128, N] product
//   C_app[track, det]     = 1 - mean(top-k over t of sims)            epilogue, straight out of TMEM
//
// Precision: the parity bar is 1e-5 relative on C_app, which a single BF16 or TF32 product (2^-8 / 2^-10 relative per
// operand) cannot meet.  Every unit vector is therefore split into three BF16 terms x = hi + mid + lo (24 mantissa bits in
// all, each residual exact in float32) and the six products of weight >= 2^-16 are accumulated in float32 in TMEM:
// hi*hi, hi*mid, mid*hi, hi*lo, lo*hi, mid*mid (what is dropped is 2^-24 relative).  Six BF16 MMAs per K step cost the
// same tensor time as the alternative three TF32 MMAs and lose less.
//
// Kernels:
//   app_tc_prep_kernel   one warp per row: normalise (same float32 operations as cost::unit_row), split, and write the row
//                        into a global "shared-memory image" of its 128-row tile: [split][K chunk of 8][row][8 bf16] -- the
//                        canonical K-major no-swizzle UMMA layout, so the main kernel stages a tile with ONE bulk copy.
//   app_tc_kernel        CTA per (4 tracks x 32 bank rows = 128 accumulator rows, 128 detections): cp.async.bulk of the two
//                        96 KB images onto an mbarrier, 48 tcgen05.mma (M 128, N 128, K 16, cta_group::1) issued by one
//                        thread, tcgen05.commit, then warp w reads TMEM lanes 32w .. 32w+31 -- exactly the 32 bank rows of
//                        track w -- with tcgen05.ld and reduces each detection column's top-k over the lanes with
//                        redux.sync / ballot (the same selection as the float32 kernels, largest first).
#include <cuda_bf16.h>

#include "assoc_cost.cuh"

namespace b200 {
namespace {

constexpr int kRows = 128;                       // rows of a tile (accumulator rows / detections)
constexpr int kTrackRows = 32;                   // bank rows per track inside a tile (hist_max <= 32 on this path)
constexpr int kChunks = cost::kD / 8;            // 16 K chunks of 8 bf16 (16 bytes)
constexpr int kSplitBytes = kChunks * kRows * 16;        // 32 KB: one split of one tile
constexpr int kImageBytes = 3 * kSplitBytes;             // 96 KB: hi | mid | lo
constexpr int kLBO = kRows * 16;                 // next K chunk of the same row
constexpr int kSBO = 8 * 16;                     // next group of eight rows
constexpr int kTcSmem = 2 * kImageBytes + 64;

__device__ __forceinline__ void split3(float x, __nv_bfloat16* hi, __nv_bfloat16* mid, __nv_bfloat16* lo) {
    *hi = __float2bfloat16_rn(x);
    const float r1 = __fsub_rn(x, __bfloat162float(*hi));
    *mid = __float2bfloat16_rn(r1);
    const float r2 = __fsub_rn(r1, __bfloat162float(*mid));
    *lo = __float2bfloat16_rn(r2);
}

// rows: which = 0 -> bank rows of track (item / 32), row t = item % 32 (zero beyond the track's length; the fallback row
// stands in for an empty bank, mainTracking.py:180-182); which = 1 -> detection rows.
// RB = rows of a detection tile: 128 (app_tc_kernel) or 64 (app_tc_walk_kernel); bank tiles always have 128 rows.
template <int RB>
__global__ void __launch_bounds__(256)
app_tc_prep_kernel(const float* __restrict__ bank, const int32_t* __restrict__ bank_len, const float* __restrict__ fallback,
                   const float* __restrict__ det, int M, int N, int T, unsigned char* __restrict__ imgA,
                   unsigned char* __restrict__ imgB, int m_tiles, int n_tiles) {
    const int lane = threadIdx.x & 31;
    const long long rowsA = (long long)m_tiles * kRows, rowsB = (long long)n_tiles * RB;
    for (long long item = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); item < rowsA + rowsB; item += (long long)gridDim.x * 8) {
        float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        unsigned char* img;
        int row, tile_rows = kRows;
        if (item < rowsA) {
            const int m = (int)(item / kTrackRows), t = (int)(item % kTrackRows);
            img = imgA + (size_t)(item / kRows) * kImageBytes;
            row = (int)(item % kRows);
            if (m < M) {
                const int len = min(bank_len[m], T);
                if (t < len) v = reinterpret_cast<const float4*>(bank + ((size_t)m * T + t) * cost::kD)[lane];
                else if (len <= 0 && fallback && t == 0) v = reinterpret_cast<const float4*>(fallback + (size_t)m * cost::kD)[lane];
            }
        } else {
            const long long j = item - rowsA;
            img = imgB + (size_t)(j / RB) * (3 * kChunks * RB * 16);
            row = (int)(j % RB);
            tile_rows = RB;
            if (j < N) v = reinterpret_cast<const float4*>(det + (size_t)j * cost::kD)[lane];
        }
        v = cost::unit_row(v);                   // a zero row stays zero (0 / 1e-12)
        __nv_bfloat16 h[3][4];
        split3(v.x, &h[0][0], &h[1][0], &h[2][0]);
        split3(v.y, &h[0][1], &h[1][1], &h[2][1]);
        split3(v.z, &h[0][2], &h[1][2], &h[2][2]);
        split3(v.w, &h[0][3], &h[1][3], &h[2][3]);
        // element k = 4 * lane .. 4 * lane + 3 of the row: K chunk lane / 2, second half of the chunk for odd lanes
        unsigned char* dst = img + (size_t)(lane >> 1) * (tile_rows * 16) + (size_t)row * 16 + (lane & 1) * 8;
#pragma unroll
        for (int s = 0; s < 3; ++s)
            *reinterpret_cast<uint2*>(dst + (size_t)s * (kChunks * tile_rows * 16)) = *reinterpret_cast<const uint2*>(&h[s][0]);
    }
}

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void tc_mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tc_bulk_load(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// K-major, no swizzle (cute::UMMA::SmemDescriptor, version 1): start address, leading (K chunk) and stride (8-row group)
// byte offsets, all without their four low bits.
__device__ __forceinline__ unsigned long long umma_desc(unsigned smem_addr, int lbo = kLBO) {
    return (unsigned long long)((smem_addr >> 4) & 0x3fffu) | ((unsigned long long)((lbo >> 4) & 0x3fff) << 16) |
           ((unsigned long long)((kSBO >> 4) & 0x3fff) << 32) | (1ull << 46);
}
// kind::f16 instruction descriptor: D float32, A and B bfloat16, both K-major, N = 128, M = 128.
constexpr unsigned kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(kRows >> 3) << 17) | ((unsigned)(kRows >> 4) << 24);

__global__ void __launch_bounds__(128, 1)
app_tc_kernel(const unsigned char* __restrict__ imgA, const unsigned char* __restrict__ imgB,
              const int32_t* __restrict__ bank_len, int has_fallback, int M, int N, int T, int topk, int topk_mean,
              float* __restrict__ C_app, int ldc) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* sA = smem;
    unsigned char* sB = smem + kImageBytes;
    const unsigned bar_load = smem_u32(smem + 2 * kImageBytes), bar_mma = bar_load + 8;
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(smem + 2 * kImageBytes + 16);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile_n = blockIdx.x, tile_m = blockIdx.y;

    if (warp == 0) {                             // 128 accumulator columns (float32) for the 128 x 128 tile
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(128u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    if (threadIdx.x == 32) {
        tc_mbar_init(bar_load, 1);
        tc_mbar_init(bar_mma, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const unsigned tmem = *tmem_slot;

    if (threadIdx.x == 0) {
        tc_mbar_expect_tx(bar_load, 2u * kImageBytes);
        tc_bulk_load(smem_u32(sA), imgA + (size_t)tile_m * kImageBytes, kImageBytes, bar_load);
        tc_bulk_load(smem_u32(sB), imgB + (size_t)tile_n * kImageBytes, kImageBytes, bar_load);
        tc_mbar_wait(bar_load, 0);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        // six split products, smallest first; eight K steps of 16 each
        const int pa[6] = {2, 0, 1, 1, 0, 0}, pb[6] = {0, 2, 1, 0, 1, 0};
        unsigned accumulate = 0;
#pragma unroll
        for (int p = 0; p < 6; ++p) {
            const unsigned a0 = smem_u32(sA) + pa[p] * kSplitBytes, b0 = smem_u32(sB) + pb[p] * kSplitBytes;
#pragma unroll
            for (int ks = 0; ks < kChunks / 2; ++ks) {
                const unsigned long long da = umma_desc(a0 + ks * 2 * kLBO), db = umma_desc(b0 + ks * 2 * kLBO);
                asm volatile(
                    "{\n\t.reg .pred p;\n\t"
                    "setp.ne.b32 p, %4, 0;\n\t"
                    "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                    ::"r"(tmem), "l"(da), "l"(db), "r"(kIdesc), "r"(accumulate) : "memory");
                accumulate = 1;
            }
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar_mma) : "memory");
    }
    __syncwarp();
    tc_mbar_wait(bar_mma, 0);
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");

    // ---- epilogue: warp w = track 4 * tile_m + w.  tcgen05.ld hands lane t the similarities of bank row t for 32 detection
    // columns; a 32 x 32 transpose through shared memory (the operand images are dead by now) gives lane j the 32 rows of
    // column j, and the top-k becomes a thread-local sorted insertion: no shuffles, 32 independent columns per warp.
    // (The first version reduced every column across lanes with redux.sync / ballot: a ~90-cycle dependent chain per round,
    // 30 us per CTA.) ----
    const int m = tile_m * (kRows / kTrackRows) + warp;
    int len = 0;
    if (m < M) {
        len = min(bank_len[m], T);
        if (len <= 0 && has_fallback) len = 1;
    }
    const int kk = topk_mean ? min(topk, len) : min(1, len);
    const float kNegInf = -__int_as_float(0x7f800000);
    float* tile = reinterpret_cast<float*>(smem) + warp * (32 * 33);
    for (int c0 = 0; c0 < kRows; c0 += 32) {
        unsigned r[32];
        const unsigned taddr = tmem + ((unsigned)(warp * 32) << 16) + (unsigned)c0;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32"
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
            " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
              "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
              "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
              "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
        __syncwarp();                            // the previous chunk's reads of `tile` are done
#pragma unroll
        for (int j = 0; j < 32; ++j) tile[lane * 33 + j] = __uint_as_float(r[j]);
        __syncwarp();
        float c = 1.0f;                          // :183-186 / :197-199: an empty bank or topk <= 0 gives a row of ones
        if (kk > 0 && kk <= 5) {
            float t0 = kNegInf, t1 = kNegInf, t2 = kNegInf, t3 = kNegInf, t4 = kNegInf;     // the five largest, descending
#pragma unroll
            for (int t = 0; t < 32; ++t) {
                float x = t < len ? tile[t * 33 + lane] : kNegInf;
                float hi;
                hi = fmaxf(t0, x); x = fminf(t0, x); t0 = hi;
                hi = fmaxf(t1, x); x = fminf(t1, x); t1 = hi;
                hi = fmaxf(t2, x); x = fminf(t2, x); t2 = hi;
                hi = fmaxf(t3, x); x = fminf(t3, x); t3 = hi;
                t4 = fmaxf(t4, x);
            }
            float sum = t0;                      // largest first (:196-202)
            if (kk > 1) sum = __fadd_rn(sum, t1);
            if (kk > 2) sum = __fadd_rn(sum, t2);
            if (kk > 3) sum = __fadd_rn(sum, t3);
            if (kk > 4) sum = __fadd_rn(sum, t4);
            c = __fsub_rn(1.0f, __fdiv_rn(sum, (float)kk));
        } else if (kk > 5) {                     // any k: k rounds of "largest not yet taken"
            unsigned taken = 0u;
            float sum = 0.0f;
            for (int q = 0; q < kk; ++q) {
                float best = kNegInf;
                int arg = 0;
                for (int t = 0; t < len; ++t) {
                    const float x = tile[t * 33 + lane];
                    if (!((taken >> t) & 1u) && x > best) { best = x; arg = t; }
                }
                taken |= 1u << arg;
                sum = __fadd_rn(sum, best);
            }
            c = __fsub_rn(1.0f, __fdiv_rn(sum, (float)kk));
        }
        const int n = tile_n * kRows + c0 + lane;
        if (m < M && n < N) C_app[(size_t)m * ldc + n] = c;
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(128u) : "memory");
}

// ---- second form, for problems with at least 100 bank tiles (400 tracks): a CTA keeps its bank image resident and WALKS the
// detection tiles, warp-specialised.  In the kernel above a CTA loads 192 KB, multiplies and runs its epilogue one after the
// other, once; the tensor pipe is busy 18 % of the time.  Here a CTA owns one bank tile (4 tracks x 32 rows, 96 KB, loaded
// once) and steps through all detection tiles of 64 rows (48 KB each, two buffers, two TMEM accumulators of 64 columns):
//   warp 8 (one thread)  bulk copies and tcgen05.mma: it only ever waits for "detection tile landed" and "accumulator free",
//                        so the tensor core runs one tile ahead of the epilogue;
//   warps 0-7            epilogue: warp w waits for "accumulator full", reads TMEM lanes 32 (w % 4) .. + 31 (track w % 4 of
//                        the tile) and columns 32 (w / 4) .. + 31 of the tile, reduces the top-k and signals "accumulator free".
// No CTA-wide barrier inside the loop.  BASELINE config 4: 30.1 us (first form) -> 23.4 us, whole call 49 -> 40 us.
// (First version of this form: thread 0 issued the products AND ran its share of the epilogue, with a __syncthreads per
// step: ncu showed the other warps 46 % of their time at that barrier; 28.5 us.  Then, each measured and none of them the
// limit: the products' issue loop (descriptors rebuilt per product inside an ELECT loop, 13 -> 8 instructions per
// UTCHMMA), the L2 traffic of the detection tiles (half-tile multicast between CTA pairs: 24.5 us; cluster-wide multicast
// with cluster barriers: 57 / 56 / 99 us for clusters of 2 / 4 / 8), L2 hot-spotting (every CTA pair now starts its walk
// at a different tile).  What is left is shared-memory bandwidth: per step the six products read 288 KB of operands out
// of shared memory while 48 KB land and the epilogue transposes 64 KB through it -- ~3 100 cycles at 128 B/clk before
// any contention.  profiles/r02_app_cost_tc.md.  Next: a wider detection tile per product (fewer re-reads of the bank
// image), which needs the two-CTA form of the instruction to fit in shared memory.)
constexpr int kWalkCols = 64;                                 // detections per step
constexpr int kWalkLBO = kWalkCols * 16;                      // next K chunk inside a 64-row image
constexpr int kWalkSplitBytes = kChunks * kWalkCols * 16;     // 16 KB
constexpr int kWalkImageBytes = 3 * kWalkSplitBytes;          // 48 KB
constexpr int kWalkEpiWarps = 8;
constexpr int kWalkThreads = (kWalkEpiWarps + 1) * 32;
constexpr int kWalkScratch = kWalkEpiWarps * 32 * 33 * 4;
constexpr int kWalkSmem = kImageBytes + 2 * kWalkImageBytes + kWalkScratch + 96;
constexpr unsigned kIdescWalk = (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(kWalkCols >> 3) << 17) | ((unsigned)(kRows >> 4) << 24);

__device__ __forceinline__ void tc_mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}

__global__ void __launch_bounds__(kWalkThreads, 1)
app_tc_walk_kernel(const unsigned char* __restrict__ imgA, const unsigned char* __restrict__ imgB,
                   const int32_t* __restrict__ bank_len, int has_fallback, int M, int N, int T, int topk, int topk_mean,
                   float* __restrict__ C_app, int ldc, int n_steps) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* sA = smem;
    unsigned char* sB = smem + kImageBytes;                                   // two buffers of kWalkImageBytes
    float* scratch = reinterpret_cast<float*>(smem + kImageBytes + 2 * kWalkImageBytes);
    const unsigned bar0 = smem_u32(smem + kImageBytes + 2 * kWalkImageBytes + kWalkScratch);
    // bar0: bank image landed; +8 / +16: detection buffer landed; +24 / +32: accumulator full; +40 / +48: accumulator free;
    // +56 / +64: the products that read detection buffer 0 / 1 have completed in EVERY CTA of the cluster
    unsigned* tmem_slot = reinterpret_cast<unsigned*>(smem + kImageBytes + 2 * kWalkImageBytes + kWalkScratch + 72);
    // A cluster of two CTAs (two bank tiles) shares the delivery of the detection tiles: each CTA fetches HALF of every tile
    // and the copy engine delivers it to the same place in both CTAs (.multicast::cluster), which halves the L2 traffic of
    // the detection images.  No cluster-wide barrier in the loop: "buffer free everywhere" is an mbarrier that both CTAs'
    // tcgen05.commit arrive on (commit with .multicast::cluster), "tile landed" counts the bytes of both halves.
    unsigned rank, nrank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(nrank));
    const unsigned short cta_mask = (unsigned short)((1u << nrank) - 1u);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tile_m = blockIdx.x;
    // Every CTA (pair) starts its walk at a different detection tile: if all of them asked L2 for the same 48 KB at the same
    // time, the few L2 slices that hold those lines would serve 128 SMs while the rest of the L2 idles.
    const int first_tile = (int)((unsigned)tile_m / nrank) % n_steps;

    if (warp == 0) {                             // two accumulators of 64 float32 columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "r"(128u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    if (tid == 32) {
        tc_mbar_init(bar0, 1);
        tc_mbar_init(bar0 + 8, 1); tc_mbar_init(bar0 + 16, 1);
        tc_mbar_init(bar0 + 24, 1); tc_mbar_init(bar0 + 32, 1);
        tc_mbar_init(bar0 + 40, kWalkEpiWarps); tc_mbar_init(bar0 + 48, kWalkEpiWarps);
        tc_mbar_init(bar0 + 56, nrank); tc_mbar_init(bar0 + 64, nrank);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (nrank > 1)                               // the peer's barriers exist before anything is delivered to them
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const unsigned tmem = *tmem_slot;

    if (warp == kWalkEpiWarps) {
        // ---- producer: bulk copies + tcgen05.mma.  The whole warp walks the loop so that every operand is warp-uniform
        // (uniform registers feed UTCHMMA / UBLKCP directly; with operands computed by one lane inside a divergent branch
        // ptxas wraps each of them in an ELECT / R2UR / BRA.U.ANY loop); lane 0 alone issues. ----
        const bool leader = lane == 0;
        const unsigned tm = __shfl_sync(0xffffffffu, tmem, 0);
        auto load_b = [&](int step) {            // leader only
            const int buf = step & 1;
            const int tile_n = (first_tile + step) % n_steps;
            tc_mbar_expect_tx(bar0 + 8 + 8 * buf, (unsigned)kWalkImageBytes);
            if (nrank > 1) {                     // my share of the tile, delivered to every CTA of the cluster
                const unsigned part = (unsigned)kWalkImageBytes / nrank;
                const unsigned dst = smem_u32(sB + buf * kWalkImageBytes) + rank * part;
                const unsigned char* src = imgB + (size_t)tile_n * kWalkImageBytes + (size_t)rank * part;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;\n"
                             ::"r"(dst), "l"(src), "r"(part), "r"(bar0 + 8 + 8 * buf), "h"(cta_mask) : "memory");
            } else {
                tc_bulk_load(smem_u32(sB + buf * kWalkImageBytes), imgB + (size_t)tile_n * kWalkImageBytes, kWalkImageBytes,
                             bar0 + 8 + 8 * buf);
            }
        };
        if (leader) {
            tc_mbar_expect_tx(bar0, (unsigned)kImageBytes);
            tc_bulk_load(smem_u32(sA), imgA + (size_t)tile_m * kImageBytes, kImageBytes, bar0);
            load_b(0);
            if (n_steps > 1) load_b(1);
        }
        __syncwarp();
        tc_mbar_wait(bar0, 0);
        const unsigned long long dA = umma_desc(smem_u32(sA));
        for (int step = 0; step < n_steps; ++step) {
            const int buf = step & 1;
            const unsigned use = (unsigned)((step >> 1) & 1);                 // parity of this use of buffer / accumulator `buf`
            if (step >= 2) tc_mbar_wait(bar0 + 40 + 8 * buf, use ^ 1u);       // the epilogue of step - 2 has released the accumulator
            tc_mbar_wait(bar0 + 8 + 8 * buf, use);                            // the detection tile has landed
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            // six split products, smallest first; eight K steps of 16 each.  A descriptor is the tile's base descriptor plus
            // a compile-time constant in its 14-bit address field.
            const int pa[6] = {2, 0, 1, 1, 0, 0}, pb[6] = {0, 2, 1, 0, 1, 0};
            const unsigned acc = tm + (unsigned)(buf * kWalkCols);
            const unsigned long long dB = umma_desc(smem_u32(sB + buf * kWalkImageBytes), kWalkLBO);
            if (leader) {
                unsigned accumulate = 0;
#pragma unroll
                for (int p = 0; p < 6; ++p) {
#pragma unroll
                    for (int ks = 0; ks < kChunks / 2; ++ks) {
                        const unsigned long long da = dA + (unsigned long long)((pa[p] * kSplitBytes + ks * 2 * kLBO) >> 4);
                        const unsigned long long db = dB + (unsigned long long)((pb[p] * kWalkSplitBytes + ks * 2 * kWalkLBO) >> 4);
                        asm volatile(
                            "{\n\t.reg .pred p;\n\t"
                            "setp.ne.b32 p, %4, 0;\n\t"
                            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                            ::"r"(acc), "l"(da), "l"(db), "r"(kIdescWalk), "r"(accumulate) : "memory");
                        accumulate = 1;
                    }
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
                             ::"r"(bar0 + 24 + 8 * buf) : "memory");
                if (nrank > 1)                   // ... and tell every CTA of the cluster that this buffer has been read here
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n"
                                 ::"r"(bar0 + 56 + 8 * buf), "h"(cta_mask) : "memory");
            }
            __syncwarp();
            // the products of step - 1 have finished reading the other detection buffer (in every CTA that receives what
            // is loaded into it): refill it with tile step + 1
            if (step >= 1 && step + 1 < n_steps) {
                if (nrank > 1) tc_mbar_wait(bar0 + 56 + 8 * (buf ^ 1), (unsigned)(((step - 1) >> 1) & 1));
                else tc_mbar_wait(bar0 + 24 + 8 * (buf ^ 1), (unsigned)(((step - 1) >> 1) & 1));
                if (leader) load_b(step + 1);
                __syncwarp();
            }
        }
    } else {
        // ---- epilogue warps ----
        const int q = warp & 3, half = warp >> 2;
        const int m = tile_m * (kRows / kTrackRows) + q;
        int len = 0;
        if (m < M) {
            len = min(bank_len[m], T);
            if (len <= 0 && has_fallback) len = 1;
        }
        const int kk = topk_mean ? min(topk, len) : min(1, len);
        const float kNegInf = -__int_as_float(0x7f800000);
        float* tile = scratch + warp * (32 * 33);
        for (int step = 0; step < n_steps; ++step) {
            const int buf = step & 1;
            tc_mbar_wait(bar0 + 24 + 8 * buf, (unsigned)((step >> 1) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            unsigned r[32];
            const unsigned taddr = tmem + ((unsigned)(q * 32) << 16) + (unsigned)(buf * kWalkCols + half * 32);
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32"
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15,"
                " %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
                : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                  "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
                  "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                  "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                : "r"(taddr)
                : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
            // the accumulator is in registers: hand it back to the tensor core before the reduction
            asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
            __syncwarp();                        // also: the previous step's reads of `tile` are done
            if (lane == 0) tc_mbar_arrive(bar0 + 40 + 8 * buf);
#pragma unroll
            for (int j = 0; j < 32; ++j) tile[lane * 33 + j] = __uint_as_float(r[j]);
            __syncwarp();
            float c = 1.0f;                      // :183-186 / :197-199: an empty bank or topk <= 0 gives a row of ones
            if (kk > 0 && kk <= 5) {
                float t0 = kNegInf, t1 = kNegInf, t2 = kNegInf, t3 = kNegInf, t4 = kNegInf;     // the five largest, descending
#pragma unroll
                for (int t = 0; t < 32; ++t) {
                    float x = t < len ? tile[t * 33 + lane] : kNegInf;
                    float hi;
                    hi = fmaxf(t0, x); x = fminf(t0, x); t0 = hi;
                    hi = fmaxf(t1, x); x = fminf(t1, x); t1 = hi;
                    hi = fmaxf(t2, x); x = fminf(t2, x); t2 = hi;
                    hi = fmaxf(t3, x); x = fminf(t3, x); t3 = hi;
                    t4 = fmaxf(t4, x);
                }
                float sum = t0;                  // largest first (:196-202)
                if (kk > 1) sum = __fadd_rn(sum, t1);
                if (kk > 2) sum = __fadd_rn(sum, t2);
                if (kk > 3) sum = __fadd_rn(sum, t3);
                if (kk > 4) sum = __fadd_rn(sum, t4);
                c = __fsub_rn(1.0f, __fdiv_rn(sum, (float)kk));
            } else if (kk > 5) {                 // any k: k rounds of "largest not yet taken"
                unsigned taken = 0u;
                float sum = 0.0f;
                for (int qq = 0; qq < kk; ++qq) {
                    float best = kNegInf;
                    int arg = 0;
                    for (int t = 0; t < len; ++t) {
                        const float x = tile[t * 33 + lane];
                        if (!((taken >> t) & 1u) && x > best) { best = x; arg = t; }
                    }
                    taken |= 1u << arg;
                    sum = __fadd_rn(sum, best);
                }
                c = __fsub_rn(1.0f, __fdiv_rn(sum, (float)kk));
            }
            const int n = ((first_tile + step) % n_steps) * kWalkCols + half * 32 + lane;
            if (m < M && n < N) C_app[(size_t)m * ldc + n] = c;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (nrank > 1)                               // no CTA leaves while its peer may still deliver to it or arrive on its barriers
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(128u) : "memory");
}

}  // namespace

// Device-side entry used by b200_app_cost_topk_f32 and the tracker: returns 1 when the tensor-core path does not apply
// (bank deeper than 32 rows, or a problem too small to be worth two launches).
int app_cost_tc(const float* bank, const int32_t* bank_len, const float* fallback, const float* det, int M, int N, int T,
                int topk, int use_topk_mean, float* C_app, int ldc, cudaStream_t st) {
    if (T > kTrackRows || (long long)M * N < 64 * 64) return 1;
    static bool configured[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    if (!configured[dev]) {
        B200_CUDA(cudaFuncSetAttribute(app_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmem));
        B200_CUDA(cudaFuncSetAttribute(app_tc_walk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWalkSmem));
        configured[dev] = true;
    }
    const int m_tiles = (M * kTrackRows + kRows - 1) / kRows;
    // Enough bank tiles to give most SMs their own (>= 100 = 400 tracks): each CTA keeps its bank tile and walks the
    // detection tiles; fewer: a CTA per (bank tile, detection tile) pair fills the GPU better.  B200TRACK_TC_KERNEL=1|2
    // forces a form (tests).
    bool walk = m_tiles >= 100;
    if (const char* e = getenv("B200TRACK_TC_KERNEL")) walk = atoi(e) == 2;
    const int rb = walk ? kWalkCols : kRows;
    const int n_tiles = (N + rb - 1) / rb;
    const size_t imgB_bytes = (size_t)n_tiles * (walk ? kWalkImageBytes : kImageBytes);
    cudaMemPool_t pool = nullptr;
    int rc = scratch_pool(&pool);
    if (rc) return rc;
    unsigned char* img = nullptr;
    B200_CUDA(cudaMallocFromPoolAsync(reinterpret_cast<void**>(&img), (size_t)m_tiles * kImageBytes + imgB_bytes, pool, st));
    unsigned char* imgA = img;
    unsigned char* imgB = img + (size_t)m_tiles * kImageBytes;
    const long long rows = (long long)m_tiles * kRows + (long long)n_tiles * rb;
    const unsigned blocks = (unsigned)((rows + 7) / 8 < 148 * 8 ? (rows + 7) / 8 : 148 * 8);
    if (walk) app_tc_prep_kernel<kWalkCols><<<blocks, 256, 0, st>>>(bank, bank_len, fallback, det, M, N, T, imgA, imgB, m_tiles, n_tiles);
    else app_tc_prep_kernel<kRows><<<blocks, 256, 0, st>>>(bank, bank_len, fallback, det, M, N, T, imgA, imgB, m_tiles, n_tiles);
    rc = check_launch("app_tc_prep_kernel");
    if (rc == B200_OK) {
        if (walk) {
            // B200TRACK_TC_CLUSTER=2: pairs of bank tiles share the delivery of the detection tiles (half-tile multicast).
            // Measured at BASELINE config 4: 24.5 us against 23.4 us without -- the kernel is bound by shared-memory
            // bandwidth (operand reads of the products + the landing copy + the epilogue's transposes), not by L2 -- so
            // it is off by default and kept as a tested option.
            int cl = 1;
            if (const char* e = getenv("B200TRACK_TC_CLUSTER")) cl = (atoi(e) == 2 && m_tiles % 2 == 0) ? 2 : 1;
            launch_ex(app_tc_walk_kernel, dim3((unsigned)m_tiles), dim3(kWalkThreads), kWalkSmem, st, false, cl,
                      (const unsigned char*)imgA, (const unsigned char*)imgB, bank_len, (int)(fallback != nullptr), M, N, T, topk,
                      use_topk_mean, C_app, ldc, n_tiles);
            rc = check_launch("app_tc_walk_kernel");
        } else {
            app_tc_kernel<<<dim3(n_tiles, m_tiles), 128, kTcSmem, st>>>(imgA, imgB, bank_len, fallback != nullptr, M, N, T, topk,
                                                                       use_topk_mean, C_app, ldc);
            rc = check_launch("app_tc_kernel");
        }
    }
    B200_CUDA(cudaFreeAsync(img, st));
    return rc;
}

}  // namespace b200

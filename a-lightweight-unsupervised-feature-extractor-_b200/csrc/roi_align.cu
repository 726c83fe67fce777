// ROI Align forward for sm_100a.
//
// Replaces torchvision.ops.roi_align as the reference calls it (tracking.py:214,
// infer.py:163, trainingCard.py:71): [B,C,H,W] fp32 map + [K,5] rois -> [K,C,PH,PW].
//
// Design (DESIGN.md section "ROI Align"): the work unit is one warp per
// (ROI, 32-channel tile), lane = channel.  Bilinear sampling is separable, and the
// sampling weights depend on the ROI only, not on the channel, so each warp
//   1. turns the ROI's PH*gh + PW*gw sample positions into two small dense weight
//      tables Wy[FY][PH], Wx[FX][PW] over the ROI's footprint (FY x FX map cells);
//   2. stages the footprint of its 32 channels into shared memory as V[cell][channel] with
//      cp.async (NHWC: one coalesced 128 B request per cell; NCHW: lanes run along x inside
//      a row segment so a request touches the fewest lines, transposed by the destination
//      address), issued before step 1's arithmetic so the round trip overlaps it;
//   3. accumulates out[ph][pw] = sum_x Wx[x][pw] * (sum_y Wy[y][ph] * V[y][x]) in
//      registers (PH*PW accumulators per lane, every map value read exactly once);
//   4. writes its [32][PH*PW] result tile -- contiguous in the NCHW output -- to shared
//      memory and hands it to the TMA engine as ONE bulk async store
//      (cp.async.bulk.global.shared::cta), so output traffic is full-line writes.
// Footprints larger than the staging capacity, and output sizes without a template
// instantiation, take exact but slower paths.  Sample coordinates are evaluated with
// the same operation order as torchvision and without FMA contraction so that cell
// selection agrees with the CPU op.
//
// Forward kernels (roi_align_dispatch -> launch_tile), for output sizes 10x10 and 7x7:
//   roi_align_tile_kernel      fewer than 16 384 tiles or fewer than four channel tiles: steps 1-4 fused, one tile
//                              per warp (single-stream latency);
//   roi_prep_kernel            all other launches: step 1 once per ROI instead of once per channel tile, then the
//                              first of these that applies:
//   roi_align_tma_kernel         float32 NCHW map (tma_applies): the footprint arrives as TMA tensor boxes, a warp
//                                walks 2-16 tiles with the next tile's boxes in flight;
//   roi_align_pipe_kernel        channels-last map whose alignment allows it (launch_pipe): software pipeline over
//                                tiles with two footprint buffers (16-byte cp.async.cg copies of tile n+1 while
//                                tile n accumulates);
//   roi_align_multi_kernel       everything else (half NCHW maps, alignments the two above cannot take): the tile body
//                                with a warp walking eight tiles (next ROI record loaded during the current tile,
//                                bulk-store wait deferred);
//   roi_align_generic_kernel   other output sizes: one thread per output element.
// Output is NCHW like the reference's, or channels-last on request (b200_roi_align_fwd_ex): lane = channel then
// stores whole lines straight from the accumulators.
//
// Backward kernels (roi_align_bwd_dispatch -> launch_bwd; see "ROI Align backward" below), same output sizes:
//   roi_align_bwd_tile_kernel  small launches as above: tables built per warp, scalar red.global.add per cell;
//   roi_prep_kernel            all other launches, then
//   roi_align_bwd_tma_kernel     float32 NCHW grad_in (tma_applies, 16-byte grad_out chunks): TMA reduce-add of
//                                each tile's gradient boxes, followed by roi_align_bwd_tile_kernel for the tiles
//                                roi_prep_kernel did not stage;
//   roi_align_bwd_tile_kernel    otherwise (channels-last grad_in, alignment), with the prep records;
//   roi_align_bwd_generic_kernel  other output sizes: one thread per grad_out element.
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include <type_traits>

namespace b200 {
namespace {

// Launch shape of the tile, multi-tile and backward tile kernels.  This value, the CTAs per SM below and the tiles per
// warp of the walking kernels were chosen by the sweeps in profiles/r01_roi_ncu_summary.md, r02_roi_ncu_summary.md and
// r02_roi_variant_sweep_*.txt.
constexpr int kWarpsPerCta = 2;
constexpr int kMinCtasPerSm = 6;  // register cap of the tile / multi-tile / pipelined kernels: 5 and 7 are slower
constexpr int kFootCap = 8;     // max footprint rows / cols on the staged path (<= 64 cells x 32 ch = 8 KB)
constexpr int kCellCap = kFootCap * kFootCap;

// Element type of the map and of the output: float, or __half storage with float arithmetic.
template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ldf<__half>(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }

struct Geom {
    float sw, sh, bw, bh, count;
    int gh, gw, b;
};

__device__ __forceinline__ Geom roi_geometry(const float* __restrict__ r, float scale, int sr,
                                             int aligned, int PH, int PW) {
    Geom g;
    const float off = aligned ? 0.5f : 0.0f;
    g.b = (int)r[0];
    g.sw = __fsub_rn(__fmul_rn(r[1], scale), off);
    g.sh = __fsub_rn(__fmul_rn(r[2], scale), off);
    const float ew = __fsub_rn(__fmul_rn(r[3], scale), off);
    const float eh = __fsub_rn(__fmul_rn(r[4], scale), off);
    float rw = __fsub_rn(ew, g.sw), rh = __fsub_rn(eh, g.sh);
    if (!aligned) {
        rw = fmaxf(rw, 1.0f);
        rh = fmaxf(rh, 1.0f);
    }
    g.bh = __fdiv_rn(rh, (float)PH);
    g.bw = __fdiv_rn(rw, (float)PW);
    g.gh = sr > 0 ? sr : (int)ceilf(g.bh);
    g.gw = sr > 0 ? sr : (int)ceilf(g.bw);
    const int n = g.gh * g.gw;
    g.count = (float)(n > 1 ? n : 1);
    return g;
}

// start + p*bin + (i + .5)*bin/grid, rounded step by step like the reference op.
__device__ __forceinline__ float sample_pos(float start, int p, float bin, int i, int grid) {
    const float a = __fadd_rn(start, __fmul_rn((float)p, bin));
    const float b = __fdiv_rn(__fmul_rn((float)i + 0.5f, bin), (float)grid);
    return __fadd_rn(a, b);
}

struct Tap {
    int lo, hi;
    float wlo, whi;
    bool valid;
};

__device__ __forceinline__ Tap make_tap(float v, int dim) {
    Tap t;
    t.valid = (v >= -1.0f) && (v <= (float)dim);   // false for NaN as well
    if (!(v > 0.0f)) v = 0.0f;
    int lo = (int)fminf(v, (float)dim);
    if (lo >= dim - 1) {
        lo = dim - 1;
        t.hi = lo;
        v = (float)lo;
    } else {
        t.hi = lo + 1;
    }
    t.lo = lo;
    t.whi = __fsub_rn(v, (float)lo);
    t.wlo = __fsub_rn(1.0f, t.whi);
    return t;
}

// Rows (or columns) of the map touched by any valid sample of one axis.  Sample positions are
// monotone in (p, i), so the two extreme samples bound every other one; clamping them to the
// validity window [-1, dim] gives a footprint that covers every valid tap (it may be one cell
// larger than strictly needed, which only adds zero weights).
__device__ __forceinline__ void axis_footprint(float start, float bin, int P, int grid, int dim, int* lo,
                                               int* n) {
    *lo = 0;
    *n = 0;
    if (grid <= 0) return;
    const float a = sample_pos(start, 0, bin, 0, grid), b = sample_pos(start, P - 1, bin, grid - 1, grid);
    const float mn = fmaxf(fminf(a, b), -1.0f), mx = fminf(fmaxf(a, b), (float)dim);
    if (!(mn <= mx) || a != a || b != b) return;
    const Tap t0 = make_tap(mn, dim), t1 = make_tap(mx, dim);
    *lo = t0.lo;
    *n = t1.hi - t0.lo + 1;
}

__device__ __forceinline__ void cp_async4_s(unsigned smem_addr, const void* gsrc) {     // shared-space address
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(smem_addr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16_s(unsigned smem_addr, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_addr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void sts_f32(unsigned smem_addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;\n" ::"r"(smem_addr), "f"(v) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.wait_all;\n" ::: "memory");
}

// One bulk async copy shared -> global issued by a single lane (TMA engine, SASS UBLKCP).  The
// source tile may be overwritten only after bulk_store_wait_read() on the issuing lane.  (An L2 evict-first hint on
// these stores, and on the footprint loads, was measured neutral or slower: profiles/r02_l2_hint_sweep.txt.)
__device__ __forceinline__ void bulk_store_issue(void* gdst, const void* ssrc, unsigned bytes) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gdst), "r"(s),
                 "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
}

// Per-ROI record of the two-kernel path: the 16 channel tiles of a ROI share one geometry / footprint /
// weight-table computation (roi_prep_kernel) instead of repeating it.
struct __align__(16) RoiPrep {
    int b, ymin, xmin, FY;
    int FX, staged, xmask, pad1;    // staged = 0: footprint too large, the tile computes everything itself;
                                    // xmask: bit x set = footprint column x carries weight (all FX of them unless widened)
};

template <int PH, int PW>
struct TileSmem {
    static constexpr int kPHP = (PH + 3) & ~3;
    static constexpr int kPWP = (PW + 3) & ~3;
    static constexpr int kOutFloats = 32 * PH * PW;
    static constexpr int kStageFloats = kCellCap * 32;
    static constexpr int kMainFloats = kOutFloats > kStageFloats ? kOutFloats : kStageFloats;
    static constexpr int kTabFloats = kFootCap * (kPHP + kPWP);
    static constexpr int kFloatsPerWarp = kMainFloats + kTabFloats;
    static constexpr int kBytesPerCta = kFloatsPerWarp * 4 * kWarpsPerCta;
};

// acc[ph][pw] += sum_x Wx[x][pw] * (sum_r Wy[r][ph] * V[r][x]); V comes from `loadv`.
template <int PH, int PW, typename LoadV>
__device__ __forceinline__ void separable_accumulate(float (&acc)[PH][PW], const float* sWy, const float* sWx,
                                                     int FY, int FX, LoadV loadv) {
    constexpr int PHP = (PH + 3) & ~3, PWP = (PW + 3) & ~3;
    for (int x = 0; x < FX; ++x) {
        float ty[PH];
#pragma unroll
        for (int a = 0; a < PH; ++a) ty[a] = 0.0f;
        for (int r = 0; r < FY; ++r) {
            const float v = loadv(r, x);
            const float4* w4 = reinterpret_cast<const float4*>(sWy + r * PHP);
#pragma unroll
            for (int q = 0; q < PHP / 4; ++q) {
                const float4 w = w4[q];
                if (4 * q + 0 < PH) ty[4 * q + 0] = fmaf(w.x, v, ty[4 * q + 0]);
                if (4 * q + 1 < PH) ty[4 * q + 1] = fmaf(w.y, v, ty[4 * q + 1]);
                if (4 * q + 2 < PH) ty[4 * q + 2] = fmaf(w.z, v, ty[4 * q + 2]);
                if (4 * q + 3 < PH) ty[4 * q + 3] = fmaf(w.w, v, ty[4 * q + 3]);
            }
        }
        const float4* w4 = reinterpret_cast<const float4*>(sWx + x * PWP);
#pragma unroll
        for (int q = 0; q < PWP / 4; ++q) {
            const float4 w = w4[q];
            const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (4 * q + e < PW) {
#pragma unroll
                    for (int a = 0; a < PH; ++a) acc[a][4 * q + e] = fmaf(wv[e], ty[a], acc[a][4 * q + e]);
                }
        }
    }
}

// Zeroes and fills the dense weight tables Wy[rows][PHP], Wx[cols][PWP] (one warp; lanes 0-15: y, 16-31: x;
// lane p owns column p of its table).  The mean over samples rides on the x weights.
template <int PH, int PW>
__device__ __forceinline__ void build_tables(const Geom& g, float inv, int H, int W, int ymin, int xmin, int FY,
                                             float* sWy, float* sWx, int n_floats, int lane) {
    constexpr int PHP = (PH + 3) & ~3, PWP = (PW + 3) & ~3;
    for (int i = lane; i < n_floats; i += 32) sWy[i] = 0.0f;      // sWx follows sWy in memory
    __syncwarp();
    const int axis = lane >> 4, p = lane & 15;
    const int Pn = axis ? PW : PH, grid = axis ? g.gw : g.gh, dim = axis ? W : H;
    const float start = axis ? g.sw : g.sh, bin = axis ? g.bw : g.bh;
    float* tab = (axis ? sWx : sWy) + p;
    const int stride = axis ? PWP : PHP, lo0 = axis ? xmin : ymin;
    const float ws = axis ? inv : 1.0f;
    if (p < Pn && FY)
        for (int i = 0; i < grid; ++i) {
            const Tap t = make_tap(sample_pos(start, p, bin, i, grid), dim);
            if (t.valid) {
                tab[(t.lo - lo0) * stride] += t.wlo * ws;
                tab[(t.hi - lo0) * stride] += t.whi * ws;
            }
        }
}

// Two-kernel path, first kernel: one warp per ROI computes footprint + tables once for all channel tiles.
template <int PH, int PW>
__global__ void __launch_bounds__(128)
roi_prep_kernel(const float* __restrict__ rois, long long K, int B, int H, int W, float scale, int sr, int aligned,
                RoiPrep* __restrict__ prep, float* __restrict__ tabs, int xalign) {
    using L = TileSmem<PH, PW>;
    __shared__ __align__(16) float sTabs[4][L::kTabFloats];
    // programmatic dependent launch: the tile kernel that follows may become resident now and wait (griddepcontrol.wait)
    // for this grid to finish, instead of paying its launch latency after it
    asm volatile("griddepcontrol.launch_dependents;");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long k = (long long)blockIdx.x * 4 + warp;
    if (k >= K) return;
    const Geom g = roi_geometry(rois + 5 * k, scale, sr, aligned, PH, PW);
    const float inv = __fdiv_rn(1.0f, g.count);
    int ymin, xmin, FY, FX;
    axis_footprint(g.sh, g.bh, PH, g.gh, H, &ymin, &FY);
    axis_footprint(g.sw, g.bw, PW, g.gw, W, &xmin, &FX);
    if (g.b < 0 || g.b >= B || FY == 0 || FX == 0) FY = FX = 0;
    // TMA consumers (roi_align_tma_kernel) can only start a box on a 16-byte boundary of a map row: the footprint is
    // widened to the left to the previous multiple of `xalign` cells; the added columns get zero weights and a clear
    // bit in the column mask, so they are never multiplied.
    int xoff = 0;
    if (xalign > 1 && FX) {
        xoff = xmin & (xalign - 1);
        xmin -= xoff;
        FX += xoff;
    }
    const bool staged = FY <= kFootCap && FX <= kFootCap;
    if (staged) {
        float* t = sTabs[warp];
        build_tables<PH, PW>(g, inv, H, W, ymin, xmin, FY, t, t + kFootCap * L::kPHP, L::kTabFloats, lane);
        __syncwarp();
        float* dst = tabs + (size_t)k * L::kTabFloats;
        for (int i = lane; i < L::kTabFloats / 4; i += 32)
            reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(t)[i];
    }
    if (lane == 0) {
        RoiPrep h;
        h.b = g.b; h.ymin = ymin; h.xmin = xmin; h.FY = FY; h.FX = FX; h.staged = staged ? 1 : 0;
        h.xmask = FX ? (((1 << (FX - xoff)) - 1) << xoff) : 0;
        h.pad1 = 0;
        prep[k] = h;
    }
}

// One (ROI k, channels c0 .. c0+cn) tile, start to finish, by one warp.  sMain: L::kMainFloats floats (V staging /
// big tables, later the output tile), sTab: L::kTabFloats floats; both private to the warp.
// MULTI (a warp that walks several tiles, roi_align_multi_kernel): the ROI's record arrives in registers (rec0 /
// rec1, loaded while the previous tile was computed) and the bulk store of the output tile is not waited for at
// the end; `*pending` says that sMain may still be being read, and the wait happens in the next call right
// before sMain is written again, i.e. after that tile's address arithmetic.
template <int PH, int PW, bool NHWC, typename T, bool PREP, bool OCL = false, bool MULTI = false>
__device__ __forceinline__ void process_tile(const T* __restrict__ feat, int B, int C, int H, int W,
                                             const float* __restrict__ rois, float scale, int sr, int aligned,
                                             T* __restrict__ out, long long k, int c0, int cn,
                                             const RoiPrep* __restrict__ prep, const float* __restrict__ prep_tabs,
                                             float* sMain, float* sTab, int lane, int4 rec0 = make_int4(0, 0, 0, 0),
                                             int4 rec1 = make_int4(0, 0, 0, 0), bool* pending = nullptr) {
    constexpr bool kF32 = sizeof(T) == 4;
    using L = TileSmem<PH, PW>;
    constexpr int PHP = L::kPHP, PWP = L::kPWP, NB = PH * PW;
    static_assert(PH <= 16 && PW <= 16, "one lane per output row/column");
    Geom g;
    float inv = 0.0f;
    int ymin = 0, xmin = 0, FY = 0, FX = 0;
    bool pre = false;                         // footprint and tables come from roi_prep_kernel
    if (PREP) {
        const int4 h0 = MULTI ? rec0 : reinterpret_cast<const int4*>(prep + k)[0];
        const int4 h1 = MULTI ? rec1 : reinterpret_cast<const int4*>(prep + k)[1];
        if (h1.y) {
            pre = true;
            g.b = h0.x; ymin = h0.y; xmin = h0.z; FY = h0.w; FX = h1.x;
        }
    }
    if (!pre) {
        g = roi_geometry(rois + 5 * k, scale, sr, aligned, PH, PW);
        // mean over samples: 1/count is exact for the power-of-two counts of sampling_ratio 1, 2, 4; otherwise
        // within 1 ulp of the reference's division
        inv = __fdiv_rn(1.0f, g.count);
        axis_footprint(g.sh, g.bh, PH, g.gh, H, &ymin, &FY);
        axis_footprint(g.sw, g.bw, PW, g.gw, W, &xmin, &FX);
        if (g.b < 0 || g.b >= B || FY == 0 || FX == 0) FY = FX = 0;      // nothing sampled: zeros
    }
    const bool staged = FY <= kFootCap && FX <= kFootCap;
    // Larger footprints keep their (bigger) weight tables in the output-tile area and read V
    // straight from global memory; only absurdly large ones take the per-bin path.
    const bool direct = !staged && (FY * PHP + FX * PWP) <= L::kMainFloats;

    float acc[PH][PW];
#pragma unroll
    for (int a = 0; a < PH; ++a)
#pragma unroll
        for (int b = 0; b < PW; ++b) acc[a][b] = 0.0f;

    if (MULTI && !OCL) {                       // the previous tile's bulk store must have left sMain
        if (*pending && lane == 0) bulk_store_wait_read();
        *pending = false;
        __syncwarp();
    }
    if (staged || direct) {
        float* sV = sMain;
        // ---- stage V[cell][channel], fully asynchronous, BEFORE the weight tables are built so the
        // global-memory round trip overlaps that work.  Cell (r, x) of channel c lands at
        // (r*FX + x)*32 + ((c + skew(x)) & 31): the skew makes both the channel-fastest reads of the
        // accumulation loop and the x-fastest NCHW writes bank-conflict free. -------------------------
        int nxp = 1;
        while (nxp < FX) nxp <<= 1;                                  // lanes per row segment: 1, 2, 4, 8
        const int cper = 32 / (nxp > 32 ? 32 : nxp), xmask = nxp - 1;
        if (staged && FY) {
            // running pointers / shared addresses: one 64-bit add and one 32-bit add per request
            const unsigned sv = (unsigned)__cvta_generic_to_shared(sV);
            if (NHWC) {
                const T* row = feat + (((size_t)g.b * H + ymin) * W + xmin) * C + c0 + lane;
                unsigned dst = sv;
                if (lane < cn)
                    for (int r = 0; r < FY; ++r, row += (size_t)W * C) {
                        const T* src = row;
#pragma unroll 4
                        for (int x = 0; x < FX; ++x, src += C, dst += 128) {
                            const unsigned a = dst + 4u * ((lane + (x & xmask) * cper) & 31);
                            if (kF32) cp_async4_s(a, src);
                            else sts_f32(a, ldf<T>(src));          // 16-bit storage: converting load
                        }
                    }
            } else {
                const int xi = lane & xmask, cs = lane / nxp;        // lane = (channel sub-index, x)
                const size_t plane = (size_t)H * W, cstep = plane * cper;
                const T* row = feat + (((size_t)g.b * C + c0 + cs) * H + ymin) * W + xmin + xi;
                unsigned dst = sv + 128u * xi;
                const int skew0 = cs + xi * cper;
                if (xi < FX)
                    for (int r = 0; r < FY; ++r, row += W, dst += 128u * FX) {
                        const T* src = row;
                        int sk = skew0;
#pragma unroll 4
                        for (int c = cs; c < cn; c += cper, src += cstep, sk += cper) {
                            if (kF32) cp_async4_s(dst + 4u * (sk & 31), src);
                            else sts_f32(dst + 4u * (sk & 31), ldf<T>(src));
                        }
                    }
            }
        }
        // ---- dense separable weight tables over the footprint ----------------------------------------
        float* sWy = staged ? sTab : sMain;
        float* sWx = sWy + (staged ? kFootCap : FY) * PHP;
        if (pre) {                             // ready-made: one more asynchronous copy
            const unsigned st = (unsigned)__cvta_generic_to_shared(sTab);
            const float* src = prep_tabs + (size_t)k * L::kTabFloats;
            for (int i = lane; i < L::kTabFloats / 4; i += 32) cp_async16_s(st + 16u * i, src + 4 * i);
        } else {
            build_tables<PH, PW>(g, inv, H, W, ymin, xmin, FY, sWy, sWx,
                                 staged ? L::kTabFloats : FY * PHP + FX * PWP, lane);
        }
        if (staged) {
            cp_async_wait_all();
            __syncwarp();
            separable_accumulate<PH, PW>(acc, sWy, sWx, FY, FX, [&](int r, int x) {
                return sV[(r * FX + x) * 32 + ((lane + (x & xmask) * cper) & 31)];
            });
        } else {
            __syncwarp();
            const int cl = lane < cn ? lane : 0;                     // idle lanes re-read channel 0
            const T* base = NHWC ? feat + (((size_t)g.b * H + ymin) * W + xmin) * C + c0 + cl
                                 : feat + (((size_t)g.b * C + c0 + cl) * H + ymin) * W + xmin;
            const size_t rs = NHWC ? (size_t)W * C : (size_t)W, xs = NHWC ? (size_t)C : 1;
            separable_accumulate<PH, PW>(acc, sWy, sWx, FY, FX,
                                         [&](int r, int x) { return ldf<T>(base + r * rs + x * xs); });
        }
        __syncwarp();                          // every lane is done with V / the tables in sMain
    } else {
        // ---- exact last-resort path: per-bin direct 4-tap sampling ------------------------------
        const size_t ps = NHWC ? (size_t)C : 1;
        const T* base = feat + (NHWC ? (size_t)g.b * H * W * C + c0 + lane
                                     : ((size_t)g.b * C + c0 + lane) * H * W);
#pragma unroll 1
        for (int bin = 0; bin < NB; ++bin) {
            const int a = bin / PW, b = bin - a * PW;
            float s = 0.0f;
            for (int iy = 0; iy < g.gh; ++iy) {
                const Tap ty = make_tap(sample_pos(g.sh, a, g.bh, iy, g.gh), H);
                for (int ix = 0; ix < g.gw; ++ix) {
                    const Tap tx = make_tap(sample_pos(g.sw, b, g.bw, ix, g.gw), W);
                    if (ty.valid && tx.valid && lane < cn) {
                        const float v1 = ldf<T>(base + ((size_t)ty.lo * W + tx.lo) * ps);
                        const float v2 = ldf<T>(base + ((size_t)ty.lo * W + tx.hi) * ps);
                        const float v3 = ldf<T>(base + ((size_t)ty.hi * W + tx.lo) * ps);
                        const float v4 = ldf<T>(base + ((size_t)ty.hi * W + tx.hi) * ps);
                        s += ty.wlo * tx.wlo * v1 + ty.wlo * tx.whi * v2 + ty.whi * tx.wlo * v3 +
                             ty.whi * tx.whi * v4;
                    }
                }
            }
            sMain[lane * NB + bin] = s;        // parked in the output tile, scaled below
        }
        __syncwarp();
#pragma unroll
        for (int a = 0; a < PH; ++a)
#pragma unroll
            for (int b = 0; b < PW; ++b) acc[a][b] = sMain[lane * NB + a * PW + b] * inv;
        __syncwarp();
    }

    if (OCL) {
        // ---- channels-last result [K][PH][PW][C]: the 32 lanes of a bin are 32 consecutive channels, so every
        // store instruction is one full 128-byte (64-byte for half) line straight from the accumulators ----------
        T* gl = out + (size_t)k * NB * C + c0 + lane;
        if (lane < cn) {
#pragma unroll
            for (int a = 0; a < PH; ++a)
#pragma unroll
                for (int b = 0; b < PW; ++b) gl[(size_t)(a * PW + b) * C] = from_f<T>(acc[a][b]);
        }
        return;
    }
    // ---- output tile to shared memory (the accumulators already hold the mean) ------------------------
    if (kF32) {
        float* myrow = sMain + lane * NB;
        if ((NB & 3) == 0) {
#pragma unroll
            for (int q = 0; q < NB / 4; ++q)
                reinterpret_cast<float4*>(myrow)[q] =
                    make_float4(acc[(4 * q) / PW][(4 * q) % PW], acc[(4 * q + 1) / PW][(4 * q + 1) % PW],
                                acc[(4 * q + 2) / PW][(4 * q + 2) % PW], acc[(4 * q + 3) / PW][(4 * q + 3) % PW]);
        } else {
#pragma unroll
            for (int i = 0; i < NB; ++i) myrow[i] = acc[i / PW][i % PW];
        }
    } else {                                   // 16-bit output: one rounding of the fp32 result
        __half* myrow = reinterpret_cast<__half*>(sMain) + lane * NB;
        if ((NB & 1) == 0) {
#pragma unroll
            for (int q = 0; q < NB / 2; ++q)
                reinterpret_cast<__half2*>(myrow)[q] = __floats2half2_rn(acc[(2 * q) / PW][(2 * q) % PW],
                                                                         acc[(2 * q + 1) / PW][(2 * q + 1) % PW]);
        } else {
#pragma unroll
            for (int i = 0; i < NB; ++i) myrow[i] = __float2half_rn(acc[i / PW][i % PW]);
        }
    }

    // ---- one contiguous [cn][PH*PW] chunk of the NCHW output -----------------------------------
    T* gdst = out + ((size_t)k * C + c0) * NB;
    const unsigned bytes = (unsigned)cn * NB * (unsigned)sizeof(T);
    const bool bulk = ((reinterpret_cast<uintptr_t>(gdst) & 15) == 0) && (bytes & 15u) == 0;
    if (bulk) {
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            bulk_store_issue(gdst, sMain, bytes);
            if (!MULTI) bulk_store_wait_read();           // shared memory must outlive the copy's read
        }
        if (MULTI) *pending = true;
    } else {
        __syncwarp();
        const T* tile = reinterpret_cast<const T*>(sMain);
        for (int i = lane; i < cn * NB; i += 32) gdst[i] = tile[i];
    }
}

template <int PH, int PW, bool NHWC, typename T, bool PREP, bool OCL>
__global__ void __launch_bounds__(kWarpsPerCta * 32, (kMinCtasPerSm * 2 + kWarpsPerCta - 1) / kWarpsPerCta)
roi_align_tile_kernel(const T* __restrict__ feat, int B, int C, int H, int W,
                      const float* __restrict__ rois, long long K, float scale, int sr, int aligned,
                      T* __restrict__ out, int ctiles, const RoiPrep* __restrict__ prep,
                      const float* __restrict__ prep_tabs) {
    using L = TileSmem<PH, PW>;
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Warps are independent: no block-wide barriers anywhere below.
    const long long wi = (long long)blockIdx.x * kWarpsPerCta + warp;
    if (wi >= K * ctiles) return;
    float* sMain = smem + (size_t)warp * L::kFloatsPerWarp;
    const unsigned wi32 = (unsigned)wi;       // the launcher keeps the tile count below 2^31
    const long long k = wi32 / (unsigned)ctiles;
    const int c0 = (int)(wi32 % (unsigned)ctiles) * 32;
    process_tile<PH, PW, NHWC, T, PREP, OCL>(feat, B, C, H, W, rois, scale, sr, aligned, out, k, c0, min(32, C - c0),
                                             prep, prep_tabs, sMain, sMain + L::kMainFloats, lane);
}

// Large launches that cannot use the pipelined kernel below (NCHW maps, half storage, 7x7): the tile kernel with a
// warp walking a few tiles.  Nothing is double-buffered, but the next ROI record is loaded during the current
// tile and the wait for the output tile's bulk store moves behind the next tile's address arithmetic, which
// takes two of the three exposed round trips off the critical path; tiles are handed out in groups the size of
// the resident warp set as in the pipelined kernel.
constexpr int kMultiTilesPerWarp = 8;
template <int PH, int PW, bool NHWC, typename T, bool OCL>
__global__ void __launch_bounds__(kWarpsPerCta * 32, (kMinCtasPerSm * 2 + kWarpsPerCta - 1) / kWarpsPerCta)
roi_align_multi_kernel(const T* __restrict__ feat, int B, int C, int H, int W, const float* __restrict__ rois,
                       long long K, float scale, int sr, int aligned, T* __restrict__ out, int ctiles,
                       const RoiPrep* __restrict__ prep, const float* __restrict__ prep_tabs, int group_warps,
                       int tiles_per_warp) {
    using L = TileSmem<PH, PW>;
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned gw = blockIdx.x * kWarpsPerCta + warp, grp = gw / (unsigned)group_warps;
    const unsigned stride = (unsigned)group_warps, window = stride * (unsigned)tiles_per_warp;
    unsigned t = grp * window + (gw - grp * stride);
    const unsigned total = (unsigned)min((long long)(grp + 1) * window, K * ctiles);
    if (t >= total) return;
    asm volatile("griddepcontrol.wait;" ::: "memory");      // roi_prep_kernel's records and tables are complete and visible
    float* sMain = smem + (size_t)warp * L::kFloatsPerWarp;
    unsigned k = t / (unsigned)ctiles;
    int4 h0 = reinterpret_cast<const int4*>(prep + k)[0], h1 = reinterpret_cast<const int4*>(prep + k)[1];
    bool pending = false;
    for (;;) {
        const unsigned tn = t + stride;
        const bool have_next = tn < total;
        unsigned kn = 0;
        int4 n0 = make_int4(0, 0, 0, 0), n1 = n0;
        if (have_next) {
            kn = tn / (unsigned)ctiles;
            n0 = reinterpret_cast<const int4*>(prep + kn)[0];
            n1 = reinterpret_cast<const int4*>(prep + kn)[1];
        }
        const int c0 = (int)(t - k * (unsigned)ctiles) * 32;
        process_tile<PH, PW, NHWC, T, true, OCL, true>(feat, B, C, H, W, rois, scale, sr, aligned, out, (long long)k, c0,
                                                       min(32, C - c0), prep, prep_tabs, sMain, sMain + L::kMainFloats,
                                                       lane, h0, h1, &pending);
        if (!have_next) break;
        t = tn; k = kn; h0 = n0; h1 = n1;
    }
    if (pending && lane == 0) bulk_store_wait_read();
}

// ---- software-pipelined persistent kernel: large float32 launches -------------------------------------
// Once roi_prep_kernel has done the per-ROI work, a tile in the kernel above is three dependent memory round
// trips (record -> footprint + tables -> drain of the bulk store) around ~1 000 instructions of arithmetic,
// and the 168-register warps that sit through them cap an SM at 12 tiles in flight.  Here a warp walks a run
// of consecutive tiles and keeps TWO footprint buffers: while it accumulates tile n from
// one, the cp.asyncs of tile n+1 fill the other and the record of tile n+2 is on its way to registers.  The
// buffers fit because there is no separate output tile: the buffer whose V has just been consumed stages the
// result, 16 channels (one contiguous 16*PH*PW*4-byte block of the NCHW output) at a time, and the warp
// copies it out with coalesced 16-byte streaming stores.  (Storing straight from registers -- lane c owns
// the row of channel c0+c -- is a 400-byte-stride scatter: 32 wavefronts per store instruction, 395 us
// instead of 232 us on the bench launch.)  Tiles whose footprint does not fit a buffer flush the pipeline
// and go through process_tile() with the warp's whole shared-memory region.
constexpr int kPipeWarps = 2;
constexpr int kPipeTilesPerWarp = 8;

template <int PH, int PW>
struct PipeSmem {
    using L = TileSmem<PH, PW>;
    static constexpr int kBufFloats = kCellCap * 32 + L::kTabFloats;       // V | Wy | Wx of one tile
    static constexpr int kFloatsPerWarp = 2 * kBufFloats;
    static constexpr int kBytesPerCta = kFloatsPerWarp * 4 * kPipeWarps;
    static_assert(kFloatsPerWarp >= L::kFloatsPerWarp, "the fallback path needs an output tile + tables");
};

// Starts the copies of one tile of a channels-last map: V[cell][channel] in the map's element type (no skew
// needed: a cell's 32 channels are one 128-byte -- half: 64-byte -- line in both the map and the buffer) and the
// ROI's ready-made weight tables.  With a full, 16-byte aligned tile, 16-byte copies move four (half: eight)
// cells per warp instruction; the 4-byte fallback exists for float only (`pipe_can_stage`).
template <int PH, int PW, typename T>
__device__ __forceinline__ void pipe_issue(const T* __restrict__ feat, int C, int H, int W, const int4 h0,
                                           const int4 h1, long long k, int c0, int cn, bool vec16,
                                           const float* __restrict__ prep_tabs, unsigned sv, int lane) {
    using L = TileSmem<PH, PW>;
    constexpr int kEs = (int)sizeof(T), kLpc = 32 * kEs / 16, kCpi = 32 / kLpc;     // lanes per cell, cells per instruction
    const int b = h0.x, ymin = h0.y, xmin = h0.z, FY = h0.w, FX = h1.x;
    const float* tsrc = prep_tabs + (size_t)k * L::kTabFloats;
    for (int i = lane; i < L::kTabFloats / 4; i += 32) cp_async16_s(sv + 4u * (kCellCap * 32) + 16u * i, tsrc + 4 * i);
    const int cells = FY * FX;
    if (vec16 && cn == 32) {
        int m = lane / kLpc, x = m, r = 0;
        while (x >= FX && r < FY) { x -= FX; ++r; }
        const T* src = feat + (((size_t)b * H + ymin + r) * W + xmin + x) * C + c0 + (lane % kLpc) * (16 / kEs);
        const size_t step = (size_t)kCpi * C, wrap = (size_t)(W - FX) * C;
        unsigned dst = sv + (unsigned)(32 * kEs) * m + 16u * (lane % kLpc);
        for (; m < cells; m += kCpi, dst += (unsigned)(32 * kEs * kCpi)) {
            cp_async16_s(dst, src);
            x += kCpi;
            src += step;
            while (x >= FX) { x -= FX; src += wrap; }
        }
    } else if (kEs == 4 && lane < cn) {
        const T* row = feat + (((size_t)b * H + ymin) * W + xmin) * C + c0 + lane;
        unsigned dst = sv + 4u * lane;
        for (int r = 0; r < FY; ++r, row += (size_t)W * C) {
            const T* src = row;
#pragma unroll 4
            for (int x = 0; x < FX; ++x, src += C, dst += 128) cp_async4_s(dst, src);
        }
    }
}

// A tile can go through the pipeline if roi_prep_kernel staged its footprint and, for half maps, the 16-byte
// copy applies (there is no 2-byte cp.async); other tiles take process_tile() between two pipeline flushes.
template <typename T>
__device__ __forceinline__ bool pipe_can_stage(const int4 rec1, bool vec16, int cn) {
    return rec1.y != 0 && (sizeof(T) == 4 || (vec16 && cn == 32));
}

template <int PH, int PW, bool OCL, typename T>
__global__ void __launch_bounds__(kPipeWarps * 32, (kMinCtasPerSm * 2 + kPipeWarps - 1) / kPipeWarps)
roi_align_pipe_kernel(const T* __restrict__ feat, int B, int C, int H, int W, const float* __restrict__ rois,
                      long long K, float scale, int sr, int aligned, T* __restrict__ out, int ctiles,
                      const RoiPrep* __restrict__ prep, const float* __restrict__ prep_tabs, int group_warps,
                      int tiles_per_warp) {
    using L = TileSmem<PH, PW>;
    using P = PipeSmem<PH, PW>;
    constexpr int PHP = L::kPHP, NB = PH * PW, kEs = (int)sizeof(T);
    static_assert(OCL || (NB * kEs) % (kEs == 4 ? 16 : 4) == 0, "vector stores of a lane's output row");
    extern __shared__ __align__(16) float smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* base = smem + (size_t)warp * P::kFloatsPerWarp;
    const unsigned sbase = (unsigned)__cvta_generic_to_shared(base);
    // Warps are taken in groups of `group_warps` (what the device holds at once); a group covers a window of
    // group_warps * tiles_per_warp consecutive tiles, warp i of the group taking tiles i, i + group_warps, ... of
    // the window, so at any time the resident warps work on neighbouring ROIs (same maps, same DRAM pages), and
    // a warp retires after tiles_per_warp tiles so that other streams' kernels (the association chain) get SM
    // slots every few tens of microseconds.
    const unsigned gw = blockIdx.x * kPipeWarps + warp, grp = gw / (unsigned)group_warps;
    const unsigned stride = (unsigned)group_warps, window = stride * (unsigned)tiles_per_warp;
    unsigned t = grp * window + (gw - grp * stride);
    const unsigned total = (unsigned)min((long long)(grp + 1) * window, K * ctiles);
    if (t >= total) return;
    asm volatile("griddepcontrol.wait;" ::: "memory");      // roi_prep_kernel's records and tables are complete and visible

    // current tile (a*), next tile (n*): ROI index, first channel, prep record
    unsigned ka = t / (unsigned)ctiles;
    int ca = (int)(t - ka * (unsigned)ctiles) * 32;
    int4 a0 = reinterpret_cast<const int4*>(prep + ka)[0], a1 = reinterpret_cast<const int4*>(prep + ka)[1];
    const bool vec16 = ((C * kEs) & 15) == 0 && (reinterpret_cast<uintptr_t>(feat) & 15) == 0;
    if (pipe_can_stage<T>(a1, vec16, min(32, C - ca)))
        pipe_issue<PH, PW, T>(feat, C, H, W, a0, a1, ka, ca, min(32, C - ca), vec16, prep_tabs, sbase, lane);
    asm volatile("cp.async.commit_group;\n" ::: "memory");
    unsigned tn = t + stride, kn = 0;
    int cnx = 0;
    int4 n0 = make_int4(0, 0, 0, 0), n1 = n0;
    if (tn < total) {
        kn = tn / (unsigned)ctiles;
        cnx = (int)(tn - kn * (unsigned)ctiles) * 32;
        n0 = reinterpret_cast<const int4*>(prep + kn)[0];
        n1 = reinterpret_cast<const int4*>(prep + kn)[1];
    }
    int par = 0;
    for (;;) {
        const bool have_next = tn < total;
        const int cn = min(32, C - ca);
        if (!pipe_can_stage<T>(a1, vec16, cn)) {           // footprint too large for a buffer (or no 16-byte copy): nothing is in flight, use the whole region
            process_tile<PH, PW, true, T, false, OCL>(feat, B, C, H, W, rois, scale, sr, aligned, out, (long long)ka,
                                                      ca, cn, nullptr, nullptr, base, base + L::kMainFloats, lane);
            __syncwarp();
        }
        if (have_next && pipe_can_stage<T>(n1, vec16, min(32, C - cnx)))
            pipe_issue<PH, PW, T>(feat, C, H, W, n0, n1, kn, cnx, min(32, C - cnx), vec16, prep_tabs,
                                  sbase + 4u * (unsigned)((par ^ 1) * P::kBufFloats), lane);
        asm volatile("cp.async.commit_group;\n" ::: "memory");
        // record of the tile after next: requested after the accumulation below (the accumulators leave no room for
        // eight more live registers) and in registers by the time the copy-out is done
        const unsigned tm = tn + stride;
        unsigned km = 0;
        int cm = 0;
        int4 m0 = make_int4(0, 0, 0, 0), m1 = m0;
        auto load_after_next = [&]() {
            if (have_next && tm < total) {
                km = tm / (unsigned)ctiles;
                cm = (int)(tm - km * (unsigned)ctiles) * 32;
                m0 = reinterpret_cast<const int4*>(prep + km)[0];
                m1 = reinterpret_cast<const int4*>(prep + km)[1];
            }
        };
        if (pipe_can_stage<T>(a1, vec16, cn)) {
            asm volatile("cp.async.wait_group 1;\n" ::: "memory");
            __syncwarp();
            const T* sV = reinterpret_cast<const T*>(base + par * P::kBufFloats);
            const float* sWy = base + par * P::kBufFloats + kCellCap * 32;
            const int FY = a0.w, FX = a1.x;
            float acc[PH][PW];
#pragma unroll
            for (int a = 0; a < PH; ++a)
#pragma unroll
                for (int bq = 0; bq < PW; ++bq) acc[a][bq] = 0.0f;
            separable_accumulate<PH, PW>(acc, sWy, sWy + kFootCap * PHP, FY, FX, [&](int r, int x) {
                return to_f32(sV[(r * FX + x) * 32 + lane]);
            });
            load_after_next();
            if (OCL) {          // channels-last result: full-line stores straight from the accumulators
                T* gl = out + (size_t)ka * NB * C + ca + lane;
                if (lane < cn) {
#pragma unroll
                    for (int a = 0; a < PH; ++a)
#pragma unroll
                        for (int bq = 0; bq < PW; ++bq) gl[(size_t)(a * PW + bq) * C] = from_f<T>(acc[a][bq]);
                }
            }
            __syncwarp();       // V of this tile is dead: its buffer now stages the output, 16 channels at a time
            T* so = reinterpret_cast<T*>(base + par * P::kBufFloats);
#pragma unroll
            for (int h = 0; h < (OCL ? 0 : 2); ++h) {
                if ((lane >> 4) == h) {
                    if (kEs == 4) {
                        float4* row = reinterpret_cast<float4*>(so + (lane & 15) * NB);
#pragma unroll
                        for (int q = 0; q < NB / 4; ++q)
                            row[q] = make_float4(acc[(4 * q) / PW][(4 * q) % PW], acc[(4 * q + 1) / PW][(4 * q + 1) % PW],
                                                 acc[(4 * q + 2) / PW][(4 * q + 2) % PW],
                                                 acc[(4 * q + 3) / PW][(4 * q + 3) % PW]);
                    } else {    // half: one rounding of the fp32 result
                        __half2* row = reinterpret_cast<__half2*>(so + (lane & 15) * NB);
#pragma unroll
                        for (int q = 0; q < NB / 2; ++q)
                            row[q] = __floats2half2_rn(acc[(2 * q) / PW][(2 * q) % PW], acc[(2 * q + 1) / PW][(2 * q + 1) % PW]);
                    }
                }
                __syncwarp();
                const int nch = min(16, cn - 16 * h);                 // contiguous [nch][PH*PW] block of the result
                float4* g4 = reinterpret_cast<float4*>(out + ((size_t)ka * C + ca + 16 * h) * NB);
                const float4* s4 = reinterpret_cast<const float4*>(so);
                if (nch == 16) {                                      // loads in batches of four, then their stores
                    constexpr int kN4 = 16 * NB * kEs / 16, kIt = (kN4 + 31) / 32;
#pragma unroll
                    for (int i0 = 0; i0 < kIt; i0 += 4) {
                        float4 v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (i0 + u < kIt && (32 * (i0 + u + 1) <= kN4 || lane + 32 * (i0 + u) < kN4))
                                v[u] = s4[lane + 32 * (i0 + u)];
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if (i0 + u < kIt && (32 * (i0 + u + 1) <= kN4 || lane + 32 * (i0 + u) < kN4))
                                __stcs(g4 + lane + 32 * (i0 + u), v[u]);
                    }
                } else {        // ragged last tile (float only: half tiles with cn < 32 are not staged)
                    for (int i = lane; i < nch * NB * kEs / 16; i += 32) __stcs(g4 + i, s4[i]);
                }
                __syncwarp();
            }
            __syncwarp();       // every lane is done with this buffer before the next iteration refills it
        } else {
            load_after_next();
        }
        if (!have_next) break;
        t = tn; ka = kn; ca = cnx; a0 = n0; a1 = n1;
        tn = tm; kn = km; cnx = cm; n0 = m0; n1 = m1;
        par ^= 1;
    }
}


// ---- TMA-staged pipelined kernel: large launches on NCHW maps --------------------------------------------
// The plane-strided footprint of an NCHW map (FY rows x FX floats in each of 32 channel planes) is exactly a
// box of a 4-D tensor (W, H, C, B): one cp.async.bulk.tensor (SASS UTMALDG) moves it with no LSU wavefronts and
// no per-element address arithmetic, which were the two costs of the LDGSTS staging above.  What the hardware
// dictates (tools/tma_probe.cu, profiles/r02_roi_ncu_summary.md):
//   * a box can only start on a 16-byte boundary of a map row (an inner coordinate that is not a multiple of
//     16 bytes raises "illegal instruction"), so roi_prep_kernel widens the footprint to the left to a multiple
//     of four cells and records which columns really carry weight (RoiPrep::xmask); the others are skipped,
//     not multiplied by zero;
//   * the TMA unit works row by row and a warp's next instruction waits until the unit has accepted the box, so
//     the number of box rows, not bytes, is the cost: boxes are 32 bytes wide (eight cells: every widened
//     footprint of the staged path fits one box) and come in three heights, 1 / 3 / 5 rows (three tensor maps),
//     the smallest that covers the footprint; taller footprints (6-8 rows) take a second box below.
// A box lands in shared memory as V[channel][row][8 cells]; with an ODD row count the 128-bit reads of one half
// row by the 8 lanes of a quarter-warp (lane = channel, stride rows * 32 B) fall on four bank groups: two
// wavefronts per read, of which there are only two per footprint row.  Coordinates beyond the map are zero-filled
// by the TMA unit.  The contraction keeps the rows of four columns in registers and runs column-outer
// (tma_accumulate).  The ROI's ready-made weight tables arrive on the same mbarrier with one cp.async.bulk.  A
// warp walks `tiles_per_warp` tiles and keeps the footprint of the NEXT tile in flight while it accumulates the
// current one (two table slots; the V region is shared by the two tiles in flight, growing from both ends, and a
// tile that does not fit beside its predecessor is simply requested after it has been consumed), stages its
// [32][PH*PW] result in a separate output tile and hands that to the TMA engine as one bulk store whose
// completion is awaited only when the next result is ready.  Tiles the prep kernel did not stage go through
// process_tile() with the output tile as scratch.
constexpr int kTmaRows = 5;                                // rows of the tallest box
constexpr int kTmaCols = 8;                                // cells per box row (32 bytes)
constexpr int kTmaRowBytes = kTmaCols * 4 * 32;            // one box row of all 32 channels in shared memory
constexpr int kTmaVRows = 10;                              // V region in box rows: two tiles of <= 5 rows in flight
constexpr int kTmaVBytes = kTmaVRows * kTmaRowBytes;
struct TmaMaps {                                           // the same map with boxes of 1, 3 and 5 rows
    CUtensorMap m[3];
};
__device__ __forceinline__ int tma_box_rows(int rows) { return rows <= 1 ? 1 : rows <= 3 ? 3 : 5; }
// CTA shape and register cap of the TMA kernels (profiles/r02_roi_variant_sweep_*.txt, r02_roi_ncu_summary.md)
constexpr int kTmaWarps = 2;
constexpr int kTmaRegs = 216;

template <int PH, int PW>
struct TmaSmem {
    using L = TileSmem<PH, PW>;
    static constexpr int kTabBytes = L::kTabFloats * 4;
    static constexpr int kOutBytes = L::kMainFloats * 4;                  // output tile; process_tile()'s sMain on the fallback
    static constexpr int kOffTab = kTmaVBytes, kOffOut = kOffTab + 2 * kTabBytes, kOffBar = kOffOut + kOutBytes;
    static constexpr int kBytesPerWarp = (kOffBar + 16 + 127) & ~127;
    static constexpr int kBytesPerCta = kBytesPerWarp * kTmaWarps;
    static_assert(kTabBytes % 16 == 0 && kOffOut % 16 == 0 && kOffBar % 8 == 0, "bulk-copy alignment");
};

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_box_4d(unsigned dst, const CUtensorMap* tm, int x, int y, int c, int b, unsigned bar) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];\n"
                 ::"r"(dst), "l"(tm), "r"(x), "r"(y), "r"(c), "r"(b), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_load(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// Box rows a staged tile occupies in the V region (0 for a ROI that samples nothing): one box of 1 / 3 / 5 rows, plus a
// second one for footprints of 6-8 rows.
__device__ __forceinline__ int tma_tile_rows(const int4 h0, const int4 h1) {
    const int FY = h0.w, FX = h1.x;
    if (FY == 0 || FX == 0) return 0;
    return FY > kTmaRows ? kTmaRows + tma_box_rows(FY - kTmaRows) : tma_box_rows(FY);
}

__device__ __forceinline__ bool elect_one() {
    unsigned p;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(p)::"memory");
    return p != 0;
}
__device__ __forceinline__ int bcast0(int v) { return __shfl_sync(0xffffffffu, v, 0); }

// One elected lane requests everything tile (k, c0) needs: the weight tables of ROI k and the footprint boxes.  Called by
// the whole (converged) warp; the operands are broadcast from lane 0 first so that they are provably warp-uniform and
// go to the TMA instructions through uniform registers directly (with per-lane values ptxas wraps every UTMALDG /
// UBLKCP in an ELECT / R2UR.BROADCAST loop, which showed up as 11 % of all stall samples).
template <int PH, int PW>
__device__ __forceinline__ void tma_issue(const TmaMaps* tm, const int4 h0, const int4 h1, unsigned k, int c0,
                                          const float* __restrict__ prep_tabs, unsigned sv, unsigned stab, unsigned bar) {
    using S = TmaSmem<PH, PW>;
    const int b = bcast0(h0.x), ymin = bcast0(h0.y), xmin = bcast0(h0.z), FY = bcast0(h0.w), FX = bcast0(h1.x);
    const unsigned ku = (unsigned)bcast0((int)k);
    const int cu = bcast0(c0);
    const unsigned svu = (unsigned)bcast0((int)sv), stabu = (unsigned)bcast0((int)stab), baru = (unsigned)bcast0((int)bar);
    const bool any = FY != 0 && FX != 0;
    const int r0 = FY > kTmaRows ? kTmaRows : tma_box_rows(FY);                 // rows of the first box
    const int r1 = FY > kTmaRows ? tma_box_rows(FY - kTmaRows) : 0;            // rows of the box below it
    if (elect_one()) {
        mbar_expect_tx(baru, (unsigned)(S::kTabBytes + (any ? (r0 + r1) * kTmaRowBytes : 0)));
        bulk_load(stabu, prep_tabs + (size_t)ku * S::L::kTabFloats, S::kTabBytes, baru);
        if (any) {
            tma_box_4d(svu, &tm->m[r0 >> 1], xmin, ymin, cu, b, baru);
            if (r1) tma_box_4d(svu + kTmaRows * kTmaRowBytes, &tm->m[r1 >> 1], xmin, ymin + kTmaRows, cu, b, baru);
        }
    }
    __syncwarp();
}

// Separable contraction over V[channel][row][8 cells] as the TMA boxes lay it out (see above).  Per box and half row
// (four columns of this lane's channel) the rows are read once as 128-bit values into registers (rows beyond the
// footprint as zeros, never as map data); then, column-outer like separable_accumulate: for every column that
// carries weight (one uniform test per column and box, not per row), ty[ph] = sum_r Wy[r][ph] * V[r][x] and
// acc[ph][pw] += Wx[x][pw] * ty[ph].
template <int PH, int PW>
__device__ __forceinline__ void tma_accumulate(float (&acc)[PH][PW], const unsigned char* sV, const float* sWy,
                                               const float* sWx, int FY, int FX, int xmask, int lane) {
    constexpr int PHP = (PH + 3) & ~3, PWP = (PW + 3) & ~3;
    const int nrb = FY > kTmaRows ? 2 : 1, ncb = FX > 4 ? 2 : 1;
    for (int rb = 0; rb < nrb; ++rb) {
        const int rows = FY - rb * kTmaRows;                          // footprint rows from this box's first row on
        const int brow = rb ? tma_box_rows(rows) : (nrb == 2 ? kTmaRows : tma_box_rows(rows));   // rows of the box itself
        const unsigned char* mine = sV + rb * (kTmaRows * kTmaRowBytes) + lane * (brow * 32);
        const float* wy0 = sWy + rb * kTmaRows * PHP;
        for (int cb = 0; cb < ncb; ++cb) {
            float v[kTmaRows][4];
#pragma unroll
            for (int i = 0; i < kTmaRows; ++i) {
                float4 q = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                if (i < rows) q = *reinterpret_cast<const float4*>(mine + i * 32 + cb * 16);
                v[i][0] = q.x; v[i][1] = q.y; v[i][2] = q.z; v[i][3] = q.w;
            }
            const int bits = (xmask >> (4 * cb)) & 15;
#pragma unroll
            for (int xi = 0; xi < 4; ++xi) {
                if ((bits >> xi) & 1) {                               // uniform
                    float ty[PH];
#pragma unroll
                    for (int a = 0; a < PH; ++a) ty[a] = 0.0f;
#pragma unroll
                    for (int i = 0; i < kTmaRows; ++i) {
                        // rows past the table (only possible in the second row box) have no weights: their data is zero
                        const int r = (rb * kTmaRows + i < kFootCap) ? i : 0;
                        const float4* w4 = reinterpret_cast<const float4*>(wy0 + r * PHP);
#pragma unroll
                        for (int q = 0; q < PHP / 4; ++q) {
                            const float4 w = w4[q];
                            if (4 * q + 0 < PH) ty[4 * q + 0] = fmaf(w.x, v[i][xi], ty[4 * q + 0]);
                            if (4 * q + 1 < PH) ty[4 * q + 1] = fmaf(w.y, v[i][xi], ty[4 * q + 1]);
                            if (4 * q + 2 < PH) ty[4 * q + 2] = fmaf(w.z, v[i][xi], ty[4 * q + 2]);
                            if (4 * q + 3 < PH) ty[4 * q + 3] = fmaf(w.w, v[i][xi], ty[4 * q + 3]);
                        }
                    }
                    const float4* w4 = reinterpret_cast<const float4*>(sWx + (4 * cb + xi) * PWP);
#pragma unroll
                    for (int q = 0; q < PWP / 4; ++q) {
                        const float4 w = w4[q];
                        const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (4 * q + e < PW) {
#pragma unroll
                                for (int a2 = 0; a2 < PH; ++a2) acc[a2][4 * q + e] = fmaf(wv[e], ty[a2], acc[a2][4 * q + e]);
                            }
                    }
                }
            }
        }
    }
}

template <int PH, int PW, bool OCL>
__global__ void __maxnreg__(kTmaRegs)
roi_align_tma_kernel(const __grid_constant__ TmaMaps tmap, const float* __restrict__ feat, int B, int C, int H, int W,
                     const float* __restrict__ rois, long long K, float scale, int sr, int aligned, float* __restrict__ out,
                     int ctiles, const RoiPrep* __restrict__ prep, const float* __restrict__ prep_tabs, int group_warps,
                     int tiles_per_warp) {
    using L = TileSmem<PH, PW>;
    using S = TmaSmem<PH, PW>;
    constexpr int PHP = L::kPHP, NB = PH * PW;
    extern __shared__ __align__(128) unsigned char smem_tma[];
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // provably warp-uniform
    unsigned char* base = smem_tma + (size_t)warp * S::kBytesPerWarp;
    const unsigned sbase = (unsigned)__cvta_generic_to_shared(base);
    const unsigned sbar = sbase + S::kOffBar;
    float* sOut = reinterpret_cast<float*>(base + S::kOffOut);
    const unsigned gw = blockIdx.x * kTmaWarps + warp, grp = gw / (unsigned)group_warps;
    const unsigned stride = (unsigned)group_warps, window = stride * (unsigned)tiles_per_warp;
    unsigned t = grp * window + (gw - grp * stride);
    const unsigned total = (unsigned)min((long long)(grp + 1) * window, K * ctiles);
    if (t >= total) return;
    asm volatile("griddepcontrol.wait;" ::: "memory");      // roi_prep_kernel's records and tables are complete and visible
    if (lane == 0) {
        mbar_init(sbar, 1);
        mbar_init(sbar + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncwarp();

    // current tile (a*), next tile (n*): ROI index, first channel, prep record
    unsigned ka = t / (unsigned)ctiles;
    int ca = (int)(t - ka * (unsigned)ctiles) * 32;
    int4 a0 = reinterpret_cast<const int4*>(prep + ka)[0], a1 = reinterpret_cast<const int4*>(prep + ka)[1];
    unsigned tn = t + stride, kn = 0;
    int cnx = 0;
    int4 n0 = make_int4(0, 0, 0, 0), n1 = n0;
    if (tn < total) {
        kn = tn / (unsigned)ctiles;
        cnx = (int)(tn - kn * (unsigned)ctiles) * 32;
        n0 = reinterpret_cast<const int4*>(prep + kn)[0];
        n1 = reinterpret_cast<const int4*>(prep + kn)[1];
    }
    int par = 0;                       // slot of the current tile: table slot, mbarrier, end of the V region it grows from
    unsigned phase = 0;                // bit p = parity the next wait on mbarrier p expects
    bool pending = false;              // the bulk store of the previous result may still be reading sOut
    bool cur_issued = false;
    // V offset of a tile with `nb` boxes in slot p: slot 0 grows up from the start, slot 1 down from the end
    auto v_off = [&](int p, int nr) { return p ? (unsigned)(kTmaVBytes - nr * kTmaRowBytes) : 0u; };
    if (a1.y) {
        tma_issue<PH, PW>(&tmap, a0, a1, ka, ca, prep_tabs, sbase + v_off(0, tma_tile_rows(a0, a1)),
                          sbase + S::kOffTab, sbar);
        cur_issued = true;
    }
    for (;;) {
        const bool have_next = tn < total;
        const int cn = min(32, C - ca);
        const int nba = a1.y ? tma_tile_rows(a0, a1) : 0;                      // box rows of the current / next tile
        const int nbn = (have_next && n1.y) ? tma_tile_rows(n0, n1) : 0;
        // the next tile's footprint is requested now if it fits beside the current one, else once that is consumed
        bool next_issued = false;
        if (have_next && n1.y && nba + nbn <= kTmaVRows) {
            tma_issue<PH, PW>(&tmap, n0, n1, kn, cnx, prep_tabs, sbase + v_off(par ^ 1, nbn),
                              sbase + S::kOffTab + (par ^ 1) * S::kTabBytes, sbar + 8 * (par ^ 1));
            next_issued = true;
        }
        // record of the tile after next: requested after the accumulation (register pressure), see roi_align_pipe_kernel
        const unsigned tm = tn + stride;
        unsigned km = 0;
        int cm = 0;
        int4 m0 = make_int4(0, 0, 0, 0), m1 = m0;
        auto load_after_next = [&]() {
            if (have_next && tm < total) {
                km = tm / (unsigned)ctiles;
                cm = (int)(tm - km * (unsigned)ctiles) * 32;
                m0 = reinterpret_cast<const int4*>(prep + km)[0];
                m1 = reinterpret_cast<const int4*>(prep + km)[1];
            }
        };
        if (a1.y) {
            if (!cur_issued) {         // only when the previous iteration could not fit it beside its own tile
                tma_issue<PH, PW>(&tmap, a0, a1, ka, ca, prep_tabs, sbase + v_off(par, nba),
                                  sbase + S::kOffTab + par * S::kTabBytes, sbar + 8 * par);
            }
            mbar_wait(sbar + 8 * par, (phase >> par) & 1u);
            phase ^= 1u << par;
            const float* sWy = reinterpret_cast<const float*>(base + S::kOffTab + par * S::kTabBytes);
            const int FY = a0.w, FX = a1.x;
            float acc[PH][PW];
#pragma unroll
            for (int a = 0; a < PH; ++a)
#pragma unroll
                for (int bq = 0; bq < PW; ++bq) acc[a][bq] = 0.0f;
            if (nba) tma_accumulate<PH, PW>(acc, base + v_off(par, nba), sWy, sWy + kFootCap * PHP, FY, FX, a1.z, lane);
            load_after_next();
            __syncwarp();              // V and the tables of this slot are dead
            if (have_next && n1.y && !next_issued && nbn <= kTmaVRows) {
                tma_issue<PH, PW>(&tmap, n0, n1, kn, cnx, prep_tabs, sbase + v_off(par ^ 1, nbn),
                                  sbase + S::kOffTab + (par ^ 1) * S::kTabBytes, sbar + 8 * (par ^ 1));
                next_issued = true;
            }
            if (OCL) {                 // channels-last result: full-line stores straight from the accumulators
                float* gl = out + (size_t)ka * NB * C + ca + lane;
                if (lane < cn) {
#pragma unroll
                    for (int a = 0; a < PH; ++a)
#pragma unroll
                        for (int bq = 0; bq < PW; ++bq) gl[(size_t)(a * PW + bq) * C] = acc[a][bq];
                }
            } else {
                if (pending && lane == 0) bulk_store_wait_read();
                pending = false;
                __syncwarp();
                float* myrow = sOut + lane * NB;
                if ((NB & 3) == 0) {
#pragma unroll
                    for (int q = 0; q < NB / 4; ++q)
                        reinterpret_cast<float4*>(myrow)[q] =
                            make_float4(acc[(4 * q) / PW][(4 * q) % PW], acc[(4 * q + 1) / PW][(4 * q + 1) % PW],
                                        acc[(4 * q + 2) / PW][(4 * q + 2) % PW], acc[(4 * q + 3) / PW][(4 * q + 3) % PW]);
                } else {
#pragma unroll
                    for (int i = 0; i < NB; ++i) myrow[i] = acc[i / PW][i % PW];
                }
                float* gdst = out + ((size_t)ka * C + ca) * NB;
                const unsigned bytes = (unsigned)cn * NB * 4u;
                if (((reinterpret_cast<uintptr_t>(gdst) & 15) == 0) && (bytes & 15u) == 0) {
                    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
                    __syncwarp();
                    if (lane == 0) bulk_store_issue(gdst, sOut, bytes);
                    pending = true;
                } else {
                    __syncwarp();
                    for (int i = lane; i < cn * NB; i += 32) gdst[i] = sOut[i];
                    __syncwarp();
                }
            }
        } else {
            // footprint larger than the staged path: everything through the generic tile body, the output tile as scratch
            process_tile<PH, PW, false, float, true, OCL, true>(feat, B, C, H, W, rois, scale, sr, aligned, out, (long long)ka,
                                                                ca, cn, prep, prep_tabs, sOut,
                                                                reinterpret_cast<float*>(base + S::kOffTab + par * S::kTabBytes),
                                                                lane, a0, a1, &pending);
            load_after_next();
            __syncwarp();
            if (have_next && n1.y && !next_issued && nbn <= kTmaVRows) {
                tma_issue<PH, PW>(&tmap, n0, n1, kn, cnx, prep_tabs, sbase + v_off(par ^ 1, nbn),
                                  sbase + S::kOffTab + (par ^ 1) * S::kTabBytes, sbar + 8 * (par ^ 1));
                next_issued = true;
            }
        }
        if (!have_next) break;
        t = tn; ka = kn; ca = cnx; a0 = n0; a1 = n1;
        tn = tm; kn = km; cnx = cm; n0 = m0; n1 = m1;
        cur_issued = next_issued;
        par ^= 1;
    }
    if (pending && lane == 0) bulk_store_wait_read();
}

// Any output size / any parameters: one thread per output element, direct sampling.
template <bool NHWC, typename T>
__global__ void __launch_bounds__(256)
roi_align_generic_kernel(const T* __restrict__ feat, int B, int C, int H, int W,
                         const float* __restrict__ rois, long long total, int PH, int PW, float scale,
                         int sr, int aligned, T* __restrict__ out, int out_cl) {
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        // idx is the linear index of the output element in its own layout ([K][C][PH][PW] or [K][PH][PW][C])
        int pw, ph, c;
        if (out_cl) {
            c = (int)(idx % C); pw = (int)((idx / C) % PW); ph = (int)((idx / ((long long)C * PW)) % PH);
        } else {
            pw = (int)(idx % PW); ph = (int)((idx / PW) % PH); c = (int)((idx / ((long long)PW * PH)) % C);
        }
        const long long k = idx / ((long long)PW * PH * C);
        const Geom g = roi_geometry(rois + 5 * k, scale, sr, aligned, PH, PW);
        float s = 0.0f;
        if (g.b >= 0 && g.b < B) {
            const size_t ps = NHWC ? (size_t)C : 1;
            const T* base = feat + (NHWC ? (size_t)g.b * H * W * C + c : ((size_t)g.b * C + c) * H * W);
            for (int iy = 0; iy < g.gh; ++iy) {
                const Tap ty = make_tap(sample_pos(g.sh, ph, g.bh, iy, g.gh), H);
                for (int ix = 0; ix < g.gw; ++ix) {
                    const Tap tx = make_tap(sample_pos(g.sw, pw, g.bw, ix, g.gw), W);
                    if (ty.valid && tx.valid) {
                        const float v1 = ldf<T>(base + ((size_t)ty.lo * W + tx.lo) * ps);
                        const float v2 = ldf<T>(base + ((size_t)ty.lo * W + tx.hi) * ps);
                        const float v3 = ldf<T>(base + ((size_t)ty.hi * W + tx.lo) * ps);
                        const float v4 = ldf<T>(base + ((size_t)ty.hi * W + tx.hi) * ps);
                        s += ty.wlo * tx.wlo * v1 + ty.wlo * tx.whi * v2 + ty.whi * tx.wlo * v3 +
                             ty.whi * tx.whi * v4;
                    }
                }
            }
        }
        out[idx] = from_f<T>(__fdiv_rn(s, g.count));
    }
}


// ---- per-device launch state ---------------------------------------------------------------------------
// Function attributes (the dynamic shared-memory opt-in), occupancy and the scratch pool belong to a device,
// not to the process: a host application may drive several GPUs from one process.  Each kernel instantiation
// keeps one slot per device ordinal; a race between two host threads writes the same values twice.
constexpr int kMaxDevices = 64;

inline int device_ordinal() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
    return dev;
}

// Warps of Kern the current device holds at once (and the shared-memory opt-in, once per device).
template <auto Kern>
int resident_warps_of(int warps_per_cta, int smem_bytes, int* out) {
    static int cache[kMaxDevices];
    const int dev = device_ordinal();
    if (!cache[dev]) {
        int sms = 0, per_sm = 0;
        B200_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        B200_CUDA(cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, Kern, warps_per_cta * 32, smem_bytes));
        cache[dev] = sms * (per_sm > 0 ? per_sm : 1) * warps_per_cta;
    }
    *out = cache[dev];
    return B200_OK;
}

// Warps a launch of the walking kernels (multi-tile, pipelined, TMA) needs: they are taken in groups of `resident`
// (what the device holds at once), each group covering a window of resident * tiles_per_warp consecutive tiles; the
// last window may need fewer warps than a group.
long long walker_warps(long long tiles, int resident, int tiles_per_warp) {
    const long long window = (long long)resident * tiles_per_warp;
    const long long groups = (tiles + window - 1) / window;
    const long long last = tiles - (groups - 1) * window;                 // tiles in the last window
    return (groups - 1) * resident + (last < resident ? last : resident);
}

// Tiles per warp of the TMA kernels, both directions: 16 amortise a warp's start-up (mbarrier init, first un-overlapped
// load) best, but a warp that walks 16 tiles lives ~60 us; a launch of only a few waves (8 streams of BASELINE config 5:
// 16 384 tiles) would then hold every SM slot from start to end and the association kernels of the other stream could
// not start beside it.  Keep at least four waves of warps, and never fewer than 2 tiles per warp.
constexpr int kTmaMaxTilesPerWarp = 16;
int tma_tiles_per_warp(long long tiles, int resident) {
    const long long tpw = tiles / ((long long)resident * 4);
    return (int)(tpw < 2 ? 2 : tpw > kTmaMaxTilesPerWarp ? kTmaMaxTilesPerWarp : tpw);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    static std::atomic<void*> cached{nullptr};
    void* fn = cached.load(std::memory_order_acquire);
    if (!fn) {
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            fn = nullptr;
        cached.store(fn, std::memory_order_release);
    }
    return reinterpret_cast<EncodeTiledFn>(fn);
}

// The TMA kernels apply to float32 NCHW tensors whose rows are a multiple of 16 bytes (the tensor map's stride rule) with
// a 16-byte aligned base and dimensions inside the descriptor's limits.  (Half maps would need a 16-column window: not
// built, they stay on the multi-tile kernel.)
bool tma_applies(const float* map, int C, int H, int W) {
    if (((size_t)W * 4) % 16 || (reinterpret_cast<uintptr_t>(map) & 15)) return false;
    if ((unsigned long long)C * H * W * 4 >= (1ull << 40)) return false;
    return encode_tiled_fn() != nullptr;
}
constexpr int kTmaXAlign = 4;                    // cells per 16 bytes of a float32 map row

// The three tensor maps of the TMA kernels over a float32 [B,C,H,W] tensor: boxes of kTmaCols cells x 1 / 3 / 5 rows x
// 32 channels.  False if the driver refuses one.
bool encode_box_maps(const float* map, int B, int C, int H, int W, TmaMaps* out) {
    EncodeTiledFn encode = encode_tiled_fn();
    if (!encode) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)C, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4, (cuuint64_t)C * H * W * 4};
    const cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
    for (int i = 0; i < 3; ++i) {
        const cuuint32_t box[4] = {(cuuint32_t)kTmaCols, (cuuint32_t)(2 * i + 1), 32u, 1u};
        const CUresult r = encode(&out->m[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(map), dims, strides,
                                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                  CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return false;
    }
    return true;
}

// Below this many tiles one fused kernel is faster (the prep kernel costs a dependent launch); above it the
// per-ROI work is done once by roi_prep_kernel and shared by the ROI's channel tiles.
constexpr long long kPrepMinTiles = 16384;

// The two-kernel path of both directions: roi_prep_kernel fills stream-ordered scratch (K records + K tables), then
// `consume(prep, tabs)` launches the kernels that read it, then the scratch is freed behind them.  Returns the first
// error, else what `consume` returns.
template <int PH, int PW, typename Consume>
int with_prep(const float* rois, long long K, int B, int H, int W, float scale, int sr, int aligned, int xalign,
              cudaStream_t st, Consume consume) {
    using L = TileSmem<PH, PW>;
    cudaMemPool_t pool = nullptr;
    int rc = scratch_pool(&pool);
    if (rc) return rc;
    char* ws = nullptr;
    const size_t rec = (size_t)K * sizeof(RoiPrep), tab = (size_t)K * L::kTabFloats * sizeof(float);
    B200_CUDA(cudaMallocFromPoolAsync(reinterpret_cast<void**>(&ws), rec + tab, pool, st));
    RoiPrep* prep = reinterpret_cast<RoiPrep*>(ws);
    float* tabs = reinterpret_cast<float*>(ws + rec);
    roi_prep_kernel<PH, PW><<<(unsigned)((K + 3) / 4), 128, 0, st>>>(rois, K, B, H, W, scale, sr, aligned, prep, tabs,
                                                                     xalign);
    rc = check_launch("roi_prep_kernel");
    if (rc == B200_OK) rc = consume(prep, tabs);
    B200_CUDA(cudaFreeAsync(ws, st));
    return rc;
}

// The tile kernels that follow roi_prep_kernel in the stream are launched as its programmatic dependents (launch_ex with
// pdl): they become resident while the prep kernel still runs and wait for it with griddepcontrol.wait before they read a
// record (-1.8 us per launch).  Measured A/B on the overlapped 64-stream step (profiles/r02_roi_pdl_ab.txt): channels-last
// 221.0 -> 220.4 us, but NCHW 235.4 -> 238.9 us -- the early-resident TMA CTAs take the SM slots that the association
// chain's first kernel, released by the same event a few microseconds later, would otherwise get first -- so the TMA
// kernel stays an ordinary launch.

// Launches the TMA-staged kernel (the caller has checked tma_applies); returns 1 when it cannot.
template <int PH, int PW, bool OCL>
int launch_tma(const float* feat, int B, int C, int H, int W, const float* rois, long long K, float scale, int sr,
               int aligned, float* out, int ctiles, const RoiPrep* prep, const float* tabs, long long tiles,
               cudaStream_t st) {
    constexpr int smem_bytes = TmaSmem<PH, PW>::kBytesPerCta;
    TmaMaps tmap;
    if ((reinterpret_cast<uintptr_t>(tabs) & 15) || !encode_box_maps(feat, B, C, H, W, &tmap)) return 1;
    constexpr auto kern = roi_align_tma_kernel<PH, PW, OCL>;
    int resident = 0;
    const int rc = resident_warps_of<kern>(kTmaWarps, smem_bytes, &resident);
    if (rc) return rc;
    const int tpw = tma_tiles_per_warp(tiles, resident);
    const long long warps = walker_warps(tiles, resident, tpw);
    launch_ex(kern, dim3((unsigned)((warps + kTmaWarps - 1) / kTmaWarps)), dim3(kTmaWarps * 32), (size_t)smem_bytes, st, false, 0,
              tmap, feat, B, C, H, W, rois, K, scale, sr, aligned, out, ctiles, prep, tabs, resident, tpw);
    return check_launch("roi_align_tma_kernel");
}

// Launches the pipelined kernel when it applies (channels-last map; NCHW output needs 16-byte rows of a lane's result
// and a 16-byte aligned base; half maps need 16-byte copies); returns 1 when it does not.
template <int PH, int PW, bool NHWC, bool OCL, typename T>
int launch_pipe(const T* feat, int B, int C, int H, int W, const float* rois, long long K, float scale, int sr,
                int aligned, T* out, int ctiles, const RoiPrep* prep, const float* tabs, long long tiles,
                cudaStream_t st) {
    // Channels-last maps only: with NCHW maps the 4-byte plane-strided staging already keeps the LSU pipe ~40 %
    // busy, and the extra shared-memory pass of the copy-out makes the pipelined kernel slower than the tiled one
    // (g64 launch: 275 us vs 232 us); channels-last has the headroom (191 us vs 208 us).
    if constexpr (NHWC && (OCL || (PH * PW * sizeof(T)) % (sizeof(T) == 4 ? 16 : 4) == 0)) {
        using P = PipeSmem<PH, PW>;
        if (!OCL && ((reinterpret_cast<uintptr_t>(out) & 15) || (sizeof(T) == 2 && (C & 1)))) return 1;
        if (sizeof(T) == 2 && ((C & 7) || (reinterpret_cast<uintptr_t>(feat) & 15))) return 1;   // half: 16-byte copies only
        constexpr auto kern = roi_align_pipe_kernel<PH, PW, OCL, T>;
        int resident_warps = 0;
        const int rcw = resident_warps_of<kern>(kPipeWarps, P::kBytesPerCta, &resident_warps);
        if (rcw) return rcw;
        const long long warps = walker_warps(tiles, resident_warps, kPipeTilesPerWarp);
        launch_ex(kern, dim3((unsigned)((warps + kPipeWarps - 1) / kPipeWarps)), dim3(kPipeWarps * 32), (size_t)P::kBytesPerCta, st,
                  true, 0, feat, B, C, H, W, rois, K, scale, sr, aligned, out, ctiles, prep, tabs, resident_warps,
                  (int)kPipeTilesPerWarp);
        return check_launch("roi_align_pipe_kernel");
    } else {
        return 1;
    }
}

template <int PH, int PW, bool NHWC, bool OCL, typename T>
int launch_tile(const T* feat, int B, int C, int H, int W, const float* rois, long long K,
                float scale, int sr, int aligned, T* out, cudaStream_t st) {
    using L = TileSmem<PH, PW>;
    static bool configured[kMaxDevices];     // per instantiation and device; the attribute is idempotent
    auto fused = roi_align_tile_kernel<PH, PW, NHWC, T, false, OCL>;
    const int dev = device_ordinal();
    if (!configured[dev]) {
        B200_CUDA(cudaFuncSetAttribute(fused, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kBytesPerCta));
        configured[dev] = true;
    }
    const int ctiles = (C + 31) / 32;
    const long long warps = K * ctiles;
    const long long blocks = (warps + kWarpsPerCta - 1) / kWarpsPerCta;
    if (blocks > 0x7fffffffLL) return fail(B200_EINVAL, "roi_align: too many ROI tiles (%lld)", blocks);
    if (warps < kPrepMinTiles || ctiles < 4) {
        fused<<<(unsigned)blocks, kWarpsPerCta * 32, L::kBytesPerCta, st>>>(feat, B, C, H, W, rois, K, scale, sr,
                                                                            aligned, out, ctiles, nullptr, nullptr);
        return check_launch("roi_align_tile_kernel");
    }
    constexpr bool kTmaLayout = !NHWC && std::is_same_v<T, float>;
    bool use_tma = false;
    if constexpr (kTmaLayout) use_tma = tma_applies(feat, C, H, W);
    return with_prep<PH, PW>(rois, K, B, H, W, scale, sr, aligned, use_tma ? kTmaXAlign : 1, st,
                             [&](const RoiPrep* prep, const float* tabs) {
        int rc = 1;
        if constexpr (kTmaLayout)
            if (use_tma) rc = launch_tma<PH, PW, OCL>(feat, B, C, H, W, rois, K, scale, sr, aligned, out, ctiles, prep, tabs, warps, st);
        if (rc == 1) rc = launch_pipe<PH, PW, NHWC, OCL>(feat, B, C, H, W, rois, K, scale, sr, aligned, out, ctiles, prep, tabs, warps, st);
        if (rc == 1) {                       // no TMA / pipelined kernel for this layout / type / size / alignment
            constexpr auto multi = roi_align_multi_kernel<PH, PW, NHWC, T, OCL>;
            int resident_warps = 0;
            rc = resident_warps_of<multi>(kWarpsPerCta, L::kBytesPerCta, &resident_warps);
            if (rc == B200_OK) {
                const long long nw = walker_warps(warps, resident_warps, kMultiTilesPerWarp);
                launch_ex(multi, dim3((unsigned)((nw + kWarpsPerCta - 1) / kWarpsPerCta)), dim3(kWarpsPerCta * 32),
                          (size_t)L::kBytesPerCta, st, true, 0, feat, B, C, H, W, rois, K, scale, sr, aligned, out, ctiles, prep,
                          tabs, resident_warps, kMultiTilesPerWarp);
                rc = check_launch("roi_align_multi_kernel");
            }
        }
        return rc;
    });
}

// ---- dispatch shared by both directions -----------------------------------------------------------------------
template <int V> using IntC = std::integral_constant<int, V>;
template <bool V> using BoolC = std::integral_constant<bool, V>;

// Output sizes with tile kernels (10x10, 7x7) go to tiled(IntC<PH>, IntC<PW>, BoolC<a>, BoolC<b>), where a and b are the
// two layout flags the launchers take as template parameters; every other size goes to generic().
template <typename Tiled, typename Generic>
int dispatch_size(int PH, int PW, bool a, bool b, Tiled tiled, Generic generic) {
    auto layouts = [&](auto ph, auto pw) {
        if (a) return b ? tiled(ph, pw, BoolC<true>(), BoolC<true>()) : tiled(ph, pw, BoolC<true>(), BoolC<false>());
        return b ? tiled(ph, pw, BoolC<false>(), BoolC<true>()) : tiled(ph, pw, BoolC<false>(), BoolC<false>());
    };
    if (PH == 10 && PW == 10) return layouts(IntC<10>(), IntC<10>());
    if (PH == 7 && PW == 7) return layouts(IntC<7>(), IntC<7>());
    return generic();
}

// Shape and pointer checks of both directions; `op` starts every message, `map` names the [B,C,H,W] tensor.  Pointers
// are not looked at when there are no ROIs.
int check_shapes(const char* op, const char* map, int B, int C, int H, int W, int PH, int PW, int64_t K, bool null_ptr) {
    B200_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "%s: bad %s shape [%d,%d,%d,%d]", op, map, B, C, H, W);
    B200_REQUIRE(PH > 0 && PW > 0, "%s: bad output size (%d,%d)", op, PH, PW);
    B200_REQUIRE(K >= 0, "%s: negative ROI count", op);
    B200_REQUIRE(K == 0 || !null_ptr, "%s: null pointer", op);
    return B200_OK;
}

// Grid of the generic kernels: one thread per element, at most 32 CTAs of 256 threads per SM (grid-stride loop).
unsigned generic_blocks(long long total) {
    const long long want = (total + 255) / 256;
    return (unsigned)(want < (long long)kSMs * 32 ? want : (long long)kSMs * 32);
}

// Calls fn(float()) or fn(__half()) for a B200_DTYPE_* of the map / gradient; EINVAL for any other.
template <typename Fn>
int with_dtype(int dtype, const char* op, Fn fn) {
    if (dtype == B200_DTYPE_F32) return fn(float());
    if (dtype == B200_DTYPE_F16) return fn(__half());
    return fail(B200_EINVAL, "%s: bad dtype %d", op, dtype);
}

template <typename T>
int roi_align_dispatch(const T* feat, int layout, int B, int C, int H, int W, const float* rois, int64_t K, int PH,
                       int PW, float spatial_scale, int sampling_ratio, int aligned, T* out, int out_layout,
                       void* stream) {
    B200_REQUIRE(layout == B200_LAYOUT_NCHW || layout == B200_LAYOUT_NHWC, "roi_align: bad layout %d", layout);
    B200_REQUIRE(out_layout == B200_LAYOUT_NCHW || out_layout == B200_LAYOUT_NHWC, "roi_align: bad output layout %d",
                 out_layout);
    if (const int rc = check_shapes("roi_align", "feature", B, C, H, W, PH, PW, K, !feat || !rois || !out)) return rc;
    if (K == 0) return B200_OK;
    cudaStream_t st = as_stream(stream);
    const bool nhwc = layout == B200_LAYOUT_NHWC, ocl = out_layout == B200_LAYOUT_NHWC;
    return dispatch_size(
        PH, PW, nhwc, ocl,
        [&](auto ph, auto pw, auto map_cl, auto out_cl) {
            return launch_tile<ph, pw, map_cl, out_cl, T>(feat, B, C, H, W, rois, K, spatial_scale, sampling_ratio, aligned,
                                                          out, st);
        },
        [&] {
            const long long total = (long long)K * C * PH * PW;
            const auto kern = nhwc ? roi_align_generic_kernel<true, T> : roi_align_generic_kernel<false, T>;
            kern<<<generic_blocks(total), 256, 0, st>>>(feat, B, C, H, W, rois, total, PH, PW, spatial_scale, sampling_ratio,
                                                        aligned, out, ocl);
            return check_launch("roi_align_generic_kernel");
        });
}

// ---- ROI Align backward (torchvision's _roi_align_backward) ---------------------------------------------------
// The forward pass contracts a footprint with two weight tables, out[ph][pw] = sum_y,x Wy[y][ph] Wx[x][pw] V[y][x];
// the gradient is its transpose, G[y][x] = sum_ph Wy[y][ph] * (sum_pw Wx[x][pw] * g[ph][pw]), ADDED into grad_in because
// the footprints of different ROIs overlap.  Same work unit (one warp per (ROI, 32-channel tile), lane = channel), same
// tables (built per warp, or once per ROI by roi_prep_kernel), G[8][8] in registers.  Kernels, by launch:
//   roi_align_bwd_tile_kernel  small launches (tables built per warp), and on large ones with prep tables whenever the
//                              TMA kernel does not apply; scalar red.global.add per cell (NHWC grad_in: one 128-byte line
//                              per warp instruction);
//   roi_align_bwd_tma_kernel   large launches into float32 NCHW grad_in: G is written to shared memory in the forward
//                              pass's box layout V[channel][row][8 cells] and added to the map by the TMA engine
//                              (cp.reduce.async.bulk.tensor .add, SASS UTMAREDG), 1 / 3 / 5-row boxes as in the forward
//                              kernel; the grad_out chunk and the tables of the next tile arrive while the current one
//                              contracts;
//   footprints the staged path cannot hold take torchvision's algorithm (per-sample scalar atomics) inside the tile
//   kernel -- after the TMA kernel, in a launch of their own, so that generic-proxy atomics and TMA reductions never
//   target the same cells concurrently; roi_align_bwd_generic_kernel: output sizes without a template, one thread per
//   grad_out element, the same algorithm.
// The order of the additions is not fixed, so the result is not bit-reproducible.
__device__ __forceinline__ void red_add(float* p, float v) { atomicAdd(p, v); }     // result unused: RED

// grad_in += the four taps of one sample, scaled like torchvision: (g * w) / count.
__device__ __forceinline__ void bwd_sample(float* __restrict__ gi, size_t ps, int W, const Tap& ty, const Tap& tx, float g,
                                           float count) {
    if (!(ty.valid && tx.valid)) return;
    red_add(gi + ((size_t)ty.lo * W + tx.lo) * ps, __fdiv_rn(g * (ty.wlo * tx.wlo), count));
    red_add(gi + ((size_t)ty.lo * W + tx.hi) * ps, __fdiv_rn(g * (ty.wlo * tx.whi), count));
    red_add(gi + ((size_t)ty.hi * W + tx.lo) * ps, __fdiv_rn(g * (ty.whi * tx.wlo), count));
    red_add(gi + ((size_t)ty.hi * W + tx.hi) * ps, __fdiv_rn(g * (ty.whi * tx.whi), count));
}

// Element (k, c, bin) of grad_out, stored [K][C][PH*PW] or channels-last [K][PH*PW][C].
template <typename T, bool GCL>
__device__ __forceinline__ float grad_at(const T* __restrict__ go, long long k, int C, int NB, int c, int bin) {
    return ldf<T>(GCL ? go + ((size_t)k * NB + bin) * C + c : go + ((size_t)k * C + c) * NB + bin);
}

// G[y][x] = sum_ph Wy[y][ph] * sum_pw Wx[x][pw] * g(ph, pw) over the 8 x 8 staged footprint (rows / columns outside the
// footprint have zero weights, so their G is zero).
template <int PH, int PW, typename LoadG>
__device__ __forceinline__ void bwd_contract(float (&G)[kFootCap][kFootCap], const float* sWy, const float* sWx, LoadG loadg) {
    constexpr int PHP = (PH + 3) & ~3, PWP = (PW + 3) & ~3;
#pragma unroll
    for (int y = 0; y < kFootCap; ++y)
#pragma unroll
        for (int x = 0; x < kFootCap; ++x) G[y][x] = 0.0f;
#pragma unroll 1
    for (int ph = 0; ph < PH; ++ph) {
        float g[PW];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) g[pw] = loadg(ph, pw);
        float t[kFootCap];
#pragma unroll
        for (int x = 0; x < kFootCap; ++x) {
            const float4* w4 = reinterpret_cast<const float4*>(sWx + x * PWP);
            float s = 0.0f;
#pragma unroll
            for (int q = 0; q < PWP / 4; ++q) {
                const float4 w = w4[q];
                if (4 * q + 0 < PW) s = fmaf(w.x, g[4 * q + 0], s);
                if (4 * q + 1 < PW) s = fmaf(w.y, g[4 * q + 1], s);
                if (4 * q + 2 < PW) s = fmaf(w.z, g[4 * q + 2], s);
                if (4 * q + 3 < PW) s = fmaf(w.w, g[4 * q + 3], s);
            }
            t[x] = s;
        }
#pragma unroll
        for (int y = 0; y < kFootCap; ++y) {
            const float wy = sWy[y * PHP + ph];
#pragma unroll
            for (int x = 0; x < kFootCap; ++x) G[y][x] = fmaf(wy, t[x], G[y][x]);
        }
    }
}

// Tiles of a footprint the staged path cannot hold: every sample of every bin, lane = channel.
template <int PH, int PW, typename T, bool GCL, bool ICL>
__device__ __forceinline__ void bwd_tile_exact(const T* __restrict__ go, const float* __restrict__ rois, long long k, int c0,
                                               int cn, float scale, int sr, int aligned, float* __restrict__ gi, int B,
                                               int C, int H, int W, int lane) {
    const Geom g = roi_geometry(rois + 5 * k, scale, sr, aligned, PH, PW);
    if (g.b < 0 || g.b >= B || lane >= cn) return;
    const int c = c0 + lane;
    float* base = gi + (ICL ? (size_t)g.b * H * W * C + c : ((size_t)g.b * C + c) * H * W);
    const size_t ps = ICL ? (size_t)C : 1;
#pragma unroll 1
    for (int bin = 0; bin < PH * PW; ++bin) {
        const int ph = bin / PW, pw = bin - ph * PW;
        const float gv = grad_at<T, GCL>(go, k, C, PH * PW, c, bin);
        for (int iy = 0; iy < g.gh; ++iy) {
            const Tap ty = make_tap(sample_pos(g.sh, ph, g.bh, iy, g.gh), H);
            for (int ix = 0; ix < g.gw; ++ix)
                bwd_sample(base, ps, W, ty, make_tap(sample_pos(g.sw, pw, g.bw, ix, g.gw), W), gv, g.count);
        }
    }
}

// One warp per (ROI, 32-channel tile).  MODE 0: tables built by the warp (small launches); 1: footprint and tables from
// roi_prep_kernel; 2: as 1 but only the tiles roi_prep_kernel did not stage (the rest went through the TMA kernel).
template <int PH, int PW, typename T, bool GCL, bool ICL, int MODE>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
roi_align_bwd_tile_kernel(const T* __restrict__ go, const float* __restrict__ rois, long long K, float scale, int sr,
                          int aligned, float* __restrict__ gi, int B, int C, int H, int W, int ctiles,
                          const RoiPrep* __restrict__ prep, const float* __restrict__ prep_tabs) {
    using L = TileSmem<PH, PW>;
    __shared__ __align__(16) float sTabs[kWarpsPerCta][L::kTabFloats];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long wi = (long long)blockIdx.x * kWarpsPerCta + warp;
    if (wi >= K * ctiles) return;
    const long long k = wi / ctiles;
    const int c0 = (int)(wi - k * ctiles) * 32, cn = min(32, C - c0);
    float* sWy = sTabs[warp];
    float* sWx = sWy + kFootCap * L::kPHP;
    int b, ymin, xmin, FY, FX;
    bool staged;
    if (MODE == 0) {
        const Geom g = roi_geometry(rois + 5 * k, scale, sr, aligned, PH, PW);
        axis_footprint(g.sh, g.bh, PH, g.gh, H, &ymin, &FY);
        axis_footprint(g.sw, g.bw, PW, g.gw, W, &xmin, &FX);
        if (g.b < 0 || g.b >= B || FY == 0 || FX == 0) return;
        b = g.b;
        staged = FY <= kFootCap && FX <= kFootCap;
        if (staged) build_tables<PH, PW>(g, __fdiv_rn(1.0f, g.count), H, W, ymin, xmin, FY, sWy, sWx, L::kTabFloats, lane);
    } else {
        const int4 h0 = reinterpret_cast<const int4*>(prep + k)[0], h1 = reinterpret_cast<const int4*>(prep + k)[1];
        b = h0.x; ymin = h0.y; xmin = h0.z; FY = h0.w; FX = h1.x;
        staged = h1.y != 0;
        if (MODE == 2 && staged) return;
        if (staged) {
            if (FY == 0) return;
            const float4* src = reinterpret_cast<const float4*>(prep_tabs + (size_t)k * L::kTabFloats);
            for (int i = lane; i < L::kTabFloats / 4; i += 32) reinterpret_cast<float4*>(sWy)[i] = src[i];
        }
    }
    if (!staged) {
        bwd_tile_exact<PH, PW, T, GCL, ICL>(go, rois, k, c0, cn, scale, sr, aligned, gi, B, C, H, W, lane);
        return;
    }
    __syncwarp();
    const int c = c0 + (lane < cn ? lane : 0);
    float G[kFootCap][kFootCap];
    bwd_contract<PH, PW>(G, sWy, sWx, [&](int ph, int pw) {
        return lane < cn ? grad_at<T, GCL>(go, k, C, PH * PW, c, ph * PW + pw) : 0.0f;
    });
    if (lane >= cn) return;
    float* base = gi + (ICL ? (((size_t)b * H + ymin) * W + xmin) * C + c : (((size_t)b * C + c) * H + ymin) * W + xmin);
    const size_t rs = ICL ? (size_t)W * C : (size_t)W, xs = ICL ? (size_t)C : 1;
#pragma unroll
    for (int y = 0; y < kFootCap; ++y)
        if (y < FY) {
#pragma unroll
            for (int x = 0; x < kFootCap; ++x)
                if (x < FX) red_add(base + y * rs + x * xs, G[y][x]);
        }
}

template <bool GCL, typename T>
__global__ void __launch_bounds__(256)
roi_align_bwd_generic_kernel(const T* __restrict__ go, const float* __restrict__ rois, long long total, int PH, int PW,
                             float scale, int sr, int aligned, float* __restrict__ gi, int ICL, int B, int C, int H, int W) {
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        // idx is the linear index of the grad_out element in its own layout ([K][C][PH][PW] or [K][PH][PW][C])
        int pw, ph, c;
        if (GCL) {
            c = (int)(idx % C); pw = (int)((idx / C) % PW); ph = (int)((idx / ((long long)C * PW)) % PH);
        } else {
            pw = (int)(idx % PW); ph = (int)((idx / PW) % PH); c = (int)((idx / ((long long)PW * PH)) % C);
        }
        const long long k = idx / ((long long)PW * PH * C);
        const Geom g = roi_geometry(rois + 5 * k, scale, sr, aligned, PH, PW);
        if (g.b < 0 || g.b >= B) continue;
        const float gv = to_f32(go[idx]);
        float* base = gi + (ICL ? (size_t)g.b * H * W * C + c : ((size_t)g.b * C + c) * H * W);
        const size_t ps = ICL ? (size_t)C : 1;
        for (int iy = 0; iy < g.gh; ++iy) {
            const Tap ty = make_tap(sample_pos(g.sh, ph, g.bh, iy, g.gh), H);
            for (int ix = 0; ix < g.gw; ++ix)
                bwd_sample(base, ps, W, ty, make_tap(sample_pos(g.sw, pw, g.bw, ix, g.gw), W), gv, g.count);
        }
    }
}

// Per-warp shared memory of the TMA kernel: two slots of (grad_out chunk, tables) -- the current tile and the next --
// and one box buffer of up to 8 rows (a 5-row box and the 1 / 3-row box below it).
template <int PH, int PW, typename T>
struct BwdTmaSmem {
    using L = TileSmem<PH, PW>;
    static constexpr int kGBytes = (32 * PH * PW * (int)sizeof(T) + 15) & ~15;
    static constexpr int kTabBytes = L::kTabFloats * 4;
    static constexpr int kSlotBytes = (kGBytes + kTabBytes + 127) & ~127;
    static constexpr int kOffBox = 2 * kSlotBytes, kOffBar = kOffBox + kFootCap * kTmaRowBytes;   // box: 128-byte aligned
    static constexpr int kBytesPerWarp = (kOffBar + 16 + 127) & ~127;
    static_assert(kTabBytes % 16 == 0, "bulk-copy alignment");
};
constexpr int kBwdTmaWarps = 2;

__device__ __forceinline__ void tma_reduce_add_4d(const CUtensorMap* tm, unsigned src, int x, int y, int c, int b) {
    asm volatile("cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2, %3, %4}], [%5];\n"
                 ::"l"(tm), "r"(x), "r"(y), "r"(c), "r"(b), "r"(src) : "memory");
}

// Requests tile (k, c0)'s tables and, with an NCHW grad_out, its contiguous [cn][PH*PW] chunk on one mbarrier.
template <int PH, int PW, typename T, bool GCL>
__device__ __forceinline__ void bwd_tma_issue(const T* __restrict__ go, int C, unsigned k, int c0, const float* prep_tabs,
                                              unsigned sslot, unsigned bar) {
    using S = BwdTmaSmem<PH, PW, T>;
    constexpr int NB = PH * PW;
    const unsigned ku = (unsigned)bcast0((int)k), su = (unsigned)bcast0((int)sslot), baru = (unsigned)bcast0((int)bar);
    const int cu = bcast0(c0), cn = min(32, C - cu);
    const unsigned gbytes = GCL ? 0u : (unsigned)(cn * NB * (int)sizeof(T));
    if (elect_one()) {
        mbar_expect_tx(baru, (unsigned)S::kTabBytes + gbytes);
        bulk_load(su + S::kGBytes, prep_tabs + (size_t)ku * S::L::kTabFloats, S::kTabBytes, baru);
        if (!GCL) bulk_load(su, go + ((size_t)ku * C + cu) * NB, gbytes, baru);
    }
    __syncwarp();
}

// Large launches into a float32 NCHW grad_in (tma_applies).  Tiles are handed out as in roi_align_tma_kernel; tiles that
// roi_prep_kernel did not stage are left to a later roi_align_bwd_tile_kernel<MODE 2> launch.
template <int PH, int PW, typename T, bool GCL>
__global__ void __launch_bounds__(kBwdTmaWarps * 32)
roi_align_bwd_tma_kernel(const __grid_constant__ TmaMaps tmap, const T* __restrict__ go, long long K, int C, int ctiles,
                         const RoiPrep* __restrict__ prep, const float* __restrict__ prep_tabs, int group_warps,
                         int tiles_per_warp) {
    using S = BwdTmaSmem<PH, PW, T>;
    constexpr int NB = PH * PW, PHP = S::L::kPHP;
    extern __shared__ __align__(128) unsigned char smem_bwd[];
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    unsigned char* base = smem_bwd + (size_t)warp * S::kBytesPerWarp;
    const unsigned sbase = (unsigned)__cvta_generic_to_shared(base);
    const unsigned sbar = sbase + S::kOffBar, sbox = sbase + S::kOffBox;
    const unsigned gw = blockIdx.x * kBwdTmaWarps + warp, grp = gw / (unsigned)group_warps;
    const unsigned stride = (unsigned)group_warps, window = stride * (unsigned)tiles_per_warp;
    unsigned t = grp * window + (gw - grp * stride);
    const unsigned total = (unsigned)min((long long)(grp + 1) * window, K * ctiles);
    if (t >= total) return;
    if (lane == 0) {
        mbar_init(sbar, 1);
        mbar_init(sbar + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncwarp();
    auto wanted = [](int4 h0, int4 h1) { return h1.y != 0 && h0.w != 0; };     // staged and sampling something
    unsigned ka = t / (unsigned)ctiles;
    int ca = (int)(t - ka * (unsigned)ctiles) * 32;
    int4 a0 = reinterpret_cast<const int4*>(prep + ka)[0], a1 = reinterpret_cast<const int4*>(prep + ka)[1];
    if (wanted(a0, a1)) bwd_tma_issue<PH, PW, T, GCL>(go, C, ka, ca, prep_tabs, sbase, sbar);
    int par = 0;
    unsigned phase = 0;                // bit p = parity the next wait on mbarrier p expects
    bool pending = false;              // a reduction may still be reading the box buffer
    for (;;) {
        const unsigned tn = t + stride;
        const bool have_next = tn < total;
        unsigned kn = 0;
        int cnx = 0;
        int4 n0 = make_int4(0, 0, 0, 0), n1 = n0;
        if (have_next) {
            kn = tn / (unsigned)ctiles;
            cnx = (int)(tn - kn * (unsigned)ctiles) * 32;
            n0 = reinterpret_cast<const int4*>(prep + kn)[0];
            n1 = reinterpret_cast<const int4*>(prep + kn)[1];
            // slot par ^ 1 was consumed by the previous tile (the warp converged after reading it)
            if (wanted(n0, n1))
                bwd_tma_issue<PH, PW, T, GCL>(go, C, kn, cnx, prep_tabs, sbase + (par ^ 1) * S::kSlotBytes, sbar + 8 * (par ^ 1));
        }
        if (wanted(a0, a1)) {
            mbar_wait(sbar + 8 * par, (phase >> par) & 1u);
            phase ^= 1u << par;
            const unsigned char* slot = base + par * S::kSlotBytes;
            const float* sWy = reinterpret_cast<const float*>(slot + S::kGBytes);
            const T* sg = reinterpret_cast<const T*>(slot);
            const int cn = min(32, C - ca);
            const int c = ca + (lane < cn ? lane : 0);
            float G[kFootCap][kFootCap];
            bwd_contract<PH, PW>(G, sWy, sWy + kFootCap * PHP, [&](int ph, int pw) {
                if (lane >= cn) return 0.0f;
                return GCL ? grad_at<T, true>(go, ka, C, NB, c, ph * PW + pw) : to_f32(sg[lane * NB + ph * PW + pw]);
            });
            __syncwarp();              // this slot is free for the tile after next
            if (pending && lane == 0) bulk_store_wait_read();
            __syncwarp();
            // G -> box buffer: rows 0-4 (or fewer) in the first box [32][r0][8], rows 5-7 in the second box [32][r1][8]
            const int FY = a0.w, ymin = a0.y, xmin = a0.z, b = a0.x;
            const int r0 = FY > kTmaRows ? kTmaRows : tma_box_rows(FY);
            const int r1 = FY > kTmaRows ? tma_box_rows(FY - kTmaRows) : 0;
            unsigned char* box0 = base + S::kOffBox + lane * (r0 * 32);
            unsigned char* box1 = base + S::kOffBox + kTmaRows * kTmaRowBytes + lane * (r1 * 32);
#pragma unroll
            for (int y = 0; y < kFootCap; ++y) {
                if (y < r0 || (y >= kTmaRows && y < kTmaRows + r1)) {
                    float4* row = reinterpret_cast<float4*>(y < kTmaRows ? box0 + y * 32 : box1 + (y - kTmaRows) * 32);
                    row[0] = make_float4(G[y][0], G[y][1], G[y][2], G[y][3]);
                    row[1] = make_float4(G[y][4], G[y][5], G[y][6], G[y][7]);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                tma_reduce_add_4d(&tmap.m[r0 >> 1], sbox, xmin, ymin, ca, b);
                if (r1) tma_reduce_add_4d(&tmap.m[r1 >> 1], sbox + kTmaRows * kTmaRowBytes, xmin, ymin + kTmaRows, ca, b);
                asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
            }
            pending = true;
        }
        if (!have_next) break;
        t = tn; ka = kn; ca = cnx; a0 = n0; a1 = n1;
        par ^= 1;
    }
    if (pending && lane == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
    __syncwarp();
}

template <int PH, int PW, typename T, bool GCL, bool ICL, int MODE>
int launch_bwd_tile(const T* go, const float* rois, long long K, float scale, int sr, int aligned, float* gi, int B, int C,
                    int H, int W, int ctiles, const RoiPrep* prep, const float* tabs, cudaStream_t st) {
    const long long blocks = (K * ctiles + kWarpsPerCta - 1) / kWarpsPerCta;
    roi_align_bwd_tile_kernel<PH, PW, T, GCL, ICL, MODE><<<(unsigned)blocks, kWarpsPerCta * 32, 0, st>>>(
        go, rois, K, scale, sr, aligned, gi, B, C, H, W, ctiles, prep, tabs);
    return check_launch("roi_align_bwd_tile_kernel");
}

// Launches the TMA kernel (the caller has checked tma_applies); returns 1 when it cannot.
template <int PH, int PW, typename T, bool GCL>
int launch_bwd_tma(const T* go, long long K, float* gi, int B, int C, int H, int W, int ctiles, const RoiPrep* prep,
                   const float* tabs, long long tiles, cudaStream_t st) {
    constexpr int smem_bytes = BwdTmaSmem<PH, PW, T>::kBytesPerWarp * kBwdTmaWarps;
    TmaMaps tmap;
    if ((reinterpret_cast<uintptr_t>(tabs) & 15) || !encode_box_maps(gi, B, C, H, W, &tmap)) return 1;
    constexpr auto kern = roi_align_bwd_tma_kernel<PH, PW, T, GCL>;
    int resident = 0;
    const int rc = resident_warps_of<kern>(kBwdTmaWarps, smem_bytes, &resident);
    if (rc) return rc;
    const int tpw = tma_tiles_per_warp(tiles, resident);
    const long long warps = walker_warps(tiles, resident, tpw);
    kern<<<(unsigned)((warps + kBwdTmaWarps - 1) / kBwdTmaWarps), kBwdTmaWarps * 32, smem_bytes, st>>>(
        tmap, go, K, C, ctiles, prep, tabs, resident, tpw);
    return check_launch("roi_align_bwd_tma_kernel");
}

template <int PH, int PW, typename T, bool GCL, bool ICL>
int launch_bwd(const T* go, const float* rois, long long K, float scale, int sr, int aligned, float* gi, int B, int C, int H,
               int W, cudaStream_t st) {
    const int ctiles = (C + 31) / 32;
    const long long tiles = K * ctiles;
    if ((tiles + kWarpsPerCta - 1) / kWarpsPerCta > 0x7fffffffLL || tiles >= (1LL << 32))
        return fail(B200_EINVAL, "roi_align_backward: too many ROI tiles (%lld)", tiles);
    if (tiles < kPrepMinTiles || ctiles < 4)
        return launch_bwd_tile<PH, PW, T, GCL, ICL, 0>(go, rois, K, scale, sr, aligned, gi, B, C, H, W, ctiles, nullptr,
                                                       nullptr, st);
    // the TMA kernel also bulk-loads NCHW grad_out chunks [cn][PH*PW]: each must be whole 16-byte units at a 16-byte boundary
    const bool use_tma = !ICL && tma_applies(gi, C, H, W) &&
                         (GCL || (((size_t)C * PH * PW * sizeof(T)) & 15) == 0 && (reinterpret_cast<uintptr_t>(go) & 15) == 0);
    return with_prep<PH, PW>(rois, K, B, H, W, scale, sr, aligned, use_tma ? kTmaXAlign : 1, st,
                             [&](const RoiPrep* prep, const float* tabs) {
        int rc = 1;
        if constexpr (!ICL) {
            if (use_tma) {
                rc = launch_bwd_tma<PH, PW, T, GCL>(go, K, gi, B, C, H, W, ctiles, prep, tabs, tiles, st);
                if (rc == B200_OK)
                    rc = launch_bwd_tile<PH, PW, T, GCL, ICL, 2>(go, rois, K, scale, sr, aligned, gi, B, C, H, W, ctiles,
                                                                 prep, tabs, st);
            }
        }
        // no TMA kernel (channels-last grad_in, alignment): the tile kernel with the prep records
        if (rc == 1)
            rc = launch_bwd_tile<PH, PW, T, GCL, ICL, 1>(go, rois, K, scale, sr, aligned, gi, B, C, H, W, ctiles, prep,
                                                         tabs, st);
        return rc;
    });
}

template <typename T>
int roi_align_bwd_dispatch(const T* go, int go_layout, const float* rois, int64_t K, int PH, int PW, float scale, int sr,
                           int aligned, float* gi, int layout, int B, int C, int H, int W, void* stream) {
    B200_REQUIRE(layout == B200_LAYOUT_NCHW || layout == B200_LAYOUT_NHWC, "roi_align_backward: bad layout %d", layout);
    B200_REQUIRE(go_layout == B200_LAYOUT_NCHW || go_layout == B200_LAYOUT_NHWC,
                 "roi_align_backward: bad grad_out layout %d", go_layout);
    if (const int rc = check_shapes("roi_align_backward", "input", B, C, H, W, PH, PW, K, !go || !rois || !gi)) return rc;
    if (K == 0) return B200_OK;
    cudaStream_t st = as_stream(stream);
    const bool gcl = go_layout == B200_LAYOUT_NHWC, icl = layout == B200_LAYOUT_NHWC;
    return dispatch_size(
        PH, PW, gcl, icl,
        [&](auto ph, auto pw, auto go_cl, auto gi_cl) {
            return launch_bwd<ph, pw, T, go_cl, gi_cl>(go, rois, K, scale, sr, aligned, gi, B, C, H, W, st);
        },
        [&] {
            const long long total = (long long)K * C * PH * PW;
            const auto kern = gcl ? roi_align_bwd_generic_kernel<true, T> : roi_align_bwd_generic_kernel<false, T>;
            kern<<<generic_blocks(total), 256, 0, st>>>(go, rois, total, PH, PW, scale, sr, aligned, gi, icl, B, C, H, W);
            return check_launch("roi_align_bwd_generic_kernel");
        });
}

// ---- box preparation in front of ROI Align (tracking.py:209-213, trainingCard.py:38-69) as one launch -----------
// torch.minimum / maximum / clamp propagate NaN; fminf / fmaxf do not.
__device__ __forceinline__ float t_min(float a, float b) { return (a != a || b != b) ? __int_as_float(0x7fc00000) : fminf(a, b); }
__device__ __forceinline__ float t_max(float a, float b) { return (a != a || b != b) ? __int_as_float(0x7fc00000) : fmaxf(a, b); }
__device__ __forceinline__ float t_clamp(float v, float lo, float hi) { return v != v ? v : fminf(fmaxf(v, lo), hi); }

__global__ void roi_boxes_prep_kernel(const float* __restrict__ boxes, long long n, int stride,
                                      const int32_t* __restrict__ batch_index, int mode, float sx, float sy, float xmax,
                                      float ymax, float min_size, float* __restrict__ rois) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* b = boxes + i * stride;
    float x1 = b[0], y1 = b[1], x2 = b[2], y2 = b[3];
    if (mode == B200_BOXES_TRAINING) {
        const float ax = t_min(x1, x2), bx = t_max(x1, x2), ay = t_min(y1, y2), by = t_max(y1, y2);   // :44-48
        x1 = t_clamp(__fmul_rn(ax, sx), 0.f, xmax);                                                   // :51-62
        x2 = t_clamp(__fmul_rn(bx, sx), 0.f, xmax);
        y1 = t_clamp(__fmul_rn(ay, sy), 0.f, ymax);
        y2 = t_clamp(__fmul_rn(by, sy), 0.f, ymax);
        if (min_size > 0.f) {                                                                         // :64-68
            x2 = t_clamp(t_max(x2, __fadd_rn(x1, min_size)), 0.f, xmax);
            y2 = t_clamp(t_max(y2, __fadd_rn(y1, min_size)), 0.f, ymax);
        }
    }
    float* r = rois + i * 5;
    r[0] = batch_index ? (float)batch_index[i] : 0.f;
    r[1] = x1; r[2] = y1; r[3] = x2; r[4] = y2;
}

}  // namespace
}  // namespace b200

extern "C" int b200_roi_boxes_prep_f32(const float* boxes, int64_t n, int box_stride, const int32_t* batch_index, int mode,
                                       int img_h, int img_w, int Hf, int Wf, float enforce_min_size, float* rois,
                                       void* stream) {
    B200_REQUIRE(n >= 0 && box_stride >= 4, "roi_boxes_prep: need n >= 0 and at least 4 columns per box (got %d)", box_stride);
    B200_REQUIRE(mode == B200_BOXES_INPUT || mode == B200_BOXES_TRAINING, "roi_boxes_prep: bad mode %d", mode);
    if (n == 0) return B200_OK;
    B200_REQUIRE(boxes && rois, "roi_boxes_prep: null pointer");
    float sx = 1.f, sy = 1.f;
    if (mode == B200_BOXES_TRAINING) {
        B200_REQUIRE(img_h > 0 && img_w > 0 && Hf > 0 && Wf > 0, "roi_boxes_prep: bad image / map size");
        sx = (float)((double)Wf / (double)img_w);      // the reference multiplies a float32 tensor by a Python float
        sy = (float)((double)Hf / (double)img_h);
    }
    const unsigned blocks = (unsigned)((n + 127) / 128);
    b200::roi_boxes_prep_kernel<<<blocks, 128, 0, b200::as_stream(stream)>>>(
        boxes, n, box_stride, batch_index, mode, sx, sy, (float)(Wf - 1), (float)(Hf - 1), enforce_min_size, rois);
    return b200::check_launch("roi_boxes_prep_kernel");
}

extern "C" int b200_roi_align_fwd_f32(const float* feat, int layout, int B, int C, int H, int W,
                                      const float* rois, int64_t K, int PH, int PW, float spatial_scale,
                                      int sampling_ratio, int aligned, float* out, void* stream) {
    return b200::roi_align_dispatch<float>(feat, layout, B, C, H, W, rois, K, PH, PW, spatial_scale, sampling_ratio,
                                           aligned, out, B200_LAYOUT_NCHW, stream);
}

extern "C" int b200_roi_align_fwd_f16(const void* feat, int layout, int B, int C, int H, int W,
                                      const float* rois, int64_t K, int PH, int PW, float spatial_scale,
                                      int sampling_ratio, int aligned, void* out, void* stream) {
    return b200::roi_align_dispatch<__half>(static_cast<const __half*>(feat), layout, B, C, H, W, rois, K, PH, PW,
                                            spatial_scale, sampling_ratio, aligned, static_cast<__half*>(out),
                                            B200_LAYOUT_NCHW, stream);
}

extern "C" int b200_roi_align_fwd_ex(const void* feat, int dtype, int layout, int B, int C, int H, int W,
                                     const float* rois, int64_t K, int PH, int PW, float spatial_scale,
                                     int sampling_ratio, int aligned, void* out, int out_layout, void* stream) {
    return b200::with_dtype(dtype, "roi_align", [&](auto zero) {
        using T = decltype(zero);
        return b200::roi_align_dispatch<T>(static_cast<const T*>(feat), layout, B, C, H, W, rois, K, PH, PW, spatial_scale,
                                           sampling_ratio, aligned, static_cast<T*>(out), out_layout, stream);
    });
}

extern "C" int b200_roi_align_bwd_ex(const void* grad_out, int dtype, int grad_out_layout, const float* rois, int64_t K,
                                     int PH, int PW, float spatial_scale, int sampling_ratio, int aligned, float* grad_in,
                                     int layout, int B, int C, int H, int W, void* stream) {
    return b200::with_dtype(dtype, "roi_align_backward", [&](auto zero) {
        using T = decltype(zero);
        return b200::roi_align_bwd_dispatch<T>(static_cast<const T*>(grad_out), grad_out_layout, rois, K, PH, PW,
                                               spatial_scale, sampling_ratio, aligned, grad_in, layout, B, C, H, W, stream);
    });
}

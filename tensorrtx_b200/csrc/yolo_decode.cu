// yolo_decode.cu -- YoloLayer_TRT hot path for sm_100a.
//
// Replaces CalDetection/forwardGpu of yolov8/plugin/yololayer.cu:178-316 (anchor-free) and
// yolov5/plugin/yololayer.cu:161-227 (anchor-based) with
//   (1) ONE streaming "scan" launch over all strides and images: 128-bit coalesced loads along the
//       anchor axis, class range sliced across the warps of a CTA, the reference's class loop kept
//       in the logit domain with ONE sigmoid per surviving anchor (bit-identical result, see
//       scan_classes / finish_best), warp ballot/scan compaction into a per-tile slot range (no
//       atomics, deterministic order);
//   (2) a tiny "pack" launch that turns the per-tile candidates into the reference's plugin
//       buffer [count, Detection rows] (only used by the drop-in plugin ABI; the fused NMS
//       kernel in nms.cu consumes the tiles directly).
//
// Roofline: HBM-bound.  Algorithmic bytes per image = sum_l C*g_l*sizeof(in)  (SURVEY 8d).
#include <math.h>

#include "yolo_layout.cuh"

namespace trtx {

thread_local int g_last_cuda_error = 0;

// --------------------------------------------------------------------------------------------
// scan_classes: running (max logit, first argmax, max before it) over `nrows` channel rows for VEC
// adjacent anchors (Best / finish_best in yolo_layout.cuh turn that into the reference's result
//     for i: p = Logist(x_i); if (p > max) { max = p; cls = i; }          (yololayer.cu:195-201)
// bit for bit).  Hot loop: one fmaxf per element, one compare per group of U rows; a group is replayed
// -- branch-free, 4 instructions per element, no sigmoid -- only when it raises some anchor's running
// maximum above the gate logit, i.e. around real candidates.
// --------------------------------------------------------------------------------------------
template <typename T, int VEC, int U>
__device__ __forceinline__ void scan_classes(const T* __restrict__ row0, size_t g, int nrows, int cls0, Best<VEC>& s) {
    const T* p = row0;
#pragma unroll 1
    for (int r = 0; r < nrows; r += U) {
        if constexpr (VEC == 4) {
            float4 v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (r + u < nrows)
                    v[u] = Elem<T>::ld4(p + (size_t)u * g);
                else
                    v[u] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
            }
            // one max per anchor over the U rows and ONE branch per group (fmaxf ignores NaN, like `p > max`)
            float4 m = v[0];
#pragma unroll
            for (int u = 1; u < U; ++u) {
                m.x = fmaxf(m.x, v[u].x);
                m.y = fmaxf(m.y, v[u].y);
                m.z = fmaxf(m.z, v[u].z);
                m.w = fmaxf(m.w, v[u].w);
            }
            // replay only the anchors whose running maximum rises (usually one of the four, around a real candidate):
            // U sequential updates for that anchor instead of 4*U for the quad; ONE branch in the common (no hit) case
#if defined(TRTX_SCAN_PROBE) && TRTX_SCAN_PROBE == 2  // experiment build: streaming + maxima only
            if (true) {
                s.bx[0] = fmaxf(s.bx[0], m.x), s.bx[1] = fmaxf(s.bx[1], m.y), s.bx[2] = fmaxf(s.bx[2], m.z), s.bx[3] = fmaxf(s.bx[3], m.w);
                p += (size_t)U * g;
                continue;
            }
#endif
            if (!((m.x > s.bx[0]) | (m.y > s.bx[1]) | (m.z > s.bx[2]) | (m.w > s.bx[3]))) {
                p += (size_t)U * g;
                continue;
            }
            if (m.x > s.bx[0]) {
#pragma unroll
                for (int u = 0; u < U; ++u) update_one<VEC>(s, 0, v[u].x, cls0 + r + u);
            }
            if (m.y > s.bx[1]) {
#pragma unroll
                for (int u = 0; u < U; ++u) update_one<VEC>(s, 1, v[u].y, cls0 + r + u);
            }
            if (m.z > s.bx[2]) {
#pragma unroll
                for (int u = 0; u < U; ++u) update_one<VEC>(s, 2, v[u].z, cls0 + r + u);
            }
            if (m.w > s.bx[3]) {
#pragma unroll
                for (int u = 0; u < U; ++u) update_one<VEC>(s, 3, v[u].w, cls0 + r + u);
            }
        } else {
            float v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) v[u] = (r + u < nrows) ? Elem<T>::ld1(p + (size_t)u * g) : -INFINITY;
            float m = v[0];
#pragma unroll
            for (int u = 1; u < U; ++u) m = fmaxf(m, v[u]);
            if (m > s.bx[0]) {
#pragma unroll
                for (int u = 0; u < U; ++u) update_one<VEC>(s, 0, v[u], cls0 + r + u);
            }
        }
        p += (size_t)U * g;
    }
}

// --------------------------------------------------------------------------------------------
// fp16 inputs, 8 anchors per lane (one 16-byte load per lane and channel row = 512 contiguous bytes per warp-row, the same
// request size as the fp32 path at half the requests per anchor).  The running maximum is ALSO kept as packed half2 so that
// the hot loop is 4 HMNMX2 per row for 8 anchors with no fp16 -> fp32 conversion at all: max and `>` on halfs are exact and
// order-preserving (hmax2 ignores NaN like fmaxf, hgt2 is false on NaN like `p > max`).  The half2 mirror of an anchor
// that has not been raised yet is x_lo rounded DOWN to half, so the packed test can only over-report; the exact decision
// is the per-anchor replay on the fp32 state (half -> float is exact), identical to the fp32 path from there on.
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ __half2 u32_as_h2(uint32_t u) { return *reinterpret_cast<__half2*>(&u); }

template <int U>
__device__ __forceinline__ void scan_classes_h8(const __half* __restrict__ row0, size_t g, int nrows, int cls0, Best<8>& s) {
    __half2 bxh[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) bxh[k] = __halves2half2(__float2half_rd(s.bx[2 * k]), __float2half_rd(s.bx[2 * k + 1]));
    const __half* p = row0;
#pragma unroll 1
    for (int r = 0; r < nrows; r += U) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (r + u < nrows)
                v[u] = ldg_stream_h8(p + (size_t)u * g);
            else
                v[u] = make_uint4(0xFC00FC00u, 0xFC00FC00u, 0xFC00FC00u, 0xFC00FC00u);  // -inf
        }
        __half2 m[4] = {u32_as_h2(v[0].x), u32_as_h2(v[0].y), u32_as_h2(v[0].z), u32_as_h2(v[0].w)};
#pragma unroll
        for (int u = 1; u < U; ++u) {
            m[0] = __hmax2(m[0], u32_as_h2(v[u].x));
            m[1] = __hmax2(m[1], u32_as_h2(v[u].y));
            m[2] = __hmax2(m[2], u32_as_h2(v[u].z));
            m[3] = __hmax2(m[3], u32_as_h2(v[u].w));
        }
        unsigned hit[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) hit[k] = __hgt2_mask(m[k], bxh[k]);
        p += (size_t)U * g;
        if (!(hit[0] | hit[1] | hit[2] | hit[3])) continue;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!hit[k]) continue;
            if (hit[k] & 0xffffu) {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const uint32_t w = k == 0 ? v[u].x : (k == 1 ? v[u].y : (k == 2 ? v[u].z : v[u].w));
                    update_one<8>(s, 2 * k, __low2float(u32_as_h2(w)), cls0 + r + u);
                }
            }
            if (hit[k] >> 16) {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const uint32_t w = k == 0 ? v[u].x : (k == 1 ? v[u].y : (k == 2 ? v[u].z : v[u].w));
                    update_one<8>(s, 2 * k + 1, __high2float(u32_as_h2(w)), cls0 + r + u);
                }
            }
            bxh[k] = __halves2half2(__float2half_rd(s.bx[2 * k]), __float2half_rd(s.bx[2 * k + 1]));
        }
    }
}

// --------------------------------------------------------------------------------------------
// Anchor-free scan (yolov8 family).  grid = B * tiles_per_image CTAs of SLICES warps.
// --------------------------------------------------------------------------------------------
template <typename T, int VEC, int SLICES, int U>
__global__ void __launch_bounds__(32 * SLICES) yolo_v8_scan_kernel(const __grid_constant__ YoloArgs a) {
    TRTX_TL(a, kTlScan);
    constexpr int TILE = 32 * VEC;
    __shared__ float s_m[SLICES > 1 ? SLICES - 1 : 1][TILE];   // per class slice: max logit,
    __shared__ float s_m2[SLICES > 1 ? SLICES - 1 : 1][TILE];  // max logit before its class,
    __shared__ int s_c[SLICES > 1 ? SLICES - 1 : 1][TILE];     // its class

    const int b = blockIdx.x / a.tiles_per_image;
    const int t = blockIdx.x - b * a.tiles_per_image;
    int l = 0;
    while (l + 1 < a.num_levels && t >= a.lv[l + 1].tile_begin) ++l;
    const LevelArg& L = a.lv[l];
    const int tile = t - L.tile_begin;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int a0 = tile * TILE + lane * VEC;  // first cell handled by this lane
    const size_t g = (size_t)L.g;
    const bool active = a0 < L.g;  // vector paths: g % VEC == 0, so a0 < g implies the whole group is in range
    const T* base = reinterpret_cast<const T*>(L.in) + (size_t)b * a.C * g;

    Best<VEC> s;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
        s.bx[j] = a.x_lo;
        s.b2[j] = a.x_lo;
        s.bc[j] = 0;
    }
    const int per = (a.nc + SLICES - 1) / SLICES;
    const int c0 = warp * per;
    const int c1 = min(a.nc, c0 + per);
    // box rows of this tile.  prefetch_box = 3: warp 0 loads them into registers up front, so the epilogue of a tile
    // with candidates has no dependent memory round trip left (the kernel's tail is such an epilogue);
    // 2: only pull them towards L2; 1: load on demand.
    float d[4][VEC];
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int j = 0; j < VEC; ++j) d[k][j] = 0.0f;
    auto load_box = [&]() {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if constexpr (VEC == 8) {
                const uint4 v = ldg_stream_h8(reinterpret_cast<const __half*>(base) + (size_t)k * g + a0);
                const float2 f0 = __half22float2(u32_as_h2(v.x)), f1 = __half22float2(u32_as_h2(v.y));
                const float2 f2 = __half22float2(u32_as_h2(v.z)), f3 = __half22float2(u32_as_h2(v.w));
                d[k][0] = f0.x, d[k][1] = f0.y, d[k][2] = f1.x, d[k][3] = f1.y;
                d[k][4] = f2.x, d[k][5] = f2.y, d[k][6] = f3.x, d[k][7] = f3.y;
            } else if constexpr (VEC == 4) {
                float4 v = Elem<T>::ld4(base + (size_t)k * g + a0);
                d[k][0] = v.x;
                d[k][1] = v.y;
                d[k][2] = v.z;
                d[k][3] = v.w;
            } else {
                d[k][0] = Elem<T>::ld1(base + (size_t)k * g + a0);
            }
        }
    };
    if (warp == 0 && active) {
        if (a.prefetch_box == 3) {
            load_box();
        } else if (a.prefetch_box == 2) {
#pragma unroll
            for (int k = 0; k < 4; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (size_t)k * g + a0));
        }
    }
    if (active && c1 > c0) {
        if constexpr (VEC == 8)
            scan_classes_h8<U>(reinterpret_cast<const __half*>(base) + (size_t)(4 + c0) * g + a0, g, c1 - c0, c0, s);
        else
            scan_classes<T, VEC, U>(base + (size_t)(4 + c0) * g + a0, g, c1 - c0, c0, s);
    }
    // The streaming loop is done: let a kernel launched programmatically behind this one (nms_kernel) get its CTAs placed
    // during the candidate epilogue below.  It reads nothing before its griddepcontrol.wait, which waits for this grid
    // to complete, so where this trigger sits only moves time, never results.
    asm volatile("griddepcontrol.launch_dependents;");

    if constexpr (SLICES > 1) {
        bool mine = false;
#pragma unroll
        for (int j = 0; j < VEC; ++j) mine |= s.bx[j] > a.x_lo || !(0.0f < a.gate);  // may pass the gate
        if (warp > 0) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                s_m[warp - 1][lane * VEC + j] = s.bx[j];
                s_m2[warp - 1][lane * VEC + j] = s.b2[j];
                s_c[warp - 1][lane * VEC + j] = s.bc[j];
            }
        }
        int any = __syncthreads_or(mine ? 1 : 0);
        if (!any) {
            if (threadIdx.x == 0) a.tile_count[(size_t)b * a.tiles_per_image + t] = 0;
            return;
        }
        if (warp > 0) return;
        // combine in ascending class-slice order: strict > keeps the FIRST class with the maximum
#pragma unroll
        for (int w = 1; w < SLICES; ++w) {
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                merge_one<VEC>(s, j, s_m[w - 1][lane * VEC + j], s_m2[w - 1][lane * VEC + j], s_c[w - 1][lane * VEC + j]);
        }
    }

    // the one sigmoid per anchor that can pass, gate (yololayer.cu:203: `if (max_cls_prob < 0.1) return;`),
    // warp-scan compaction
    float bp[VEC];
    unsigned flags = 0;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
        bp[j] = 0.0f;  // the reference's initial max: every logit was -inf / NaN, or below the gate logit
        if (active && (a0 + j < L.g)) {
            if (s.bx[j] > a.x_lo) {
                const T* cls_row0 = base + (size_t)4 * g + a0 + j;
                bp[j] = finish_best(s.bx[j], s.b2[j], s.bc[j], a.gate, [&](int i) { return Elem<T>::ld1(cls_row0 + (size_t)i * g); });
            }
            if (!(bp[j] < a.gate)) flags |= 1u << j;
        }
    }
    int total;
    int off = warp_excl_scan(__popc(flags), lane, &total);
    if (lane == 0) a.tile_count[(size_t)b * a.tiles_per_image + t] = total;
#if defined(TRTX_SCAN_PROBE) && TRTX_SCAN_PROBE == 1  // experiment build: no box decode / record stores
    flags = 0;
#endif
    if (flags) {
        if (a.prefetch_box != 3) load_box();
        const size_t slot0 = (size_t)b * a.slots_per_image + L.slot_begin + (size_t)tile * TILE;
        const float fs = (float)L.stride;
        // this epilogue is the kernel's tail (a lone warp, every instruction at full latency): one division per
        // lane, the other cells of the quad step along the row
        const int row0 = a0 / L.gw, col0 = a0 - row0 * L.gw;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            if (flags & (1u << j)) {
                const int e = a0 + j;
                int row = row0, col = col0 + j;
                while (col >= L.gw) {  // at most once unless the grid is narrower than the quad
                    col -= L.gw;
                    ++row;
                }
                // yololayer.cu:217-220
                float x1 = ((float)col + 0.5f - d[0][j]) * fs;
                float y1 = ((float)row + 0.5f - d[1][j]) * fs;
                float x2 = ((float)col + 0.5f + d[2][j]) * fs;
                float y2 = ((float)row + 0.5f + d[3][j]) * fs;
                store_record(a.cand, slot0 + off, x1, y1, x2, y2, bp[j], s.bc[j], L.slot_begin + e);
                ++off;
            }
        }
    }
}

// --------------------------------------------------------------------------------------------
// Anchor-based scan (yolov5 family; variant TRTX_YOLO_V3 = yolov3 / v3-spp / v4, yolov3-spp/yololayer.cu:148-191: the
// class probability is gated too (:171), boxes use exp() for w/h and the stride for x/y (:183-186), and the record's
// spare float carries the class confidence).  CTA = 4 warps over a tile of 32*VEC cells x 3 anchors.
// Objectness rows are read first; the class rows of anchor k are only streamed when some cell of
// the tile passes the objectness gate for k (the reference skips its class loop per thread,
// yololayer.cu:176-177; here the skip is per tile so that the loads stay coalesced).
// --------------------------------------------------------------------------------------------
template <typename T, int VEC, int U>
__global__ void __launch_bounds__(128) yolo_v5_scan_kernel(const __grid_constant__ YoloArgs a) {
    constexpr int TILE = 32 * VEC;
    constexpr int SLICES = 4;
    __shared__ float s_obj[3][TILE];            // objectness prob (0 if not passing)
    __shared__ float s_m[SLICES - 1][TILE];     // class slices 1..3: max logit, max logit before its class, its class
    __shared__ float s_m2[SLICES - 1][TILE];
    __shared__ int s_c[SLICES - 1][TILE];
    __shared__ float s_fp[3][TILE];             // final class prob per (k, cell)
    __shared__ int s_fc[3][TILE];
    __shared__ int s_anyk[3];

    const int b = blockIdx.x / a.tiles_per_image;
    const int t = blockIdx.x - b * a.tiles_per_image;
    int l = 0;
    while (l + 1 < a.num_levels && t >= a.lv[l + 1].tile_begin) ++l;
    const LevelArg& L = a.lv[l];
    const int tile = t - L.tile_begin;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int a0 = tile * TILE + lane * VEC;
    const size_t g = (size_t)L.g;
    const bool active = a0 < L.g;
    const int ilen = a.info_len;
    const T* base = reinterpret_cast<const T*>(L.in) + (size_t)b * a.C * g;

    if (threadIdx.x < 3) s_anyk[threadIdx.x] = 0;
    __syncthreads();
    // ---- objectness: warp k reads row k*ilen+4 ----
    if (warp < 3) {
        float x[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) x[j] = -INFINITY;
        if (active) {
            const T* p = base + ((size_t)warp * ilen + 4) * g + a0;
            if constexpr (VEC == 4) {
                float4 v = Elem<T>::ld4(p);
                x[0] = v.x;
                x[1] = v.y;
                x[2] = v.z;
                x[3] = v.w;
            } else {
                x[0] = Elem<T>::ld1(p);
            }
        }
        bool anyp = false;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            float pr = 0.0f;
            bool pass = false;
            if (active && (a0 + j < L.g) && x[j] > a.x_lo) {
                pr = logist(x[j]);
                pass = !(pr < a.gate);  // yololayer.cu:177 `if (box_prob < kIgnoreThresh) continue;`
            }
            s_obj[warp][lane * VEC + j] = pass ? pr : -1.0f;
            anyp |= pass;
        }
        if (__any_sync(0xffffffffu, anyp) && lane == 0) s_anyk[warp] = 1;
    }
    __syncthreads();
    const int anyk0 = s_anyk[0], anyk1 = s_anyk[1], anyk2 = s_anyk[2];
    if (!(anyk0 | anyk1 | anyk2)) {
        if (threadIdx.x == 0) a.tile_count[(size_t)b * a.tiles_per_image + t] = 0;
        return;
    }
    // ---- class scan for each anchor k that has a passing cell in this tile ----
    const int per = (a.nc + SLICES - 1) / SLICES;
    const int c0 = warp * per;
    const int c1 = min(a.nc, c0 + per);
#pragma unroll 1
    for (int k = 0; k < 3; ++k) {
        const int anyk = k == 0 ? anyk0 : (k == 1 ? anyk1 : anyk2);
        if (!anyk) continue;
        Best<VEC> s;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            // anchors that failed the objectness gate never update; passing ones see every running max
            s.bx[j] = (s_obj[k][lane * VEC + j] >= 0.0f) ? -INFINITY : INFINITY;
            s.b2[j] = s.bx[j];
            s.bc[j] = 0;
        }
        if (active && c1 > c0)
            scan_classes<T, VEC, U>(base + ((size_t)k * ilen + 5 + c0) * g + a0, g, c1 - c0, c0, s);
        if (warp > 0) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                s_m[warp - 1][lane * VEC + j] = s.bx[j];
                s_m2[warp - 1][lane * VEC + j] = s.b2[j];
                s_c[warp - 1][lane * VEC + j] = s.bc[j];
            }
        }
        __syncthreads();
        if (warp == 0) {
#pragma unroll
            for (int w = 1; w < SLICES; ++w) {
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                    merge_one<VEC>(s, j, s_m[w - 1][lane * VEC + j], s_m2[w - 1][lane * VEC + j], s_c[w - 1][lane * VEC + j]);
            }
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                // one sigmoid per passing anchor; the v5 class probability has no gate of its own (yololayer.cu:178-186)
                float P = 0.0f;
                if (s_obj[k][lane * VEC + j] >= 0.0f && s.bx[j] > -INFINITY) {
                    const T* cls_row0 = base + ((size_t)k * ilen + 5) * g + a0 + j;
                    P = finish_best(s.bx[j], s.b2[j], s.bc[j], 0.0f, [&](int i) { return Elem<T>::ld1(cls_row0 + (size_t)i * g); });
                }
                s_fp[k][lane * VEC + j] = P;
                s_fc[k][lane * VEC + j] = s.bc[j];
            }
        }
        __syncthreads();
    }
    if (warp > 0) return;
    // ---- compaction in ascending (cell, k) order + box decode (yololayer.cu:188-208) ----
    const bool v3 = a.variant == TRTX_YOLO_V3;
    unsigned flags = 0;
#pragma unroll
    for (int j = 0; j < VEC; ++j)
#pragma unroll
        for (int k = 0; k < 3; ++k)  // v3: `max_cls_prob < IGNORE_THRESH || box_prob < IGNORE_THRESH` -> skip
            if (s_obj[k][lane * VEC + j] >= 0.0f && !(v3 && s_fp[k][lane * VEC + j] < a.gate)) flags |= 1u << (j * 3 + k);
    int total;
    int off = warp_excl_scan(__popc(flags), lane, &total);
    if (lane == 0) a.tile_count[(size_t)b * a.tiles_per_image + t] = total;
    if (flags) {
        const size_t slot0 = (size_t)b * a.slots_per_image + L.slot_begin + (size_t)tile * TILE * 3;
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                if (flags & (1u << (j * 3 + k))) {
                    const int e = a0 + j;
                    const int row = e / L.gw, col = e - row * L.gw;
                    const T* ck = base + (size_t)k * ilen * g + e;
                    if (v3) {  // yolov3-spp/yololayer.cu:183-189
                        const float fs = (float)L.stride;
                        const float bx = ((float)col + logist(Elem<T>::ld1_cached(ck))) * fs;
                        const float by = ((float)row + logist(Elem<T>::ld1_cached(ck + g))) * fs;
                        const float bw = expf(Elem<T>::ld1_cached(ck + 2 * g)) * L.anc[2 * k];
                        const float bh = expf(Elem<T>::ld1_cached(ck + 3 * g)) * L.anc[2 * k + 1];
                        store_record(a.cand, slot0 + off, bx, by, bw, bh, s_obj[k][lane * VEC + j], s_fc[k][lane * VEC + j],
                                     L.slot_begin + e * 3 + k, s_fp[k][lane * VEC + j]);
                        ++off;
                        continue;
                    }
                    float t0 = logist(Elem<T>::ld1_cached(ck));
                    float t1 = logist(Elem<T>::ld1_cached(ck + g));
                    float t2 = logist(Elem<T>::ld1_cached(ck + 2 * g));
                    float t3 = logist(Elem<T>::ld1_cached(ck + 3 * g));
                    // yololayer.cu:196-203 (left-to-right: (..)*netw/yoloWidth)
                    float cx = ((float)col - 0.5f + 2.0f * t0) * (float)a.net_w / (float)L.gw;
                    float cy = ((float)row - 0.5f + 2.0f * t1) * (float)a.net_h / (float)L.gh;
                    float w = 2.0f * t2;
                    w = w * w * L.anc[2 * k];
                    float h = 2.0f * t3;
                    h = h * h * L.anc[2 * k + 1];
                    float conf = s_obj[k][lane * VEC + j] * s_fp[k][lane * VEC + j];
                    store_record(a.cand, slot0 + off, cx, cy, w, h, conf, s_fc[k][lane * VEC + j],
                                 L.slot_begin + e * 3 + k);
                    ++off;
                }
            }
        }
    }
}

// --------------------------------------------------------------------------------------------
// yolo26 NMS-free gather (variant TRTX_YOLO_V26, yolo26/plugin/yololayer.cu:178-245).  The input is row-major per anchor
// ([B, A, C], C = 4 + classes (+ angle)), so a tile of 32 anchors is ONE contiguous block of 32*C floats: the warp
// streams it with coalesced 128-bit loads into shared memory (row pitch C|1: conflict-free), then lane i scans the class
// scores of anchor i with the reference's loop (`conf > score` from score = 0, class -1), gates (`score < thresh`) and
// the survivors are ballot-compacted into the tile's slot range like every other scan.  HBM-bound: C*4 bytes per anchor.
// --------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(128) yolo26_gather_kernel(const __grid_constant__ YoloArgs a, int batch, int warps_per_cta) {
    extern __shared__ float s_rows[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * warps_per_cta + warp;
    if (warp >= warps_per_cta || gw >= batch * a.tiles_per_image) return;
    const int b = gw / a.tiles_per_image, t = gw - b * a.tiles_per_image;
    const LevelArg& L = a.lv[0];
    const int C = a.C, Cp = C | 1;
    float* rows = s_rows + (size_t)warp * 32 * Cp;
    const int a0 = t * 32;
    const int n = min(32, L.g - a0);
    const float* src = static_cast<const float*>(L.in) + ((size_t)b * L.g + a0) * C;
    const int total = n * C;
    if constexpr (VEC == 4) {
        constexpr int U = 7;  // loads in flight per lane
        for (int i0 = lane; i0 < total / 4; i0 += 32 * U) {
            float4 v[U];
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (i0 + 32 * u < total / 4) v[u] = ldg_stream_f4(src + 4 * (size_t)(i0 + 32 * u));
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int e = 4 * (i0 + 32 * u);
                if (e < total) {
                    const int r = e / C, c = e - r * C;  // C % 4 == 0: a float4 never straddles two anchors
                    float* q = rows + r * Cp + c;
                    q[0] = v[u].x;
                    q[1] = v[u].y;
                    q[2] = v[u].z;
                    q[3] = v[u].w;
                }
            }
        }
    } else {
        for (int e = lane; e < total; e += 32) {
            const int r = e / C, c = e - r * C;
            rows[r * Cp + c] = ldg_stream_f1(src + e);
        }
    }
    __syncwarp();
    float score = 0.0f;  // :199-209
    int cls = -1;
    const float* mine = rows + lane * Cp;
    if (lane < n) {
        for (int c = 0; c < a.nc; ++c) {
            const float conf = mine[4 + c];
            if (conf > score) {
                score = conf;
                cls = c;
            }
        }
    }
    const bool keep = lane < n && !(score < a.gate);  // :211
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) a.tile_count[(size_t)b * a.tiles_per_image + t] = __popc(bal);
    if (keep) {
        const size_t slot = (size_t)b * a.slots_per_image + a0 + __popc(bal & ((1u << lane) - 1u));
        store_record(a.cand, slot, mine[0], mine[1], mine[2], mine[3], score, cls, a0 + lane, a.is_obb ? mine[4 + a.nc] : 0.0f);
    }
}

// --------------------------------------------------------------------------------------------
// pack: per-tile candidates -> reference plugin buffer [count, Detection rows] (one CTA per image).
// Extras (seg coefficients, pose keypoints, obb) are gathered from the inputs per candidate,
// exactly the reference's per-candidate work (yololayer.cu:222-279, yolov5 :206-208).
// --------------------------------------------------------------------------------------------
template <typename T>
__device__ void write_extras_v8(const YoloArgs& a, int b, int anchor_id, float* det) {
    int l = 0;
    while (l + 1 < a.num_levels && anchor_id >= a.lv[l + 1].slot_begin) ++l;
    const LevelArg& L = a.lv[l];
    const int e = anchor_id - L.slot_begin;
    const size_t g = (size_t)L.g;
    const T* cur = reinterpret_cast<const T*>(L.in) + (size_t)b * a.C * g + e;
    const int row = e / L.gw, col = e - row * L.gw;
    const int nc = a.nc, nk = a.num_kpts;
    if (a.is_seg) {
        for (int k = 0; k < 32; ++k)
            det[6 + k] = Elem<T>::ld1_cached(cur + (size_t)(4 + nc + (a.is_pose ? nk * 3 : 0) + (a.is_obb ? 1 : 0) + k) * g);
    }
    if (a.is_pose) {
        float* kp = det + 6 + 32;
        for (int k = 0; k < nk; ++k) {
            const size_t base = (size_t)(4 + nc + (a.is_seg ? 32 : 0) + (a.is_obb ? 1 : 0) + k * 3);
            float kc = logist(Elem<T>::ld1_cached(cur + (base + 2) * g));
            // `* 2.0` is a double literal in the reference (yololayer.cu:238-239)
            float kx = (float)(((double)Elem<T>::ld1_cached(cur + base * g) * 2.0 + col) * L.stride);
            float ky = (float)(((double)Elem<T>::ld1_cached(cur + (base + 1) * g) * 2.0 + row) * L.stride);
            bool inside = kx >= det[0] && kx <= det[2] && ky >= det[1] && ky <= det[3];
            if (kc < a.kpt_thresh || !inside) {
                kp[k * 3] = -1;
                kp[k * 3 + 1] = -1;
                kp[k * 3 + 2] = -1;
            } else {
                kp[k * 3] = kx;
                kp[k * 3 + 1] = ky;
                kp[k * 3 + 2] = kc;
            }
        }
    }
    if (a.is_obb) {
        const double pi = 3.14159265358979323846;
        float d0 = Elem<T>::ld1_cached(cur), d1 = Elem<T>::ld1_cached(cur + g);
        float d2 = Elem<T>::ld1_cached(cur + 2 * g), d3 = Elem<T>::ld1_cached(cur + 3 * g);
        float ain = Elem<T>::ld1_cached(cur + (size_t)(4 + nc + (a.is_seg ? 32 : 0) + (a.is_pose ? nk * 3 : 0)) * g);
        double angle = (double)(logist(ain) - 0.25f) * pi;
        double cos1 = cos(angle), sin1 = sin(angle);
        float xf = (d2 - d0) / 2;
        float yf = (d3 - d1) / 2;
        double x = xf * cos1 - yf * sin1;
        double y = xf * sin1 + yf * cos1;
        det[0] = (float)(((double)((float)col + 0.5f) + x) * L.stride);
        det[1] = (float)(((double)((float)row + 0.5f) + y) * L.stride);
        det[2] = (d0 + d2) * L.stride;
        det[3] = (d1 + d3) * L.stride;
        det[a.det_floats - 1] = (float)angle;
    }
}

template <typename T>
__device__ void write_extras_v5(const YoloArgs& a, int b, int anchor_id, float* det) {
    if (!a.is_seg) return;
    int l = 0;
    while (l + 1 < a.num_levels && anchor_id >= a.lv[l + 1].slot_begin) ++l;
    const LevelArg& L = a.lv[l];
    const int local = anchor_id - L.slot_begin;
    const int e = local / 3, k = local - e * 3;
    const size_t g = (size_t)L.g;
    const T* ck = reinterpret_cast<const T*>(L.in) + (size_t)b * a.C * g + (size_t)k * a.info_len * g + e;
    for (int i = 0; i < 32; ++i) det[6 + i] = Elem<T>::ld1_cached(ck + (size_t)(i + 5 + a.nc) * g);
}

template <typename T>
__global__ void __launch_bounds__(256) yolo_pack_rows_kernel(const __grid_constant__ YoloArgs a, float* __restrict__ out) {
    extern __shared__ int s_prefix[];  // tiles_per_image + 1
    const int b = blockIdx.x;
    const int T_ = a.tiles_per_image;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int* cnt = a.tile_count + (size_t)b * T_;
    if (warp == 0) {
        int carry = 0;
        for (int base = 0; base < T_; base += 32) {
            int v = (base + lane < T_) ? cnt[base + lane] : 0;
            int tot;
            int ex = warp_excl_scan(v, lane, &tot);
            if (base + lane < T_) s_prefix[base + lane] = carry + ex;
            carry += tot;
        }
        if (lane == 0) s_prefix[T_] = carry;
    }
    __syncthreads();
    const int total = s_prefix[T_];
    const int out_elem = 1 + a.max_out * a.det_floats;
    float* o = out + (size_t)b * out_elem;
    if (threadIdx.x == 0) o[0] = (float)min(total, a.max_out);  // clamped (see trtx_hot.h)
    if (a.variant == TRTX_YOLO_V26)  // yolo26/plugin/yololayer.cu:258: the whole buffer is memset before the gather
        for (int i = min(total, a.max_out) * a.det_floats + threadIdx.x; i < a.max_out * a.det_floats; i += blockDim.x) o[1 + i] = 0.0f;
    const int tile_slots = a.tile_cells * a.apc;
    for (int t = warp; t < T_; t += nwarps) {
        const int n = s_prefix[t + 1] - s_prefix[t];
        if (n == 0) continue;
        int l = 0;
        while (l + 1 < a.num_levels && t >= a.lv[l + 1].tile_begin) ++l;
        const size_t slot0 =
                (size_t)b * a.slots_per_image + a.lv[l].slot_begin + (size_t)(t - a.lv[l].tile_begin) * tile_slots;
        for (int j = lane; j < n; j += 32) {
            const int rank = s_prefix[t] + j;
            if (rank >= a.max_out) continue;  // yololayer.cu:207
            float4 r0 = a.cand[2 * (slot0 + j)];
            float4 r1 = a.cand[2 * (slot0 + j) + 1];
            float* det = o + 1 + (size_t)rank * a.det_floats;
            det[0] = r0.x;
            det[1] = r0.y;
            det[2] = r0.z;
            det[3] = r0.w;
            det[4] = r1.x;
            det[5] = r1.y;
            const int anchor_id = __float_as_int(r1.z);
            if (a.variant == TRTX_YOLO_V8) {
                if (a.is_seg | a.is_pose | a.is_obb) write_extras_v8<T>(a, b, anchor_id, det);
            } else if (a.variant == TRTX_YOLO_V5) {
                write_extras_v5<T>(a, b, anchor_id, det);
            } else if (a.variant == TRTX_YOLO_V3) {
                det[6] = r1.w;  // class_confidence
            } else {            // V26: the reference memsets the buffer, so the fields gatherKernel skips are zero
                for (int f = 6; f < a.det_floats; ++f) det[f] = 0.0f;
                if (a.is_obb) det[a.det_floats - 1] = r1.w;
            }
        }
    }
}

// --------------------------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------------------------
int yolo_pick_vec(const trtx_yolo_params* p, const void* const* inputs_dev) {
    // fp16 inputs of the anchor-free layout: 8 anchors per lane (16-byte loads, packed half2 maxima) when every level allows it
    if (p->in_dtype == TRTX_F16 && p->variant == TRTX_YOLO_V8) {
        bool ok8 = true;
        for (int l = 0; l < p->num_levels && ok8; ++l)
            ok8 = (p->grid_h[l] * p->grid_w[l]) % 8 == 0 && !(inputs_dev && reinterpret_cast<uintptr_t>(inputs_dev[l]) % 16 != 0);
        if (ok8) return 8;
    }
    const size_t need = (p->in_dtype == TRTX_F16) ? 8 : 16;
    for (int l = 0; l < p->num_levels; ++l) {
        int g = p->grid_h[l] * p->grid_w[l];
        if (g % 4 != 0) return 1;
        if (inputs_dev && (reinterpret_cast<uintptr_t>(inputs_dev[l]) % need) != 0) return 1;
    }
    return 4;
}

static int validate(const trtx_yolo_params* p, int batch) {
    if (!p || batch <= 0) return TRTX_ERR_INVALID;
    if (p->variant < TRTX_YOLO_V8 || p->variant > TRTX_YOLO_V26) return TRTX_ERR_INVALID;
    if (p->num_levels <= 0 || p->num_levels > TRTX_MAX_LEVELS) return TRTX_ERR_INVALID;
    if (p->num_classes <= 0 || p->max_out <= 0 || p->det_floats < 6) return TRTX_ERR_INVALID;
    if (p->in_dtype != TRTX_F32 && p->in_dtype != TRTX_F16) return TRTX_ERR_INVALID;
    for (int l = 0; l < p->num_levels; ++l)
        if (p->grid_h[l] <= 0 || p->grid_w[l] <= 0) return TRTX_ERR_INVALID;
    if (p->variant == TRTX_YOLO_V8) {
        int need = 6 + (p->is_seg || p->is_pose || p->is_obb ? 32 : 0);
        if (p->is_pose) need = 6 + 32 + p->num_kpts * 3;
        if (p->is_obb) need = (need > 7 ? need : 7);
        if (p->det_floats < need) return TRTX_ERR_INVALID;
        if (p->is_pose && p->num_kpts <= 0) return TRTX_ERR_INVALID;
    } else if (p->variant == TRTX_YOLO_V5) {
        if (p->is_seg && p->det_floats < 38) return TRTX_ERR_INVALID;
        if (p->is_pose || p->is_obb) return TRTX_ERR_UNSUPPORTED;
    } else if (p->variant == TRTX_YOLO_V3) {
        if (p->det_floats < 7) return TRTX_ERR_INVALID;
        if (p->is_seg || p->is_pose || p->is_obb) return TRTX_ERR_UNSUPPORTED;
        for (int l = 0; l < p->num_levels; ++l)
            if (p->strides[l] <= 0) return TRTX_ERR_INVALID;
    } else {  // V26: one AoS input; seg / pose tails are "TODO" in the reference too (yololayer.cu:244)
        if (p->num_levels != 1 || p->in_dtype != TRTX_F32) return TRTX_ERR_UNSUPPORTED;
        if (p->is_seg || p->is_pose) return TRTX_ERR_UNSUPPORTED;
        if (p->is_obb && p->det_floats < 7) return TRTX_ERR_INVALID;
    }
    return TRTX_OK;
}

int yolo_fill_args(const trtx_yolo_params* p, int batch, const void* const* inputs_dev, void* workspace_dev,
                   size_t workspace_bytes, YoloArgs* a, YoloLayout* Lo) {
    int rc = validate(p, batch);
    if (rc) return rc;
    if (!inputs_dev || !workspace_dev) return TRTX_ERR_INVALID;
    for (int l = 0; l < p->num_levels; ++l)
        if (!inputs_dev[l]) return TRTX_ERR_INVALID;
    const int vec = p->variant == TRTX_YOLO_V26 ? 1 : yolo_pick_vec(p, inputs_dev);  // V26: 32-anchor tiles
    // The TMA pipeline scan splits every 128-anchor stage over four warps of 32 anchors, i.e. it runs on the
    // 32-cell tile layout (the same one as the scalar kernels, which are its fallback).
    if (p->tune_class_slices < 0 || p->tune_rows_in_flight < 0 || p->tune_tma_stages < 0 || p->tune_box_prefetch < 0 ||
        p->tune_box_prefetch > 3 || (p->tune_tma_pipeline != 0 && p->tune_tma_pipeline != 1))
        return TRTX_ERR_INVALID;
    const bool pipe = p->tune_tma_pipeline && p->variant == TRTX_YOLO_V8 && vec >= 4 && yolo_pipe_supported(p, inputs_dev);
    YoloLayout L = yolo_layout(p, batch, pipe ? 1 : vec);
    L.pipe = pipe ? 1 : 0;
    L.slices = p->tune_class_slices ? p->tune_class_slices : 2;
    L.unroll = p->tune_rows_in_flight ? p->tune_rows_in_flight : (vec == 8 ? 10 : 5);  // B200 sweep, profiles/r02c_sweep_graph.log
    L.pipe_stages = p->tune_tma_stages;
    if (workspace_bytes < L.total_bytes) return TRTX_ERR_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(workspace_dev) % 16 != 0) return TRTX_ERR_INVALID;
    memset(a, 0, sizeof(*a));
    for (int l = 0; l < p->num_levels; ++l) {
        LevelArg& v = a->lv[l];
        v.in = inputs_dev[l];
        v.gh = p->grid_h[l];
        v.gw = p->grid_w[l];
        v.g = v.gh * v.gw;
        v.stride = p->strides[l];
        v.tile_begin = L.level_tile_begin[l];
        v.slot_begin = L.level_slot_begin[l];
        for (int i = 0; i < 6; ++i) v.anc[i] = p->anchors[l][i];
    }
    a->num_levels = p->num_levels;
    a->variant = p->variant;
    a->tiles_per_image = L.tiles_per_image;
    a->slots_per_image = L.slots_per_image;
    a->tile_cells = L.tile_cells;
    a->apc = L.apc;
    a->nc = p->num_classes;
    if (p->variant == TRTX_YOLO_V8) {
        // yololayer.cu:186
        a->info_len = 4 + p->num_classes + (p->is_seg ? 32 : 0) + (p->is_pose ? p->num_kpts * 3 : 0) + (p->is_obb ? 1 : 0);
        a->C = a->info_len;
    } else if (p->variant == TRTX_YOLO_V26) {
        a->info_len = 4 + p->num_classes + (p->is_obb ? 1 : 0);  // yolo26 yololayer.cu:189-194
        a->C = a->info_len;
    } else if (p->variant == TRTX_YOLO_V3) {
        a->info_len = 5 + p->num_classes;  // yolov3-spp yololayer.cu:159
        a->C = 3 * a->info_len;
    } else {
        a->info_len = 5 + p->num_classes + (p->is_seg ? 32 : 0);  // yolov5 yololayer.cu:170-171
        a->C = 3 * a->info_len;
    }
    a->net_w = p->net_w;
    a->net_h = p->net_h;
    a->max_out = p->max_out;
    a->det_floats = p->det_floats;
    a->is_seg = p->is_seg;
    a->is_pose = p->is_pose;
    a->is_obb = p->is_obb;
    a->num_kpts = p->num_kpts;
    a->kpt_thresh = p->kpt_thresh;
    a->gate = p->gate;
    // logit below which sigmoid(x) < gate for certain (0.05 logit units of slack >> any rounding)
    if (p->gate <= 0.0f)
        a->x_lo = -INFINITY;
    else if (p->gate >= 1.0f)
        a->x_lo = 10.0f;
    else
        a->x_lo = logf(p->gate / (1.0f - p->gate)) - 0.05f;
    a->prefetch_box = p->tune_box_prefetch ? p->tune_box_prefetch : 2;
    a->tile_count = reinterpret_cast<int*>(static_cast<char*>(workspace_dev) + L.off_tile_count);
    a->cand = reinterpret_cast<float4*>(static_cast<char*>(workspace_dev) + L.off_cand);
    *Lo = L;
    return TRTX_OK;
}

template <typename T, int VEC>
static int launch_v8(const YoloArgs& a, const YoloLayout& L, int grid, cudaStream_t st) {
#define TRTX_V8_CASE(S, UU)                                                        \
    if (L.slices == S && L.unroll == UU) {                                         \
        yolo_v8_scan_kernel<T, VEC, S, UU><<<grid, 32 * S, 0, st>>>(a);            \
        return TRTX_OK;                                                            \
    }
    TRTX_V8_CASE(1, 8)
    TRTX_V8_CASE(1, 16)
    TRTX_V8_CASE(2, 4)
    TRTX_V8_CASE(2, 5)
    TRTX_V8_CASE(2, 8)
    TRTX_V8_CASE(2, 10)
    TRTX_V8_CASE(2, 20)
    TRTX_V8_CASE(4, 4)
    TRTX_V8_CASE(4, 5)
    TRTX_V8_CASE(4, 10)
    TRTX_V8_CASE(4, 20)
    TRTX_V8_CASE(8, 5)
    TRTX_V8_CASE(8, 10)
#undef TRTX_V8_CASE
    return TRTX_ERR_UNSUPPORTED;  // (slices, rows in flight) pair that is not built
}

int yolo_scan_launch(const YoloArgs& a_in, const YoloLayout& L, int in_dtype, int batch, cudaStream_t st) {
    YoloArgs a = a_in;
    TRTX_TL_TAKE(a);
    const int grid = batch * L.tiles_per_image;
    if (L.pipe) {
        const int rc = yolo_scan_pipe_launch(a, L, in_dtype, batch, st);
        if (rc != TRTX_ERR_UNSUPPORTED) return rc;  // else: scalar kernels on the same 32-cell layout
    }
    if (a.variant == TRTX_YOLO_V26) {
        const int Cp = a.C | 1;
        int wpc = 4;
        while (wpc > 1 && (size_t)wpc * 32 * Cp * sizeof(float) > 200 * 1024) wpc >>= 1;
        const size_t smem = (size_t)wpc * 32 * Cp * sizeof(float);
        if (smem > 200 * 1024) return TRTX_ERR_UNSUPPORTED;
        const bool v4 = a.C % 4 == 0 && reinterpret_cast<uintptr_t>(a.lv[0].in) % 16 == 0;
        auto kern = v4 ? yolo26_gather_kernel<4> : yolo26_gather_kernel<1>;
        if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        kern<<<(grid + wpc - 1) / wpc, 128, smem, st>>>(a, batch, wpc);
    } else if (a.variant == TRTX_YOLO_V8) {
        int rc;
        if (in_dtype == TRTX_F32)
            rc = L.vec == 4 ? launch_v8<float, 4>(a, L, grid, st) : launch_v8<float, 1>(a, L, grid, st);
        else
            rc = L.vec == 8 ? launch_v8<__half, 8>(a, L, grid, st)
                            : (L.vec == 4 ? launch_v8<__half, 4>(a, L, grid, st) : launch_v8<__half, 1>(a, L, grid, st));
        if (rc) return rc;
    } else {
        if (in_dtype == TRTX_F32) {
            if (L.vec == 4)
                yolo_v5_scan_kernel<float, 4, 10><<<grid, 128, 0, st>>>(a);
            else
                yolo_v5_scan_kernel<float, 1, 10><<<grid, 128, 0, st>>>(a);
        } else {
            if (L.vec == 4)
                yolo_v5_scan_kernel<__half, 4, 10><<<grid, 128, 0, st>>>(a);
            else
                yolo_v5_scan_kernel<__half, 1, 10><<<grid, 128, 0, st>>>(a);
        }
    }
    return check_launch();
}

}  // namespace trtx

using namespace trtx;

extern "C" {

TRTX_API const char* trtx_version(void) { return "trtx_hot 0.1 (sm_100a)"; }
TRTX_API int trtx_last_cuda_error(void) { return g_last_cuda_error; }
TRTX_API size_t trtx_abi_sizeof(int which) {
    switch (which) {
        case 0: return sizeof(trtx_yolo_params);
        case 1: return sizeof(trtx_nms_params);
        case 2: return sizeof(trtx_retina_params);
        case 3: return sizeof(trtx_image_desc);
        case 4: return sizeof(trtx_mask_params);
        case 5: return sizeof(trtx_refinedet_params);
        default: return 0;
    }
}

TRTX_API int trtx_yolo_params_init_v8(trtx_yolo_params* p, int num_classes, int net_w, int net_h, int max_out,
                                      const int* strides, int num_levels) {
    if (!p || !strides || num_levels <= 0 || num_levels > TRTX_MAX_LEVELS) return TRTX_ERR_INVALID;
    memset(p, 0, sizeof(*p));
    p->variant = TRTX_YOLO_V8;
    p->num_classes = num_classes;
    p->net_w = net_w;
    p->net_h = net_h;
    p->max_out = max_out;
    p->det_floats = 90;  // yolov8/include/types.h:4-12 with kNumberOfPoints = 17
    p->num_levels = num_levels;
    for (int i = 0; i < num_levels; ++i) {
        if (strides[i] <= 0) return TRTX_ERR_INVALID;
        p->strides[i] = strides[i];
        p->grid_h[i] = net_h / strides[i];  // yololayer.cu:294-295
        p->grid_w[i] = net_w / strides[i];
    }
    p->num_kpts = 17;
    p->gate = 0.1f;
    p->in_dtype = TRTX_F32;
    return TRTX_OK;
}

TRTX_API size_t trtx_yolo_workspace_size(const trtx_yolo_params* p, int batch) {
    if (validate(p, batch)) return 0;
    // the scalar layout has the most tiles; the candidate array is identical
    return yolo_layout(p, batch, 1).total_bytes;
}

TRTX_API int trtx_yolo_decode_enqueue(const trtx_yolo_params* p, int batch, const void* const* inputs_dev,
                                      float* output_dev, void* workspace_dev, size_t workspace_bytes,
                                      trtx_stream_t stream) {
    if (!output_dev) return TRTX_ERR_INVALID;
    YoloArgs a;
    YoloLayout L;
    int rc = yolo_fill_args(p, batch, inputs_dev, workspace_dev, workspace_bytes, &a, &L);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = yolo_scan_launch(a, L, p->in_dtype, batch, st);
    if (rc) return rc;
    const size_t smem = sizeof(int) * (size_t)(L.tiles_per_image + 1);
    if (smem > 200 * 1024) return TRTX_ERR_UNSUPPORTED;
    if (p->in_dtype == TRTX_F32) {
        if (smem > 48 * 1024)
            cudaFuncSetAttribute(yolo_pack_rows_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        yolo_pack_rows_kernel<float><<<batch, 256, smem, st>>>(a, output_dev);
    } else {
        if (smem > 48 * 1024)
            cudaFuncSetAttribute(yolo_pack_rows_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        yolo_pack_rows_kernel<__half><<<batch, 256, smem, st>>>(a, output_dev);
    }
    return check_launch();
}

}  // extern "C"

// yolo_scan_pipe.cu -- the YoloLayer scan as a persistent, TMA-fed pipeline (sm_100a).
//
// One CTA per SM, resident for the whole launch.  A producer thread streams 64-anchor tiles of the level
// tensors (all C channel rows, 21.5 KB for YOLOv8 fp32) into a ring of shared-memory stages with ONE TMA
// tensor copy per stage (cp.async.bulk.tensor.3d over a [B, C, g] tensor map, box [1, C, 64], completion
// counted on an mbarrier -- the TMA engine moves the bytes, no registers are tied up and ~200 KB per SM
// are in flight from the first cycle; columns past the end of a level are zero-filled by the engine).
// Every stage is consumed by TWO warps, each owning 32 of its anchors (one anchor per lane, conflict-free
// 128-byte LDS per channel row): scan of all class rows, gate, warp-scan compaction, box decode from the 4
// box rows already in the stage, 32-byte candidate records, then one arrive on the stage's "empty" mbarrier.
// Warps never synchronise with each other; with 10 stages that is 20 consumer warps per SM, enough
// thread-level parallelism to hide the LDS/ALU latency of the scan while TMA refills the other stages.
//
// Layouts tried before this one, kept for the record (profiles/r01b..r01d sweep logs): one 512-byte
// cp.async.bulk per channel row (84 descriptors per tile throttle the copy engine: 1.7 TB/s); one tensor
// copy per tile with all consumer warps cooperating on each tile (tiles strictly one after another:
// 2.2 TB/s); one consumer warp per stage (5 warps per SM are latency-bound: 2.7 TB/s).
// tools/tma_bench.cu measures the copy-engine ceiling of this access pattern: 5.3 TB/s.
//
// The arithmetic is the same bit-exact running-max scheme as yolo_decode.cu::scan_classes.
// HBM traffic = algorithmic bytes (every row is read exactly once); candidates add <= 4%.
#include "tma.cuh"
#include "yolo_layout.cuh"

namespace trtx {

constexpr int kTileAnchors = 64;   // anchors per TMA stage (box [1, C, 64]; 256-byte rows stream as fast as 512-byte ones)
constexpr int kMaxStages = 15;     // 2 consumer warps per stage + the producer warp <= 32 warps

struct alignas(64) TmaMaps {
    CUtensorMap m[TRTX_MAX_LEVELS];
};
template <typename T>
__device__ __forceinline__ float4 lds4(const T* p);
template <>
__device__ __forceinline__ float4 lds4<float>(const float* p) {
    return *reinterpret_cast<const float4*>(p);
}
template <>
__device__ __forceinline__ float4 lds4<__half>(const __half* p) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}

constexpr int kSubWarps = kTileAnchors / 32;  // consumer warps per stage (32 anchors each)

struct PipeGeom {
    int stile_begin[TRTX_MAX_LEVELS];  // first 128-anchor stage tile of each level within an image
    int stiles_per_image;
};

template <typename T>
__device__ __forceinline__ float lds1(const T* p);
template <>
__device__ __forceinline__ float lds1<float>(const float* p) {
    return *p;
}
template <>
__device__ __forceinline__ float lds1<__half>(const __half* p) {
    return __half2float(*p);
}

template <typename T>
__global__ void __launch_bounds__(1024, 1)
        yolo_v8_scan_pipe_kernel(const __grid_constant__ YoloArgs a, const __grid_constant__ TmaMaps maps,
                                 const __grid_constant__ PipeGeom geo, int total_stiles, int stages, int stage_bytes) {
    TRTX_TL(a, kTlScan);
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* stage_base = smem;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)stages * stage_bytes);
    uint64_t* empty_bar = full_bar + kMaxStages;

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1);           // producer's arrive.expect_tx
            mbar_init(&empty_bar[s], kSubWarps);  // the stage's consumer warps
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == stages * kSubWarps) {
        // ------------------------------ producer (one elected thread) ------------------------------
        if (lane == 0) {
            int it = 0;
            for (int Tg = blockIdx.x; Tg < total_stiles; Tg += gridDim.x, ++it) {
                const int s = it % stages;
                const uint32_t ph = (uint32_t)(it / stages) & 1u;
                mbar_wait(&empty_bar[s], ph ^ 1u);
                const int b = Tg / geo.stiles_per_image, t = Tg - b * geo.stiles_per_image;
                int l = 0;
                while (l + 1 < a.num_levels && t >= geo.stile_begin[l + 1]) ++l;
                const int col0 = (t - geo.stile_begin[l]) * kTileAnchors;
                unsigned char* dst = stage_base + (size_t)s * stage_bytes;
                mbar_arrive_expect_tx(&full_bar[s], (uint32_t)stage_bytes);  // OOB columns are zero-filled and counted
                for (int ch = 0; ch < a.C; ch += 256)                          // TMA box dims are limited to 256
                    tma_load_3d(dst + (size_t)ch * kTileAnchors * sizeof(T), &maps.m[l], col0, ch, b, &full_bar[s]);
            }
        }
        asm volatile("griddepcontrol.launch_dependents;");  // every load is issued (see yolo_v8_scan_kernel)
        return;
    }

    // ------------------------------ consumers: warp = stage * kSubWarps + part ------------------------------
    const int s = warp / kSubWarps;
    const int sub = warp - s * kSubWarps;
    const T* tile = reinterpret_cast<const T*>(stage_base + (size_t)s * stage_bytes) + sub * 32 + lane;
    int it = s;
    for (int Tg = blockIdx.x + s * gridDim.x; Tg < total_stiles; Tg += stages * gridDim.x, it += stages) {
        const uint32_t ph = (uint32_t)(it / stages) & 1u;
        const int b = Tg / geo.stiles_per_image, t = Tg - b * geo.stiles_per_image;
        int l = 0;
        while (l + 1 < a.num_levels && t >= geo.stile_begin[l + 1]) ++l;
        const LevelArg& L = a.lv[l];
        const int cell0 = (t - geo.stile_begin[l]) * kTileAnchors + sub * 32;  // first cell of this warp's 32-cell tile
        const int e = cell0 + lane;
        const bool active = e < L.g;

        mbar_wait(&full_bar[s], ph);
        Best<1> st;
        st.bx[0] = active ? a.x_lo : INFINITY;  // TMA zero-fills columns past the level: those lanes never update
        st.b2[0] = st.bx[0];
        st.bc[0] = 0;
        if (cell0 < L.g) {
            // Fast path: one max over a group of U class rows and ONE compare/branch per group (fmaxf ignores NaN,
            // exactly like the reference's `p > max` never fires on NaN); the per-class update only runs for groups
            // whose max beats the running maximum logit, i.e. around real candidates.
            const T* p = tile + (size_t)4 * kTileAnchors;
            constexpr int U = 10;
            int c = 0;
            for (; c + U <= a.nc; c += U, p += U * kTileAnchors) {
                float v[U];
#pragma unroll
                for (int u = 0; u < U; ++u) v[u] = lds1<T>(p + u * kTileAnchors);
                float m = v[0];
#pragma unroll
                for (int u = 1; u < U; ++u) m = fmaxf(m, v[u]);
                if (m > st.bx[0]) {
#pragma unroll
                    for (int u = 0; u < U; ++u) update_one<1>(st, 0, v[u], c + u);
                }
            }
            for (; c < a.nc; ++c, p += kTileAnchors) update_one<1>(st, 0, lds1<T>(p), c);
            float bp = 0.0f;  // the reference's initial max
            if (active && st.bx[0] > a.x_lo)
                bp = finish_best(st.bx[0], st.b2[0], st.bc[0], a.gate,
                                 [&](int i) { return lds1<T>(tile + (size_t)(4 + i) * kTileAnchors); });
            const bool keep = active && !(bp < a.gate);  // yololayer.cu:203
            const unsigned bal = __ballot_sync(0xffffffffu, keep);
            if (lane == 0) a.tile_count[(size_t)b * a.tiles_per_image + L.tile_begin + (cell0 >> 5)] = __popc(bal);
            if (keep) {
                const float d0 = lds1<T>(tile + 0 * kTileAnchors), d1 = lds1<T>(tile + 1 * kTileAnchors);
                const float d2 = lds1<T>(tile + 2 * kTileAnchors), d3 = lds1<T>(tile + 3 * kTileAnchors);
                const int row = e / L.gw, col = e - row * L.gw;
                const float fs = (float)L.stride;
                // yololayer.cu:217-220
                const float x1 = ((float)col + 0.5f - d0) * fs;
                const float y1 = ((float)row + 0.5f - d1) * fs;
                const float x2 = ((float)col + 0.5f + d2) * fs;
                const float y2 = ((float)row + 0.5f + d3) * fs;
                const size_t slot = (size_t)b * a.slots_per_image + L.slot_begin + cell0 + __popc(bal & ((1u << lane) - 1u));
                store_record(a.cand, slot, x1, y1, x2, y2, bp, st.bc[0], L.slot_begin + e);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);  // one of the releases the producer waits for
    }
    asm volatile("griddepcontrol.launch_dependents;");
}


template <typename T>
static int launch_pipe(const YoloArgs& a, const YoloLayout& L, int batch, cudaStream_t st) {
    EncodeTiledFn enc = tma_encoder();
    if (!enc) return TRTX_ERR_UNSUPPORTED;
    int dev = 0, sms = 0, max_smem = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    const int stage_bytes = a.C * kTileAnchors * (int)sizeof(T);
    const int fixed = 2 * kMaxStages * (int)sizeof(uint64_t);
    int stages = L.pipe_stages >= 2 && L.pipe_stages < kMaxStages ? L.pipe_stages : kMaxStages;  // tune_tma_stages
    if (stages * kSubWarps + 1 > 32) stages = 31 / kSubWarps;  // 1024-thread CTA limit
    while (stages >= 2 && (size_t)stages * stage_bytes + fixed + 128 > (size_t)max_smem) --stages;
    if (stages < 2) return TRTX_ERR_UNSUPPORTED;
    const size_t smem = (size_t)stages * stage_bytes + fixed;
    TmaMaps maps;
    memset(&maps, 0, sizeof(maps));
    for (int l = 0; l < a.num_levels; ++l) {
        const cuuint64_t gdim[3] = {(cuuint64_t)a.lv[l].g, (cuuint64_t)a.C, (cuuint64_t)batch};
        const cuuint64_t gstr[2] = {(cuuint64_t)a.lv[l].g * sizeof(T), (cuuint64_t)a.C * a.lv[l].g * sizeof(T)};
        const cuuint32_t box[3] = {(cuuint32_t)kTileAnchors, (cuuint32_t)(a.C < 256 ? a.C : 256), 1u};
        const cuuint32_t estr[3] = {1u, 1u, 1u};
        const CUresult r = enc(&maps.m[l], sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                               const_cast<void*>(a.lv[l].in), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return TRTX_ERR_UNSUPPORTED;  // caller falls back to the register-path scan
    }
    PipeGeom geo;
    memset(&geo, 0, sizeof(geo));
    for (int l = 0; l < a.num_levels; ++l) {
        geo.stile_begin[l] = geo.stiles_per_image;
        geo.stiles_per_image += (a.lv[l].g + kTileAnchors - 1) / kTileAnchors;
    }
    const int total_stiles = batch * geo.stiles_per_image;
    const int grid = total_stiles < sms ? total_stiles : sms;
    auto kern = yolo_v8_scan_pipe_kernel<T>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, 32 * (stages * kSubWarps + 1), smem, st>>>(a, maps, geo, total_stiles, stages, stage_bytes);
    return check_launch();
}

bool yolo_pipe_supported(const trtx_yolo_params* p, const void* const* inputs_dev) {
    if (p->variant != TRTX_YOLO_V8) return false;
    const int C = 4 + p->num_classes + (p->is_seg ? 32 : 0) + (p->is_pose ? p->num_kpts * 3 : 0) + (p->is_obb ? 1 : 0);
    if (C > 256 && (C % 256) != 0) return false;  // keeps the expect_tx byte count exact
    for (int l = 0; l < p->num_levels; ++l) {
        const int g = p->grid_h[l] * p->grid_w[l];
        // TMA needs 16-byte aligned bases and strides
        if (inputs_dev && reinterpret_cast<uintptr_t>(inputs_dev[l]) % 16 != 0) return false;
        if (g % (p->in_dtype == TRTX_F16 ? 8 : 4) != 0) return false;
    }
    return tma_encoder() != nullptr;
}

int yolo_scan_pipe_launch(const YoloArgs& a, const YoloLayout& L, int in_dtype, int batch, cudaStream_t st) {
    if (a.variant != TRTX_YOLO_V8 || !L.pipe || L.tile_cells != 32) return TRTX_ERR_UNSUPPORTED;
    if (in_dtype == TRTX_F32) return launch_pipe<float>(a, L, batch, st);
    return launch_pipe<__half>(a, L, batch, st);
}

}  // namespace trtx

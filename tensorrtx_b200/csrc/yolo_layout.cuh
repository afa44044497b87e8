// yolo_layout.cuh -- workspace layout + kernel argument blocks shared by the YoloLayer scan,
// the row packer and the fused NMS kernel.
//
// HBM layout (DESIGN.md section 3):
//   inputs      : per level l, [B, C, g_l] channel-major (the reference's plugin input, SURVEY 8a3)
//   tile_count  : [B, tiles_per_image] int32   -- candidates found in each 32*VEC-slot tile
//   cand        : [B, slots_per_image] records of 32 B (two float4):
//                 {b0,b1,b2,b3} {conf, cls, anchor_id (int bits), spare (v3 class confidence / v26 angle)}
//                 tile t of image b owns slots [tile_slot_begin(t), +tile_slots); its candidates are
//                 written densely from the tile's first slot, in ascending anchor order.
//   list        : [B, slots_per_image] uint2 (conf key, slot) -- scratch of the fused NMS kernel
// Because every tile writes its own count and its own slot range, compaction needs no atomics and
// no zero-initialisation, and the result is deterministic.
#pragma once
#include "common.cuh"

namespace trtx {

struct LevelArg {
    const void* in;   // level tensor
    int g;            // cells = grid_h*grid_w
    int gw;           // grid width
    int gh;
    int stride;       // v8
    int tile_begin;   // first tile index of this level within an image
    int slot_begin;   // first slot (flat anchor id) of this level within an image
    float anc[6];     // v5 anchors
};

struct YoloArgs {
    LevelArg lv[TRTX_MAX_LEVELS];
    int num_levels;
    int variant;
    int tiles_per_image;
    int slots_per_image;
    int tile_cells;  // cells per tile = 32*VEC
    int apc;         // anchors per cell: 1 (v8, v26) / 3 (v5, v3)
    int C;           // channels per image per level (v8: info_len; v5: 3*info_len_i)
    int info_len;    // v8: 4+nc+extras ; v5: 5+nc(+32)
    int nc;
    int net_w, net_h;
    int max_out, det_floats;
    int is_seg, is_pose, is_obb, num_kpts;
    float kpt_thresh;
    float gate;
    float x_lo;  // logit below which sigmoid(x) < gate for certain
    int prefetch_box;  // register scan: L2-prefetch the 4 box rows while the class rows stream
    int* tile_count;
    float4* cand;
    TRTX_TL_FIELD  // probe build: this launch's timeline record
};

struct YoloLayout {
    int vec;
    int pipe;  // 1: the TMA pipeline scan runs on this layout (tile_cells = 32, four tiles per 128-anchor stage)
    int slices, unroll, pipe_stages;  // launch tuning resolved from trtx_yolo_params.tune_* (per call, no global state)
    int tile_cells;
    int apc;
    int tiles_per_image;
    int slots_per_image;
    int level_tile_begin[TRTX_MAX_LEVELS];
    int level_slot_begin[TRTX_MAX_LEVELS];
    size_t off_tile_count;
    size_t off_cand;
    size_t off_list;  // fused NMS: per-image list of (conf key, slot id) of rows above conf_thresh
    size_t total_bytes;
};

// vec = 4 (128-bit rows) or 1 (scalar fallback for grids not divisible by 4 / unaligned pointers).
inline YoloLayout yolo_layout(const trtx_yolo_params* p, int batch, int vec) {
    YoloLayout L{};
    L.vec = vec;
    L.tile_cells = 32 * vec;
    L.apc = (p->variant == TRTX_YOLO_V5 || p->variant == TRTX_YOLO_V3) ? 3 : 1;
    int tiles = 0, slots = 0;
    for (int l = 0; l < p->num_levels; ++l) {
        int g = p->grid_h[l] * p->grid_w[l];
        L.level_tile_begin[l] = tiles;
        L.level_slot_begin[l] = slots;
        tiles += (g + L.tile_cells - 1) / L.tile_cells;
        slots += g * L.apc;
    }
    L.tiles_per_image = tiles;
    L.slots_per_image = slots;
    L.off_tile_count = 0;
    L.off_cand = align_up(sizeof(int) * (size_t)batch * tiles);
    L.off_list = L.off_cand + align_up(sizeof(float4) * 2 * (size_t)batch * slots);
    L.total_bytes = L.off_list + align_up(sizeof(uint2) * (size_t)batch * slots);
    return L;
}

// ---- device helpers shared by the scan kernels ----
// Running state of the reference's class loop
//     max = 0; cls = 0; for i: p = Logist(x_i); if (p > max) { max = p; cls = i; }        (yololayer.cu:195-201)
// kept in the LOGIT domain: bx = largest logit so far, bc = the first class holding it, b2 = largest logit seen
// BEFORE class bc.  Logist is evaluated once per surviving anchor afterwards (finish_best) instead of once per
// running maximum; DESIGN.md section 4.1 has the equivalence argument.
template <int VEC>
struct Best {
    float bx[VEC];
    float b2[VEC];
    int bc[VEC];
};

// branch-free; `x > bx` is false for NaN, like the reference's `p > max` on a NaN probability
template <int VEC>
__device__ __forceinline__ void update_one(Best<VEC>& s, int j, float x, int cls) {
    const bool up = x > s.bx[j];
    s.b2[j] = up ? s.bx[j] : s.b2[j];
    s.bc[j] = up ? cls : s.bc[j];
    s.bx[j] = up ? x : s.bx[j];
}

// fold the state of a later class slice (m, m2, c) into s: strict `>` keeps the first class holding the maximum,
// and everything the earlier slices saw lies before class c
template <int VEC>
__device__ __forceinline__ void merge_one(Best<VEC>& s, int j, float m, float m2, int c) {
    if (m > s.bx[j]) {
        s.b2[j] = fmaxf(s.bx[j], m2);
        s.bx[j] = m;
        s.bc[j] = c;
    }
}

// (max prob, class) of the reference loop from the logit-domain state.  Logist is monotone non-decreasing in fp32,
// so max prob = Logist(bx).  The reference's class is the FIRST one whose probability equals that maximum:
//   * P == 0: no probability ever beat the initial max = 0 -> class 0;
//   * otherwise class bc, unless an EARLIER class has a smaller logit with the same rounded probability (two logits
//     a few ulps apart, or both saturated at 1.0f).  The largest earlier logit is b2, so Logist(b2) != P rules that
//     out; when it does collide the class rows before bc are re-read (`ld(i)`) and the reference loop is replayed.
// Anchors below the gate return early (the caller drops them, yololayer.cu:203).
template <typename LoadRow>
__device__ __forceinline__ float finish_best(float bx, float b2, int& cls, float gate, LoadRow ld) {
    const float P = logist(bx), P2 = logist(b2);  // independent: the two evaluations overlap
    if (P < gate) return P;
    if (P == 0.0f) {
        cls = 0;
        return P;
    }
    if (P2 == P) {
        for (int i = 0; i < cls; ++i) {
            if (logist(ld(i)) == P) {
                cls = i;
                break;
            }
        }
    }
    return P;
}

// `spare`: v3 class confidence / v26 obb angle (0 elsewhere)
__device__ __forceinline__ void store_record(float4* cand, size_t slot, float b0, float b1, float b2, float b3,
                                             float conf, int cls, int anchor_id, float spare = 0.0f) {
    cand[2 * slot] = make_float4(b0, b1, b2, b3);
    cand[2 * slot + 1] = make_float4(conf, (float)cls, __int_as_float(anchor_id), spare);
}

int yolo_pick_vec(const trtx_yolo_params* p, const void* const* inputs_dev);
int yolo_fill_args(const trtx_yolo_params* p, int batch, const void* const* inputs_dev, void* workspace_dev,
                   size_t workspace_bytes, YoloArgs* a, YoloLayout* L);
int yolo_scan_launch(const YoloArgs& a, const YoloLayout& L, int in_dtype, int batch, cudaStream_t stream);
// TMA-pipelined scan (yolo_scan_pipe.cu); returns TRTX_ERR_UNSUPPORTED when the shape does not fit it
int yolo_scan_pipe_launch(const YoloArgs& a, const YoloLayout& L, int in_dtype, int batch, cudaStream_t stream);
bool yolo_pipe_supported(const trtx_yolo_params* p, const void* const* inputs_dev);

}  // namespace trtx

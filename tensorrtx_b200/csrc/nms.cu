// nms.cu -- sort + class-aware greedy NMS, one CTA (1024 threads; 512 on request on the fused YOLO path) per
// image, every image of the batch in one launch.  Replaces
//   host  nms()/batch_nms()      yolov8/src/postprocess.cpp:94-129, yolov5/src/postprocess.cpp:49-80,
//                                retinaface/common.hpp:110-130           (std::map + std::sort + erase)
//   device cuda_decode()+cuda_nms()  yolov8/src/postprocess.cu:42-111,168-179   (batch 1 only, one-shot)
//
// Phases (all on-chip after the first read of the candidates; latency/occupancy-bound, no roofline):
//   A  collect rows with conf > conf_thresh into a list (conf key, id)
//   B  if more than `pre_topk` survive: block radix-select (4 x 8-bit passes) of the top pre_topk,
//      ties at the cut broken by the smaller id (second radix select over the ids)
//   C  bitonic sort by (class asc, conf desc, box[0] asc, id asc) -- the order the reference builds with
//      std::map<float,...> + std::sort(cmp).  Up to one row per thread: rows in registers, the
//      j < 32 exchange steps are warp shuffles, only the j >= 32 steps go through shared memory
//      (1 barrier each, ping-pong buffers); more rows: plain shared-memory network.
//   D  stage boxes of the sorted rows in shared memory (SoA)
//   E  greedy NMS per CLASS SEGMENT of the sorted list (rows of different classes never interact):
//      short segments (<= 96 rows, the normal multi-class case) are claimed by single warps and
//      resolved with shuffles + ballots only -- no block barrier at all;  long segments (single-class
//      models such as retinaface, or degenerate inputs) are processed by the whole CTA in chunks of 32
//      rows: every chunk member is tested against the already-kept rows (all threads, IoU tile in
//      shared memory) and against its 31 chunk-mates (warp w = member w mod warps, lane j = mate j, one
//      __ballot_sync per member gives its suppressor bitmap); warp 0 resolves the chunk serially on
//      the 32x32 bitmap.  2 barriers per 32 rows.
//   F  block scan of the keep flags -> [count, (box, conf, cls, keep, extras)*] in sorted order.
//
// IoU arithmetic mirrors the reference's CPU functions operation by operation with round-to-nearest
// intrinsics (no FMA contraction), so kept sets agree with the host code bit for bit.
#include <string.h>

#include "yolo_layout.cuh"

namespace trtx {

// Phase stamps (clock64 per image) exist only in the probe build (tensorrtx_b200/build.py build(probe=True), used by
// tools/nms_probe.py): the release library has no profiling state at all.
#ifdef TRTX_NMS_PROBE
static thread_local long long* t_nms_stamps = nullptr;
static thread_local unsigned long long* t_tl_buf = nullptr;
static thread_local int t_tl_records = 0, t_tl_next = 0;
unsigned long long* tl_take() {
    if (!t_tl_buf || t_tl_next >= t_tl_records) return nullptr;
    return t_tl_buf + kTlRecordWords * (size_t)t_tl_next++;
}
#define TRTX_STAMP(k) do { if (a.dbg && threadIdx.x == 0) a.dbg[blockIdx.x * 16 + (k)] = clock64(); } while (0)
#else
#define TRTX_STAMP(k) do { } while (0)
#endif

// Block sizes of nms_kernel.  The general kernel (every source, box format and mode, up to kMaxSort rows) runs 1024
// threads at 60 registers, so it needs an SM of its own.  The half-SM instantiation (512 threads, <= 64 registers, 2 CTAs
// an SM by launch bounds) fits next to 5 letterbox or 8 scan CTAs; it covers the fused YOLO path (tile source, greedy,
// axis-aligned, pre_topk <= 1024, no fused gather) on request (trtx_yolo_params.tune_nms_threads = 512).  Both compute
// the same outputs: only the mapping of threads to work differs.  It is not the default: on a B200 at b32 its CTAs run
// 30-35 us next to the streaming letterbox instead of 21-24 (half the threads for the same phases), which costs more
// than placing a CTA early gains (profiles/r03a_timeline_*.log).
constexpr int kNmsThreads = 1024;
constexpr int kNmsThreadsHalf = 512;
constexpr int kMaxSort = TRTX_NMS_MAX_ROWS;  // rows entering NMS per image (>= kMaxNumOutputBbox = 1000)
// bucket sort: one histogram bin per thread (NT bins; a class id >= NT takes the bitonic paths)
constexpr int kMaxBucket = 256;           // rows per class the rank-by-counting pass accepts
constexpr int kShortSeg = 96;  // class segments up to this many rows are resolved by a single warp

struct NmsArgs {
    // source 0: plugin-format rows  [B, 1 + max_rows*det_floats]
    const float* rows;
    int max_rows;
    int det_floats;
    // source 1: YoloLayer tiles (fused path)
    int from_tiles;
    int tiles_per_image, slots_per_image, tile_slots;
    int num_levels;
    int lv_tile_begin[TRTX_MAX_LEVELS];
    int lv_slot_begin[TRTX_MAX_LEVELS];
    const int* tile_count;
    const float4* cand;
    // scratch list [B, list_stride] of (conf key, id)
    uint2* list;
    int list_stride;
    // parameters
    int box_format, mode, class_aware, tie_break_x0;
    float conf_thresh, nms_thresh;
    int pre_topk;  // rows entering NMS (<= kMaxSort)
    int max_det;
    int extra_floats, extra_offset;
#ifdef TRTX_NMS_PROBE
    long long* dbg;       // 16 clock64 stamps per image, or null
#endif
    TRTX_TL_FIELD  // probe build: this launch's timeline record
    float* out;           // [B, 1 + max_det*(7+extra)]
    int32_t* keep_index;  // [B, max_det] or null
    // multi-GPU: phase F also stores every emitted row (and the count) into the gathered buffer of EVERY rank over
    // NVLink peer memory, then the last CTA of the launch publishes a per-(rank, slot) flag (trtx_gather, trtx_hot.h)
    struct Gather {
        float* out[8];
        unsigned* flags[8];
        unsigned* ctrl;  // local: [1] CTAs done, [2] error ([0], [3] unused)
        int world, rank, slots, slot;
    } g;
};

// system-scope RELAXED accesses of the gather's publish counters: the ordering comes from kernel boundaries (or, in the variant
// fused into nms_kernel, from one __threadfence_system()), never from per-access acquire / release -- see gather_wait_kernel
__device__ __forceinline__ unsigned ld_relaxed_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys(unsigned* p, unsigned v) {
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---- IoU variants -------------------------------------------------------------------------
// Host IoUs restated by to_corners / box_area / overlaps below:
//   yolov8/src/postprocess.cpp:71-85  l,t,r,b     inter / (la + ra - inter)       (std::max(a,b) = a<b ? b : a)
//   yolov5/src/postprocess.cpp:30-43  cx,cy,w,h   corners x -/+ w/2, areas w*h
//   retinaface/common.hpp:91-104      l,t,r,b     inter / (la + ra - inter + 0.000001f)
// yolov8/src/postprocess.cu:74-87 (device box_iou of the one-shot path)
__device__ __forceinline__ float iou_oneshot(const float4 a, const float4 b) {
    float cl = fmaxf(a.x, b.x), ct = fmaxf(a.y, b.y), cr = fminf(a.z, b.z), cb = fminf(a.w, b.w);
    float c_area = __fmul_rn(fmaxf(__fsub_rn(cr, cl), 0.0f), fmaxf(__fsub_rn(cb, ct), 0.0f));
    if (c_area == 0.0f) return 0.0f;
    float a_area = __fmul_rn(fmaxf(0.0f, __fsub_rn(a.z, a.x)), fmaxf(0.0f, __fsub_rn(a.w, a.y)));
    float b_area = __fmul_rn(fmaxf(0.0f, __fsub_rn(b.z, b.x)), fmaxf(0.0f, __fsub_rn(b.w, b.y)));
    return __fdiv_rn(c_area, __fsub_rn(__fadd_rn(a_area, b_area), c_area));
}
// ---- oriented boxes (yolov8-obb): Gaussian covariance per row + ProbIoU per pair ------------------------------
// Host flavour = convariance_matrix / probiou of yolov8/src/postprocess.cpp:303-355 with its C++ promotions
// (`w*w/12.0` and every std::pow(x, 2) are double, std::cos/sin/exp(float) are float, std::log/sqrt of the mixed
// expressions are double); device flavour = postprocess.cu:113-145, all float, left to nvcc's FMA contraction like
// the reference build.  A row is kept as (cx, cy, a, b) + c.
__device__ __forceinline__ void obb_cov_host(float w, float h, float r, float& a, float& b, float& c) {
    const float A = (float)((double)__fmul_rn(w, w) / 12.0), B = (float)((double)__fmul_rn(h, h) / 12.0);
    const float cr = cosf(r), sr = sinf(r);
    const float cr2 = __fmul_rn(cr, cr), sr2 = __fmul_rn(sr, sr);
    a = __fadd_rn(__fmul_rn(A, cr2), __fmul_rn(B, sr2));
    b = __fadd_rn(__fmul_rn(A, sr2), __fmul_rn(B, cr2));
    c = __fmul_rn(__fmul_rn(__fsub_rn(A, B), cr), sr);
}
__device__ __forceinline__ float obb_probiou_host(const float4 p1, float c1, const float4 p2, float c2) {
    const float eps = 1e-7;
    const float x1 = p1.x, y1 = p1.y, a1 = p1.z, b1 = p1.w, x2 = p2.x, y2 = p2.y, a2 = p2.z, b2 = p2.w;
    const float sa = __fadd_rn(a1, a2), sb = __fadd_rn(b1, b2), sc = __fadd_rn(c1, c2);
    const double dy = (double)__fsub_rn(y1, y2), dx = (double)__fsub_rn(x1, x2), dc = (double)sc;
    const double py = __dmul_rn(dy, dy), px = __dmul_rn(dx, dx), pc = __dmul_rn(dc, dc);  // std::pow(float, 2): exact in double
    const double den = __dadd_rn(__dsub_rn((double)__fmul_rn(sa, sb), pc), (double)eps);
    const float t1 = (float)__ddiv_rn(__dadd_rn(__dmul_rn((double)sa, py), __dmul_rn((double)sb, px)), den);
    const float t2 = (float)__ddiv_rn((double)__fmul_rn(__fmul_rn(sc, __fsub_rn(x2, x1)), __fsub_rn(y1, y2)), den);
    const float s1 = sqrtf(fmaxf(__fsub_rn(__fmul_rn(a1, b1), __fmul_rn(c1, c1)), 0.0f));
    const float s2 = sqrtf(fmaxf(__fsub_rn(__fmul_rn(a2, b2), __fmul_rn(c2, c2)), 0.0f));
    const float d3 = __fadd_rn(__fmul_rn(__fmul_rn(4.0f, s1), s2), eps);
    const float t3 = (float)log(__dadd_rn(__ddiv_rn(__dsub_rn((double)__fmul_rn(sa, sb), pc), (double)d3), (double)eps));
    float bd = __fadd_rn(__fadd_rn(__fmul_rn(0.25f, t1), __fmul_rn(0.5f, t2)), __fmul_rn(0.5f, t3));
    bd = fmaxf(fminf(bd, 100.0f), eps);
    const float hd = (float)sqrt(__dadd_rn(__dsub_rn(1.0, (double)expf(-bd)), (double)eps));
    return __fsub_rn(1.0f, hd);
}
__device__ __forceinline__ void obb_cov_dev(float w, float h, float r, float& a, float& b, float& c) {  // :113-122
    float a_val = w * w / 12.0f;
    float b_val = h * h / 12.0f;
    float cos_r = cosf(r);
    float sin_r = sinf(r);
    a = a_val * cos_r * cos_r + b_val * sin_r * sin_r;
    b = a_val * sin_r * sin_r + b_val * cos_r * cos_r;
    c = (a_val - b_val) * sin_r * cos_r;
}
__device__ __forceinline__ float obb_probiou_dev(const float4 p1, float c1, const float4 p2, float c2) {  // :124-145
    const float eps = 1e-7;
    const float cx1 = p1.x, cy1 = p1.y, a1 = p1.z, b1 = p1.w, cx2 = p2.x, cy2 = p2.y, a2 = p2.z, b2 = p2.w;
    float t1 = ((a1 + a2) * powf(cy1 - cy2, 2) + (b1 + b2) * powf(cx1 - cx2, 2)) /
               ((a1 + a2) * (b1 + b2) - powf(c1 + c2, 2) + eps);
    float t2 = ((c1 + c2) * (cx2 - cx1) * (cy1 - cy2)) / ((a1 + a2) * (b1 + b2) - powf(c1 + c2, 2) + eps);
    float t3 = logf(((a1 + a2) * (b1 + b2) - powf(c1 + c2, 2)) /
                            (4 * sqrtf(fmaxf(a1 * b1 - c1 * c1, 0.0f)) * sqrtf(fmaxf(a2 * b2 - c2 * c2, 0.0f)) + eps) +
                    eps);
    float bd = 0.25f * t1 + 0.5f * t2 + 0.5f * t3;
    bd = fmaxf(fminf(bd, 100.0f), eps);
    float hd = sqrtf(1.0f - expf(-bd) + eps);
    return 1 - hd;
}

// ---- greedy NMS inner loop: boxes pre-converted to corners, areas precomputed ---------------------------------
// The three host IoUs above differ only in how corners and areas are formed and in retinaface's +1e-6; with those
// hoisted out (phase D) one test serves all.  Every operation is the reference's, in the reference's order.
__device__ __forceinline__ float4 to_corners(int fmt, const float4 b) {
    if (fmt != TRTX_BOX_CXCYWH) return b;
    // x/2 == x*0.5 exactly in binary floating point
    const float hw = __fmul_rn(b.z, 0.5f), hh = __fmul_rn(b.w, 0.5f);
    return make_float4(__fsub_rn(b.x, hw), __fsub_rn(b.y, hh), __fadd_rn(b.x, hw), __fadd_rn(b.y, hh));
}
__device__ __forceinline__ float box_area(int fmt, const float4 b) {  // b = the row as stored (before to_corners)
    if (fmt == TRTX_BOX_CXCYWH) return __fmul_rn(b.z, b.w);
    return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
}
struct IouTest {
    float thr;
    bool obb;       // rows are (cx, cy, a, b) + c: ProbIoU `>= thr` (nms_obb, postprocess.cpp:378)
    bool retina;    // denominator + 0.000001f
    bool zero_hit;  // `0.0f > thr` (disjoint boxes)
    bool fast_ok;   // the division-free test below is proven for |thr| <= 4
};
// == (iou(l, r) > thr) bit for bit.  fl(inter/denom) > thr is decided by the sign of t = inter - thr*denom (one FMA
// rounding, so sign and magnitude of t are right to 2^-24) whenever |t| > 1e-5*denom, i.e. the true quotient is at
// least ~1e-5 away from thr -- hundreds of ulps for |thr| <= 4.  Anything closer, or a non-positive / non-finite
// denominator, takes the IEEE division the reference takes.
__device__ __forceinline__ bool overlaps(const IouTest& q, const float4 l, float la, const float4 r, float ra) {
    if (q.obb) return obb_probiou_host(l, la, r, ra) >= q.thr;
    const float ib0 = l.x < r.x ? r.x : l.x;
    const float ib1 = r.z < l.z ? r.z : l.z;
    const float ib2 = l.y < r.y ? r.y : l.y;
    const float ib3 = r.w < l.w ? r.w : l.w;
    if (ib2 > ib3 || ib0 > ib1) return q.zero_hit;
    const float inter = __fmul_rn(__fsub_rn(ib1, ib0), __fsub_rn(ib3, ib2));
    float denom = __fsub_rn(__fadd_rn(la, ra), inter);
    if (q.retina) denom = __fadd_rn(denom, 0.000001f);
    const float t = __fmaf_rn(-q.thr, denom, inter);
    if (q.fast_ok && denom > 0.0f && fabsf(t) > __fmul_rn(1e-5f, denom)) return t > 0.0f;
    return __fdiv_rn(inter, denom) > q.thr;
}

// ---- candidate accessors --------------------------------------------------------------------
struct Row {
    float4 box;
    float conf;
    float cls;
    int anchor;
};
__device__ __forceinline__ Row fetch_row(const NmsArgs& a, int b, uint32_t id) {
    Row r;
    if (a.from_tiles) {
        const float4* c = a.cand + 2 * ((size_t)b * a.slots_per_image + id);
        r.box = c[0];
        float4 m = c[1];
        r.conf = m.x;
        r.cls = m.y;
        r.anchor = __float_as_int(m.z);
    } else {
        const float* p = a.rows + (size_t)b * (1 + (size_t)a.max_rows * a.det_floats) + 1 + (size_t)id * a.det_floats;
        r.box = make_float4(p[0], p[1], p[2], p[3]);
        r.conf = p[4];
        r.cls = a.box_format == TRTX_BOX_RETINA ? 0.0f : p[5];
        r.anchor = (int)id;
    }
    return r;
}

// Block-wide: find the bucket holding the `need`-th element counting from the top (descending)
// or from the bottom (ascending) of a 256-bin histogram; returns bucket, updates need to the
// rank inside that bucket.  Executed by thread 0, result broadcast through shared memory.
__device__ __forceinline__ void pick_bucket(const int* hist, bool descending, int* need_io, int* bucket_out) {
    int need = *need_io, c = 0, d;
    if (descending) {
        for (d = 255; d > 0; --d) {
            if (c + hist[d] >= need) break;
            c += hist[d];
        }
    } else {
        for (d = 0; d < 255; ++d) {
            if (c + hist[d] >= need) break;
            c += hist[d];
        }
    }
    *need_io = need - c;
    *bucket_out = d;
}

// IoU work units of a segment of m rows: row li (0-based inside the segment) needs ceil(li/8) of them
__device__ __forceinline__ int seg_units(int m) {
    const int G = (m + 6) >> 3;
    return G * (m - 1) - 4 * G * (G - 1);
}

template <int NT>
__global__ void __launch_bounds__(NT, kNmsThreads / NT) nms_kernel(const __grid_constant__ NmsArgs a) {
    constexpr int NW = NT / 32;  // warps; per-warp partials in s_wsum[0 .. NW)
    static_assert(NT % 32 == 0 && NT >= 256 && NT <= 1024, "the 256-bin histograms need >= 256 threads");
    // Programmatic dependent launch (nms_launch): this CTA may become resident while the kernel before it in the stream
    // still runs.  Nothing before this point touches global memory; the wait returns once that kernel has completed
    // and its writes are visible (a no-op after an ordinary launch).
    TRTX_TL(a, kTlNms);  // entry stamp = the CTA is resident (under PDL: possibly before the scan has completed)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // carve-up (S = row capacity, power of two >= pre_topk)
    const int S = a.pre_topk <= 1024 ? 1024 : kMaxSort;
    float4* u_box = reinterpret_cast<float4*>(smem_raw);                         // S  stash in arrival order
    float4* s_box = u_box + S;                                                   // S  sorted rows
    unsigned long long* k64 = reinterpret_cast<unsigned long long*>(s_box + S);  // S  64-bit sort keys (fast path)
    float* u_conf = reinterpret_cast<float*>(k64 + S);                           // S
    int* u_cls = reinterpret_cast<int*>(u_conf + S);                             // S
    uint32_t* u_id = reinterpret_cast<uint32_t*>(u_cls + S);                     // S
    float* s_conf = reinterpret_cast<float*>(u_id + S);                          // S
    int* s_cls = reinterpret_cast<int*>(s_conf + S);                             // S
    uint32_t* s_id = reinterpret_cast<uint32_t*>(s_cls + S);                     // S
    int* s_seg = reinterpret_cast<int*>(s_id + S);                               // S   short class segments (start<<16 | len)
    int* s_long = s_seg + S;                                                     // S/2 long class segments
    unsigned short* s_pos = reinterpret_cast<unsigned short*>(s_long + S / 2);   // S   slow path: stash position riding along
    unsigned char* s_keep = reinterpret_cast<unsigned char*>(s_pos + S);         // S   keep flags
    unsigned short* s_unit = reinterpret_cast<unsigned short*>(s_keep + S);      // S*12 IoU work units (row << 4 | group of 8)
    float* s_area = reinterpret_cast<float*>(s_unit + S * (kShortSeg / 8));      // S   box areas (greedy mode)
    int* s_tpre = reinterpret_cast<int*>(s_area + S);                            // tiles_per_image + 1 (fused path)
    unsigned short* s_krow = reinterpret_cast<unsigned short*>(u_box);  // kept rows of a long segment (the stash is dead after D)
    unsigned* s_mask = reinterpret_cast<unsigned*>(u_conf);  // 3 words per row: suppressor bitmaps (aliases u_conf/u_cls/u_id)
    int* s_rowseg = reinterpret_cast<int*>(k64);             // per row: segment start << 16 | length (aliases the sort keys)
    // slow path only: 128-bit keys live in the (not yet filled) sorted-row area
    unsigned long long* k_hi = reinterpret_cast<unsigned long long*>(s_box);
    unsigned long long* k_lo = k_hi + S;

    __shared__ int s_hist[256];
    __shared__ int s_chist[NT], s_cstart[NT];  // bucket sort: rows per class, first sorted row of a class
    __shared__ int s_n, s_need, s_bucket, s_nkept, s_nshort, s_nmed, s_nlong, s_cursor, s_bad, s_nunit;
    __shared__ unsigned s_rem;
    __shared__ unsigned s_sup[32];
    __shared__ int s_wsum[32];

    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint2* list = a.list + (size_t)b * a.list_stride;

    TRTX_STAMP(0);
    // ---------------- A: collect rows above conf_thresh, stash them in shared memory ----------------
    // greedy: `conf <= thr -> skip` (postprocess.cpp:99; false for NaN, which v8 skips too);
    // one-shot: `conf < thr -> skip` (postprocess.cu:57)
    if (tid == 0) {
        s_n = 0;
        s_bad = 0;
    }
    auto stash = [&](const Row& r, uint32_t id) {
        const int pos = atomicAdd(&s_n, 1);
        list[pos] = make_uint2(float_key(r.conf), id);  // only read back if more than pre_topk rows survive
        if (pos < S) {
            const int c = a.class_aware ? (int)r.cls : 0;
            u_box[pos] = r.box;
            u_conf[pos] = r.conf;
            u_cls[pos] = c;
            u_id[pos] = id;
            if (c < 0 || c > 0xffff) s_bad = 1;  // class does not fit the packed 64-bit key: generic sort
        }
    };
    if (a.from_tiles) {
        // prefix over the per-tile candidate counts, then one thread per candidate (binary search for its tile)
        const int T = a.tiles_per_image;
        const int* cnt = a.tile_count + (size_t)b * T;
        int carry = 0;
        for (int base = 0; base < T; base += NT) {
            const int t = base + tid;
            const int v = t < T ? cnt[t] : 0;
            int tot;
            const int ex = warp_excl_scan(v, lane, &tot);
            if (lane == 0) s_wsum[warp] = tot;
            __syncthreads();
            if (warp == 0) {
                int w = lane < NW ? s_wsum[lane] : 0, wt;
                const int wex = warp_excl_scan(w, lane, &wt);
                s_wsum[lane] = wex;
                if (lane == 0) s_need = wt;
            }
            __syncthreads();
            if (t < T) s_tpre[t] = carry + s_wsum[warp] + ex;
            carry += s_need;
            __syncthreads();
        }
        if (tid == 0) s_tpre[T] = carry;
        __syncthreads();
        // The reference plugin keeps the first max_out candidates that grab a slot (yololayer.cu:206-208) and its host
        // nms() filters THOSE by confidence: same here with "first" = ascending anchor order (what
        // trtx_yolo_decode_enqueue + trtx_nms_enqueue do through the plugin buffer), so both paths agree above max_out.
        const int n_in = min(carry, a.pre_topk);
        for (int r = tid; r < n_in; r += NT) {
            int lo = 0, hi = T;  // largest t with s_tpre[t] <= r
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (s_tpre[mid] <= r) lo = mid; else hi = mid;
            }
            const int t = lo;
            int l = 0;
            while (l + 1 < a.num_levels && t >= a.lv_tile_begin[l + 1]) ++l;
            const uint32_t id = a.lv_slot_begin[l] + (uint32_t)(t - a.lv_tile_begin[l]) * a.tile_slots + (uint32_t)(r - s_tpre[t]);
            const Row row = fetch_row(a, b, id);
            if (a.mode == TRTX_NMS_ONESHOT ? row.conf >= a.conf_thresh : row.conf > a.conf_thresh) stash(row, id);
        }
    } else {
        __syncthreads();
        const float* img = a.rows + (size_t)b * (1 + (size_t)a.max_rows * a.det_floats);
        int n_in = (int)img[0];  // `i < output[0]`
        n_in = max(0, min(n_in, a.max_rows));
        for (int i = tid; i < n_in; i += NT) {
            const Row row = fetch_row(a, b, (uint32_t)i);
            if (a.mode == TRTX_NMS_ONESHOT ? row.conf >= a.conf_thresh : row.conf > a.conf_thresh) stash(row, (uint32_t)i);
        }
    }
    __syncthreads();
    const int n_valid = s_n;
    const int M = min(n_valid, a.pre_topk);

    // ---------------- B: radix select when more than pre_topk rows survive (rare) ----------------
    if (n_valid > a.pre_topk) {
        uint32_t key_cut = 0, id_cut = 0xffffffffu;  // take key > key_cut, or key == key_cut && id <= id_cut
        uint32_t prefix = 0, mask = 0;
        if (tid == 0) s_need = a.pre_topk;
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            if (tid < 256) s_hist[tid] = 0;
            __syncthreads();
            for (int i = tid; i < n_valid; i += NT) {
                uint32_t k = list[i].x;
                if ((k & mask) == prefix) atomicAdd(&s_hist[(k >> shift) & 255], 1);
            }
            __syncthreads();
            if (tid == 0) {
                int need = s_need, d;
                pick_bucket(s_hist, true, &need, &d);
                s_need = need;
                s_bucket = d;
            }
            __syncthreads();
            prefix |= (uint32_t)s_bucket << shift;
            mask |= 255u << shift;
        }
        key_cut = prefix;
        const int need_eq = s_need;  // how many rows with key == key_cut are taken
        uint32_t ip = 0, im = 0;     // ties at the cut: take the need_eq smallest ids
        __syncthreads();
        if (tid == 0) s_need = need_eq;
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            if (tid < 256) s_hist[tid] = 0;
            __syncthreads();
            for (int i = tid; i < n_valid; i += NT) {
                uint2 e = list[i];
                if (e.x == key_cut && (e.y & im) == ip) atomicAdd(&s_hist[(e.y >> shift) & 255], 1);
            }
            __syncthreads();
            if (tid == 0) {
                int need = s_need, d;
                pick_bucket(s_hist, false, &need, &d);
                s_need = need;
                s_bucket = d;
            }
            __syncthreads();
            ip |= (uint32_t)s_bucket << shift;
            im |= 255u << shift;
        }
        id_cut = ip;
        // re-stash exactly the selected rows
        if (tid == 0) {
            s_n = 0;
            s_bad = 0;
        }
        __syncthreads();
        for (int i = tid; i < n_valid; i += NT) {
            const uint2 e = list[i];
            if (e.x > key_cut || (e.x == key_cut && e.y <= id_cut)) {
                const Row r = fetch_row(a, b, e.y);
                const int pos = atomicAdd(&s_n, 1);
                const int c = a.class_aware ? (int)r.cls : 0;
                u_box[pos] = r.box;
                u_conf[pos] = r.conf;
                u_cls[pos] = c;
                u_id[pos] = e.y;
                if (c < 0 || c > 0xffff) s_bad = 1;
            }
        }
        __syncthreads();
    }

    TRTX_STAMP(1);
    // ---------------- C: sort by (class asc, conf desc, box[0] asc, id asc) ----------------
    int S_eff = 32;
    while (S_eff < M) S_eff <<= 1;
    // fast path: packed key = class(16) | ~conf key(32) | stash position(16); exact unless two rows share
    // (class, conf) -- detected below, then the generic 128-bit sort decides by (box[0], id).
    bool generic = s_bad != 0;
    // fastest path (the detector case: many classes, a few dozen rows each): counting sort by class, then every row
    // ranks itself inside its class bucket by counting smaller keys -- no compare-exchange network.
    // Falls through to the bitonic paths when a class id is >= NT or a bucket holds more than kMaxBucket rows.
    bool bucketed = false;
    if (!generic) {
        unsigned long long* kb = reinterpret_cast<unsigned long long*>(s_box);  // keys in bucket order (rows not staged yet)
        s_chist[tid] = 0;
        __syncthreads();
        bool big = false;
        for (int base = 0; base < M; base += NT) {
            // rows arrive in tile order, so neighbouring lanes often share a class: one atomic per (warp, class)
            const int i = base + tid;
            const int c = i < M ? u_cls[i] : -1;
            const unsigned peers = __match_any_sync(0xffffffffu, c);
            const int leader = __ffs(peers) - 1;
            int first = 0;
            if (c >= NT) big = true;
            if (lane == leader && c >= 0 && c < NT) first = atomicAdd(&s_chist[c], __popc(peers));
            first = __shfl_sync(0xffffffffu, first, leader);
            if (i < M) s_pos[i] = (unsigned short)(first + __popc(peers & ((1u << lane) - 1u)));  // slot inside the bucket (any order works)
        }
        __syncthreads();
        const int h = s_chist[tid];
        int tot;
        const int ex = warp_excl_scan(h, lane, &tot);
        if (lane == 0) s_wsum[warp] = tot;
        if (!__syncthreads_or(big || h > kMaxBucket ? 1 : 0)) {
            if (warp == 0) {
                int w = lane < NW ? s_wsum[lane] : 0, wt;
                const int wex = warp_excl_scan(w, lane, &wt);
                s_wsum[lane] = wex;
            }
            __syncthreads();
            s_cstart[tid] = s_wsum[warp] + ex;
            __syncthreads();
            for (int i = tid; i < M; i += NT) {
                const int c = u_cls[i];
                kb[s_cstart[c] + s_pos[i]] =
                    ((unsigned long long)(uint32_t)c << 48) | ((unsigned long long)(uint32_t)(~float_key(u_conf[i])) << 16) | (uint32_t)i;
            }
            __syncthreads();
            // thread p owns bucket slot p: neighbouring lanes share a bucket, so the key reads below are broadcasts
            for (int p = tid; p < M; p += NT) {
                const unsigned long long mk = kb[p];
                const int c = (int)(mk >> 48);
                const int s0 = s_cstart[c], m = s_chist[c];
                int rank = 0;
#pragma unroll 4
                for (int k = 0; k < m; ++k) rank += kb[s0 + k] < mk ? 1 : 0;  // keys are distinct (stash position in the low bits)
                k64[s0 + rank] = mk;
            }
            __syncthreads();
            bool tie = false;  // same (class, conf) twice: the generic sort decides by (box[0], id)
            for (int i = tid; i < M; i += NT)
                if (i > 0 && (k64[i] >> 16) == (k64[i - 1] >> 16)) tie = true;
            generic = __syncthreads_or(tie ? 1 : 0) != 0;
            bucketed = !generic;
        }
    }
    if (!generic && !bucketed) {
        for (int i = tid; i < S_eff; i += NT)
            k64[i] = i < M ? ((unsigned long long)(uint32_t)u_cls[i] << 48) | ((unsigned long long)(uint32_t)(~float_key(u_conf[i])) << 16) | (uint32_t)i
                           : ~0ull;
        __syncthreads();
        if (S_eff <= NT) {
            // one key per thread in registers; shuffles for partner distance < 32, smem ping-pong otherwise
            unsigned long long* ex = reinterpret_cast<unsigned long long*>(s_box);  // 2 x 1024 u64 scratch (rows not staged yet)
            unsigned long long mk = tid < S_eff ? k64[tid] : ~0ull;
            int pp = 0;
            for (int k = 2; k <= S_eff; k <<= 1) {
                for (int jj = k >> 1; jj > 0; jj >>= 1) {
                    unsigned long long ok;
                    if (jj >= 32) {
                        ex[pp * NT + tid] = mk;
                        __syncthreads();
                        ok = ex[pp * NT + (tid ^ jj)];
                        pp ^= 1;
                    } else {
                        ok = __shfl_xor_sync(0xffffffffu, mk, jj);
                    }
                    const bool want_min = (((tid & k) == 0) == ((tid & jj) == 0));
                    if (want_min == (ok < mk)) mk = ok;
                }
            }
            __syncthreads();
            if (tid < S_eff) k64[tid] = mk;
            __syncthreads();
        } else {
            for (int k = 2; k <= S_eff; k <<= 1) {
                for (int jj = k >> 1; jj > 0; jj >>= 1) {
                    for (int i = tid; i < S_eff; i += NT) {
                        const int ixj = i ^ jj;
                        if (ixj > i) {
                            const unsigned long long x = k64[i], y = k64[ixj];
                            if ((x > y) == ((i & k) == 0)) {
                                k64[i] = y;
                                k64[ixj] = x;
                            }
                        }
                    }
                    __syncthreads();
                }
            }
        }
        bool tie = false;
        for (int i = tid; i < M; i += NT)
            if (i > 0 && (k64[i] >> 16) == (k64[i - 1] >> 16)) tie = true;
        generic = __syncthreads_or(tie ? 1 : 0) != 0;
    }
    if (generic) {
        for (int i = tid; i < S_eff; i += NT) {
            if (i < M) {
                k_hi[i] = ((unsigned long long)(uint32_t)u_cls[i] << 32) | (uint32_t)(~float_key(u_conf[i]));
                k_lo[i] = ((unsigned long long)(a.tie_break_x0 ? float_key(u_box[i].x) : 0u) << 32) | u_id[i];
            } else {
                k_hi[i] = ~0ull;
                k_lo[i] = ~0ull;
            }
            s_pos[i] = (unsigned short)i;
        }
        __syncthreads();
        for (int k = 2; k <= S_eff; k <<= 1) {
            for (int jj = k >> 1; jj > 0; jj >>= 1) {
                for (int i = tid; i < S_eff; i += NT) {
                    const int ixj = i ^ jj;
                    if (ixj > i) {
                        const unsigned long long ah = k_hi[i], al = k_lo[i], bh = k_hi[ixj], bl = k_lo[ixj];
                        const bool gt = ah > bh || (ah == bh && al > bl);
                        if (gt == ((i & k) == 0)) {
                            k_hi[i] = bh;
                            k_lo[i] = bl;
                            k_hi[ixj] = ah;
                            k_lo[ixj] = al;
                            const unsigned short t0 = s_pos[i];
                            s_pos[i] = s_pos[ixj];
                            s_pos[ixj] = t0;
                        }
                    }
                }
                __syncthreads();
            }
        }
        for (int i = tid; i < M; i += NT) k64[i] = s_pos[i];  // permutation in the low 16 bits, like the fast path
        __syncthreads();  // the 128-bit keys (in the sorted-row area) are dead from here on
    }

    TRTX_STAMP(2);
    // ---------------- D: permute the stash into sorted order ----------------
    const bool greedy = a.mode == TRTX_NMS_GREEDY;
    IouTest iq;
    iq.thr = a.nms_thresh;
    iq.obb = a.box_format == TRTX_BOX_OBB;
    iq.retina = a.box_format == TRTX_BOX_RETINA;
    iq.zero_hit = 0.0f > a.nms_thresh;
    iq.fast_ok = fabsf(a.nms_thresh) <= 4.0f;
    for (int i = tid; i < M; i += NT) {
        const int pos = (int)(k64[i] & 0xffffull);
        const float4 bx = u_box[pos];
        if (a.box_format == TRTX_BOX_OBB) {  // covariance of the row's Gaussian, once per row; the angle is the first extra float
            const float ang = a.rows[(size_t)b * (1 + (size_t)a.max_rows * a.det_floats) + 1 + (size_t)u_id[pos] * a.det_floats +
                                     a.extra_offset];
            float ca, cb, cc;
            if (greedy)
                obb_cov_host(bx.z, bx.w, ang, ca, cb, cc);
            else
                obb_cov_dev(bx.z, bx.w, ang, ca, cb, cc);
            s_box[i] = make_float4(bx.x, bx.y, ca, cb);
            s_area[i] = cc;
        } else if (greedy) {  // the host IoUs work on corners and areas: form both once per row instead of once per pair
            s_box[i] = to_corners(a.box_format, bx);
            s_area[i] = box_area(a.box_format, bx);
        } else {
            s_box[i] = bx;
        }
        s_conf[i] = u_conf[pos];
        s_cls[i] = u_cls[pos];
        s_id[i] = u_id[pos];
        s_keep[i] = 0;
    }
    if (tid == 0) {
        s_nkept = 0;
        s_rem = 0;
        s_nshort = 0;
        s_nmed = 0;
        s_nlong = 0;
        s_cursor = 0;
        s_nunit = 0;
    }
    __syncthreads();
    TRTX_STAMP(8);

    const int R = 7 + a.extra_floats;
    float* o = a.out + (size_t)b * (1 + (size_t)a.max_det * R);
    int32_t* oidx = a.keep_index ? a.keep_index + (size_t)b * a.max_det : nullptr;
    // gathered buffers: [slots][world*B][1 + max_det*R]; this image's block on every rank
    const int gworld = a.g.world;
    const size_t goff = gworld ? ((size_t)a.g.slot * gworld * gridDim.x + (size_t)a.g.rank * gridDim.x + b) * (1 + (size_t)a.max_det * R) : 0;

    if (greedy) {
        // ---------------- E: class segments ----------------
        if (bucketed) {
            // the class histogram already is the segment table
            for (int i = tid; i < M; i += NT) {
                const int c = s_cls[i], m = s_chist[c];
                s_rowseg[i] = m > kShortSeg ? 0 : ((s_cstart[c] << 16) | m);
            }
            const int m = s_chist[tid], p0 = s_cstart[tid];
            if (m > kShortSeg)
                s_long[atomicAdd(&s_nlong, 1)] = (p0 << 16) | m;
            else if (m > 32)
                s_seg[S - 1 - atomicAdd(&s_nmed, 1)] = (p0 << 16) | m;
            else if (m > 0)
                s_seg[atomicAdd(&s_nshort, 1)] = (p0 << 16) | m;
            if (m > 1 && m <= kShortSeg) s_pos[p0] = (unsigned short)atomicAdd(&s_nunit, seg_units(m));
        } else
        for (int i = tid; i < M; i += NT) {
            if (i == 0 || s_cls[i] != s_cls[i - 1]) {
                int e = i + 1;
                while (e < M && s_cls[e] == s_cls[i]) ++e;
                const int m = e - i;
                // every row learns its segment (start << 16 | length; 0 = long segment, handled by the whole CTA)
                for (int r = i; r < e; ++r) s_rowseg[r] = m > kShortSeg ? 0 : ((i << 16) | m);
                if (m > kShortSeg)
                    s_long[atomicAdd(&s_nlong, 1)] = (i << 16) | m;  // M <= 2048: start and length fit 16 bits
                else if (m > 32)
                    s_seg[S - 1 - atomicAdd(&s_nmed, 1)] = (i << 16) | m;  // medium segments: taken first (longest-first scheduling)
                else
                    s_seg[atomicAdd(&s_nshort, 1)] = (i << 16) | m;
                if (m > 1 && m <= kShortSeg) s_pos[i] = (unsigned short)atomicAdd(&s_nunit, seg_units(m));
            }
        }
        __syncthreads();
        TRTX_STAMP(3);
        // ---- long segments: whole CTA, chunks of 32 ----
        const int n_long = s_nlong;
        for (int ls = 0; ls < n_long; ++ls) {
            const int p0 = s_long[ls] >> 16, m = s_long[ls] & 0xffff;
            int n_kept = 0;
            for (int c0 = 0; c0 < m; c0 += 32) {
                const int nchunk = min(32, m - c0);
                const int P = 32 * n_kept;
                for (int p = tid; p < P; p += NT) {
                    const int i = p & 31, k = p >> 5;
                    const int kr = s_krow[k];
                    if (i < nchunk && overlaps(iq, s_box[kr], s_area[kr], s_box[p0 + c0 + i], s_area[p0 + c0 + i]))
                        atomicOr(&s_rem, 1u << i);
                }
                for (int i = warp; i < 32; i += NW) {  // chunk member i: warp i % NW, lane = mate
                    const int jx = lane;
                    bool hit = false;
                    if (i < nchunk && jx < i)
                        hit = overlaps(iq, s_box[p0 + c0 + jx], s_area[p0 + c0 + jx], s_box[p0 + c0 + i], s_area[p0 + c0 + i]);
                    const unsigned mm = __ballot_sync(0xffffffffu, hit);
                    if (lane == 0) s_sup[i] = mm;
                }
                __syncthreads();
                if (warp == 0) {
                    const unsigned my = s_sup[lane];
                    unsigned alive = ~s_rem & (nchunk == 32 ? 0xffffffffu : ((1u << nchunk) - 1u));
                    for (unsigned rem = alive; rem != 0u;) {
                        const int jx = __ffs(rem) - 1;
                        const unsigned kill = __ballot_sync(0xffffffffu, (my >> jx) & 1u);
                        alive &= ~kill;
                        rem = alive & ~((2u << jx) - 1u);
                    }
                    if ((alive >> lane) & 1u) {
                        const int pos = n_kept + __popc(alive & ((1u << lane) - 1u));
                        s_krow[pos] = (unsigned short)(p0 + c0 + lane);
                        s_keep[p0 + c0 + lane] = 1;
                    }
                    if (lane == 0) {
                        s_nkept = n_kept + __popc(alive);
                        s_rem = 0;
                    }
                }
                __syncthreads();
                n_kept = s_nkept;
            }
        }
        TRTX_STAMP(4);
        // ---- short / medium segments (<= kShortSeg rows) ----
        // (1) IoU of every row against the earlier rows of its segment -> suppressor bitmap per row (bit j = row start+j
        //     overlaps it).  Work unit = (row, group g of 8 earlier rows) = one byte of the bitmap.  The units of all
        //     segments go into one list so the threads share them evenly whatever the segment lengths are; inside
        //     a segment they are ordered group-major, so neighbouring lanes hold neighbouring rows and test them
        //     against the SAME 8 earlier rows (shared-memory broadcasts instead of 128-byte-stride bank conflicts).
        for (int i = tid; i < M; i += NT) {
            const int rs = s_rowseg[i];
            if (rs == 0) continue;
            const int p0 = rs >> 16, m = rs & 0xffff, li = i - p0;
#pragma unroll
            for (int w = 0; w < kShortSeg / 32; ++w) s_mask[i * (kShortSeg / 32) + w] = 0u;
            const int ub = s_pos[p0] + li - 1;
            for (int g = 0; g * 8 < li; ++g)  // group g holds rows 8g+1 .. m-1 of the segment, after groups 0..g-1
                s_unit[ub + g * (m - 1) - 4 * g * (g - 1) - 8 * g] = (unsigned short)((i << 4) | g);
        }
        __syncthreads();
        TRTX_STAMP(9);
        {
            const int n_unit = s_nunit;
            unsigned char* mask_bytes = reinterpret_cast<unsigned char*>(s_mask);
            for (int u = tid; u < n_unit; u += NT) {
                const int e = s_unit[u], i = e >> 4, g = e & 15;
                const int p0 = s_rowseg[i] >> 16, li = i - p0;
                const float4 bi = s_box[i];
                const float ai = s_area[i];
                unsigned bits = 0u;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int jx = g * 8 + k;
                    if (jx < li && overlaps(iq, s_box[p0 + jx], s_area[p0 + jx], bi, ai)) bits |= 1u << k;
                }
                mask_bytes[i * (kShortSeg / 8) + g] = (unsigned char)bits;  // little-endian: byte g of the row's 3 words
            }
        }
        __syncthreads();
        TRTX_STAMP(7);
        // (2) one warp per segment resolves the greedy order on the bitmaps: 32 rows per step, ballots only
        const int n_short = s_nshort, n_med = s_nmed;
        for (;;) {
            int sidx = 0;
            if (lane == 0) sidx = atomicAdd(&s_cursor, 1);
            sidx = __shfl_sync(0xffffffffu, sidx, 0);
            if (sidx >= n_med + n_short) break;
            const int ent = sidx < n_med ? s_seg[S - 1 - sidx] : s_seg[sidx - n_med];
            const int p0 = ent >> 16, m = ent & 0xffff;
            unsigned kept[kShortSeg / 32] = {0u, 0u, 0u};
#pragma unroll
            for (int c = 0; c < kShortSeg / 32; ++c) {
                if (c * 32 >= m) break;
                const int nchunk = min(32, m - c * 32);
                const bool in = lane < nchunk;
                const int row = p0 + c * 32 + lane;
                unsigned mw[kShortSeg / 32] = {0u, 0u, 0u};
                if (in) {
#pragma unroll
                    for (int w = 0; w <= c; ++w) mw[w] = s_mask[row * (kShortSeg / 32) + w];
                }
                bool removed = false;
#pragma unroll
                for (int w = 0; w < c; ++w) removed |= (mw[w] & kept[w]) != 0u;  // suppressed by a kept row of an earlier chunk
                unsigned alive = __ballot_sync(0xffffffffu, in && !removed);
                const unsigned mymask = mw[c];
                for (unsigned rem = alive; rem != 0u;) {  // visit surviving rows only: one ballot per kept row
                    const int jx = __ffs(rem) - 1;
                    const unsigned kill = __ballot_sync(0xffffffffu, (mymask >> jx) & 1u);  // later rows that row jx suppresses
                    alive &= ~kill;
                    rem = alive & ~((2u << jx) - 1u);
                }
                kept[c] = alive;
                if ((alive >> lane) & 1u) s_keep[row] = 1;
            }
        }
        __syncthreads();
    } else {
        // one-shot: dropped iff some earlier same-class row (higher conf) overlaps (postprocess.cu:89-111)
        for (int i = tid; i < M; i += NT) {
            const int ci = s_cls[i];
            const float4 bi = s_box[i];
            bool keep = true;
            for (int jx = i - 1; jx >= 0 && s_cls[jx] == ci; --jx) {
                if (iq.obb ? obb_probiou_dev(bi, s_area[i], s_box[jx], s_area[jx]) > a.nms_thresh
                           : iou_oneshot(bi, s_box[jx]) > a.nms_thresh) {
                    keep = false;
                    break;
                }
            }
            s_keep[i] = keep ? 1 : 0;
        }
        __syncthreads();
    }

    TRTX_STAMP(5);
    // ---------------- F: block scan of the output flags, rows in sorted (class, conf) order ----------------
    // greedy: only kept rows are emitted; one-shot: every row is emitted with its keep flag
    int carry = 0;
    for (int base = 0; base < M; base += NT) {
        const int i = base + tid;
        const bool emit = i < M && (a.mode == TRTX_NMS_ONESHOT || s_keep[i]);
        const unsigned bal = __ballot_sync(0xffffffffu, emit);
        if (lane == 0) s_wsum[warp] = __popc(bal);
        __syncthreads();
        if (warp == 0) {
            int v = lane < NW ? s_wsum[lane] : 0, tot;
            const int ex = warp_excl_scan(v, lane, &tot);
            s_wsum[lane] = ex;
            if (lane == 0) s_nkept = tot;
        }
        __syncthreads();
        const int k = carry + s_wsum[warp] + __popc(bal & ((1u << lane) - 1u));
        if (emit && k < a.max_det) {
            // rows that were turned into corners / covariances for the overlap tests are emitted as they came in
            const float4 bx = a.box_format == TRTX_BOX_OBB || (greedy && a.box_format == TRTX_BOX_CXCYWH)
                                  ? fetch_row(a, b, s_id[i]).box
                                  : s_box[i];
            float* row = o + 1 + (size_t)k * R;
            row[0] = bx.x;
            row[1] = bx.y;
            row[2] = bx.z;
            row[3] = bx.w;
            row[4] = s_conf[i];
            row[5] = (float)s_cls[i];
            row[6] = s_keep[i] ? 1.0f : 0.0f;
            if (oidx) oidx[k] = a.from_tiles ? __float_as_int(a.cand[2 * ((size_t)b * a.slots_per_image + s_id[i]) + 1].z)
                                             : (int)s_id[i];
            if (a.extra_floats && !a.from_tiles) {
                const float* src = a.rows + (size_t)b * (1 + (size_t)a.max_rows * a.det_floats) + 1 +
                                   (size_t)s_id[i] * a.det_floats + a.extra_offset;
                for (int e = 0; e < a.extra_floats; ++e) row[7 + e] = src[e];
            }
        }
        carry += s_nkept;
        __syncthreads();
    }
    const int n_rows_out = min(carry, a.max_det);
    if (tid == 0) o[0] = (float)n_rows_out;
    // rows >= count are zero (the reference memsets its decode buffer, yolov8_det.cpp:106)
    for (int i = n_rows_out * R + tid; i < a.max_det * R; i += NT) o[1 + i] = 0.0f;
    if (oidx)
        for (int i = n_rows_out + tid; i < a.max_det; i += NT) oidx[i] = -1;
    if (gworld) {
        // The image's block [count, rows...] is contiguous and was just written to `o` by this CTA: copy its live part to every
        // rank's gathered buffer with lane-consecutive stores (full 128-byte NVLink writes instead of one 4-byte packet per
        // float; rows past `count` are NOT cleared on the peers -- consumers read `count` rows).
        __syncthreads();
        const int live = 1 + n_rows_out * R;
        for (int p = 0; p < gworld; ++p) {
            float* dstp = a.g.out[p] + goff;
            for (int i = tid; i < live; i += NT) dstp[i] = i == 0 ? (float)n_rows_out : o[i];
        }
        __syncthreads();  // CTA-scope order of all peer stores before thread 0's system-scope fence (cumulative)
        if (tid == 0) {
            // gpu-scope fences order this CTA's stores before its count and the last CTA's view of all counts before the flag;
            // the ONE system-scope operation is the release store of the flag (a system-scope fence under the step's HBM
            // traffic costs several microseconds each: tools/gather_probe.py)
            __threadfence();
            if (atomicAdd(&a.g.ctrl[1], 1u) == gridDim.x - 1) {  // last CTA of the launch: publish
                a.g.ctrl[1] = 0u;
                __threadfence_system();  // the ONE system-scope fence of the launch; the counters follow as relaxed stores
                const size_t fi = (size_t)a.g.rank * a.g.slots + a.g.slot;  // this rank's publish counter of the slot, on every rank
                const unsigned v = *reinterpret_cast<volatile unsigned*>(a.g.flags[a.g.rank] + fi) + 1u;
                for (int p = 0; p < gworld; ++p) st_relaxed_sys(a.g.flags[p] + fi, v);
            }
        }
    }
    TRTX_STAMP(6);
}

// Completes a gather of `nslots` slots on this rank: spins until every rank's publish counter of each slot has reached this
// rank's own (its own publish precedes this kernel in stream order).  One warp; gives up after ~2 s of SM clocks (ctrl[2] = 1)
// instead of hanging the GPU.  The polls are RELAXED system-scope loads and there is no fence: whatever reads the gathered rows
// is a later kernel (or copy) of the stream, and the kernel boundary orders it after these loads.  (Measured, tools/
// gather_probe.py and profiles/r02e_gather.log: every system-scope fence or release / acquire executed while the step's
// kernels stream at ~6 TB/s stalls the whole step by several microseconds.)
__global__ void __launch_bounds__(64) gather_wait_kernel(NmsArgs::Gather g, int nslots) {
    const int lane = threadIdx.x;  // one thread per (rank, slot): world * nslots <= 64
    const unsigned* fl = g.flags[g.rank];
    bool ok = true;
    if (lane < g.world * nslots) {
        const int r = lane / nslots, sl = g.slot + lane - r * nslots;
        const unsigned expected = ld_relaxed_sys(fl + (size_t)g.rank * g.slots + sl);
        const unsigned* f = fl + (size_t)r * g.slots + sl;
        const long long t0 = clock64();
        while ((int)(ld_relaxed_sys(f) - expected) < 0) {
            __nanosleep(200);
            if (clock64() - t0 > 4000000000ll) {
                ok = false;
                break;
            }
        }
    }
    if (!ok) g.ctrl[2] = 1u;
}

// The publish as SEPARATE small kernels (default of PeerGather.push): (1) gather_copy_kernel -- a few 256-thread CTAs that
// co-reside with the step's streaming kernels -- copies the live part of every image's block of the local compact outputs
// into the slots on every rank: plain stores, no fence, no flag; (2) gather_publish_kernel -- one warp -- bumps this rank's
// publish counter of every slot on every rank with relaxed system-scope stores.  The ordering "rows before counter" is the
// KERNEL BOUNDARY between the two (a grid's writes, peer writes included, are performed at system scope before a dependent
// grid of the stream starts), so no thread ever executes a system-scope fence.  Neither kernel waits for anybody.
struct PushSrc {
    const float* src[8];  // local compact outputs of n consecutive steps -> slots slot .. slot+n-1
    int n;
};
__global__ void __launch_bounds__(256) gather_copy_kernel(NmsArgs::Gather g, PushSrc ps, int batch, int cols, int max_det, int R) {
    // one CTA per (step, image): the kernel is a chain of dependent latencies (count -> rows -> stores), so its duration is one
    // such chain, not their sum (8 CTAs walking 16 blocks each took ~40 us under the step's traffic and, because the NMS that
    // overwrites a block has to wait for this copy, stalled the scan -> NMS chain by that much: profiles/r02e_gather.log)
    const int tid = threadIdx.x;
    const int w = blockIdx.x;
    const int k = w / batch, b = w - k * batch;
    const float* src = ps.src[k] + (size_t)b * cols;
    const int n = min(max((int)src[0], 0), max_det);
    const int live = 1 + n * R;
    const size_t off = (((size_t)(g.slot + k) * g.world + g.rank) * batch + b) * cols;
    constexpr int U = 4;  // rows in flight per thread: all loads first, then the stores to every rank
    for (int i0 = tid; i0 < live; i0 += 256 * U) {
        float v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = (i0 + u * 256 < live) ? src[i0 + u * 256] : 0.0f;
        for (int p = 0; p < g.world; ++p) {
            float* dst = g.out[p] + off;
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (i0 + u * 256 < live) dst[i0 + u * 256] = v[u];
        }
    }
}
__global__ void __launch_bounds__(64) gather_publish_kernel(NmsArgs::Gather g, int nslots) {
    const int lane = threadIdx.x;  // one thread per (destination rank, slot): world * nslots <= 64
    if (lane >= g.world * nslots) return;
    const int p = lane / nslots, k = lane - p * nslots;
    const size_t fi = (size_t)g.rank * g.slots + g.slot + k;  // this rank's publish counter of the slot, on every rank
    // the local copy of the counter is only ever written by this rank's publishes, which are stream-ordered
    const unsigned v = ld_relaxed_sys(g.flags[g.rank] + fi) + 1u;
    __syncwarp();  // (every lane has read the old local value before lane p == rank overwrites it)
    __syncthreads();
    st_relaxed_sys(g.flags[p] + fi, v);
}

static size_t nms_smem_bytes(int pre_topk, int tiles = 0) {
    const size_t S = pre_topk <= 1024 ? 1024 : kMaxSort;
    return S * (16 + 16 + 8 + 6 * 4 + 4 + 2 + 2 + 1 + 2 * (kShortSeg / 8) + 4) + 64 + sizeof(int) * (size_t)(tiles + 1);
}

static int nms_validate(const trtx_nms_params* q) {
    if (!q) return TRTX_ERR_INVALID;
    if (q->box_format < 0 || q->box_format > TRTX_BOX_OBB) return TRTX_ERR_INVALID;
    if (q->box_format == TRTX_BOX_OBB && q->extra_floats < 1) return TRTX_ERR_INVALID;  // the angle travels as the first extra
    if (q->mode != TRTX_NMS_GREEDY && q->mode != TRTX_NMS_ONESHOT) return TRTX_ERR_INVALID;
    if (q->max_det <= 0 || q->extra_floats < 0 || q->extra_offset < 0) return TRTX_ERR_INVALID;
    return TRTX_OK;
}

// The half-SM kernel covers the fused YOLO source in greedy mode with axis-aligned boxes and at most 1024 rows, without
// the gather fused into the kernel.
static bool nms_half_ok(const NmsArgs& a) {
    return a.from_tiles && a.mode == TRTX_NMS_GREEDY && a.box_format != TRTX_BOX_OBB && a.pre_topk <= 1024 && a.g.world == 0;
}

template <int NT>
static cudaError_t nms_launch_nt(const NmsArgs& a, int batch, size_t smem, cudaStream_t st) {
    // per-device function attribute; cheap and idempotent, so set on every call (no global state).
    // 227 KB per CTA minus the kernel's static shared memory (histograms, <= ~18 KB)
    constexpr size_t kMaxDynSmem = (227 - 20) * 1024;
    cudaFuncSetAttribute(nms_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynSmem);
    // Programmatic dependent launch: the CTAs may be placed (and run up to griddepcontrol.wait) while the previous kernel
    // of the stream -- the scan, which triggers once its streaming loop is done -- finishes its tail, instead of after
    // it.  Stream capture turns the attribute into a programmatic graph edge.
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(batch);
    cfg.blockDim = dim3(NT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
#ifdef TRTX_NMS_NO_PDL  // experiment build (tools/step_timeline.py): the ordinary launch, for before / after timelines
    cfg.numAttrs = 0;
#endif
    cudaError_t e = cudaLaunchKernelEx(&cfg, nms_kernel<NT>, a);
    if (e == cudaErrorNotSupported || e == cudaErrorInvalidValue) {  // a driver without PDL: ordinary launch
        (void)cudaGetLastError();
        cfg.numAttrs = 0;
        e = cudaLaunchKernelEx(&cfg, nms_kernel<NT>, a);
    }
    return e;
}

// threads: 0 / 1024 = the general kernel; 512 = the half-SM one (TRTX_ERR_UNSUPPORTED where it does not cover the call)
static int nms_launch(NmsArgs& a, int batch, cudaStream_t st, int threads = 0) {
#ifdef TRTX_NMS_PROBE
    a.dbg = t_nms_stamps;
#endif
    TRTX_TL_TAKE(a);
    if (a.pre_topk > kMaxSort) return TRTX_ERR_UNSUPPORTED;
    if (threads != 0 && threads != kNmsThreads && threads != kNmsThreadsHalf) return TRTX_ERR_UNSUPPORTED;
    const bool half = threads == kNmsThreadsHalf;
    if (half && !nms_half_ok(a)) return TRTX_ERR_UNSUPPORTED;
    const size_t smem = nms_smem_bytes(a.pre_topk, a.from_tiles ? a.tiles_per_image : 0);
    if (smem > (227 - 20) * 1024) return TRTX_ERR_UNSUPPORTED;
    const cudaError_t e = half ? nms_launch_nt<kNmsThreadsHalf>(a, batch, smem, st) : nms_launch_nt<kNmsThreads>(a, batch, smem, st);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        g_last_cuda_error = (int)e;
        return TRTX_ERR_CUDA;
    }
    return check_launch();
}

}  // namespace trtx

using namespace trtx;

extern "C" {

#ifdef TRTX_NMS_PROBE
// probe build only: device buffer of 16*batch int64 receiving clock64 phase stamps of nms_kernel (this thread's launches)
TRTX_API int trtx_probe_set_nms_stamps(void* p) {
    t_nms_stamps = static_cast<long long*>(p);
    return TRTX_OK;
}
// probe build only: device buffer of `records` timeline records (common.cuh) for this thread's next launches; null: off
TRTX_API int trtx_probe_set_timeline(void* p, int records) {
    t_tl_buf = static_cast<unsigned long long*>(p);
    t_tl_records = p ? records : 0;
    t_tl_next = 0;
    return TRTX_OK;
}
TRTX_API size_t trtx_probe_timeline_record_words() { return kTlRecordWords; }
#endif

TRTX_API size_t trtx_nms_workspace_size(const trtx_nms_params* p, int batch, int max_rows) {
    if (nms_validate(p) || batch <= 0 || max_rows <= 0) return 0;
    return align_up(sizeof(uint2) * (size_t)batch * max_rows);
}

TRTX_API int trtx_nms_enqueue(const trtx_nms_params* p, int batch, const float* plugin_out_dev, int max_rows,
                              int det_floats, float* compact_out_dev, int32_t* keep_index_dev, void* workspace_dev,
                              size_t workspace_bytes, trtx_stream_t stream) {
    int rc = nms_validate(p);
    if (rc) return rc;
    if (batch <= 0 || max_rows <= 0 || det_floats < 5 || !plugin_out_dev || !compact_out_dev || !workspace_dev)
        return TRTX_ERR_INVALID;
    if (p->extra_floats && p->extra_offset + p->extra_floats > det_floats) return TRTX_ERR_INVALID;
    if (p->box_format != TRTX_BOX_RETINA && det_floats < 6) return TRTX_ERR_INVALID;
    if (workspace_bytes < trtx_nms_workspace_size(p, batch, max_rows)) return TRTX_ERR_WORKSPACE;
    NmsArgs a{};
    a.rows = plugin_out_dev;
    a.max_rows = max_rows;
    a.det_floats = det_floats;
    a.from_tiles = 0;
    a.list = static_cast<uint2*>(workspace_dev);
    a.list_stride = max_rows;
    a.box_format = p->box_format;
    a.mode = p->mode;
    a.class_aware = p->class_aware && p->box_format != TRTX_BOX_RETINA;
    a.tie_break_x0 = p->tie_break_x0;
    a.conf_thresh = p->conf_thresh;
    a.nms_thresh = p->nms_thresh;
    a.pre_topk = max_rows < kMaxSort ? max_rows : kMaxSort;
    a.max_det = p->max_det;
    a.extra_floats = p->extra_floats;
    a.extra_offset = p->extra_offset;
    a.out = compact_out_dev;
    a.keep_index = keep_index_dev;
    return nms_launch(a, batch, static_cast<cudaStream_t>(stream));
}

// shared by the fused call and its split form
static int fill_gather(const trtx_gather* g, NmsArgs::Gather* o) {
    memset(o, 0, sizeof(*o));
    if (!g) return TRTX_OK;
    if (g->world < 1 || g->world > 8 || g->rank < 0 || g->rank >= g->world || g->slots < 1 || g->slot < 0 || g->slot >= g->slots ||
        !g->ctrl_dev)
        return TRTX_ERR_INVALID;
    for (int r = 0; r < g->world; ++r) {
        if (!g->out_dev[r] || !g->flags_dev[r]) return TRTX_ERR_INVALID;
        o->out[r] = g->out_dev[r];
        o->flags[r] = g->flags_dev[r];
    }
    o->ctrl = g->ctrl_dev;
    o->world = g->world;
    o->rank = g->rank;
    o->slots = g->slots;
    o->slot = g->slot;
    return TRTX_OK;
}

static int yolo_nms_tiles(const trtx_yolo_params* p, const trtx_nms_params* q, int batch, const YoloArgs& ya,
                          const YoloLayout& L, float* compact_out_dev, int32_t* keep_index_dev, void* workspace_dev,
                          cudaStream_t st, const trtx_gather* gather = nullptr) {
    if (q->box_format == TRTX_BOX_OBB) return TRTX_ERR_UNSUPPORTED;  // the tile records carry no angle: use the plugin-row source
    NmsArgs a{};
    a.from_tiles = 1;
    a.tiles_per_image = L.tiles_per_image;
    a.slots_per_image = L.slots_per_image;
    a.tile_slots = L.tile_cells * L.apc;
    a.num_levels = p->num_levels;
    for (int l = 0; l < p->num_levels; ++l) {
        a.lv_tile_begin[l] = L.level_tile_begin[l];
        a.lv_slot_begin[l] = L.level_slot_begin[l];
    }
    a.tile_count = ya.tile_count;
    a.cand = ya.cand;
    a.list = reinterpret_cast<uint2*>(static_cast<char*>(workspace_dev) + L.off_list);
    a.list_stride = L.slots_per_image;
    a.box_format = q->box_format;
    a.mode = q->mode;
    a.class_aware = q->class_aware;
    a.tie_break_x0 = q->tie_break_x0;
    a.conf_thresh = q->conf_thresh;
    a.nms_thresh = q->nms_thresh;
    a.pre_topk = p->max_out;  // the reference's plugin capacity bounds what reaches nms()
    a.max_det = q->max_det;
    a.out = compact_out_dev;
    a.keep_index = keep_index_dev;
    const int rc = fill_gather(gather, &a.g);
    if (rc) return rc;
    return nms_launch(a, batch, st, p->tune_nms_threads);
}

TRTX_API int trtx_yolo_decode_nms_enqueue(const trtx_yolo_params* p, const trtx_nms_params* q, int batch,
                                          const void* const* inputs_dev, float* compact_out_dev,
                                          int32_t* keep_index_dev, void* workspace_dev, size_t workspace_bytes,
                                          trtx_stream_t stream) {
    int rc = nms_validate(q);
    if (rc) return rc;
    if (!compact_out_dev) return TRTX_ERR_INVALID;
    if (q->extra_floats) return TRTX_ERR_UNSUPPORTED;  // extras need the plugin-format rows (use the two-stage path)
    YoloArgs ya;
    YoloLayout L;
    rc = yolo_fill_args(p, batch, inputs_dev, workspace_dev, workspace_bytes, &ya, &L);
    if (rc) return rc;
    if (p->max_out > kMaxSort) return TRTX_ERR_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = yolo_scan_launch(ya, L, p->in_dtype, batch, st);
    if (rc) return rc;
    return yolo_nms_tiles(p, q, batch, ya, L, compact_out_dev, keep_index_dev, workspace_dev, st);
}

TRTX_API int trtx_yolo_decode_nms_gather_enqueue(const trtx_yolo_params* p, const trtx_nms_params* q, int batch,
                                                 const void* const* inputs_dev, float* compact_out_dev, int32_t* keep_index_dev,
                                                 void* workspace_dev, size_t workspace_bytes, const trtx_gather* gather,
                                                 trtx_stream_t stream) {
    int rc = nms_validate(q);
    if (rc) return rc;
    if (!compact_out_dev || !gather) return TRTX_ERR_INVALID;
    if (q->extra_floats) return TRTX_ERR_UNSUPPORTED;
    YoloArgs ya;
    YoloLayout L;
    rc = yolo_fill_args(p, batch, inputs_dev, workspace_dev, workspace_bytes, &ya, &L);
    if (rc) return rc;
    if (p->max_out > kMaxSort) return TRTX_ERR_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    rc = yolo_scan_launch(ya, L, p->in_dtype, batch, st);
    if (rc) return rc;
    return yolo_nms_tiles(p, q, batch, ya, L, compact_out_dev, keep_index_dev, workspace_dev, st, gather);
}

TRTX_API int trtx_gather_wait_many_enqueue(const trtx_gather* gather, int nslots, trtx_stream_t stream) {
    NmsArgs::Gather g;
    int rc = fill_gather(gather, &g);
    if (rc || !gather) return rc ? rc : TRTX_ERR_INVALID;
    if (nslots < 1 || nslots > 8 || gather->slot + nslots > gather->slots) return TRTX_ERR_INVALID;
    gather_wait_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream)>>>(g, nslots);
    return check_launch();
}
TRTX_API int trtx_gather_wait_enqueue(const trtx_gather* gather, trtx_stream_t stream) {
    return trtx_gather_wait_many_enqueue(gather, 1, stream);
}

TRTX_API int trtx_gather_push_many_enqueue(const trtx_gather* gather, const float* const* compact_outs_dev, int n, int batch, int max_det,
                                           int extra_floats, trtx_stream_t stream) {
    NmsArgs::Gather g;
    int rc = fill_gather(gather, &g);
    if (rc || !gather || !compact_outs_dev || batch <= 0 || max_det <= 0 || extra_floats < 0) return rc ? rc : TRTX_ERR_INVALID;
    if (n < 1 || n > 8 || gather->slot + n > gather->slots) return TRTX_ERR_INVALID;
    PushSrc ps{};
    ps.n = n;
    for (int k = 0; k < n; ++k) {
        if (!compact_outs_dev[k]) return TRTX_ERR_INVALID;
        ps.src[k] = compact_outs_dev[k];
    }
    if (n * g.world > 64) return TRTX_ERR_UNSUPPORTED;
    const int R = 7 + extra_floats;
    const int work = n * batch;
    gather_copy_kernel<<<work, 256, 0, static_cast<cudaStream_t>(stream)>>>(g, ps, batch, 1 + max_det * R, max_det, R);
    gather_publish_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream)>>>(g, n);
    return check_launch();
}
TRTX_API int trtx_gather_push_enqueue(const trtx_gather* gather, const float* compact_out_dev, int batch, int max_det,
                                      int extra_floats, trtx_stream_t stream) {
    return trtx_gather_push_many_enqueue(gather, &compact_out_dev, 1, batch, max_det, extra_floats, stream);
}

// ---- peer memory for the gather: cudaMalloc + CUDA IPC (one process per GPU on one NVSwitch node) ----
TRTX_API int trtx_peer_alloc(size_t bytes, void** dev_ptr, unsigned char handle[64]) {
    if (!bytes || !dev_ptr || !handle) return TRTX_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) e = cudaMemset(p, 0, bytes);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        g_last_cuda_error = (int)e;
        if (p) cudaFree(p);
        return TRTX_ERR_CUDA;
    }
    memcpy(handle, &h, 64);
    *dev_ptr = p;
    return TRTX_OK;
}
TRTX_API int trtx_peer_open(const unsigned char handle[64], void** dev_ptr) {
    if (!handle || !dev_ptr) return TRTX_ERR_INVALID;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    const cudaError_t e = cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        g_last_cuda_error = (int)e;
        return TRTX_ERR_CUDA;
    }
    return TRTX_OK;
}
TRTX_API int trtx_peer_close(void* dev_ptr) { return cudaIpcCloseMemHandle(dev_ptr) == cudaSuccess ? TRTX_OK : TRTX_ERR_CUDA; }
TRTX_API int trtx_peer_free(void* dev_ptr) { return cudaFree(dev_ptr) == cudaSuccess ? TRTX_OK : TRTX_ERR_CUDA; }

TRTX_API int trtx_yolo_scan_enqueue(const trtx_yolo_params* p, int batch, const void* const* inputs_dev,
                                    void* workspace_dev, size_t workspace_bytes, trtx_stream_t stream) {
    YoloArgs ya;
    YoloLayout L;
    int rc = yolo_fill_args(p, batch, inputs_dev, workspace_dev, workspace_bytes, &ya, &L);
    if (rc) return rc;
    return yolo_scan_launch(ya, L, p->in_dtype, batch, static_cast<cudaStream_t>(stream));
}

TRTX_API int trtx_yolo_nms_after_scan_enqueue(const trtx_yolo_params* p, const trtx_nms_params* q, int batch,
                                              const void* const* inputs_dev, float* compact_out_dev,
                                              int32_t* keep_index_dev, void* workspace_dev, size_t workspace_bytes,
                                              trtx_stream_t stream) {
    int rc = nms_validate(q);
    if (rc) return rc;
    if (!compact_out_dev) return TRTX_ERR_INVALID;
    if (q->extra_floats) return TRTX_ERR_UNSUPPORTED;
    YoloArgs ya;
    YoloLayout L;
    rc = yolo_fill_args(p, batch, inputs_dev, workspace_dev, workspace_bytes, &ya, &L);
    if (rc) return rc;
    if (p->max_out > kMaxSort) return TRTX_ERR_UNSUPPORTED;
    return yolo_nms_tiles(p, q, batch, ya, L, compact_out_dev, keep_index_dev, workspace_dev,
                          static_cast<cudaStream_t>(stream));
}

}  // extern "C"

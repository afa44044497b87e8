// refinedet.cu -- RefineDet post-process for sm_100a: two-stage prior decode + per-class greedy NMS.
// Replaces PriorBox / decode / nms and the driver glue of refinedet/refinedet.cpp:553-790.  The reference runs it as
// tensor-library ops in fp64 for batch 1: per class a sort, then a host loop with ~20 small launches and 4 device-to-host
// syncs per kept box.  Here every image of the batch goes through three launches:
//   refinedet_decode_kernel  one warp per 32 priors: both decodes in fp64 -> corners [B,P,4] in the workspace, and one
//                            32-bit candidate mask per (image, class, tile) from a warp-transposed odm_conf tile
//   refinedet_nms_kernel     one 1024-thread CTA per (class, image): candidates in prior order from the masks, top_k
//                            select + sort, greedy NMS in chunks of 32
//   refinedet_pack_kernel    prefix over the classes' kept counts -> compact rows, zeroed tail
//
// Exactness (DESIGN.md section 4, "RefineDet"):
//  * Every fp64 operation is rounded on its own (__d*_rn), because the reference's eager ops never fuse.  exp is CUDA's
//    fp64 exp, which the reference's tensor library calls on the GPU too.
//  * `x > (double)t` for a float x and a float threshold t is the float compare `x > t`; NaN is never a candidate.
//    The reference's `odm_conf * (0/1 mask) > mask_thresh` (:741-760) reduces to `arm > obj_thresh && odm > conf_thresh`
//    for every input: a masked value is 0, -0 or NaN, none of which passes.
//  * The IoU uses the suppressor's corners rounded to float (`.item().toFloat()`, :674-677) as clamp bounds, the
//    tensor library's clamp (NaN bound -> NaN, NaN value passes through), union = (area_j - inter) + area_i and IEEE
//    division; j is dropped when !(IoU < nms_thresh), so a NaN IoU suppresses.  The test is asymmetric: i, the higher
//    ranked box, is always the suppressor.
//  * Equal scores rank the lower prior index first, at the top_k cut too (desc_key, select_sort.cuh).  The reference's
//    sort is unstable there, so parity holds on tie-free inputs.
#include <math.h>

#include <algorithm>
#include <initializer_list>

#include "common.cuh"
#include "select_sort.cuh"

namespace trtx {

constexpr int kRdDecodeWarps = 4;
constexpr int kRdPackThreads = 256;

struct RdArgs {
    const float* priors;    // [P,4]
    const float* arm_loc;   // [B,P,4]
    const float* arm_conf;  // [B,P,2]
    const float* odm_loc;   // [B,P,4]
    const float* odm_conf;  // [B,P,C]
    double4* boxes;         // [B,P] ODM corners (written for priors passing the objectness gate)
    uint32_t* masks;        // [B,C-1,T] candidate bit r of tile t = prior 32t+r
    int* kept_count;        // [B,C-1]
    int* kept_prior;        // [B,C-1,top_k] prior index of each kept row, keep order
    float* out;             // [B, 1 + max_out*7]
    int P, C, T, top_k, max_out, pitch, region;
    float obj_thresh, conf_thresh;
    double nms_thresh, v0, v1;
};

// at::clamp with scalar bounds: a NaN bound fills the result with NaN, a NaN value passes through
__device__ __forceinline__ double rd_clamp(double v, double lo, double hi) {
    if (isnan(lo) || isnan(hi)) return __longlong_as_double(0x7ff8000000000000ll);
    if (isnan(v)) return v;
    return fmin(fmax(v, lo), hi);
}

// nms(), refinedet.cpp:674-691: does kept box i drop box j?
__device__ __forceinline__ bool rd_suppress(double ix1, double iy1, double ix2, double iy2, double iarea, double jx1,
                                            double jy1, double jx2, double jy2, double jarea, double thr) {
    const double kMax = 2147483647.0, kMin = -2147483648.0;  // INT_MAX * 1.0, INT_MIN * 1.0
    const double xx1 = rd_clamp(jx1, (double)__double2float_rn(ix1), kMax);
    const double yy1 = rd_clamp(jy1, (double)__double2float_rn(iy1), kMax);
    const double xx2 = rd_clamp(jx2, kMin, (double)__double2float_rn(ix2));
    const double yy2 = rd_clamp(jy2, kMin, (double)__double2float_rn(iy2));
    const double w = rd_clamp(__dsub_rn(xx2, xx1), 0.0, kMax);
    const double h = rd_clamp(__dsub_rn(yy2, yy1), 0.0, kMax);
    const double inter = __dmul_rn(w, h);
    const double uni = __dadd_rn(__dsub_rn(jarea, inter), iarea);
    return !(__ddiv_rn(inter, uni) < thr);
}

__global__ void __launch_bounds__(kRdDecodeWarps * 32, 4) refinedet_decode_kernel(const __grid_constant__ RdArgs a, int batch) {
    extern __shared__ float s_conf[];  // [warps][32 rows][pitch]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gw = blockIdx.x * kRdDecodeWarps + warp;
    if (gw >= batch * a.T) return;  // warp-uniform; the kernel has no CTA barrier
    const int b = gw / a.T, t = gw - b * a.T;
    const int p = t * 32 + lane;
    const bool valid = p < a.P;
    const size_t row = (size_t)b * a.P + p;
    const bool obj = valid && __ldg(a.arm_conf + row * 2 + 1) > a.obj_thresh;  // :739-741
    const unsigned objm = __ballot_sync(0xffffffffu, obj);
    uint32_t* mk = a.masks + (size_t)b * (a.C - 1) * a.T + t;
    if (objm == 0) {
        for (int c = lane; c < a.C - 1; c += 32) mk[(size_t)c * a.T] = 0u;
        return;
    }
    if (obj) {
        const float4 pr = __ldg(reinterpret_cast<const float4*>(a.priors) + p);
        const float4 al = __ldg(reinterpret_cast<const float4*>(a.arm_loc) + row);
        const float4 ol = __ldg(reinterpret_cast<const float4*>(a.odm_loc) + row);
        // decode(arm_loc, prior), :606-608: c1 = p_xy + (loc_xy * v0) * p_wh, c2 = p_wh * exp(loc_wh * v1)
        const double px = pr.x, py = pr.y, pw = pr.z, ph = pr.w;
        const double ax = __dadd_rn(px, __dmul_rn(__dmul_rn((double)al.x, a.v0), pw));
        const double ay = __dadd_rn(py, __dmul_rn(__dmul_rn((double)al.y, a.v0), ph));
        const double aw = __dmul_rn(pw, exp(__dmul_rn((double)al.z, a.v1)));
        const double ah = __dmul_rn(ph, exp(__dmul_rn((double)al.w, a.v1)));
        // decode(odm_loc, ARM box, b_form_pt = true), :606-613: c3 = xy - wh/2, c4 = c3 + wh
        const double ox = __dadd_rn(ax, __dmul_rn(__dmul_rn((double)ol.x, a.v0), aw));
        const double oy = __dadd_rn(ay, __dmul_rn(__dmul_rn((double)ol.y, a.v0), ah));
        const double ow = __dmul_rn(aw, exp(__dmul_rn((double)ol.z, a.v1)));
        const double oh = __dmul_rn(ah, exp(__dmul_rn((double)ol.w, a.v1)));
        const double x1 = __dsub_rn(ox, __dmul_rn(ow, 0.5));  // wh.div(2) is exact either way
        const double y1 = __dsub_rn(oy, __dmul_rn(oh, 0.5));
        a.boxes[row] = make_double4(x1, y1, __dadd_rn(x1, ow), __dadd_rn(y1, oh));
    }
    // the tile's odm_conf rows are contiguous: coalesced loads into shared memory, then lane c-1 reads column c
    const int nrows = min(32, a.P - t * 32);
    const float* src = a.odm_conf + ((size_t)b * a.P + (size_t)t * 32) * a.C;
    float* s = s_conf + warp * 32 * a.pitch;
    for (int e = lane; e < nrows * a.C; e += 32) {
        const int r = e / a.C;
        s[r * a.pitch + (e - r * a.C)] = ldg_stream_f1(src + e);
    }
    __syncwarp();
    for (int c = 1 + lane; c < a.C; c += 32) {
        uint32_t m = 0;
        for (int r = 0; r < nrows; ++r)
            if (((objm >> r) & 1u) && s[r * a.pitch + c] > a.conf_thresh) m |= 1u << r;  // :758
        mk[(size_t)(c - 1) * a.T] = m;
    }
}

__global__ void __launch_bounds__(kSelThreads) refinedet_nms_kernel(const __grid_constant__ RdArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ SelectScratch sc;
    __shared__ int s_warp[32];
    __shared__ int s_cnt, s_nkept;
    __shared__ unsigned s_sup, s_pair[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cls = blockIdx.x, b = blockIdx.y, K = a.C - 1, T = a.T;
    unsigned long long* sel = reinterpret_cast<unsigned long long*>(smem);  // [kSelThreads] sorted candidates
    unsigned long long* ckey = sel + kSelThreads;                           // [P] candidate keys (region A) ...
    double* bx1 = reinterpret_cast<double*>(ckey);                          // ... later the sorted rows' corners
    double* by1 = bx1 + kSelThreads;
    double* bx2 = by1 + kSelThreads;
    double* by2 = bx2 + kSelThreads;
    double* bar = by2 + kSelThreads;
    int* pref = reinterpret_cast<int*>(ckey + a.region);  // [T]
    int* kept = pref + T;                                  // [kSelThreads] rows kept, keep order
    const uint32_t* mk = a.masks + ((size_t)b * K + cls) * T;

    // 1. candidates of the class in ascending prior order (`nonzero`, :759): exclusive prefix of the tiles' popcounts
    int n = 0;
    for (int base = 0; base < T; base += kSelThreads) {
        const int t = base + tid;
        const int v = t < T ? __popc(mk[t]) : 0;
        int wt;
        const int ex = warp_excl_scan(v, lane, &wt);
        if (lane == 31) s_warp[warp] = wt;
        __syncthreads();
        if (warp == 0) {
            int tot;
            const int wex = warp_excl_scan(s_warp[lane], lane, &tot);
            s_warp[lane] = wex;
            if (lane == 0) s_cnt = tot;
        }
        __syncthreads();
        if (t < T) pref[t] = n + s_warp[warp] + ex;
        n += s_cnt;
        __syncthreads();
    }
    if (n == 0) {
        if (tid == 0) a.kept_count[(size_t)b * K + cls] = 0;
        return;
    }
    const int c = cls + 1;
    for (int t = warp; t < T; t += kSelThreads / 32) {
        const uint32_t m = mk[t];
        if ((m >> lane) & 1u) {
            const int p = t * 32 + lane;
            const float score = __ldg(a.odm_conf + ((size_t)b * a.P + p) * a.C + c);
            ckey[pref[t] + __popc(m & ((1u << lane) - 1u))] = desc_key(score, (uint32_t)p);
        }
    }
    __syncthreads();

    // 2. the top_k highest scores (:648-656), then sorted by score descending, prior ascending
    const int m = min(n, a.top_k);
    if (n > a.top_k) {
        uint32_t key_cut, id_cut;
        auto key = [&](int i) { return ~(uint32_t)(ckey[i] >> 32); };
        block_select_topk(key, n, a.top_k, sc, &key_cut, &id_cut);
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        for (int i = tid; i < n; i += kSelThreads) {
            const uint32_t k = key(i);
            if (k > key_cut || (k == key_cut && (uint32_t)i <= id_cut)) sel[atomicAdd(&s_cnt, 1)] = ckey[i];
        }
    } else {
        for (int i = tid; i < n; i += kSelThreads) sel[i] = ckey[i];
    }
    int S = 1;
    while (S < m) S <<= 1;
    for (int i = m + tid; i < S; i += kSelThreads) sel[i] = ~0ull;
    __syncthreads();
    block_bitonic_sort_u64(sel, S);

    // 3. corners and areas of the sorted rows (region A is free again)
    for (int r = tid; r < m; r += kSelThreads) {
        const double4 q = a.boxes[(size_t)b * a.P + (uint32_t)sel[r]];
        bx1[r] = q.x;
        by1[r] = q.y;
        bx2[r] = q.z;
        by2[r] = q.w;
        bar[r] = __dmul_rn(__dsub_rn(q.z, q.x), __dsub_rn(q.w, q.y));  // area, :645
    }
    if (tid == 0) {
        s_nkept = 0;
        s_sup = 0;
    }
    __syncthreads();

    // 4. greedy NMS (:658-693) in chunks of 32 rows.  Row j = base + lane of the chunk is tested by every warp against
    //    a slice of the rows kept before the chunk; warp w also tests row base + w against the rows after it in the
    //    chunk.  One thread then resolves the chunk in rank order.
    for (int base = 0; base < m; base += 32) {
        const int j = base + lane;
        const int nk = s_nkept;
        bool sup = false, pair = false;
        if (j < m) {
            const double jx1 = bx1[j], jy1 = by1[j], jx2 = bx2[j], jy2 = by2[j], ja = bar[j];
            for (int k = warp; k < nk && !sup; k += 32) {
                const int i = kept[k];
                sup = rd_suppress(bx1[i], by1[i], bx2[i], by2[i], bar[i], jx1, jy1, jx2, jy2, ja, a.nms_thresh);
            }
            const int i = base + warp;  // < j < m when lane > warp
            pair = lane > warp &&
                   rd_suppress(bx1[i], by1[i], bx2[i], by2[i], bar[i], jx1, jy1, jx2, jy2, ja, a.nms_thresh);
        }
        const unsigned sb = __ballot_sync(0xffffffffu, sup), pb = __ballot_sync(0xffffffffu, pair);
        if (lane == 0) {
            s_pair[warp] = pb;
            if (sb) atomicOr(&s_sup, sb);
        }
        __syncthreads();
        if (tid == 0) {
            const int len = min(32, m - base);
            unsigned alive = (len == 32 ? 0xffffffffu : (1u << len) - 1u) & ~s_sup;
            for (int i = 0; i < len; ++i)
                if ((alive >> i) & 1u) alive &= ~s_pair[i];
            int k = nk;
            for (; alive; alive &= alive - 1u) kept[k++] = base + __ffs(alive) - 1;
            s_nkept = k;
            s_sup = 0;
        }
        __syncthreads();
    }

    // 5. kept rows of the class.  The reference's `score_my[0] < conf_thresh` (:774) cannot fire: every candidate's
    //    score already passed `> conf_thresh` (the same 0.01 literal) at :758.
    const int nk = s_nkept;
    int* dst = a.kept_prior + ((size_t)b * K + cls) * a.top_k;
    for (int r = tid; r < nk; r += kSelThreads) dst[r] = (int)(uint32_t)sel[kept[r]];
    if (tid == 0) a.kept_count[(size_t)b * K + cls] = nk;
}

// grid (B, G): every CTA computes the class prefix; rows and the zeroed tail are split over the G CTAs of an image
__global__ void __launch_bounds__(kRdPackThreads) refinedet_pack_kernel(const __grid_constant__ RdArgs a) {
    __shared__ int s_pref[TRTX_REFINEDET_MAX_CLASSES];
    const int b = blockIdx.x, K = a.C - 1;
    const int tid = threadIdx.x, lane = tid & 31;
    const int* cnt = a.kept_count + (size_t)b * K;
    if (tid == 0) {
        int acc = 0;
        for (int k = 0; k < K; ++k) {
            s_pref[k] = acc;
            acc += cnt[k];
        }
        s_pref[K] = acc;
    }
    __syncthreads();
    const int total = min(s_pref[K], a.max_out);
    float* o = a.out + (size_t)b * (1 + (size_t)a.max_out * 7);
    if (blockIdx.y == 0 && tid == 0) o[0] = (float)total;
    const int gwarp = blockIdx.y * (kRdPackThreads / 32) + (tid >> 5);
    const int nwarps = gridDim.y * (kRdPackThreads / 32);
    for (int k = gwarp; k < K; k += nwarps) {  // classes ascending, rows in keep order (:756-790)
        const int start = s_pref[k], nk = min(s_pref[k + 1], a.max_out) - start;
        const int* kp = a.kept_prior + ((size_t)b * K + k) * a.top_k;
        for (int q = lane; q < nk; q += 32) {
            const int p = kp[q];
            const double4 bx = a.boxes[(size_t)b * a.P + p];
            float* r = o + 1 + (size_t)(start + q) * 7;
            r[0] = __double2float_rn(bx.x);  // the host reads the double rows as float, :799-803
            r[1] = __double2float_rn(bx.y);
            r[2] = __double2float_rn(bx.z);
            r[3] = __double2float_rn(bx.w);
            r[4] = __ldg(a.odm_conf + ((size_t)b * a.P + p) * a.C + k + 1);
            r[5] = (float)(k + 1);
            r[6] = 1.0f;
        }
    }
    const size_t end = 1 + (size_t)a.max_out * 7;
    for (size_t e = 1 + (size_t)total * 7 + (size_t)blockIdx.y * kRdPackThreads + tid; e < end;
         e += (size_t)gridDim.y * kRdPackThreads)
        o[e] = 0.0f;
}

struct RdLayout {
    int T, pitch, region;
    size_t off_masks, off_count, off_kept, total, nms_smem, decode_smem;
};
static bool rd_valid(const trtx_refinedet_params* p, int batch) {
    return p && batch > 0 && p->num_priors > 0 && p->num_classes >= 2 && p->top_k >= 1 &&
           p->top_k <= TRTX_REFINEDET_MAX_TOPK && p->max_out >= 1;
}
static RdLayout rd_layout(const trtx_refinedet_params* p, int batch) {
    RdLayout L{};
    const size_t B = (size_t)batch, K = (size_t)p->num_classes - 1;
    L.T = (p->num_priors + 31) / 32;
    L.pitch = p->num_classes | 1;  // odd: the column reads of a warp hit 32 different banks
    L.region = p->num_priors > 5 * kSelThreads ? p->num_priors : 5 * kSelThreads;
    L.off_masks = align_up(sizeof(double4) * B * p->num_priors);
    L.off_count = L.off_masks + align_up(sizeof(uint32_t) * B * K * L.T);
    L.off_kept = L.off_count + align_up(sizeof(int) * B * K);
    L.total = L.off_kept + align_up(sizeof(int) * B * K * p->top_k);
    L.nms_smem = sizeof(unsigned long long) * ((size_t)kSelThreads + L.region) + sizeof(int) * ((size_t)L.T + kSelThreads);
    L.decode_smem = sizeof(float) * kRdDecodeWarps * 32 * L.pitch;
    return L;
}

}  // namespace trtx

using namespace trtx;

extern "C" {

TRTX_API int trtx_refinedet_priors(int image_size, int num_levels, const int* feature_maps, const int* steps,
                                   const int* min_sizes, const float* aspect_ratios, float* out_host) {
    if (image_size <= 0 || num_levels <= 0 || num_levels > TRTX_MAX_LEVELS || !feature_maps || !steps || !min_sizes ||
        !aspect_ratios)
        return 0;
    long long n = 0;
    for (int k = 0; k < num_levels; ++k) {
        if (feature_maps[k] <= 0 || steps[k] <= 0) return 0;
        n += 3LL * feature_maps[k] * feature_maps[k];
    }
    if (n > 0x7fffffff) return 0;
    if (!out_host) return (int)n;
    float* o = out_host;
    for (int k = 0; k < num_levels; ++k) {  // PriorBox, :561-589, in its float / double rounding
        const int f = feature_maps[k];
        const float ar = aspect_ratios[k];
        const double sq = sqrt((double)ar);  // `sqrt(ar)` binds to the double overload there
        for (int i = 0; i < f; ++i) {
            for (int j = 0; j < f; ++j) {
                const float f_k = (float)(image_size * 1.0 / steps[k]);
                const float cx = (float)((j + 0.5) / f_k);
                const float cy = (float)((i + 0.5) / f_k);
                const float s_k = (float)(min_sizes[k] * 1.0 / image_size);
                const float v[12] = {cx, cy, s_k, s_k, cx, cy, (float)(s_k * 1.0 * sq), (float)(s_k * 1.0 / sq),
                                     cx, cy, (float)(s_k * 1.0 / sq), (float)(s_k * 1.0 * sq)};
                for (int e = 0; e < 12; ++e)  // m_prior.clamp(0, 1), :594 (NaN passes through)
                    *o++ = v[e] != v[e] ? v[e] : fminf(fmaxf(v[e], 0.0f), 1.0f);
            }
        }
    }
    return (int)n;
}

TRTX_API size_t trtx_refinedet_workspace_size(const trtx_refinedet_params* p, int batch) {
    if (!rd_valid(p, batch)) return 0;
    return rd_layout(p, batch).total;
}

TRTX_API int trtx_refinedet_detect_enqueue(const trtx_refinedet_params* p, int batch, const float* priors_dev,
                                           const float* arm_loc_dev, const float* arm_conf_dev, const float* odm_loc_dev,
                                           const float* odm_conf_dev, float* output_dev, void* workspace_dev,
                                           size_t workspace_bytes, trtx_stream_t stream) {
    if (!rd_valid(p, batch) || !priors_dev || !arm_loc_dev || !arm_conf_dev || !odm_loc_dev || !odm_conf_dev ||
        !output_dev || !workspace_dev)
        return TRTX_ERR_INVALID;
    if (p->num_classes > TRTX_REFINEDET_MAX_CLASSES) return TRTX_ERR_UNSUPPORTED;
    for (const float* q : {priors_dev, arm_loc_dev, odm_loc_dev})  // float4 rows
        if (reinterpret_cast<uintptr_t>(q) % 16 != 0) return TRTX_ERR_INVALID;
    if (reinterpret_cast<uintptr_t>(arm_conf_dev) % 8 != 0) return TRTX_ERR_INVALID;
    const RdLayout L = rd_layout(p, batch);
    if (L.nms_smem > 200 * 1024) return TRTX_ERR_UNSUPPORTED;
    if (workspace_bytes < L.total) return TRTX_ERR_WORKSPACE;
    RdArgs a{};
    a.priors = priors_dev;
    a.arm_loc = arm_loc_dev;
    a.arm_conf = arm_conf_dev;
    a.odm_loc = odm_loc_dev;
    a.odm_conf = odm_conf_dev;
    char* ws = static_cast<char*>(workspace_dev);
    a.boxes = reinterpret_cast<double4*>(ws);
    a.masks = reinterpret_cast<uint32_t*>(ws + L.off_masks);
    a.kept_count = reinterpret_cast<int*>(ws + L.off_count);
    a.kept_prior = reinterpret_cast<int*>(ws + L.off_kept);
    a.out = output_dev;
    a.P = p->num_priors;
    a.C = p->num_classes;
    a.T = L.T;
    a.top_k = p->top_k;
    a.max_out = p->max_out;
    a.pitch = L.pitch;
    a.region = L.region;
    a.obj_thresh = p->obj_thresh;
    a.conf_thresh = p->conf_thresh;
    a.nms_thresh = (double)p->nms_thresh;
    a.v0 = (double)p->variance[0];
    a.v1 = (double)p->variance[1];
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    const int warps = batch * L.T;
    refinedet_decode_kernel<<<(warps + kRdDecodeWarps - 1) / kRdDecodeWarps, kRdDecodeWarps * 32, L.decode_smem, st>>>(
            a, batch);
    int rc = check_launch();
    if (rc) return rc;
    cudaFuncSetAttribute(refinedet_nms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.nms_smem);
    rc = check_launch();
    if (rc) return rc;
    refinedet_nms_kernel<<<dim3(p->num_classes - 1, batch), kSelThreads, L.nms_smem, st>>>(a);
    rc = check_launch();
    if (rc) return rc;
    const size_t out_floats = 1 + (size_t)p->max_out * 7;
    const int g = (int)std::min<size_t>(16, std::max<size_t>(1, out_floats / (kRdPackThreads * 16)));
    refinedet_pack_kernel<<<dim3(batch, g), kRdPackThreads, 0, st>>>(a);
    return check_launch();
}

}  // extern "C"

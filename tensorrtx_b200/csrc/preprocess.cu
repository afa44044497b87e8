// preprocess.cu -- batched letterbox warp-affine + BGR->RGB + /255 + HWC->CHW (+fp16) for sm_100a.
// Replaces warpaffine_kernel / cuda_preprocess / cuda_batch_preprocess, yolov8/src/preprocess.cu:7-127
// (identical bodies in yolov5/7/9/10/11/12/13/26), which launch once per image and synchronise the
// stream after every image (:119-127).  Here: ONE launch for the whole batch, per-image descriptors
// and affine matrices in the kernel parameter block (no H2D copy of metadata); a warp covers 32
// adjacent destination columns and every thread produces a strip of rows of its column.  Measured and
// rejected (profiles/): 4 adjacent pixels per lane (L1 sector-bound), staging the source band in shared
// memory (2x slower).
//
// Roofline: HBM-bound; algorithmic bytes per image = src_w*src_h*3 (u8 read once) +
// 3*dst_w*dst_h*sizeof(out) (SURVEY 8d: 6 144 000 B for 640x640 -> 640x640 fp32).
//
// Arithmetic follows the reference kernel statement by statement (including its `+0.5f` source
// offset without a matching `-0.5f`, preprocess.cu:22-23) and, like the reference's own nvcc build,
// leaves the bilinear sums to the default FMA contraction (<= 1 ulp from the uncontracted oracle).
#include <limits.h>
#include <math.h>
#include <string.h>

#include "tma.cuh"

namespace trtx {

constexpr int kMaxImagesPerLaunch = 128;

struct PreImage {
    const uint8_t* src;
    int sw, sh, pitch;
    int dst_idx;  // image slot in dst
    float m[6];   // d2s
};
struct PreArgs {
    PreImage img[kMaxImagesPerLaunch];
    int dw, dh;
    TRTX_TL_FIELD  // probe build: this launch's timeline record
};

// x / 255.0f, correctly rounded, in 3 FP instructions instead of the IEEE division subroutine:
// q0 = x*r, e = fma(-255, q0, x), q = fma(e, r, q0) with r = RN(1/255).  Verified EXHAUSTIVELY against
// x/255.0f for every float in [0, 65536) (1.2e9 values, tools/verify_div255.c) -- bit-identical.
__device__ __forceinline__ float div255(float x) {
    const float r = 1.0f / 255.0f;
    const float q0 = __fmul_rn(x, r);
    return __fmaf_rn(__fmaf_rn(-255.0f, q0, x), r, q0);
}

// One thread = ONE destination column x kRowsPerThread destination rows; the 32 lanes of a warp are 32 adjacent
// columns, so a warp-level byte load spans 32 px * 3 B = 96 B = 3-4 sectors and the planar stores are 128 contiguous
// bytes per warp.  ncu (profiles/r01k_letterbox_ncu.txt) shows the kernel bound by INSTRUCTION ISSUE (81 % issue
// active, 136 SASS instructions per pixel before the fast path below), not by HBM, and a rolled, row-serial variant
// with fewer instructions was slower still (too few loads in flight): so everything is straight-line code that
// issues all of a strip's loads before the first use.
//   * the letterbox matrix has no rotation (m[1] = m[3] = -0.0f, preprocess.cu:99-104), so everything that depends on
//     the column only (src_x, x taps, horizontal weights, byte offsets, validity) is computed once per thread;
//   * the bilinear sum is written as the reference writes it and left to nvcc's default FMA contraction, exactly
//     like the reference's own build: the output is BIT-IDENTICAL to the reference kernel's
//     (tests/test_vs_reference_gpu.py::test_preprocess_vs_reference_kernel).

// u8 -> f32 without the conversion (XU) pipe: for 0 <= i < 2^23, 2^23 + i is exactly representable with i in the
// mantissa, so OR-ing i into the bits of 2^23 and subtracting 2^23 gives float(i) exactly (two full-rate instructions).
// The fast path converts every other sample this way so that neither the XU pipe nor the issue slots saturate.
__device__ __forceinline__ float u8_to_float_alu(uint32_t i) { return __uint_as_float(0x4B000000u | i) - 8388608.0f; }

constexpr int kRowsPerThread = 4;  // 8-row strips measured slower (profiles/r01k_lb_probe.log)

// __launch_bounds__(256, 8): 32 registers -> 64 resident warps per SM.  The kernel is latency-bound once the instruction
// count is down (no pipe above 60 %), and occupancy is what hides it: 59.4 us at 60 registers, 53.7 at 40, 51.9 at 32.
template <typename OutT>
__global__ void __launch_bounds__(256, 8) letterbox_kernel(const __grid_constant__ PreArgs a, OutT* __restrict__ dst) {
    TRTX_TL(a, kTlLetterbox);
    constexpr int R = kRowsPerThread;
    const int b = blockIdx.z;
    const PreImage& im = a.img[b];
    const int dx = blockIdx.x * blockDim.x + threadIdx.x;
    const int dy0 = (blockIdx.y * blockDim.y + threadIdx.y) * R;
    if (dx >= a.dw || dy0 >= a.dh) return;
    const size_t area = (size_t)a.dw * a.dh;
    OutT* base = dst + (size_t)im.dst_idx * 3 * area + (size_t)dy0 * a.dw + dx;
    const float cv = 128.0f;  // const_value_st (:115)
    const uint8_t* __restrict__ img = im.src;
    const int sw = im.sw, sh = im.sh;

    // preprocess.cu:22 (src_x), evaluated with the thread's first dy: m[1]*dy is +-0 for every dy
    const float src_x = im.m[0] * (float)dx + im.m[1] * (float)dy0 + im.m[2] + 0.5f;
    const bool x_out = src_x <= -1 || src_x >= sw;
    const int x_low = (int)floorf(src_x);
    const int x_high = x_low + 1;
    const float lx = src_x - (float)x_low, hx = 1 - lx;
    const bool xl = x_low >= 0, xh = x_high < sw;
    const float xm = im.m[3] * (float)dx;

    // bgr -> rgb, /255 (:64-74); planar stores, 128 B per warp and plane
    auto emit = [&](int r, float c0, float c1, float c2) {
        OutT* o = base + (size_t)r * a.dw;
        if constexpr (sizeof(OutT) == 4) {
            o[0] = div255(c2);
            o[area] = div255(c1);
            o[2 * area] = div255(c0);
        } else {
            o[0] = __float2half_rn(div255(c2));
            o[area] = __float2half_rn(div255(c1));
            o[2 * area] = __float2half_rn(div255(c0));
        }
    };

    float src_y[R];
    int y_low[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        src_y[r] = xm + im.m[4] * (float)(dy0 + r) + im.m[5] + 0.5f;  // :23
        y_low[r] = (int)floorf(src_y[r]);
    }
    // Fast path (warp-uniform but for the image's left/right edge): a full strip whose rows step through CONSECUTIVE
    // source rows, all taps inside the image -- any letterbox that does not shrink the image, e.g. the 640x640 ->
    // 640x640 benchmark.  The R+1 source rows are loaded once (one address per row: the right tap is the next pixel)
    // and shared by neighbouring destination rows: (R+1)*6 loads and conversions instead of R*12, no clamps, no selects.
    bool fast = dy0 + R <= a.dh && xl && xh && y_low[0] >= 0 && y_low[0] + R < sh;
#pragma unroll
    for (int r = 1; r < R; ++r) fast = fast && y_low[r] == y_low[0] + r;
    if (fast) {
        const uint8_t* p = img + (size_t)y_low[0] * (size_t)im.pitch + (uint32_t)x_low * 3u;
        float t[R + 1][6];
#pragma unroll
        for (int s = 0; s <= R; ++s) {
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                const uint32_t v = __ldg(p + k);
                t[s][k] = ((s * 6 + k) & 1) ? u8_to_float_alu(v) : (float)v;
            }
            p += im.pitch;
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float ly = src_y[r] - (float)y_low[r], hy = 1 - ly;
            const float w1 = hy * hx, w2 = hy * lx, w3 = ly * hx, w4 = ly * lx;
            // :59-61 (left-to-right; nvcc contracts to mul + 3 fma, as in the reference build)
            emit(r, w1 * t[r][0] + w2 * t[r][3] + w3 * t[r + 1][0] + w4 * t[r + 1][3],
                 w1 * t[r][1] + w2 * t[r][4] + w3 * t[r + 1][1] + w4 * t[r + 1][4],
                 w1 * t[r][2] + w2 * t[r][5] + w3 * t[r + 1][2] + w4 * t[r + 1][5]);
        }
        return;
    }

    // General path (borders, shrinking letterboxes): source coordinates are CLAMPED into the image and the 12 bytes
    // always loaded (one address per tap, channels through immediate offsets, no divergent border path); out-of-image
    // taps are then replaced by the border value with selects, which is what the reference's pointer redirection to
    // `const_value` does (preprocess.cu:38-57).
    const uint32_t o1 = (uint32_t)min(max(x_low, 0), sw - 1) * 3u, o2 = (uint32_t)min(max(x_high, 0), sw - 1) * 3u;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        if (dy0 + r >= a.dh) break;
        float c0 = cv, c1 = cv, c2 = cv;
        if (!(x_out || src_y[r] <= -1 || src_y[r] >= sh)) {
            const int y_high = y_low[r] + 1;
            const float ly = src_y[r] - (float)y_low[r], hy = 1 - ly;
            const float w1 = hy * hx, w2 = hy * lx, w3 = ly * hx, w4 = ly * lx;
            const bool r0ok = y_low[r] >= 0, r1ok = y_high < sh;
            const uint32_t row0 = (uint32_t)max(y_low[r], 0) * (uint32_t)im.pitch;  // images < 4 GiB
            const uint32_t row1 = (uint32_t)min(y_high, sh - 1) * (uint32_t)im.pitch;
            const bool k1 = r0ok && xl, k2 = r0ok && xh, k3 = r1ok && xl, k4 = r1ok && xh;
            const uint8_t* p1 = img + (row0 + o1);
            const uint8_t* p2 = img + (row0 + o2);
            const uint8_t* p3 = img + (row1 + o1);
            const uint8_t* p4 = img + (row1 + o2);
            float v1[3], v2[3], v3[3], v4[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float t1 = (float)(uint32_t)__ldg(p1 + k);
                const float t2 = (float)(uint32_t)__ldg(p2 + k);
                const float t3 = (float)(uint32_t)__ldg(p3 + k);
                const float t4 = (float)(uint32_t)__ldg(p4 + k);
                v1[k] = k1 ? t1 : cv;
                v2[k] = k2 ? t2 : cv;
                v3[k] = k3 ? t3 : cv;
                v4[k] = k4 ? t4 : cv;
            }
            c0 = w1 * v1[0] + w2 * v2[0] + w3 * v3[0] + w4 * v4[0];
            c1 = w1 * v1[1] + w2 * v2[1] + w3 * v3[1] + w4 * v4[1];
            c2 = w1 * v1[2] + w2 * v2[2] + w3 * v3[2] + w4 * v4[2];
        }
        emit(r, c0, c1, c2);
    }
}


// =====================================================================================================================
// Unit-scale letterbox, TMA-staged (the 640x640 -> 640x640 benchmark and every source that fits the network input in
// one dimension: scale == 1, the image is only translated / padded).
//
// With scale == 1 the d2s matrix is {1, -0, tx, -0, 1, ty} with 2*tx, 2*ty integers (preprocess.cu:98-110), so for every
// destination pixel  x_low = dx + ox,  y_low = dy + oy  and the bilinear fractions lx, ly are image-wide constants in
// {0, 0.5}: the four weights are products of {0, 0.5, 1}, every product w*u8 and every partial sum of the reference's
// expression (preprocess.cu:59-61) is exact in fp32, hence the result does not depend on evaluation order or FMA
// contraction, and "tap outside the image -> 128" (preprocess.cu:38-57) also reproduces the fully-outside case
// (:25-30: the weights sum to exactly 1).  The kernel is therefore bit-identical to the reference by construction;
// tests assert array_equal against the reference's compiled kernel.
//
// A CTA owns a TW x TH destination tile.  Its (TH+1) x (TW+1)-pixel source window is fetched by ONE TMA tensor copy
// (u8 tensor map over the image, box [kBoxBytes, TH+1]; rows/columns outside the image arrive as zeros and are patched
// to 128 by the few border tiles) -- no per-lane byte loads, no address arithmetic per tap.  Each thread then produces
// 4 ADJACENT pixels x 4 rows: per source row 4 conflict-free LDS.32 (15 bytes = 5 BGR pixels), every byte converted
// once with one PRMT (byte -> mantissa of 2^23) + one FADD and shared by the 2x2 destination pixels that use it, and
// one 16-byte store per plane and row (8 bytes for fp16 output).  Half-warps take row groups 4 rows apart, which puts
// their LDS on disjoint banks (4 * 52 words = 16 mod 32).
// Instructions per destination pixel: ~33 (the per-lane-byte-load kernel above: 79).
constexpr int kUnitTW = 64;                   // destination columns per CTA = 16 lanes x 4 pixels
constexpr int kUnitBoxBytes = 208;            // >= (kUnitTW + 1) * 3 = 195, multiple of 16 (TMA inner box extent)
constexpr int kMaxUnitImages = 64;

struct UnitImage {
    int ox, oy;    // x_low(dx = 0), y_low(dy = 0)
    int sw, sh;
    int map, z;    // tensor map index, image coordinate inside that map
    int dst_idx;
    float lx, ly;  // bilinear fractions (0 or 0.5), constant over the image
};
struct alignas(64) UnitArgs {
    CUtensorMap map[kMaxUnitImages];
    UnitImage img[kMaxUnitImages];
    int dw, dh;
    TRTX_TL_FIELD  // probe build: this launch's timeline record
};

template <typename OutT, int WARPS>
__global__ void __launch_bounds__(WARPS * 32) letterbox_unit_kernel(const __grid_constant__ UnitArgs a, OutT* __restrict__ dst) {
    TRTX_TL(a, kTlLetterbox);
    constexpr int TW = kUnitTW, TH = WARPS * 8, BOXW = kUnitBoxBytes, ROWS = TH + 1;
    __shared__ __align__(128) uint8_t box[ROWS * BOXW];
    __shared__ uint64_t bar;
    const int tid = threadIdx.x;
    const UnitImage& im = a.img[blockIdx.z];
    const int dx0 = blockIdx.x * TW, dy0 = blockIdx.y * TH;
    const int sx0 = dx0 + im.ox, sy0 = dy0 + im.oy;  // source pixel under the tile's first tap
    const int sw = im.sw, sh = im.sh;
    const bool all_out = sx0 + TW < 0 || sx0 >= sw || sy0 + TH < 0 || sy0 >= sh;
    const bool interior = sx0 >= 0 && sx0 + TW < sw && sy0 >= 0 && sy0 + TH < sh;

    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (!all_out) {
        if (tid == 0) {
            mbar_arrive_expect_tx(&bar, ROWS * BOXW);
            tma_load_3d(box, &a.map[im.map], sx0 * 3, sy0, im.z, &bar);
        }
        mbar_wait(&bar, 0);
        if (!interior) {
            // border tile: pixels of the window outside the image -> const_value_st = 128 (preprocess.cu:115)
            for (int i = tid; i < ROWS * (TW + 1); i += WARPS * 32) {
                const int r = i / (TW + 1), c = i - r * (TW + 1);
                const int y = sy0 + r, x = sx0 + c;
                if (y < 0 || y >= sh || x < 0 || x >= sw) {
                    uint8_t* q = box + r * BOXW + c * 3;
                    q[0] = 128;
                    q[1] = 128;
                    q[2] = 128;
                }
            }
            __syncthreads();
        }
    } else {  // pure padding tile: every tap is the border value
        for (int i = tid; i < ROWS * BOXW / 4; i += WARPS * 32) reinterpret_cast<uint32_t*>(box)[i] = 0x80808080u;
        __syncthreads();
    }

    const int lane = tid & 31, warp = tid >> 5;
    const int k = lane & 15;
    const int r0 = warp * 8 + (lane >> 4) * 4;  // half-warps 4 rows apart: disjoint banks
    const int dx = dx0 + 4 * k;
    if (dx >= a.dw) return;
    const float lx = im.lx, ly = im.ly, hx = 1 - lx, hy = 1 - ly;
    const float w1 = hy * hx, w2 = hy * lx, w3 = ly * hx, w4 = ly * lx;  // preprocess.cu:34-35
    const size_t area = (size_t)a.dw * a.dh;
    OutT* o = dst + (size_t)im.dst_idx * 3 * area + (size_t)(dy0 + r0) * a.dw + dx;
    const uint8_t* p = box + r0 * BOXW + 12 * k;

    auto load_row = [&](const uint8_t* q, float (&t)[15]) {
        uint32_t w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) w[j] = reinterpret_cast<const uint32_t*>(q)[j];
#pragma unroll
        for (int i = 0; i < 15; ++i)  // byte i -> float: 2^23 + v is exact with v in the mantissa
            t[i] = __uint_as_float(__byte_perm(w[i >> 2], 0x4B000000u, 0x7650u + (i & 3))) - 8388608.0f;
    };
    float top[15], bot[15];
    load_row(p, top);
    const int rows = a.dh - (dy0 + r0);  // rows of this strip inside the destination
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        load_row(p + (r + 1) * BOXW, bot);
        if (r < rows) {
            float v[3][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int c = 0; c < 3; ++c)  // :59-61, bgr -> rgb and /255 :64-74
                    v[c][j] = div255(w1 * top[3 * j + c] + w2 * top[3 * j + 3 + c] + w3 * bot[3 * j + c] + w4 * bot[3 * j + 3 + c]);
            OutT* orow = o + (size_t)r * a.dw;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                OutT* q = orow + (size_t)(2 - c) * area;
                if constexpr (sizeof(OutT) == 4) {
                    *reinterpret_cast<float4*>(q) = make_float4(v[c][0], v[c][1], v[c][2], v[c][3]);
                } else {
                    const __half2 h0 = __floats2half2_rn(v[c][0], v[c][1]), h1 = __floats2half2_rn(v[c][2], v[c][3]);
                    uint2 u;
                    u.x = *reinterpret_cast<const uint32_t*>(&h0);
                    u.y = *reinterpret_cast<const uint32_t*>(&h1);
                    *reinterpret_cast<uint2*>(q) = u;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 15; ++i) top[i] = bot[i];
    }
}

// Host: does this image take the unit-scale path?  (scale == 1 exactly, half-integer translation, TMA-compatible.)
static bool unit_scale_image(const trtx_image_desc& d, const float m[6], UnitImage* u) {
    if (!(m[0] == 1.0f && m[4] == 1.0f && m[1] == 0.0f && m[3] == 0.0f)) return false;
    const float tx = m[2] + 0.5f, ty = m[5] + 0.5f;
    if (!(fabsf(tx) < 1048576.0f && fabsf(ty) < 1048576.0f)) return false;
    if (2.0f * tx != rintf(2.0f * tx) || 2.0f * ty != rintf(2.0f * ty)) return false;
    if (reinterpret_cast<uintptr_t>(d.data_dev) % 16 != 0 || d.pitch % 16 != 0) return false;  // TMA base / stride
    u->ox = (int)floorf(tx);
    u->oy = (int)floorf(ty);
    // TMA fetches the box from byte column 3 * (64 * tile + ox): the start of a box must be 16-byte aligned in global memory
    // (an unaligned start is an illegal instruction on sm_100a), so horizontal offsets that are not a multiple of 16 pixels
    // (e.g. a 624-wide source centred in 640) take the general kernel
    if (u->ox % 16 != 0) return false;
    u->lx = tx - floorf(tx);
    u->ly = ty - floorf(ty);
    u->sw = d.width;
    u->sh = d.height;
    return true;
}

static bool encode_image_map(CUtensorMap* map, const uint8_t* base, int sw, int sh, int pitch, int n, size_t image_stride,
                             int box_rows) {
    EncodeTiledFn enc = tma_encoder();
    if (!enc) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)sw * 3u, (cuuint64_t)sh, (cuuint64_t)n};
    const cuuint64_t gstr[2] = {(cuuint64_t)pitch, (cuuint64_t)image_stride};
    const cuuint32_t bdim[3] = {(cuuint32_t)kUnitBoxBytes, (cuuint32_t)box_rows, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(base), gdim, gstr, bdim, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

constexpr int kUnitWarps = 4;

// Launch the unit-scale kernel for `n` images (descriptors d[i], unit info u[i] already filled but for map/z).
// Returns TRTX_ERR_UNSUPPORTED when no tensor map can be made (caller falls back to the general kernel).
static int launch_unit(const trtx_image_desc* const* d, UnitImage* u, int n, void* dst, int dw, int dh, int out_dtype,
                       cudaStream_t st) {
    UnitArgs a;
    a.dw = dw;
    a.dh = dh;
    constexpr int box_rows = kUnitWarps * 8 + 1;
    // one 3-D map for the whole group when the images are equally sized and equally spaced (a frame ring / one batch
    // tensor): one encode instead of n
    bool uniform = n > 1;
    const ptrdiff_t step = n > 1 ? d[1]->data_dev - d[0]->data_dev : 0;
    for (int i = 1; i < n && uniform; ++i)
        uniform = d[i]->width == d[0]->width && d[i]->height == d[0]->height && d[i]->pitch == d[0]->pitch &&
                  d[i]->data_dev - d[i - 1]->data_dev == step;
    uniform = uniform && step > 0 && step % 16 == 0 && (size_t)step >= (size_t)d[0]->pitch * (size_t)d[0]->height;
    if (uniform) {
        if (!encode_image_map(&a.map[0], d[0]->data_dev, d[0]->width, d[0]->height, d[0]->pitch, n, (size_t)step, box_rows))
            return TRTX_ERR_UNSUPPORTED;
    }
    for (int i = 0; i < n; ++i) {
        if (uniform) {
            u[i].map = 0;
            u[i].z = i;
        } else {
            if (!encode_image_map(&a.map[i], d[i]->data_dev, d[i]->width, d[i]->height, d[i]->pitch, 1,
                                  (size_t)d[i]->pitch * (size_t)d[i]->height, box_rows))
                return TRTX_ERR_UNSUPPORTED;
            u[i].map = i;
            u[i].z = 0;
        }
        a.img[i] = u[i];
    }
    dim3 grid((dw + kUnitTW - 1) / kUnitTW, (dh + kUnitWarps * 8 - 1) / (kUnitWarps * 8), n);
    TRTX_TL_TAKE(a);
    if (out_dtype == TRTX_F32)
        letterbox_unit_kernel<float, kUnitWarps><<<grid, kUnitWarps * 32, 0, st>>>(a, static_cast<float*>(dst));
    else
        letterbox_unit_kernel<__half, kUnitWarps><<<grid, kUnitWarps * 32, 0, st>>>(a, static_cast<__half*>(dst));
    return check_launch();
}

}  // namespace trtx

using namespace trtx;

extern "C" {

// preprocess.cu:98-110 + cv::invertAffineTransform (CV_32F branch)
TRTX_API void trtx_letterbox_matrix(int sw, int sh, int dw, int dh, float d2s[6]) {
    float a = dh / (float)sh, b = dw / (float)sw;
    float scale = a < b ? a : b;  // std::min
    float s2d[6];
    s2d[0] = scale;
    s2d[1] = 0;
    s2d[2] = (float)(-scale * sw * 0.5 + dw * 0.5);
    s2d[3] = 0;
    s2d[4] = scale;
    s2d[5] = (float)(-scale * sh * 0.5 + dh * 0.5);
    /* cv::invertAffineTransform, CV_32F branch, as OpenCV >= 4.x evaluates it with softfloat/softdouble
     * (pinned against cv2 4.13 on 3000 sizes, tests/test_oracle_cpu.py): the determinant and the
     * A = M*D products are FLOAT operations (softfloat::operator* converts D to float), 1/D and the
     * translation terms are double. */
    float p0 = s2d[0] * s2d[4], p1 = s2d[1] * s2d[3];
    float det = p0 - p1;
    double D = (double)det;
    D = D != 0 ? 1. / D : 0;
    float Df = (float)D;
    float fA11 = s2d[4] * Df, fA22 = s2d[0] * Df, fA12 = (-s2d[1]) * Df, fA21 = (-s2d[3]) * Df;
    double A11 = fA11, A22 = fA22, A12 = fA12, A21 = fA21;
    double b1 = -A11 * s2d[2] - A12 * s2d[5];
    double b2 = -A21 * s2d[2] - A22 * s2d[5];
    d2s[0] = (float)A11;
    d2s[1] = (float)A12;
    d2s[2] = (float)b1;
    d2s[3] = (float)A21;
    d2s[4] = (float)A22;
    d2s[5] = (float)b2;
}

// get_rect: the inverse of the letterbox for a detection box -- yolov8/src/postprocess.cpp:6-36 (TRTX_YOLO_V8: l,t,r,b,
// clamped to the image) and yolov5/src/postprocess.cpp:4-29 (TRTX_YOLO_V5: cx,cy,w,h).  Host arithmetic, statement
// by statement: the two ratios are double divisions stored to float, the rest is float, round() sees doubles.
TRTX_API int trtx_get_rect(int variant, int net_w, int net_h, int img_w, int img_h, const float bbox[4], int rect[4]) {
    if (!bbox || !rect || net_w <= 0 || net_h <= 0 || img_w <= 0 || img_h <= 0) return TRTX_ERR_INVALID;
    if (variant != TRTX_YOLO_V8 && variant != TRTX_YOLO_V5) return TRTX_ERR_INVALID;
    float l, r, t, b;
    const float r_w = (float)(net_w / (img_w * 1.0));
    const float r_h = (float)(net_h / (img_h * 1.0));
    const bool by_w = r_h > r_w;  // the width fills the network input: vertical padding
    const float ratio = by_w ? r_w : r_h;
    const float pad = by_w ? (net_h - r_w * img_h) / 2 : (net_w - r_h * img_w) / 2;
    if (variant == TRTX_YOLO_V8) {
        l = bbox[0];
        r = bbox[2];
        t = bbox[1];
        b = bbox[3];
    } else {
        l = bbox[0] - bbox[2] / 2.f;
        r = bbox[0] + bbox[2] / 2.f;
        t = bbox[1] - bbox[3] / 2.f;
        b = bbox[1] + bbox[3] / 2.f;
    }
    if (by_w) {
        t = t - pad;
        b = b - pad;
    } else {
        l = l - pad;
        r = r - pad;
    }
    l = l / ratio;
    r = r / ratio;
    t = t / ratio;
    b = b / ratio;
    if (variant == TRTX_YOLO_V8) {
        l = 0.0f > l ? 0.0f : l;
        t = 0.0f > t ? 0.0f : t;
        const int rw = (int)round((double)(r - l)), rl = (int)round((double)l);
        const int rh = (int)round((double)(b - t)), rt = (int)round((double)t);
        const int width = rw < img_w - rl ? rw : img_w - rl, height = rh < img_h - rt ? rh : img_h - rt;
        rect[0] = rl;
        rect[1] = rt;
        rect[2] = width > 0 ? width : 0;
        rect[3] = height > 0 ? height : 0;
    } else {
        rect[0] = (int)round((double)l);
        rect[1] = (int)round((double)t);
        rect[2] = (int)round((double)(r - l));
        rect[3] = (int)round((double)(b - t));
    }
    return TRTX_OK;
}

// get_rect_adapt_landmark, yolov8/src/postprocess.cpp:38-69, statement by statement (ratios: double division stored to float;
// `(kInputH - r_w * img.rows) / 2`: int - float*int in float, then / 2).
TRTX_API int trtx_get_rect_adapt_landmark(int net_w, int net_h, int img_w, int img_h, const float bbox[4], float* lmk,
                                          int num_kpts, int rect[4]) {
    if (!bbox || !rect || (num_kpts > 0 && !lmk) || num_kpts < 0 || net_w <= 0 || net_h <= 0 || img_w <= 0 || img_h <= 0)
        return TRTX_ERR_INVALID;
    float l, r, t, b;
    const float r_w = (float)(net_w / (img_w * 1.0));
    const float r_h = (float)(net_h / (img_h * 1.0));
    if (r_h > r_w) {
        l = bbox[0] / r_w;
        r = bbox[2] / r_w;
        t = (bbox[1] - (net_h - r_w * img_h) / 2) / r_w;
        b = (bbox[3] - (net_h - r_w * img_h) / 2) / r_w;
        for (int i = 0; i < num_kpts * 3; i += 3) {
            lmk[i] /= r_w;
            lmk[i + 1] = (lmk[i + 1] - (net_h - r_w * img_h) / 2) / r_w;
        }
    } else {
        l = (bbox[0] - (net_w - r_h * img_w) / 2) / r_h;
        r = (bbox[2] - (net_w - r_h * img_w) / 2) / r_h;
        t = bbox[1] / r_h;
        b = bbox[3] / r_h;
        for (int i = 0; i < num_kpts * 3; i += 3) {
            lmk[i] = (lmk[i] - (net_w - r_h * img_w) / 2) / r_h;
            lmk[i + 1] /= r_h;
        }
    }
    l = 0.0f > l ? 0.0f : l;
    t = 0.0f > t ? 0.0f : t;
    const int rw = (int)round((double)(r - l)), rl = (int)round((double)l);
    const int rh = (int)round((double)(b - t)), rt = (int)round((double)t);
    const int width = rw < img_w - rl ? rw : img_w - rl, height = rh < img_h - rt ? rh : img_h - rt;
    rect[0] = rl;
    rect[1] = rt;
    rect[2] = width > 0 ? width : 0;
    rect[3] = height > 0 ? height : 0;
    return TRTX_OK;
}

// get_rect_adapt_landmark of RetinaFace, retinaface/common.hpp:65-89, statement by statement: box AND the 5 landmarks (x, y pairs) of
// a face mapped from the letterboxed network input back to the original image; the box corners are TRUNCATED to int (`int l =
// bbox[0] / r_w`), not rounded, and not clamped to the image.
TRTX_API int trtx_retina_get_rect_adapt_landmark(int input_w, int input_h, int img_w, int img_h, const float bbox[4], float lmk[10],
                                                 int rect[4]) {
    if (!bbox || !lmk || !rect || input_w <= 0 || input_h <= 0 || img_w <= 0 || img_h <= 0) return TRTX_ERR_INVALID;
    int l, r, t, b;
    float r_w = input_w / (img_w * 1.0);
    float r_h = input_h / (img_h * 1.0);
    if (r_h > r_w) {
        l = bbox[0] / r_w;
        r = bbox[2] / r_w;
        t = (bbox[1] - (input_h - r_w * img_h) / 2) / r_w;
        b = (bbox[3] - (input_h - r_w * img_h) / 2) / r_w;
        for (int i = 0; i < 10; i += 2) {
            lmk[i] /= r_w;
            lmk[i + 1] = (lmk[i + 1] - (input_h - r_w * img_h) / 2) / r_w;
        }
    } else {
        l = (bbox[0] - (input_w - r_h * img_w) / 2) / r_h;
        r = (bbox[2] - (input_w - r_h * img_w) / 2) / r_h;
        t = bbox[1] / r_h;
        b = bbox[3] / r_h;
        for (int i = 0; i < 10; i += 2) {
            lmk[i] = (lmk[i] - (input_w - r_h * img_w) / 2) / r_h;
            lmk[i + 1] /= r_h;
        }
    }
    rect[0] = l, rect[1] = t, rect[2] = r - l, rect[3] = b - t;
    return TRTX_OK;
}

// process_decode_ptr_host, yolov8/src/postprocess.cpp:131-147
TRTX_API int trtx_process_decode_ptr_host(const float* decode_ptr_host, int bbox_element, int count, float* rows_out) {
    if (!decode_ptr_host || !rows_out || bbox_element < 7 || count < 0) return -TRTX_ERR_INVALID;
    int n = 0;
    for (int i = 0; i < count; ++i) {
        const float* p = decode_ptr_host + 1 + (size_t)i * bbox_element;
        if ((int)p[6] == 1) {  // `int keep_flag = decode_ptr_host[basic_pos + 6]`
            for (int k = 0; k < 6; ++k) rows_out[(size_t)n * 6 + k] = p[k];
            ++n;
        }
    }
    return n;
}

// process_decode_ptr_host_obb (yolov8/src/postprocess.cpp:273-290): the same for oriented boxes -- 7 floats per kept row, the angle
// from column 7 of the 8-float rows cuda_decode_obb writes (postprocess.cu:31-39)
TRTX_API int trtx_process_decode_ptr_host_obb(const float* decode_ptr_host, int bbox_element, int count, float* rows_out) {
    if (!decode_ptr_host || !rows_out || bbox_element < 8 || count < 0) return -TRTX_ERR_INVALID;
    int n = 0;
    for (int i = 0; i < count; ++i) {
        const float* p = decode_ptr_host + 1 + (size_t)i * bbox_element;
        if ((int)p[6] == 1) {
            for (int k = 0; k < 6; ++k) rows_out[(size_t)n * 7 + k] = p[k];
            rows_out[(size_t)n * 7 + 6] = p[7];
            ++n;
        }
    }
    return n;
}

TRTX_API int trtx_preprocess_batch_enqueue(const trtx_image_desc* images_host, int batch, void* dst_dev, int dst_w,
                                           int dst_h, int out_dtype, trtx_stream_t stream) {
    if (!images_host || batch <= 0 || !dst_dev || dst_w <= 0 || dst_h <= 0) return TRTX_ERR_INVALID;
    if (out_dtype != TRTX_F32 && out_dtype != TRTX_F16) return TRTX_ERR_INVALID;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    for (int i = 0; i < batch; ++i) {
        const trtx_image_desc& d = images_host[i];
        if (!d.data_dev || d.width <= 0 || d.height <= 0 || d.pitch < 3 * d.width) return TRTX_ERR_INVALID;
    }
    // vector stores of the unit-scale kernel: 4 pixels per thread and plane
    const bool unit_ok = dst_w % 4 == 0 && reinterpret_cast<uintptr_t>(dst_dev) % 16 == 0;
    PreArgs g;  // general-path group
    g.dw = dst_w;
    g.dh = dst_h;
    int ng = 0;
    const trtx_image_desc* ud[kMaxUnitImages];
    UnitImage uu[kMaxUnitImages];
    int nu = 0;
    auto flush_general = [&]() -> int {
        if (!ng) return TRTX_OK;
        constexpr int R = kRowsPerThread;
        dim3 block(128, 2, 1);  // 128 columns x (2 x R) rows per block
        dim3 grid((dst_w + 127) / 128, (dst_h + 2 * R - 1) / (2 * R), ng);
        TRTX_TL_TAKE(g);
        if (out_dtype == TRTX_F32)
            letterbox_kernel<float><<<grid, block, 0, st>>>(g, static_cast<float*>(dst_dev));
        else
            letterbox_kernel<__half><<<grid, block, 0, st>>>(g, static_cast<__half*>(dst_dev));
        ng = 0;
        return check_launch();
    };
    auto add_general = [&](int i) -> int {
        const trtx_image_desc& d = images_host[i];
        PreImage& im = g.img[ng++];
        im.src = d.data_dev;
        im.sw = d.width;
        im.sh = d.height;
        im.pitch = d.pitch;
        im.dst_idx = i;
        trtx_letterbox_matrix(d.width, d.height, dst_w, dst_h, im.m);
        return ng == kMaxImagesPerLaunch ? flush_general() : TRTX_OK;
    };
    auto flush_unit = [&]() -> int {
        if (!nu) return TRTX_OK;
        int rc = launch_unit(ud, uu, nu, dst_dev, dst_w, dst_h, out_dtype, st);
        if (rc == TRTX_ERR_UNSUPPORTED) {  // no tensor map (driver without the encoder): general kernel
            rc = TRTX_OK;
            for (int j = 0; j < nu && rc == TRTX_OK; ++j) rc = add_general(uu[j].dst_idx);
        }
        nu = 0;
        return rc;
    };
    for (int i = 0; i < batch; ++i) {
        const trtx_image_desc& d = images_host[i];
        float m[6];
        trtx_letterbox_matrix(d.width, d.height, dst_w, dst_h, m);
        int rc = TRTX_OK;
        if (unit_ok && unit_scale_image(d, m, &uu[nu])) {
            ud[nu] = &d;
            uu[nu].dst_idx = i;
            if (++nu == kMaxUnitImages) rc = flush_unit();
        } else {
            rc = add_general(i);
        }
        if (rc) return rc;
    }
    int rc = flush_unit();
    if (rc) return rc;
    return flush_general();
}

}  // extern "C"

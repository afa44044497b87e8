/* refinedet_oracle.c -- plain-C fp64 restatement of RefineDet's post-process (refinedet/refinedet.cpp:553-790):
 * PriorBox is not restated here (the library's host trtx_refinedet_priors is pinned against the reference's table);
 * decode (:600-619) twice, the candidate gate (:738-760), per-class nms() (:632-695) and the output rows (:796-813).
 * TEST INFRASTRUCTURE ONLY.  Built with -ffp-contract=off so that every operation is rounded on its own, like the
 * reference's eager tensor ops.  exp is glibc's, which may differ from CUDA's fp64 exp in the last bit.
 * Equal scores rank the lower prior index first (the reference's sort is unstable there). */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#define API __attribute__((visibility("default")))

typedef struct {
    double score;
    int index;
} Cand;

static int cand_cmp(const void* a, const void* b) { /* score descending, index ascending */
    const Cand* x = (const Cand*)a;
    const Cand* y = (const Cand*)b;
    if (x->score != y->score) return x->score > y->score ? -1 : 1;
    return x->index - y->index;
}

/* at::clamp with scalar bounds: a NaN bound gives NaN, a NaN value passes through */
static double clampd(double v, double lo, double hi) {
    if (isnan(lo) || isnan(hi)) return NAN;
    if (isnan(v)) return v;
    return fmin(fmax(v, lo), hi);
}

/* does kept box i (suppressor) drop box j?  nms(), :674-692 */
static int suppress(const double* bi, double area_i, const double* bj, double area_j, float overlap) {
    const double xx1 = clampd(bj[0], (double)(float)bi[0], 2147483647.0);
    const double yy1 = clampd(bj[1], (double)(float)bi[1], 2147483647.0);
    const double xx2 = clampd(bj[2], -2147483648.0, (double)(float)bi[2]);
    const double yy2 = clampd(bj[3], -2147483648.0, (double)(float)bi[3]);
    const double w = clampd(xx2 - xx1, 0.0, 2147483647.0);
    const double h = clampd(yy2 - yy1, 0.0, 2147483647.0);
    const double inter = w * h;
    const double uni = (area_j - inter) + area_i;
    return !(inter / uni < (double)overlap);
}

/* decode(loc, prior) of :600-619 for one row; corners = b_form_pt */
static void decode(const double* prior, const float* loc, double v0, double v1, int corners, double* o) {
    const double c1x = prior[0] + ((double)loc[0] * v0) * prior[2];
    const double c1y = prior[1] + ((double)loc[1] * v0) * prior[3];
    const double c2w = prior[2] * exp((double)loc[2] * v1);
    const double c2h = prior[3] * exp((double)loc[3] * v1);
    if (corners) {
        o[0] = c1x - c2w / 2;
        o[1] = c1y - c2h / 2;
        o[2] = o[0] + c2w;
        o[3] = o[1] + c2h;
    } else {
        o[0] = c1x;
        o[1] = c1y;
        o[2] = c2w;
        o[3] = c2h;
    }
}

/* nms() of :632-695 on n boxes [n,4] (x1, y1, x2, y2) with scores [n]: the top_k highest scores (ties: lower index
 * first), greedy, keep = indices into boxes in keep order.  Returns the kept count. */
API int oracle_refinedet_nms(const double* boxes, const double* scores, int n, float overlap, int top_k, int64_t* keep) {
    if (n <= 0) return 0;
    Cand* cand = (Cand*)malloc(sizeof(Cand) * (size_t)n);
    char* alive = (char*)malloc((size_t)n);
    double* area = (double*)malloc(sizeof(double) * (size_t)n);
    for (int i = 0; i < n; ++i) {
        cand[i].score = scores[i];
        cand[i].index = i;
        area[i] = (boxes[4 * i + 2] - boxes[4 * i]) * (boxes[4 * i + 3] - boxes[4 * i + 1]);  /* :645 */
    }
    qsort(cand, (size_t)n, sizeof(Cand), cand_cmp);
    const int m = n < top_k ? n : top_k;
    int count = 0;
    for (int i = 0; i < m; ++i) alive[i] = 1;
    for (int i = 0; i < m; ++i) {
        if (!alive[i]) continue;
        const int bi = cand[i].index;
        keep[count++] = bi;
        for (int j = i + 1; j < m; ++j) {
            const int bj = cand[j].index;
            if (alive[j] && suppress(boxes + 4 * (size_t)bi, area[bi], boxes + 4 * (size_t)bj, area[bj], overlap))
                alive[j] = 0;
        }
    }
    free(cand);
    free(alive);
    free(area);
    return count;
}

/* One image.  rows: capacity (C-1)*top_k rows of 6 floats (x1, y1, x2, y2, score, label) in the reference's order;
 * prior_out (may be NULL): the prior index of each row.  Returns the number of rows, or -1 on bad arguments. */
API int oracle_refinedet_image(const float* priors, const float* arm_loc, const float* arm_conf, const float* odm_loc,
                               const float* odm_conf, int P, int C, float obj_thresh, float conf_thresh, float nms_thresh,
                               int top_k, float v0f, float v1f, float* rows, int32_t* prior_out) {
    if (P <= 0 || C < 2 || top_k < 1) return -1;
    const double v0 = v0f, v1 = v1f;
    double* box = (double*)malloc(sizeof(double) * 4 * (size_t)P);
    double* cbox = (double*)malloc(sizeof(double) * 4 * (size_t)P);
    double* cscore = (double*)malloc(sizeof(double) * (size_t)P);
    int* cprior = (int*)malloc(sizeof(int) * (size_t)P);
    int64_t* keep = (int64_t*)malloc(sizeof(int64_t) * (size_t)P);
    for (int p = 0; p < P; ++p) {  /* :747-750 */
        double pr[4] = {priors[4 * p], priors[4 * p + 1], priors[4 * p + 2], priors[4 * p + 3]}, arm[4];
        decode(pr, arm_loc + 4 * (size_t)p, v0, v1, 0, arm);
        decode(arm, odm_loc + 4 * (size_t)p, v0, v1, 1, box + 4 * (size_t)p);
    }
    int nrows = 0;
    for (int c = 1; c < C; ++c) {  /* :756-790; candidates in ascending prior order (nonzero) */
        int n = 0;
        for (int p = 0; p < P; ++p) {
            const float s = odm_conf[(size_t)p * C + c];
            if (arm_conf[2 * (size_t)p + 1] > obj_thresh && s > conf_thresh) {
                for (int e = 0; e < 4; ++e) cbox[4 * n + e] = box[4 * (size_t)p + e];
                cscore[n] = s;
                cprior[n] = p;
                ++n;
            }
        }
        const int k = oracle_refinedet_nms(cbox, cscore, n, nms_thresh, top_k, keep);
        for (int r = 0; r < k; ++r) {  /* the host reads the double rows as float, :796-813 */
            const int q = (int)keep[r];
            float* o = rows + 6 * (size_t)nrows;
            for (int e = 0; e < 4; ++e) o[e] = (float)cbox[4 * q + e];
            o[4] = (float)cscore[q];
            o[5] = (float)c;
            if (prior_out) prior_out[nrows] = cprior[q];
            ++nrows;
        }
    }
    free(box);
    free(cbox);
    free(cscore);
    free(cprior);
    free(keep);
    return nrows;
}

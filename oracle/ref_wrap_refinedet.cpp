// ref_wrap_refinedet.cpp -- C entry points around the REFERENCE's own PriorBox / decode / nms (refinedet/refinedet.cpp,
// extracted by oracle/refinedet.mk into _ref/refinedet_postprocess.inc) and a restatement of its driver glue
// (doInference, :729-790), run for one image per call.  Test and benchmark infrastructure only.
//   ref_refinedet_priors   PriorBox() -> [6375,4] doubles on the host (needs a GPU: PriorBox calls .cuda())
//   ref_refinedet_nms      nms() on CPU double tensors
//   ref_refinedet_image    :729-790 on device inputs; rows (x1,y1,x2,y2,score,label) in double, host-synchronous like
//                          the reference (it ends with the .cpu() copy of :793)
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <sstream>
#include <vector>
#include <chrono>
#include "cuda_runtime_api.h"

#include <torch/script.h>
#include "torch/torch.h"
#include "torch/jit.h"

#include "refinedet_postprocess.inc"

#define API __attribute__((visibility("default")))

extern "C" {

API int ref_refinedet_priors(double* out) {
    torch::Tensor t = PriorBox().cpu().contiguous();
    std::memcpy(out, t.data_ptr<double>(), sizeof(double) * t.numel());
    return (int)t.size(0);
}

API int ref_refinedet_nms(const double* boxes, const double* scores, int n, float overlap, int top_k, int64_t* keep_out) {
    torch::Tensor b = torch::from_blob(const_cast<double*>(boxes), {n, 4}, torch::kFloat64).clone();
    torch::Tensor s = torch::from_blob(const_cast<double*>(scores), {n}, torch::kFloat64).clone();
    torch::Tensor keep;
    int count = 0;
    nms(b, s, keep, count, overlap, top_k);
    if (count) std::memcpy(keep_out, keep.slice(0, 0, count).contiguous().data_ptr<int64_t>(), sizeof(int64_t) * count);
    return count;
}

// priors_host: [P,4] doubles, or NULL for the reference's own PriorBox() (P = 6375).  Returns the row count (rows beyond
// `cap` are not written), or -1 on an error of the tensor library.
API int ref_refinedet_image(const double* priors_host, int P, int C, const float* arm_loc_dev, const float* arm_conf_dev,
                            const float* odm_loc_dev, const float* odm_conf_dev, double* rows_out, int cap) {
    try {
        torch::Tensor m_prior = priors_host
                ? torch::from_blob(const_cast<double*>(priors_host), {P, 4}, torch::kFloat64).clone().cuda()
                : PriorBox();
        auto f32 = torch::TensorOptions().dtype(torch::kFloat32).device(torch::kCUDA);
        // :733-736 (from_blob over the engine's device buffers)
        torch::Tensor arm_loc = torch::from_blob(const_cast<float*>(arm_loc_dev), {P, 4}, f32).toType(torch::kFloat64).unsqueeze(0);
        torch::Tensor arm_conf = torch::from_blob(const_cast<float*>(arm_conf_dev), {P, 2}, f32).toType(torch::kFloat64).unsqueeze(0);
        torch::Tensor odm_loc = torch::from_blob(const_cast<float*>(odm_loc_dev), {P, 4}, f32).toType(torch::kFloat64).unsqueeze(0);
        torch::Tensor odm_conf = torch::from_blob(const_cast<float*>(odm_conf_dev), {P, C}, f32).toType(torch::kFloat64).unsqueeze(0);
        // :738-790
        float obj_threshed = 0.01;
        torch::Tensor arm_object_conf = arm_conf.squeeze(0).select(1, 1);
        torch::Tensor object_index = arm_object_conf > obj_threshed;
        object_index = object_index.unsqueeze(1);
        torch::Tensor object_index_1 = object_index.expand_as(odm_conf.squeeze(0)).toType(torch::kFloat64);
        auto filter_odm_conf = odm_conf.squeeze(0).toType(torch::kFloat64) * object_index_1;
        torch::Tensor conf_preds_ = filter_odm_conf.clone().toType(torch::kFloat64);
        torch::Tensor conf_preds = conf_preds_.transpose(1, 0).toType(torch::kFloat64);
        torch::Tensor default_m = decode(arm_loc[0], m_prior);
        bool b_form_pt = true;
        torch::Tensor decode_boxes_m = decode(odm_loc[0], default_m, b_form_pt);
        float conf_thresh = 0.01;
        float mask_thresh = 0.01;
        torch::Tensor result_out;
        for (int i = 1; i < C; i++) {
            torch::Tensor c_mask_m = conf_preds[i] > mask_thresh;
            torch::Tensor nonzero_index = torch::nonzero(c_mask_m);
            torch::Tensor score_m = torch::index_select(conf_preds[i], 0, nonzero_index.squeeze(1));
            torch::Tensor boxes_m = torch::index_select(decode_boxes_m, 0, nonzero_index.squeeze(1));
            torch::Tensor keep;
            int count = 0;
            float overlap = 0.45;
            int top_k = 1000;
            nms(boxes_m, score_m, keep, count, overlap, top_k);
            if (0 == count) continue;
            keep = keep.slice(0, 0, count).clone();
            torch::Tensor score_my = score_m.index_select(0, keep);
            torch::Tensor boxes_my = boxes_m.index_select(0, keep);
            if (score_my[0].item().toFloat() < conf_thresh) continue;
            torch::Tensor label_tensor = torch::full_like(score_my.unsqueeze(1), i);
            torch::Tensor result_ = torch::cat({boxes_my.toType(torch::kFloat64), score_my.unsqueeze(1).toType(torch::kFloat64),
                                                label_tensor.toType(torch::kFloat64)}, 1);
            result_out = 0 == result_out.numel() ? result_.clone() : torch::cat({result_out, result_}, 0);
        }
        if (0 == result_out.numel()) return 0;
        result_out = result_out.cpu().contiguous();
        const int n = (int)result_out.size(0);
        std::memcpy(rows_out, result_out.data_ptr<double>(), sizeof(double) * 6 * (size_t)std::min(n, cap));
        return n;
    } catch (const std::exception& e) {
        std::cerr << "ref_refinedet_image: " << e.what() << std::endl;
        return -1;
    }
}

}  // extern "C"

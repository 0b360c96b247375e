// aa_window.cuh -- the fp32 window of one output index: start, length and normalised weights.
//
// The per-index body of the K1 table kernel aa_tables_fwd_f32 (aa_tables.cu), shared with the crops kernel
// (aa_crops.cu), which computes the tables of its own tile in shared memory: both call this one function, so the
// two cannot drift.  Follows HelperInterpBase::_compute_indices_weights_aa
// (the reference's step_two_dot_two/aa_interpolation_impl.h:194-281) with every operation an explicit
// round-to-nearest intrinsic, so nvcc can neither contract nor reassociate (tests/test_tables_gpu.py).
#pragma once

#include "aa_common.cuh"

namespace aa {

__host__ __device__ inline double base_half(int filter) {  // interp_size * 0.5  (:208)
  return filter == AA_FILTER_BOX ? 0.5 : (filter == AA_FILTER_TRIANGLE ? 1.0 : 2.0);
}

#ifdef __CUDACC__
__device__ __forceinline__ float filt_f32(int filter, float x) {
  if (filter == AA_FILTER_BOX) return (x > -0.5f && x <= 0.5f) ? 1.0f : 0.0f;  // :367-372
  if (x < 0.0f) x = -x;
  if (filter == AA_FILTER_TRIANGLE) {  // :292-300, `1.0 - x` in double
    return x < 1.0f ? __double2float_rn(__dsub_rn(1.0, (double)x)) : 0.0f;
  }
  if (x < 1.0f) {  // :417 all double: ((a+2)x - (a+3)) x x + 1, a = -0.5
    double xd = (double)x;
    double t = __dsub_rn(__dmul_rn(1.5, xd), 2.5);
    t = __dmul_rn(t, xd);
    t = __dmul_rn(t, xd);
    return __double2float_rn(__dadd_rn(t, 1.0));
  }
  if (x < 2.0f) {  // :420 polynomial in float, final *a in double
    float p = __fsub_rn(x, 5.0f);
    p = __fmul_rn(p, x);
    p = __fadd_rn(p, 8.0f);
    p = __fmul_rn(p, x);
    p = __fsub_rn(p, 4.0f);
    return __double2float_rn(__dmul_rn((double)p, -0.5));
  }
  return 0.0f;
}

// Output index i of an axis of `in` samples: *xmin_o, *xsize_o and wr[0..K) (normalised, zero padded to K).
// `scale` = area_pixel_compute_scale<float>, one IEEE division done by the host (h_scale_f32).
__device__ __forceinline__ void aa_window_f32(int64_t in, int filter, float scale, int K, int64_t i,
                                              int32_t* __restrict__ xmin_o, int32_t* __restrict__ xsize_o,
                                              float* __restrict__ wr) {
  const double bh = base_half(filter);
  const float support = (scale >= 1.0f) ? __double2float_rn(__dmul_rn(bh, (double)scale)) : (float)bh;  // :208-209
  const float invscale = (scale >= 1.0f) ? __double2float_rn(__ddiv_rn(1.0, (double)scale)) : 1.0f;     // :242
  const float center = __double2float_rn(__dmul_rn((double)scale, __dadd_rn((double)i, 0.5)));         // :253
  long long xmin = __double2ll_rz(__dadd_rn((double)__fsub_rn(center, support), 0.5));                  // :254
  if (xmin < 0) xmin = 0;
  long long xmax = __double2ll_rz(__dadd_rn((double)__fadd_rn(center, support), 0.5));                  // :255-257
  if (xmax > in) xmax = in;
  xmax -= xmin;
  *xmin_o = (int32_t)xmin;
  *xsize_o = (int32_t)xmax;
  float total = 0.0f;
  long long j = 0;
  for (; j < xmax && j < K; j++) {
    float d = __fsub_rn(__ll2float_rn(j + xmin), center);                                               // :266
    float arg = __double2float_rn(__dmul_rn(__dadd_rn((double)d, 0.5), (double)invscale));
    float wj = filt_f32(filter, arg);
    wr[j] = wj;
    total = __fadd_rn(total, wj);                                                                      // :268
  }
  const long long nt = j;
  if (total != 0.0f)
    for (j = 0; j < nt; j++) wr[j] = __fdiv_rn(wr[j], total);                                           // :270-274
  for (j = nt; j < K; j++) wr[j] = 0.0f;                                                                // :276-278
}
#endif

}  // namespace aa

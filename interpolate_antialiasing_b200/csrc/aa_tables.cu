// aa_tables.cu -- K1: the per-axis index/weight table builder as a tiny sm_100a kernel, plus the
// per-device table cache.
//
// Replaces HelperInterpBase::_compute_indices_weights_aa and the three filter helpers
// (/root/reference/step_two_dot_two/aa_interpolation_impl.h:194-281, :292-300, :367-372, :410-424)
// and torch's area_pixel_compute_scale (ATen/native/UpSample.h).  The reference evaluates the
// tables in mixed fp32/fp64 by C++ promotion rules on x86-64 without FMA; every operation below is
// an explicit round-to-nearest intrinsic (__fmul_rn, __dadd_rn, ...) so nvcc can neither contract
// nor reassociate, and the integer tables AND the weights come out bit-identical
// (tests/test_tables_gpu.py).  Compile this TU without --use_fast_math.
#include <math.h>

#include <map>
#include <mutex>
#include <tuple>

#include "aa_common.cuh"
#include "aa_window.cuh"

namespace aa {

// ------------------------------------------------------------------------------------------------
// scalar recipe shared by host (launch planning) and device (the tables)
// ------------------------------------------------------------------------------------------------
// host versions: plain IEEE float/double operators (no a*b+c pattern exists in them)
// area_pixel_compute_scale<scalar_t> + compute_scales_value (ATen/native/UpSample.h): a caller-provided scale factor
// (`scale_factors`, aa_interpolation_impl.h:735,740-742) replaces in/out by 1/scale_factor unless align_corners.
static float h_scale_f32(int64_t in, int64_t out, int align, double user_scale = 0.0) {
  if (align) return out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.0f;
  if (user_scale > 0.0) return (float)(1.0 / user_scale);
  return (float)in / (float)out;
}
static double h_scale_f64(int64_t in, int64_t out, int align, double user_scale = 0.0) {
  if (align) return out > 1 ? (double)(in - 1) / (double)(out - 1) : 0.0;
  if (user_scale > 0.0) return 1.0 / user_scale;
  return (double)in / (double)out;
}
static float h_support_f32(float scale, int filter) {
  return (scale >= 1.0f) ? (float)(base_half(filter) * (double)scale) : (float)base_half(filter);
}
static double h_support_f64(double scale, int filter) {
  return (scale >= 1.0) ? base_half(filter) * scale : base_half(filter);
}

int host_interp_size(int64_t in, int64_t out, int filter, int align, int dtype, double user_scale) {
  if (dtype == AA_F64) {
    double s = h_support_f64(h_scale_f64(in, out, align, user_scale), filter);
    return (int)ceilf((float)s) * 2 + 1;  // ceilf() of a double converts to float first (:210)
  }
  float s = h_support_f32(h_scale_f32(in, out, align, user_scale), filter);
  return (int)ceilf(s) * 2 + 1;
}

float host_scale_f32(int64_t in, int64_t out, int align) { return h_scale_f32(in, out, align); }

// Integer tables on the host: the same IEEE operations as the device kernels below (this TU is compiled with
// -ffp-contract=off and x86-64 SSE arithmetic has no excess precision), so launch planning never has to read the
// device tables back.  tests/test_tables_gpu.py holds the two bit-identical.
void host_int_tables(int64_t in, int64_t out, int filter, int align, int dtype, double user_scale, int32_t* xmin_o,
                     int32_t* xsize_o) {
  if (dtype == AA_F64) {
    const double scale = h_scale_f64(in, out, align, user_scale);
    const double support = h_support_f64(scale, filter);
    for (int64_t i = 0; i < out; i++) {
      const double center = scale * ((double)i + 0.5);
      long long xmin = (long long)((center - support) + 0.5);
      if (xmin < 0) xmin = 0;
      long long xmax = (long long)((center + support) + 0.5);
      if (xmax > in) xmax = in;
      xmin_o[i] = (int32_t)xmin;
      xsize_o[i] = (int32_t)(xmax - xmin);
    }
    return;
  }
  const float scale = h_scale_f32(in, out, align, user_scale);
  const float support = h_support_f32(scale, filter);
  for (int64_t i = 0; i < out; i++) {
    const float center = (float)((double)scale * ((double)i + 0.5));
    long long xmin = (long long)((double)(center - support) + 0.5);
    if (xmin < 0) xmin = 0;
    long long xmax = (long long)((double)(center + support) + 0.5);
    if (xmax > in) xmax = in;
    xmin_o[i] = (int32_t)xmin;
    xsize_o[i] = (int32_t)(xmax - xmin);
  }
}

// ------------------------------------------------------------------------------------------------
// device filters, explicit rounding
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double filt_f64(int filter, double x) {
  if (filter == AA_FILTER_BOX) return (x > -0.5 && x <= 0.5) ? 1.0 : 0.0;
  if (x < 0.0) x = -x;
  if (filter == AA_FILTER_TRIANGLE) return x < 1.0 ? __dsub_rn(1.0, x) : 0.0;
  if (x < 1.0) {
    double t = __dsub_rn(__dmul_rn(1.5, x), 2.5);
    t = __dmul_rn(t, x);
    t = __dmul_rn(t, x);
    return __dadd_rn(t, 1.0);
  }
  if (x < 2.0) {
    double p = __dsub_rn(x, 5.0);
    p = __dmul_rn(p, x);
    p = __dadd_rn(p, 8.0);
    p = __dmul_rn(p, x);
    p = __dsub_rn(p, 4.0);
    return __dmul_rn(p, -0.5);
  }
  return 0.0;
}

// One thread per output index.  fp32 instantiation of :194-281 (aa_window.cuh).
__global__ void aa_tables_fwd_f32(int64_t in, int64_t out, int filter, float scale, int K,
                                  int32_t* __restrict__ xmin_o, int32_t* __restrict__ xsize_o,
                                  float* __restrict__ w) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out) return;
  aa_window_f32(in, filter, scale, K, i, xmin_o + i, xsize_o + i, w + i * K);
}

__global__ void aa_tables_fwd_f64(int64_t in, int64_t out, int filter, double scale, int K,
                                  int32_t* __restrict__ xmin_o, int32_t* __restrict__ xsize_o,
                                  double* __restrict__ w) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out) return;
  const double bh = base_half(filter);
  const double support = (scale >= 1.0) ? __dmul_rn(bh, scale) : bh;
  const double invscale = (scale >= 1.0) ? __ddiv_rn(1.0, scale) : 1.0;
  const double center = __dmul_rn(scale, __dadd_rn((double)i, 0.5));
  long long xmin = __double2ll_rz(__dadd_rn(__dsub_rn(center, support), 0.5));
  if (xmin < 0) xmin = 0;
  long long xmax = __double2ll_rz(__dadd_rn(__dadd_rn(center, support), 0.5));
  if (xmax > in) xmax = in;
  xmax -= xmin;
  xmin_o[i] = (int32_t)xmin;
  xsize_o[i] = (int32_t)xmax;
  double* wr = w + i * K;
  double total = 0.0;
  long long j = 0;
  for (; j < xmax && j < K; j++) {
    // (j + xmin - center + 0.5) * invscale, all double, left to right
    double arg = __dmul_rn(__dadd_rn(__dsub_rn((double)(j + xmin), center), 0.5), invscale);
    double wj = filt_f64(filter, arg);
    wr[j] = wj;
    total = __dadd_rn(total, wj);
  }
  const long long nt = j;
  if (total != 0.0)
    for (j = 0; j < nt; j++) wr[j] = __ddiv_rn(wr[j], total);
  for (j = nt; j < K; j++) wr[j] = 0.0;
}

// One thread per input index x: the transposed (adjoint) tables (the host checks the monotonicity the
// contiguous-range argument relies on, on its bit-identical copy of xmin/xsize).
template <typename T>
__global__ void aa_tables_adj(int64_t in, int64_t out, int K, int KT, const int32_t* __restrict__ xmin,
                              const int32_t* __restrict__ xsize, const T* __restrict__ w,
                              int32_t* __restrict__ omin_o, int32_t* __restrict__ osize_o,
                              T* __restrict__ wT) {
  int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= in) return;
  // omin = first o with xmin[o]+xsize[o] > x ; oend = first o with xmin[o] > x
  int64_t lo = 0, hi = out;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if ((int64_t)xmin[mid] + xsize[mid] > x) hi = mid; else lo = mid + 1;
  }
  const int64_t omin = lo;
  lo = omin; hi = out;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if ((int64_t)xmin[mid] > x) hi = mid; else lo = mid + 1;
  }
  const int64_t osz = lo - omin;
  omin_o[x] = (int32_t)omin;
  osize_o[x] = (int32_t)osz;
  T* row = wT + x * KT;
  for (int k = 0; k < KT; k++) {
    T v = (T)0;
    if (k < osz) {
      int64_t o = omin + k;
      int64_t j = x - xmin[o];
      if (j >= 0 && j < K) v = w[o * K + j];
    }
    row[k] = v;
  }
}

// One thread per input row y: the records used by the streaming kernel's vertical pass.
// Record = A weights wT[y][0..A) (k-th weight belongs to output omin[y]+k, the k-th OLDEST output row
// still open at y), followed by (first_flush_o | nflush << 24): the `nflush` oldest open outputs,
// starting at first_flush_o = omin[y], have y as the LAST row of their window.  Because the outputs
// that end at y are exactly the ones missing from row y+1's range, omin[y+1] = omin[y] + nflush.
__global__ void aa_tables_slots(int64_t in, int A, int RS, int KT, const int32_t* __restrict__ xmin,
                                const int32_t* __restrict__ xsize, const int32_t* __restrict__ omin,
                                const int32_t* __restrict__ osize, const float* __restrict__ wT,
                                float* __restrict__ slot) {
  int64_t y = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (y >= in) return;
  float* rec = slot + y * RS;
  for (int a = 0; a < RS; a++) rec[a] = 0.0f;
  const int o0 = omin[y], n = osize[y];
  int nflush = 0;
  for (int k = 0; k < n && k < A; k++) {
    const int o = o0 + k;
    rec[k] = wT[y * KT + k];
    if ((int64_t)xmin[o] + xsize[o] - 1 == y) nflush++;
  }
  rec[A] = __int_as_float(o0 | (nflush << 24));
}

// Adjoint direction: one thread per forward-output index o (= a streamed grad_out row).  The open
// grad_in rows at o are [xmin[o], xmin[o]+xsize[o]) with the forward weights; the ones that no later o
// covers (y < xmin[o+1]) finish here.
__global__ void aa_tables_slots_adj(int64_t out, int A, int RS, int K, const int32_t* __restrict__ xmin,
                                    const int32_t* __restrict__ xsize, const float* __restrict__ w,
                                    float* __restrict__ slot) {
  int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= out) return;
  float* rec = slot + o * RS;
  for (int a = 0; a < RS; a++) rec[a] = 0.0f;
  const int x0 = xmin[o], n = xsize[o];
  for (int k = 0; k < n && k < A; k++) rec[k] = w[o * K + k];
  const int end = x0 + n;
  const int nxt = (o + 1 < out) ? xmin[o + 1] : end;
  const int nflush = (nxt < end ? nxt : end) - x0;
  rec[A] = __int_as_float(x0 | (nflush << 24));
}

// Tensor-core vertical pass (aa_vmma.cu): fixed-point weights.  One block finds s = the largest shift with
// max|w| * 2^s <= 2^23 - 2^16 (so that the top digit fits an int8) and the constants that turn the three int32 limb
// sums L0, L1, L2 (as floats m_i = 1.5*2^23 + L_i, the magic-number int->float) back into
//   sum_j w_j * pixel_j = (65536*L0 + 256*L1 + L2) * 2^-s = fma(m2, c2, fma(m1, c1, fma(m0, c0, K0))),
//   c_i = 2^(16-8i-s), K0 = -1.5*2^23 * (c0 + c1 + c2)   (exact: 197379 * 2^(22-s)).
// The first two fmas are exact (their results are multiples of 2^16*c2 resp. 2^8*c2 that fit 24 bits ... 28 bits:
// the second rounds like any fp32 add), so the reconstruction carries two fp32 roundings.
__global__ void aa_tables_vq_scale(const float* __restrict__ w, int64_t n, float* __restrict__ meta) {
  __shared__ float red[256];
  float m = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, fabsf(w[i]));
  red[threadIdx.x] = m;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] = fmaxf(red[threadIdx.x], red[threadIdx.x + s]);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    m = red[0];
    int s = 22;
    if (m > 0.f) s = ilogbf(8323072.0f / m);  // floor(log2((2^23 - 2^16) / max|w|))
    s = s < 0 ? 0 : (s > 30 ? 30 : s);
    const float c2 = exp2f((float)-s), c1 = exp2f((float)(8 - s)), c0 = exp2f((float)(16 - s));
    meta[0] = c0; meta[1] = c1; meta[2] = c2;
    meta[3] = -197379.0f * exp2f((float)(22 - s));
    meta[4] = __int_as_float(s);
  }
}
// One thread per (output row, tap): three int8 digits into the row block's matrix.  Element (k, n) of a block lives at
// byte k*128 + (((n >> 4) ^ (k & 7)) << 4) + (n & 15): the 128-byte swizzle the MMA's shared-memory descriptor
// expects, applied here so that a plain bulk copy can land the matrix.  n = digit*32 + (row inside the block).
__global__ void aa_tables_vq(int64_t out, int K, int oyb, int krows, const int32_t* __restrict__ xmin,
                             const int32_t* __restrict__ xsize, const float* __restrict__ w, const float* __restrict__ meta,
                             int8_t* __restrict__ bq) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= out * K) return;
  const int64_t oy = idx / K;
  const int j = (int)(idx - oy * K);
  if (j >= xsize[oy]) return;
  const int64_t b = oy / oyb;
  const int i = (int)(oy - b * oyb);
  const int k = xmin[oy] + j - xmin[b * oyb];
  if (k < 0 || k >= krows) return;  // cannot happen: the host sized krows from the same tables
  const int s = __float_as_int(meta[4]);
  const int q = __float2int_rn(w[idx] * exp2f((float)s));  // exact product (power of two), |q| <= 2^23 - 2^16
  const int d2 = ((q + 128) & 255) - 128;
  const int q1 = (q - d2) >> 8;
  const int d1 = ((q1 + 128) & 255) - 128;
  const int d0 = (q1 - d1) >> 8;
  int8_t* row = bq + ((size_t)b * krows + k) * 128;
  const int dig[3] = {d0, d1, d2};
  for (int l = 0; l < 3; l++) {
    const int n = l * 32 + i;  // 32 accumulator columns per digit whatever the block height (16 or 32 rows)
    row[(((n >> 4) ^ (k & 7)) << 4) + (n & 15)] = (int8_t)dig[l];
  }
}

// ------------------------------------------------------------------------------------------------
// cache
// ------------------------------------------------------------------------------------------------
AxisTables::~AxisTables() {
  // Device memory is released with the owning context; freeing here is best effort.
  int cur = -1;
  if (cudaGetDevice(&cur) == cudaSuccess) {
    cudaSetDevice(device);
    if (ready) cudaEventDestroy(ready);
    if (block) cudaFree(block);  // cudaFree waits for in-flight work that may still read the tables
    if (slot) cudaFree(slot);
    if (slot_adj) cudaFree(slot_adj);
    if (vq) cudaFree(vq);
    if (vq_meta) cudaFree(vq_meta);
    cudaSetDevice(cur);
  }
}

namespace {
using Key = std::tuple<int, int64_t, int64_t, int, int, int, double>;
std::mutex g_mu;  // guards the map and the LRU clock only: tables are built outside it
std::map<Key, std::shared_ptr<AxisTables>> g_cache;
uint64_t g_clock = 0, g_next_id = 1;
struct CacheStats { int64_t hits = 0, misses = 0, evictions = 0; } g_stats;

size_t cache_capacity() {
  static const size_t cap = [] { const char* e = getenv("AA_TABLE_CACHE_MAX"); long v = e ? atol(e) : 256; return (size_t)(v < 2 ? 2 : v); }();
  return cap;
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Everything the launch planners need is computed on the host (integer tables, their transpose, the maxima); the
// device gets its own copy from the table kernels (K1), stream-ordered, with no read-back and no synchronisation.
int build_tables(AxisTables* t, cudaStream_t stream) {
  const int64_t in = t->in, out = t->out;
  const bool f64 = t->dtype == AA_F64;
  t->scale_f = h_scale_f32(in, out, t->align, t->user_scale);
  t->support_f = h_support_f32(t->scale_f, t->filter);
  t->scale_d = h_scale_f64(in, out, t->align, t->user_scale);
  t->support_d = h_support_f64(t->scale_d, t->filter);
  t->K = host_interp_size(in, out, t->filter, t->align, t->dtype, t->user_scale);
  t->h_xmin.resize(out);
  t->h_xsize.resize(out);
  t->h_omin.resize(in);
  t->h_osize.resize(in);
  host_int_tables(in, out, t->filter, t->align, t->dtype, t->user_scale, t->h_xmin.data(), t->h_xsize.data());
  int xsize_max = 0;
  bool monotone = true;
  for (int64_t o = 0; o < out; o++) {
    xsize_max = std::max(xsize_max, t->h_xsize[o]);
    if (o > 0 && (t->h_xmin[o] < t->h_xmin[o - 1] || t->h_xmin[o] + t->h_xsize[o] < t->h_xmin[o - 1] + t->h_xsize[o - 1])) monotone = false;
  }
  if (!monotone) return fail(AA_ERR_INVALID, "internal: window tables are not monotone");
  if (xsize_max > t->K) return fail(AA_ERR_INVALID, "internal: window longer than interp_size");
  // transpose of the window relation: omin[x] = first o whose window ends after x, oend[x] = first o starting after x
  int kt_max = 0;
  {
    int64_t lo = 0, hi = 0;
    for (int64_t x = 0; x < in; x++) {
      while (lo < out && (int64_t)t->h_xmin[lo] + t->h_xsize[lo] <= x) lo++;
      if (hi < lo) hi = lo;
      while (hi < out && t->h_xmin[hi] <= x) hi++;
      t->h_omin[x] = (int32_t)lo;
      t->h_osize[x] = (int32_t)(hi - lo);
      kt_max = std::max(kt_max, (int)(hi - lo));
    }
  }
  t->xsize_max = xsize_max;
  t->kt_max = kt_max;
  t->monotone = 1;
  t->KT = std::max(1, kt_max);
  const size_t es = f64 ? 8 : 4;
  size_t off = 0;
  const size_t o_xmin = off;  off = align_up(off + sizeof(int32_t) * out, 256);
  const size_t o_xsize = off; off = align_up(off + sizeof(int32_t) * out, 256);
  const size_t o_w = off;     off = align_up(off + es * out * t->K, 256);
  const size_t o_omin = off;  off = align_up(off + sizeof(int32_t) * in, 256);
  const size_t o_osize = off; off = align_up(off + sizeof(int32_t) * in, 256);
  const size_t o_wT = off;    off = align_up(off + es * in * t->KT, 256);
  AA_CUDA_TRY(cudaMalloc(&t->block, off));
  char* base = (char*)t->block;
  t->xmin = (int32_t*)(base + o_xmin);
  t->xsize = (int32_t*)(base + o_xsize);
  t->w = base + o_w;
  t->omin = (int32_t*)(base + o_omin);
  t->osize = (int32_t*)(base + o_osize);
  t->wT = base + o_wT;
  const int NT = 128;
  const unsigned gb_out = (unsigned)((out + NT - 1) / NT);
  const unsigned gb_adj = (unsigned)((in + NT - 1) / NT);
  if (f64) {
    aa_tables_fwd_f64<<<gb_out, NT, 0, stream>>>(in, out, t->filter, t->scale_d, t->K, t->xmin, t->xsize, (double*)t->w);
    AA_LAUNCH_CHECK("aa_tables_fwd_f64");
    aa_tables_adj<double><<<gb_adj, NT, 0, stream>>>(in, out, t->K, t->KT, t->xmin, t->xsize, (const double*)t->w, t->omin,
                                                      t->osize, (double*)t->wT);
    AA_LAUNCH_CHECK("aa_tables_adj<double>");
  } else {
    aa_tables_fwd_f32<<<gb_out, NT, 0, stream>>>(in, out, t->filter, t->scale_f, t->K, t->xmin, t->xsize, (float*)t->w);
    AA_LAUNCH_CHECK("aa_tables_fwd_f32");
    aa_tables_adj<float><<<gb_adj, NT, 0, stream>>>(in, out, t->K, t->KT, t->xmin, t->xsize, (const float*)t->w, t->omin,
                                                     t->osize, (float*)t->wT);
    AA_LAUNCH_CHECK("aa_tables_adj<float>");
  }
  // cross-stream publication: users on OTHER streams wait on this event until it has completed once
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(stream, &cap);
  if (cap != cudaStreamCaptureStatusNone) return fail(AA_ERR_INVALID, "table cache miss under CUDA-graph capture: call aa_warm_tables first");
  AA_CUDA_TRY(cudaEventCreateWithFlags(&t->ready, cudaEventDisableTiming));
  AA_CUDA_TRY(cudaEventRecord(t->ready, stream));
  t->build_stream = stream;
  return AA_OK;
}

// make `stream` see the finished tables (called with g_mu held)
int acquire_ready(AxisTables* t, cudaStream_t stream) {
  if (!t->ready) return AA_OK;
  const cudaError_t q = cudaEventQuery(t->ready);
  if (q == cudaSuccess) {
    cudaEventDestroy(t->ready);
    t->ready = nullptr;
    return AA_OK;
  }
  if (q != cudaErrorNotReady) return cuda_fail(q, "cudaEventQuery(table ready)");
  if (stream != t->build_stream) AA_CUDA_TRY(cudaStreamWaitEvent(stream, t->ready, 0));
  return AA_OK;
}
}  // namespace

int get_axis_tables(int device, int64_t in, int64_t out, int filter, int align, int dtype, double user_scale,
                    cudaStream_t stream, std::shared_ptr<AxisTables>* result) {
  if (in <= 0 || out <= 0) return fail(AA_ERR_INVALID, "table sizes must be positive");
  if (in >= (1ll << 31) || out >= (1ll << 31)) return fail(AA_ERR_UNSUPPORTED, "axis length >= 2^31");
  if (dtype == AA_U8) dtype = AA_F32;
  if (align || !(user_scale > 0.0)) user_scale = 0.0;  // ignored with align_corners (area_pixel_compute_scale)
  const Key key(device, in, out, filter, align ? 1 : 0, dtype, user_scale);
  {
    std::lock_guard<std::mutex> lock(g_mu);
    auto it = g_cache.find(key);
    if (it != g_cache.end()) {
      it->second->last_use = ++g_clock;
      g_stats.hits++;
      int rc = acquire_ready(it->second.get(), stream);
      if (rc != AA_OK) return rc;
      *result = it->second;
      return AA_OK;
    }
  }
  // miss: build without holding the lock (two threads missing on the same key both build; the first insert wins)
  auto t = std::make_shared<AxisTables>();
  t->device = device;
  t->in = in;
  t->out = out;
  t->filter = filter;
  t->align = align ? 1 : 0;
  t->dtype = dtype;
  t->user_scale = user_scale;
  int rc = build_tables(t.get(), stream);
  if (rc != AA_OK) return rc;
  std::vector<std::shared_ptr<AxisTables>> evicted;  // destroyed after the lock is released (cudaFree may block)
  {
    std::lock_guard<std::mutex> lock(g_mu);
    g_stats.misses++;
    auto it = g_cache.find(key);
    if (it != g_cache.end()) {
      it->second->last_use = ++g_clock;
      rc = acquire_ready(it->second.get(), stream);
      if (rc != AA_OK) return rc;
      *result = it->second;
      evicted.push_back(t);
      return AA_OK;
    }
    t->id = g_next_id++;
    t->last_use = ++g_clock;
    g_cache[key] = t;
    while (g_cache.size() > cache_capacity()) {  // LRU among entries nobody else holds
      auto victim = g_cache.end();
      for (auto c = g_cache.begin(); c != g_cache.end(); ++c)
        if (c->second.use_count() == 1 && c->second.get() != t.get() && (victim == g_cache.end() || c->second->last_use < victim->second->last_use))
          victim = c;
      if (victim == g_cache.end()) break;
      evicted.push_back(victim->second);
      g_cache.erase(victim);
      g_stats.evictions++;
    }
  }
  *result = t;
  return AA_OK;
}

void table_cache_stats(int64_t* entries, int64_t* hits, int64_t* misses, int64_t* evictions) {
  std::lock_guard<std::mutex> lock(g_mu);
  *entries = (int64_t)g_cache.size();
  *hits = g_stats.hits;
  *misses = g_stats.misses;
  *evictions = g_stats.evictions;
}

// The derived tables below are built once per AxisTables under its own mutex (not the cache lock) and published
// after a stream synchronisation ("first use only"): a later user on any stream sees complete tables.
int ensure_slot_tables(AxisTables* t, int A, cudaStream_t stream) {
  std::lock_guard<std::mutex> lock(t->mu);
  if (t->dtype != AA_F32) return fail(AA_ERR_UNSUPPORTED, "slot tables are float only");
  if (t->slot && t->slot_A == A) return AA_OK;
  if (t->slot) return fail(AA_ERR_INVALID, "internal: slot tables requested with two different A");
  if (t->out >= (1 << 24)) return fail(AA_ERR_UNSUPPORTED, "streaming path needs out < 2^24");
  const int RS = (A + 1 + 3) / 4 * 4;
  float* slot = nullptr;
  AA_CUDA_TRY(cudaMalloc(&slot, sizeof(float) * (size_t)t->in * RS));
  const int NT = 128;
  aa_tables_slots<<<(unsigned)((t->in + NT - 1) / NT), NT, 0, stream>>>(
      t->in, A, RS, t->KT, t->xmin, t->xsize, t->omin, t->osize, (const float*)t->wT, slot);
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);  // first use only
  if (e != cudaSuccess) {
    cudaFree(slot);
    return cuda_fail(e, "aa_tables_slots");
  }
  t->slot_A = A;
  t->slot_RS = RS;
  t->slot = slot;
  return AA_OK;
}

int ensure_slot_tables_adj(AxisTables* t, int A, cudaStream_t stream) {
  std::lock_guard<std::mutex> lock(t->mu);
  if (t->dtype != AA_F32) return fail(AA_ERR_UNSUPPORTED, "slot tables are float only");
  if (t->slot_adj && t->slot_adj_A == A) return AA_OK;
  if (t->slot_adj) return fail(AA_ERR_INVALID, "internal: adjoint slot tables requested with two different A");
  if (t->in >= (1 << 24)) return fail(AA_ERR_UNSUPPORTED, "streaming path needs in < 2^24");
  const int RS = (A + 1 + 3) / 4 * 4;
  float* slot = nullptr;
  AA_CUDA_TRY(cudaMalloc(&slot, sizeof(float) * (size_t)t->out * RS));
  const int NT = 128;
  aa_tables_slots_adj<<<(unsigned)((t->out + NT - 1) / NT), NT, 0, stream>>>(t->out, A, RS, t->K, t->xmin, t->xsize,
                                                                             (const float*)t->w, slot);
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);  // first use only
  if (e != cudaSuccess) {
    cudaFree(slot);
    return cuda_fail(e, "aa_tables_slots_adj");
  }
  t->slot_adj_A = A;
  t->slot_adj_RS = RS;
  t->slot_adj = slot;
  return AA_OK;
}

int ensure_vq_tables(AxisTables* t, int oyb_max, int kstep, int max_ksteps, cudaStream_t stream) {
  std::lock_guard<std::mutex> lock(t->mu);
  if (t->dtype != AA_F32) return fail(AA_ERR_UNSUPPORTED, "vq tables are float only");
  if (t->vq) return AA_OK;  // complete: the builder synchronised before publishing
  if (t->vq_ksteps < 0) return fail(AA_ERR_UNSUPPORTED, "vmma: a block of output rows spans too many input rows");
  const int64_t out = t->out;
  // block height: 32 output rows, or 16 when 32 rows would span more than max_ksteps*kstep input rows (scales > ~7x)
  int oyb = oyb_max, noyb = 0, ksteps = 0;
  for (;; oyb /= 2) {
    noyb = (int)((out + oyb - 1) / oyb);
    int span = 1;
    for (int b = 0; b < noyb; b++) {
      const int64_t o0 = (int64_t)b * oyb, o1 = std::min<int64_t>(out, o0 + oyb) - 1;
      span = std::max<int>(span, t->h_xmin[o1] + t->h_xsize[o1] - t->h_xmin[o0]);
    }
    ksteps = (span + kstep - 1) / kstep;
    if (ksteps <= max_ksteps) break;
    if (oyb <= 16) {
      t->vq_ksteps = -1;
      return fail(AA_ERR_UNSUPPORTED, "vmma: a block of output rows spans too many input rows");
    }
  }
  const int krows = ksteps * kstep;
  const size_t bytes = (size_t)noyb * krows * 128;
  int8_t* vq = nullptr;
  float* meta = nullptr;
  AA_CUDA_TRY(cudaMalloc(&vq, bytes));
  cudaError_t e = cudaMalloc(&meta, 8 * sizeof(float));
  if (e == cudaSuccess) e = cudaMemsetAsync(vq, 0, bytes, stream);
  if (e == cudaSuccess) {
    aa_tables_vq_scale<<<1, 256, 0, stream>>>((const float*)t->w, out * t->K, meta);
    const int NT = 256;
    aa_tables_vq<<<(unsigned)((out * t->K + NT - 1) / NT), NT, 0, stream>>>(out, t->K, oyb, krows, t->xmin, t->xsize,
                                                                           (const float*)t->w, meta, vq);
    count_launch(2);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);  // first use only
  if (e != cudaSuccess) {
    cudaFree(vq);
    if (meta) cudaFree(meta);
    return cuda_fail(e, "vq tables");
  }
  t->vq_meta = meta;
  t->vq_ksteps = ksteps;
  t->vq_noyb = noyb;
  t->vq_oyb = oyb;
  t->vq = vq;
  return AA_OK;
}

namespace stream_detail { void plan_clear(); }

int clear_table_cache() {
  stream_detail::plan_clear();
  vmma_plan_clear();
  tile_plan_clear();
  redo_clear();
  std::map<Key, std::shared_ptr<AxisTables>> old;
  {
    std::lock_guard<std::mutex> lock(g_mu);
    old.swap(g_cache);
  }
  return AA_OK;  // `old` is destroyed here, outside the lock
}

}  // namespace aa

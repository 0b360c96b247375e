// aa_api.cu -- the C ABI (include/aa_resize.h): validation, table cache lookups, path selection.
// No torch types, no exceptions across the boundary, no CPU fallback.
#include <algorithm>
#include <cstdlib>
#include <tuple>
#include <vector>
#include <string.h>

#include <mutex>

#include "aa_common.cuh"

namespace aa {

static thread_local std::string g_err;
static thread_local int64_t g_launches = 0;

void set_error(const std::string& msg) { g_err = msg; }
int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string("CUDA error: ") + cudaGetErrorString(e) + " (" + cudaGetErrorName(e) + ") at " + what;
  return e == cudaErrorMemoryAllocation ? AA_ERR_NOMEM : AA_ERR_CUDA;
}
void count_launch(int n) { g_launches += n; }

int classify_layout(const aa_tensor_desc& t, bool prefer_channels_last, Layout* L, bool* is_cl_out) {
  // strides of size-1 dimensions carry no information
  const bool cf = (t.w == 1 || t.stride_w == 1);
  const bool cl = (t.c == 1 || t.stride_c == 1) && (t.w == 1 || t.stride_w == t.c);
  bool use_cl;
  if (cf && cl) use_cl = prefer_channels_last;
  else if (cl) use_cl = true;
  else if (cf) use_cl = false;
  else return fail(AA_ERR_UNSUPPORTED, "tensor is neither channels_first (stride_w == 1) nor channels_last "
                                       "(stride_c == 1, stride_w == c); make it contiguous in one of the two formats");
  Layout r;
  if (use_cl) {
    // the stride of a size-1 batch dimension carries no information (torch reports arbitrary values there): 0 keeps
    // the alignment tests of the vectorised / TMA paths from tripping over it
    r.planes = t.n; r.Cp = 1; r.Ci = (int)t.c; r.stride_n = t.n == 1 ? 0 : t.stride_n; r.stride_p = 0;
    r.stride_h = (t.h == 1) ? t.w * t.c : t.stride_h;
    if (r.stride_h < t.w * t.c) return fail(AA_ERR_UNSUPPORTED, "channels_last rows overlap (stride_h < w*c)");
  } else {
    r.planes = t.n * t.c; r.Cp = (int)t.c; r.Ci = 1; r.stride_n = t.n == 1 ? 0 : t.stride_n; r.stride_p = (t.c == 1) ? 0 : t.stride_c;
    r.stride_h = (t.h == 1) ? t.w : t.stride_h;
    if (r.stride_h < t.w) return fail(AA_ERR_UNSUPPORTED, "channels_first rows overlap (stride_h < w)");
  }
  *L = r;
  if (is_cl_out) *is_cl_out = use_cl;
  return AA_OK;
}

namespace {

int check_desc(const aa_tensor_desc* t, const char* name) {
  if (!t) return fail(AA_ERR_INVALID, std::string(name) + " is null");
  if (t->n < 0 || t->c <= 0 || t->h <= 0 || t->w <= 0)
    return fail(AA_ERR_INVALID, std::string("Non-empty 4D data tensor expected but got ") + name + " with sizes [" +
                                    std::to_string(t->n) + ", " + std::to_string(t->c) + ", " + std::to_string(t->h) + ", " +
                                    std::to_string(t->w) + "]");
  if (t->n > 0 && !t->data) return fail(AA_ERR_INVALID, std::string(name) + ".data is null");
  if (t->dtype < AA_U8 || t->dtype > AA_BF16) return fail(AA_ERR_INVALID, std::string(name) + ": bad dtype");
  return AA_OK;
}
int check_filter(int filter) {
  if (filter != AA_FILTER_BOX && filter != AA_FILTER_TRIANGLE && filter != AA_FILTER_CUBIC)
    return fail(AA_ERR_INVALID, "filter must be 0 (box), 1 (triangle) or 2 (cubic)");
  return AA_OK;
}

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
    ok = err == cudaSuccess;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

BandedAxis fwd_axis(const AxisTables* t) {
  return BandedAxis{t->xmin, t->xsize, t->w, t->K, t->in, t->out, t->h_xmin.data(), t->h_xsize.data(), t->id * 2, t->device};
}
BandedAxis adj_axis(const AxisTables* t) {
  return BandedAxis{t->omin, t->osize, t->wT, t->KT, t->out, t->in, t->h_omin.data(), t->h_osize.data(), t->id * 2 + 1, t->device};
}

// AUTO policy for the tensor-core path: vertical downsampling with enough taps that the FP32-pipe kernel is
// instruction-bound (measured crossover, DESIGN.md section 6).  AA_VMMA_AUTO=0 disables, =1 forces wherever eligible.
bool vmma_auto(const AxisTables* th, const AxisTables* tw) {
  static const int mode = [] { const char* e = getenv("AA_VMMA_AUTO"); return e ? atoi(e) : -1; }();
  if (mode == 0) return false;
  if (mode == 1) return true;
  (void)tw;
  // measured on the uint8 sweep (profiles/r02_u8_paths.txt -> DESIGN.md section 6): the tensor-core kernel beats the
  // streaming, band and tile kernels at every vertical scale from 1x down to the 7x its K span allows -- except bilinear at
  // exactly 1x, where the band kernel with 32-bit pixel loads is 13 % faster (3-tap windows: nothing to amortise)
  if (th->scale_f <= 1.0f && th->xsize_max <= 3) return false;
  return th->scale_f >= 1.0f;
}

__global__ void widen_i32_i64(const int32_t* __restrict__ a, int64_t* __restrict__ b, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) b[i] = a[i];
}

// One launch: few taps on both axes (near scale 1 / upsampling) -> output-bound tile / band kernels; uint8 pixels with
// vertical downsampling -> tensor-core vertical pass; otherwise (downsampling) -> input-bound streaming kernel.
// AA_ERR_UNSUPPORTED when none of them takes the shape.
int fused_dispatch(const void* in, int in_dtype, const Layout& lin, void* out, const Layout& lout, AxisTables* th, AxisTables* tw,
                   int64_t H, int64_t W, int64_t oH, int64_t oW, uint32_t flags, const OutEpi& epi, cudaStream_t stream) {
  int rc;
  const bool want_vmma = in_dtype == AA_U8 && !(flags & (AA_FLAG_FORCE_STREAM | AA_FLAG_STREAM_TMA | AA_FLAG_STREAM_LDG)) &&
                         ((flags & AA_FLAG_VMMA) || vmma_auto(th, tw));
  if (want_vmma) {
    rc = launch_vmma(in, lin, out, lout, th, tw, H, W, oH, oW, epi, stream);
    if (rc != AA_ERR_UNSUPPORTED || (flags & AA_FLAG_VMMA)) return rc;
  }
  const bool few_taps = th->xsize_max <= 7 && tw->xsize_max <= 7;
  if (few_taps && !(flags & AA_FLAG_FORCE_STREAM)) {
    // mild vertical downsampling (1x..1.6x fewer rows): the band-walking variant; otherwise one tile per CTA
    if (oH <= H && H * 5 <= oH * 8) {
      rc = launch_band(in, in_dtype, lin, out, lout, fwd_axis(th), fwd_axis(tw), th->xsize_max, tw->xsize_max, epi, stream);
      if (rc != AA_ERR_UNSUPPORTED) return rc;
    }
    rc = launch_tile(in, in_dtype, lin, out, lout, fwd_axis(th), fwd_axis(tw), th->xsize_max, tw->xsize_max, epi, stream);
    if (rc != AA_ERR_UNSUPPORTED) return rc;
  }
  return launch_stream(in, in_dtype, lin, out, lout, th, tw, H, W, oH, oW, flags, epi, stream);
}

int two_pass(const aa_tensor_desc* in, const aa_tensor_desc* out, const Layout& lin, const Layout& lout, AxisTables* th, AxisTables* tw,
             int filter, int align, uint32_t flags, const OutEpi& epi, cudaStream_t stream) {
  if (epi.planar) return fail(AA_ERR_UNSUPPORTED, "two-pass: planar epilogue not supported");
  int rc;
  // identities H -> H and oW -> oW: the box filter at scale 1 (window = the pixel itself, weight exactly 1).  The
  // triangle / cubic tables at scale 1 would also be exact copies for finite data, but their windows hold zero-weight
  // neighbours, and 0 * NaN there spreads a non-finite pixel along the axis the pass is not supposed to touch (found by
  // scripts/fuzz_parity.py; the reference's two passes each work on one axis only, aa_interpolation_impl.h:655-679)
  (void)filter; (void)align;
  std::shared_ptr<AxisTables> ih, iw;
  if ((rc = get_axis_tables(in->device, in->h, in->h, AA_FILTER_BOX, 0, AA_F32, 0.0, stream, &ih)) != AA_OK) return rc;
  if ((rc = get_axis_tables(in->device, out->w, out->w, AA_FILTER_BOX, 0, AA_F32, 0.0, stream, &iw)) != AA_OK) return rc;
  // intermediate [n, c, H, oW] float32 in the input's memory format, dense
  Layout lt = lin;
  const int64_t row = out->w * lin.Ci;
  lt.stride_h = row;
  if (lin.Cp > 1) { lt.stride_p = in->h * row; lt.stride_n = lt.stride_p * lin.Cp; }
  else { lt.stride_p = 0; lt.stride_n = in->h * row; }
  const size_t bytes = sizeof(float) * (size_t)in->n * in->c * in->h * out->w;
  void* tmp = nullptr;
  AA_CUDA_TRY(cudaMallocAsync(&tmp, bytes, stream));
  rc = fused_dispatch(in->data, in->dtype, lin, tmp, lt, ih.get(), tw, in->h, in->w, in->h, out->w, flags & ~AA_FLAG_VMMA, OutEpi(), stream);
  if (rc == AA_OK) rc = fused_dispatch(tmp, AA_F32, lt, out->data, lout, th, iw.get(), in->h, out->w, out->h, out->w, flags & ~AA_FLAG_VMMA, epi, stream);
  const cudaError_t e = cudaFreeAsync(tmp, stream);
  if (rc == AA_OK && e != cudaSuccess) return cuda_fail(e, "cudaFreeAsync");
  return rc;
}

int forward_impl(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align, uint32_t flags,
                 cudaStream_t stream, const aa_epilogue* ex = nullptr, const aa_scales* sc = nullptr) {
  int rc;
  const RedoScope redo_scope(!(flags & AA_FLAG_ASSUME_FINITE));
  if ((rc = check_desc(in, "input")) != AA_OK) return rc;
  if ((rc = check_desc(out, "output")) != AA_OK) return rc;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  if (in->n != out->n || in->c != out->c) return fail(AA_ERR_INVALID, "input and output must agree in n and c");
  if (in->device != out->device) return fail(AA_ERR_INVALID, "input and output must live on the same device");
  if (in->dtype > AA_F64) return fail(AA_ERR_INVALID, "input dtype must be u8, f32 or f64");
  const int tdtype = in->dtype == AA_F64 ? AA_F64 : AA_F32;
  OutEpi epi;
  epi.round = (flags & AA_FLAG_ROUND_NEAREST) ? 1 : 0;
  if (tdtype == AA_F32) {
    if (out->dtype == AA_U8) epi.kind = 1;
    else if (ex && out->dtype == AA_F16) epi.kind = 2;
    else if (ex && out->dtype == AA_BF16) epi.kind = 3;
  }
  if (out->dtype != tdtype && epi.kind == 0)
    return fail(AA_ERR_INVALID, "output dtype must be f32 (or u8 with the fused clamp/round epilogue; f16/bf16 through "
                                "aa_resize_forward_ex) for u8/f32 inputs and f64 for f64 inputs");
  if (ex && ex->normalize) {
    if (tdtype != AA_F32) return fail(AA_ERR_UNSUPPORTED, "normalisation epilogue: u8/f32 inputs only");
    if (in->c > 4) return fail(AA_ERR_UNSUPPORTED, "normalisation epilogue: at most 4 channels");
    epi.norm = 1;
    for (int i = 0; i < 4; i++) { epi.scale[i] = ex->scale[i]; epi.bias[i] = ex->bias[i]; }
  }
  if (in->n == 0) return AA_OK;  // empty batch is allowed (aa_interpolation_impl.h:747-750)
  Layout lin, lout;
  bool in_cl = false, out_cl = false;
  if ((rc = classify_layout(*in, /*prefer_cl=*/false, &lin, &in_cl)) != AA_OK) return rc;
  if ((rc = classify_layout(*out, in_cl, &lout, &out_cl)) != AA_OK) return rc;
  if (in_cl != out_cl) {
    // ambiguous input (e.g. c == 1): retry with the output's format
    if ((rc = classify_layout(*in, out_cl, &lin, &in_cl)) != AA_OK) return rc;
  }
  if (in_cl != out_cl) {
    // decode-adjacent case: channels_last (HWC) input -> channels_first (planar) output, fused into the stores
    if (!(ex && in_cl && !out_cl && tdtype == AA_F32))
      return fail(AA_ERR_UNSUPPORTED, "input and output must use the same memory format (channels_last -> channels_first is "
                                      "available through aa_resize_forward_ex)");
    if (out->stride_c >= (1ll << 31) / (out->c > 0 ? out->c : 1)) return fail(AA_ERR_UNSUPPORTED, "planar output: plane stride too large");
    epi.planar = 1;
    epi.stride_c = (int)out->stride_c;
    lout = Layout();
    lout.planes = out->n; lout.Cp = 1; lout.Ci = (int)out->c; lout.stride_n = out->stride_n; lout.stride_p = 0;
    lout.stride_h = (out->h == 1) ? out->w : out->stride_h;
  }
  if (epi.norm && !in_cl && in->c > 1) {
    // the kernels take the channel of scale[c] / bias[c] from the interleaved column (channels_last); in a channels_first
    // tensor every plane would get channel 0's.  One call per channel plane, its own scale / bias in slot 0.
    auto es = [](int dt) { return (int64_t)(dt == AA_U8 ? 1 : (dt == AA_F16 || dt == AA_BF16) ? 2 : (dt == AA_F32 ? 4 : 8)); };
    for (int64_t c = 0; c < in->c; c++) {
      aa_tensor_desc di = *in, dd = *out;
      di.c = dd.c = 1;
      di.data = (char*)in->data + c * in->stride_c * es(in->dtype);
      dd.data = (char*)out->data + c * out->stride_c * es(out->dtype);
      aa_epilogue e1 = *ex;
      e1.scale[0] = ex->scale[c];
      e1.bias[0] = ex->bias[c];
      if ((rc = forward_impl(&di, &dd, filter, align, flags, stream, &e1, sc)) != AA_OK) return rc;
    }
    return AA_OK;
  }
  DeviceGuard g(in->device);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  std::shared_ptr<AxisTables> th, tw;
  if ((rc = get_axis_tables(in->device, in->h, out->h, filter, align, tdtype, sc ? sc->scale_h : 0.0, stream, &th)) != AA_OK) return rc;
  if ((rc = get_axis_tables(in->device, in->w, out->w, filter, align, tdtype, sc ? sc->scale_w : 0.0, stream, &tw)) != AA_OK) return rc;
  if ((flags & AA_FLAG_STRICT_NONFINITE) && in->dtype != AA_U8) flags |= AA_FLAG_FORCE_GENERAL;
  if (!(flags & AA_FLAG_FORCE_GENERAL) && tdtype == AA_F32) {
    rc = fused_dispatch(in->data, in->dtype, lin, out->data, lout, th.get(), tw.get(), in->h, in->w, out->h, out->w, flags, epi, stream);
    if (rc != AA_ERR_UNSUPPORTED || (flags & (AA_FLAG_FORCE_STREAM | AA_FLAG_VMMA))) return rc;
    // No fused kernel takes this shape (typically: upsampling in H, many-tap downsampling in W).  Two launches with
    // an intermediate, the reference's own structure (W pass into a temp, then H pass: aa_interpolation_impl.h:655-679),
    // each through a fused kernel with the identity on the other axis (one tap of weight 1: exact).
    rc = two_pass(in, out, lin, lout, th.get(), tw.get(), filter, align, flags, epi, stream);
    if (rc != AA_ERR_UNSUPPORTED) return rc;
  } else if (flags & AA_FLAG_FORCE_STREAM) {
    return fail(AA_ERR_UNSUPPORTED, "stream path: f32/u8 only");
  }
  return launch_general(in->data, in->dtype, lin, out->data, out->dtype, lout, fwd_axis(th.get()), fwd_axis(tw.get()),
                        /*exact=*/true, epi, stream);
}

int backward_check(const aa_tensor_desc* gout, const aa_tensor_desc* gin, Layout* lo, Layout* li) {
  int rc;
  if ((rc = check_desc(gout, "grad_output")) != AA_OK) return rc;
  if ((rc = check_desc(gin, "grad_input")) != AA_OK) return rc;
  if (gout->n != gin->n || gout->c != gin->c) return fail(AA_ERR_INVALID, "grad_output and grad_input must agree in n and c");
  if (gout->device != gin->device) return fail(AA_ERR_INVALID, "grad tensors must live on the same device");
  if ((gout->dtype != AA_F32 && gout->dtype != AA_F64) || gout->dtype != gin->dtype)
    return fail(AA_ERR_INVALID, "backward: f32 or f64, same dtype on both sides");
  bool o_cl = false, i_cl = false;
  if ((rc = classify_layout(*gout, false, lo, &o_cl)) != AA_OK) return rc;
  if ((rc = classify_layout(*gin, o_cl, li, &i_cl)) != AA_OK) return rc;
  if (o_cl != i_cl) {
    if ((rc = classify_layout(*gout, i_cl, lo, &o_cl)) != AA_OK) return rc;
    if (o_cl != i_cl) return fail(AA_ERR_UNSUPPORTED, "grad_output and grad_input must use the same memory format");
  }
  return AA_OK;
}

}  // namespace
}  // namespace aa

using namespace aa;

extern "C" {

int aa_abi_version(void) { return AA_RESIZE_ABI_VERSION; }
const char* aa_last_error(void) { return g_err.c_str(); }

int64_t aa_launch_count(int reset) {
  int64_t v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

int aa_interp_size(int64_t in_size, int64_t out_size, int filter, int align_corners, int dtype, int32_t* k) {
  int rc;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  if (!k || in_size <= 0 || out_size <= 0) return fail(AA_ERR_INVALID, "aa_interp_size: bad arguments");
  *k = host_interp_size(in_size, out_size, filter, align_corners, dtype == AA_F64 ? AA_F64 : AA_F32);
  return AA_OK;
}

int aa_host_tables(int64_t in_size, int64_t out_size, int filter, int align_corners, int dtype, double scale_factor,
                   int64_t* xmin, int64_t* xsize) {
  int rc;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  if (!xmin || !xsize || in_size <= 0 || out_size <= 0 || in_size >= (1ll << 31) || out_size >= (1ll << 31))
    return fail(AA_ERR_INVALID, "aa_host_tables: bad arguments");
  std::vector<int32_t> a((size_t)out_size), b((size_t)out_size);
  host_int_tables(in_size, out_size, filter, align_corners ? 1 : 0, dtype == AA_F64 ? AA_F64 : AA_F32,
                  (align_corners || !(scale_factor > 0.0)) ? 0.0 : scale_factor, a.data(), b.data());
  for (int64_t i = 0; i < out_size; i++) { xmin[i] = a[(size_t)i]; xsize[i] = b[(size_t)i]; }
  return AA_OK;
}

int aa_build_tables(int64_t in_size, int64_t out_size, int filter, int align_corners, int dtype, int device,
                    aa_tables_desc* dst, void* cuda_stream) {
  return aa_build_tables_sf(in_size, out_size, filter, align_corners, dtype, 0.0, device, dst, cuda_stream);
}

int aa_build_tables_sf(int64_t in_size, int64_t out_size, int filter, int align_corners, int dtype, double scale_factor,
                       int device, aa_tables_desc* dst, void* cuda_stream) {
  int rc;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  if (!dst || !dst->xmin || !dst->xsize || !dst->weights) return fail(AA_ERR_INVALID, "aa_build_tables: null destination");
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  DeviceGuard g(device);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  std::shared_ptr<AxisTables> t;
  const int td = dtype == AA_F64 ? AA_F64 : AA_F32;
  if ((rc = get_axis_tables(device, in_size, out_size, filter, align_corners, td, scale_factor, stream, &t)) != AA_OK) return rc;
  const int NT = 256;
  widen_i32_i64<<<(unsigned)((out_size + NT - 1) / NT), NT, 0, stream>>>(t->xmin, dst->xmin, out_size);
  AA_LAUNCH_CHECK("widen xmin");
  widen_i32_i64<<<(unsigned)((out_size + NT - 1) / NT), NT, 0, stream>>>(t->xsize, dst->xsize, out_size);
  AA_LAUNCH_CHECK("widen xsize");
  AA_CUDA_TRY(cudaMemcpyAsync(dst->weights, t->w, (size_t)(td == AA_F64 ? 8 : 4) * out_size * t->K,
                              cudaMemcpyDeviceToDevice, stream));
  dst->interp_size = t->K;
  return AA_OK;
}

int aa_warm_tables(int64_t in_h, int64_t in_w, int64_t out_h, int64_t out_w, int filter, int align_corners, int dtype,
                   int device, void* cuda_stream) {
  int rc;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  DeviceGuard g(device);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  std::shared_ptr<AxisTables> th, tw;
  const int td = dtype == AA_F64 ? AA_F64 : AA_F32;
  if ((rc = get_axis_tables(device, in_h, out_h, filter, align_corners, td, 0.0, stream, &th)) != AA_OK) return rc;
  if ((rc = get_axis_tables(device, in_w, out_w, filter, align_corners, td, 0.0, stream, &tw)) != AA_OK) return rc;
  if (td == AA_F32) {
    // the derived tables of every path a later forward / backward call of this shape may take
    if (th->kt_max <= 6) {
      rc = ensure_slot_tables(th.get(), th->kt_max <= 3 ? 3 : th->kt_max, stream);
      if (rc != AA_OK && rc != AA_ERR_UNSUPPORTED) return rc;
    }
    if (th->xsize_max <= 6) {
      rc = ensure_slot_tables_adj(th.get(), th->xsize_max <= 3 ? 3 : th->xsize_max, stream);
      if (rc != AA_OK && rc != AA_ERR_UNSUPPORTED) return rc;
    }
    if (dtype == AA_U8 && vmma_auto(th.get(), tw.get())) {
      rc = vmma_warm(th.get(), stream);
      if (rc != AA_OK && rc != AA_ERR_UNSUPPORTED) return rc;
    }
    if (dtype != AA_U8) {  // float inputs: the stream's list of regions to redo tap-exactly (aa_redo.cu)
      RedoList* rl = nullptr;
      if ((rc = redo_list(device, stream, &rl)) != AA_OK) return rc;
    }
  }
  // after this the tables are complete for every stream (and for CUDA-graph capture)
  AA_CUDA_TRY(cudaStreamSynchronize(stream));
  return AA_OK;
}

int aa_clear_table_cache(void) { return clear_table_cache(); }

int aa_check_device(int device) {
  if (device < 0 || device >= 64) return fail(AA_ERR_INVALID, "bad device ordinal");
  DeviceGuard g(device);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  return vmma_check_watchdog(device);
}

int aa_debug_counters(int device, uint64_t* counters16, int reset) {
  if (!counters16) return fail(AA_ERR_INVALID, "aa_debug_counters: null destination");
  DeviceGuard g(device);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  return vmma_read_counters(device, reinterpret_cast<unsigned long long*>(counters16), reset);
}

int aa_resize_forward(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                      void* cuda_stream) {
  return forward_impl(in, out, filter, align_corners, flags, (cudaStream_t)cuda_stream);
}

int aa_resize_forward_ex(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                         const aa_epilogue* epilogue, void* cuda_stream) {
  if (!epilogue) return fail(AA_ERR_INVALID, "aa_resize_forward_ex: epilogue is null (use aa_resize_forward)");
  return forward_impl(in, out, filter, align_corners, flags, (cudaStream_t)cuda_stream, epilogue);
}

int aa_resize_forward_sf(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align_corners,
                         const aa_scales* scales, uint32_t flags, void* cuda_stream) {
  return forward_impl(in, out, filter, align_corners, flags, (cudaStream_t)cuda_stream, nullptr, scales);
}

int aa_resize_forward_ragged(const aa_image_desc* images, int32_t count, int32_t dtype, int64_t channels, int32_t channels_last,
                             const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags, const aa_epilogue* epilogue,
                             void* cuda_stream, int32_t* launches_out) {
  int rc;
  if (launches_out) *launches_out = 0;
  if (count < 0 || (count > 0 && !images)) return fail(AA_ERR_INVALID, "aa_resize_forward_ragged: bad image list");
  if ((rc = check_desc(out, "output")) != AA_OK) return rc;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  if (out->n != count || out->c != channels) return fail(AA_ERR_INVALID, "output must be [count, channels, oH, oW]");
  if (dtype != AA_U8 && dtype != AA_F32 && dtype != AA_F64) return fail(AA_ERR_INVALID, "input dtype must be u8, f32 or f64");
  const int64_t es = dtype == AA_U8 ? 1 : (dtype == AA_F32 ? 4 : 8);
  for (int i = 0; i < count; i++) {
    if (!images[i].data || images[i].h <= 0 || images[i].w <= 0)
      return fail(AA_ERR_INVALID, "aa_resize_forward_ragged: image " + std::to_string(i) + " is empty");
    if (images[i].stride_h < images[i].w * (channels_last ? channels : 1))
      return fail(AA_ERR_INVALID, "aa_resize_forward_ragged: rows of image " + std::to_string(i) + " overlap");
  }
  // order: size class, then address
  std::vector<int> idx((size_t)count);
  for (int i = 0; i < count; i++) idx[(size_t)i] = i;
  auto cls = [&](int i) { const aa_image_desc& m = images[i]; return std::make_tuple(m.h, m.w, m.stride_h, channels_last ? (int64_t)1 : m.stride_c); };
  std::sort(idx.begin(), idx.end(), [&](int a, int b) {
    if (cls(a) != cls(b)) return cls(a) < cls(b);
    return a < b;
  });
  int launches = 0;
  for (size_t p = 0; p < idx.size();) {
    const int i0 = idx[p];
    // extend the run: same class, consecutive output slots, constant pointer distance
    size_t q = p + 1;
    int64_t delta = 0;
    while (q < idx.size() && cls(idx[q]) == cls(i0) && idx[q] == idx[q - 1] + 1) {
      const int64_t d = (const char*)images[idx[q]].data - (const char*)images[idx[q - 1]].data;
      if (d <= 0 || d % es) break;
      if (q == p + 1) delta = d;
      else if (d != delta) break;
      q++;
    }
    const aa_image_desc& m = images[i0];
    aa_tensor_desc di;
    di.data = m.data; di.dtype = dtype; di.device = out->device;
    di.n = (int64_t)(q - p); di.c = channels; di.h = m.h; di.w = m.w;
    di.stride_n = q - p > 1 ? delta / es : m.h * m.stride_h * (channels_last ? 1 : channels);
    di.stride_h = m.stride_h;
    if (channels_last) { di.stride_c = 1; di.stride_w = channels; }
    else { di.stride_c = m.stride_c; di.stride_w = 1; }
    aa_tensor_desc dd = *out;
    dd.n = di.n;
    dd.data = (char*)out->data + (size_t)i0 * out->stride_n * (out->dtype == AA_U8 ? 1 : (out->dtype == AA_F64 ? 8 : (out->dtype == AA_F32 ? 4 : 2)));
    rc = forward_impl(&di, &dd, filter, align_corners, flags, (cudaStream_t)cuda_stream, epilogue);
    if (rc != AA_OK) return rc;
    launches++;
    p = q;
  }
  if (launches_out) *launches_out = launches;
  return AA_OK;
}

static_assert(sizeof(aa_crop_ex) == 72, "aa_crop_ex layout (capi.CropEx and capi.crop_ex_dtype() mirror it)");
static_assert(sizeof(aa_fill) == 20, "aa_fill layout (capi.Fill mirrors it)");

// aa_resize_crops, aa_resize_crops_ex and aa_resize_crops_pad: every check before the first launch, then the crops kernel.
// `name` prefixes the messages.  With a fill (mode != AA_FILL_NONE) a window may lie anywhere its edges fit in int32.
static int resize_crops_impl(const char* name, const aa_image_desc* images, const aa_crop_ex* crops, int32_t count,
                             int32_t dtype, int64_t channels, int32_t channels_last, const aa_tensor_desc* out, int filter,
                             int align_corners, uint32_t flags, const aa_epilogue* epilogue, const aa_fill* fill,
                             void* cuda_stream, int32_t* launches_out) {
  int rc;
  const std::string nm = name;
  if (launches_out) *launches_out = 0;
  if (count < 0 || (count > 0 && (!images || !crops))) return fail(AA_ERR_INVALID, nm + ": null image or crop list");
  if ((rc = check_desc(out, "output")) != AA_OK) return rc;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  if (dtype == AA_F64) return fail(AA_ERR_UNSUPPORTED, nm + ": input dtype must be u8 or f32");
  if (dtype != AA_U8 && dtype != AA_F32) return fail(AA_ERR_INVALID, nm + ": input dtype must be u8 or f32");
  if (flags & (AA_FLAG_FORCE_STREAM | AA_FLAG_STREAM_TMA | AA_FLAG_STREAM_LDG | AA_FLAG_VMMA | AA_FLAG_FORCE_GENERAL))
    return fail(AA_ERR_UNSUPPORTED, nm + ": has one kernel; the path-forcing flags do not apply");
  if (channels < 1 || out->n != count || out->c != channels)
    return fail(AA_ERR_INVALID, nm + ": output must be [count, channels, oH, oW]");
  const int64_t ci = channels_last ? channels : 1;
  if (out->h >= (1ll << 31) || out->w * ci >= (1ll << 31)) return fail(AA_ERR_UNSUPPORTED, nm + ": output plane too large");
  if (!channels_last && channels > 65535) return fail(AA_ERR_UNSUPPORTED, nm + ": more than 65535 planar channels");
  if (fill && fill->mode != AA_FILL_NONE && fill->mode != AA_FILL_INPUT && fill->mode != AA_FILL_OUTPUT)
    return fail(AA_ERR_INVALID, nm + ": unknown fill mode " + std::to_string(fill->mode));
  const bool padded = fill && fill->mode != AA_FILL_NONE;
  if (padded && channels > 4) return fail(AA_ERR_UNSUPPORTED, nm + ": a fill takes at most 4 channels");
  OutEpi epi;
  epi.round = (flags & AA_FLAG_ROUND_NEAREST) ? 1 : 0;
  switch (out->dtype) {
    case AA_F32: epi.kind = 0; break;
    case AA_U8: epi.kind = 1; break;
    case AA_F16: epi.kind = 2; break;
    case AA_BF16: epi.kind = 3; break;
    default: return fail(AA_ERR_INVALID, nm + ": output dtype must be f32, u8, f16 or bf16");
  }
  if (epilogue && epilogue->normalize) {
    if (channels > 4) return fail(AA_ERR_UNSUPPORTED, "normalisation epilogue: at most 4 channels");
    epi.norm = 1;
    for (int i = 0; i < 4; i++) { epi.scale[i] = epilogue->scale[i]; epi.bias[i] = epilogue->bias[i]; }
  }
  // out: channels_first, or channels_last for an HWC input (the memory formats aa_resize_forward_ex accepts)
  Layout lout;
  bool out_cl = false;
  if ((rc = classify_layout(*out, channels_last != 0, &lout, &out_cl)) != AA_OK) return rc;
  if (out_cl && !channels_last && channels > 1)
    return fail(AA_ERR_UNSUPPORTED, nm + ": a planar input needs a channels_first output");
  for (int32_t i = 0; i < count; i++) {
    const aa_image_desc& m = images[i];
    const aa_crop_ex& b = crops[i];
    const std::string at = nm + ": crop " + std::to_string(i);
    if (!m.data || m.h <= 0 || m.w <= 0) return fail(AA_ERR_INVALID, at + ": image is empty");
    if (m.stride_h < m.w * ci) return fail(AA_ERR_INVALID, at + ": rows of the image overlap");
    if (b.top < 0 || b.left < 0 || b.height < 1 || b.width < 1 || b.height > m.h - b.top || b.width > m.w - b.left)
      return fail(AA_ERR_INVALID, at + ": box (top " + std::to_string(b.top) + ", left " + std::to_string(b.left) + ", height " +
                                      std::to_string(b.height) + ", width " + std::to_string(b.width) + ") is not inside its " +
                                      std::to_string(m.h) + "x" + std::to_string(m.w) + " image");
    if (b.resized_h < 1 || b.resized_w < 1)
      return fail(AA_ERR_INVALID, at + ": resized size " + std::to_string(b.resized_h) + "x" + std::to_string(b.resized_w) +
                                      " is empty");
    if (padded) {
      const int64_t lo = INT32_MIN, hi = INT32_MAX;
      if (b.crop_top < lo || b.crop_top > hi - out->h || b.crop_left < lo || b.crop_left > hi - out->w)
        return fail(AA_ERR_UNSUPPORTED, at + ": window (top " + std::to_string(b.crop_top) + ", left " +
                                            std::to_string(b.crop_left) + ", " + std::to_string(out->h) + "x" +
                                            std::to_string(out->w) + ") has an edge outside int32");
    } else if (b.crop_top < 0 || b.crop_left < 0 || b.crop_top > b.resized_h - out->h || b.crop_left > b.resized_w - out->w)
      return fail(AA_ERR_INVALID, at + ": window (top " + std::to_string(b.crop_top) + ", left " + std::to_string(b.crop_left) +
                                      ", " + std::to_string(out->h) + "x" + std::to_string(out->w) + ") is not inside the " +
                                      std::to_string(b.resized_h) + "x" + std::to_string(b.resized_w) + " resized image");
    if (b.flip & ~3) return fail(AA_ERR_INVALID, at + ": flip has bits other than 0 (horizontal) and 1 (vertical)");
    if (b.height >= (1ll << 31) || b.width >= (1ll << 31)) return fail(AA_ERR_UNSUPPORTED, at + ": box too large");
    if (b.resized_h >= (1ll << 31) || b.resized_w >= (1ll << 31)) return fail(AA_ERR_UNSUPPORTED, at + ": resized size too large");
    if (host_interp_size(b.height, b.resized_h, filter, align_corners, AA_F32) > kCropMaxTaps ||
        host_interp_size(b.width, b.resized_w, filter, align_corners, AA_F32) > kCropMaxTaps)
      return fail(AA_ERR_UNSUPPORTED, at + ": window longer than " + std::to_string(kCropMaxTaps) + " taps (downscale too large)");
  }
  if (count == 0) return AA_OK;
  DeviceGuard g(out->device);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  int32_t launches = 0;
  rc = launch_crops(name, images, crops, count, dtype, channels, channels_last, out, filter, align_corners ? 1 : 0, epi,
                    fill, (cudaStream_t)cuda_stream, &launches);
  if (launches_out) *launches_out = launches;
  return rc;
}

int aa_resize_crops_ex(const aa_image_desc* images, const aa_crop_ex* crops, int32_t count, int32_t dtype, int64_t channels,
                       int32_t channels_last, const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                       const aa_epilogue* epilogue, void* cuda_stream, int32_t* launches_out) {
  return resize_crops_impl("aa_resize_crops_ex", images, crops, count, dtype, channels, channels_last, out, filter,
                           align_corners, flags, epilogue, nullptr, cuda_stream, launches_out);
}

int aa_resize_crops_pad(const aa_image_desc* images, const aa_crop_ex* crops, int32_t count, int32_t dtype, int64_t channels,
                        int32_t channels_last, const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                        const aa_epilogue* epilogue, const aa_fill* fill, void* cuda_stream, int32_t* launches_out) {
  return resize_crops_impl("aa_resize_crops_pad", images, crops, count, dtype, channels, channels_last, out, filter,
                           align_corners, flags, epilogue, fill, cuda_stream, launches_out);
}

int aa_resize_crops(const aa_image_desc* images, const aa_crop* crops, int32_t count, int32_t dtype, int64_t channels,
                    int32_t channels_last, const aa_tensor_desc* out, int filter, int align_corners, uint32_t flags,
                    const aa_epilogue* epilogue, void* cuda_stream, int32_t* launches_out) {
  // each box resized to the output size, the window at the origin
  std::vector<aa_crop_ex> ex(crops && count > 0 ? (size_t)count : 0);
  for (size_t i = 0; i < ex.size(); i++) {
    const aa_crop& b = crops[i];
    ex[i] = aa_crop_ex{b.top, b.left, b.height, b.width, out ? out->h : 0, out ? out->w : 0, 0, 0, b.hflip ? 1 : 0};
  }
  return resize_crops_impl("aa_resize_crops", images, crops ? ex.data() : nullptr, count, dtype, channels, channels_last, out,
                           filter, align_corners, flags, epilogue, nullptr, cuda_stream, launches_out);
}

static int backward_impl(const aa_tensor_desc* gout, const aa_tensor_desc* gin, int filter, int align_corners, uint32_t flags,
                         void* cuda_stream, const aa_scales* sc) {
  int rc;
  const RedoScope redo_scope(!(flags & AA_FLAG_ASSUME_FINITE));
  Layout lo, li;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  if ((rc = backward_check(gout, gin, &lo, &li)) != AA_OK) return rc;
  if (gout->n == 0) return AA_OK;
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  DeviceGuard g(gout->device);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  std::shared_ptr<AxisTables> th, tw;
  if ((rc = get_axis_tables(gout->device, gin->h, gout->h, filter, align_corners, gout->dtype, sc ? sc->scale_h : 0.0, stream, &th)) != AA_OK) return rc;
  if ((rc = get_axis_tables(gout->device, gin->w, gout->w, filter, align_corners, gout->dtype, sc ? sc->scale_w : 0.0, stream, &tw)) != AA_OK) return rc;
  if (gout->dtype == AA_F32 && !(flags & AA_FLAG_FORCE_GENERAL)) {
    // few adjoint taps (the forward was a downsampling): write-bound tile kernel; many taps (the forward was
    // an upsampling): the backward is the input-bound direction -> streaming kernel with the roles swapped
    if (!(flags & AA_FLAG_FORCE_STREAM)) {
      rc = launch_tile(gout->data, gout->dtype, lo, gin->data, li, adj_axis(th.get()), adj_axis(tw.get()), th->kt_max,
                       tw->kt_max, OutEpi(), stream);
      if (rc != AA_ERR_UNSUPPORTED) return rc;
    }
    rc = launch_stream_adjoint(gout->data, lo, gin->data, li, th.get(), tw.get(), stream);
    if (rc != AA_ERR_UNSUPPORTED || (flags & AA_FLAG_FORCE_STREAM)) return rc;
  }
  return launch_general(gout->data, gout->dtype, lo, gin->data, gin->dtype, li, adj_axis(th.get()), adj_axis(tw.get()),
                        /*exact=*/false, OutEpi(), stream);
}

int aa_resize_backward(const aa_tensor_desc* gout, const aa_tensor_desc* gin, int filter, int align_corners, uint32_t flags,
                       void* cuda_stream) {
  return backward_impl(gout, gin, filter, align_corners, flags, cuda_stream, nullptr);
}
int aa_resize_backward_sf(const aa_tensor_desc* gout, const aa_tensor_desc* gin, int filter, int align_corners,
                          const aa_scales* scales, uint32_t flags, void* cuda_stream) {
  return backward_impl(gout, gin, filter, align_corners, flags, cuda_stream, scales);
}

int aa_resize_backward_nonaa_bilinear(const aa_tensor_desc* gout, const aa_tensor_desc* gin, int align_corners,
                                      void* cuda_stream) {
  int rc;
  Layout lo, li;
  if ((rc = backward_check(gout, gin, &lo, &li)) != AA_OK) return rc;
  if (gout->n == 0) return AA_OK;
  DeviceGuard g(gout->device);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  return launch_backward_nonaa(gout->data, gin->data, gout->dtype, lo, li, gout->h, gout->w, gin->h, gin->w, align_corners,
                               (cudaStream_t)cuda_stream);
}

// ---- host-buffer entries: chunked H2D -> resize -> D2H on rotating streams -------------------------
namespace {
struct HostCtx {
  static constexpr int NS = 3;
  std::mutex mu;  // one host call at a time per device
  cudaStream_t streams[NS] = {};
  void* din[NS] = {};
  void* dout[NS] = {};
  size_t cap_in = 0, cap_out = 0;
  bool init = false;
};
HostCtx g_host_ctx[64];

// dense NCHW (fmt 0) or NHWC (fmt 1) check for host buffers: the staging copies are flat memcpys
int dense_format(const aa_tensor_desc* t, int* fmt) {
  auto ok = [](int64_t size, int64_t stride, int64_t want) { return size == 1 || stride == want; };
  const bool cf = ok(t->w, t->stride_w, 1) && ok(t->h, t->stride_h, t->w) && ok(t->c, t->stride_c, t->h * t->w) &&
                  ok(t->n, t->stride_n, t->c * t->h * t->w);
  const bool cl = ok(t->c, t->stride_c, 1) && ok(t->w, t->stride_w, t->c) && ok(t->h, t->stride_h, t->w * t->c) &&
                  ok(t->n, t->stride_n, t->c * t->h * t->w);
  if (!cf && !cl) return AA_ERR_UNSUPPORTED;
  *fmt = (cf && cl) ? -1 : (cl ? 1 : 0);  // -1: both readings describe the same bytes
  return AA_OK;
}
void dense_strides(aa_tensor_desc* t, int fmt) {
  if (fmt == 1) { t->stride_c = 1; t->stride_w = t->c; t->stride_h = t->w * t->c; t->stride_n = t->h * t->w * t->c; }
  else { t->stride_w = 1; t->stride_h = t->w; t->stride_c = t->h * t->w; t->stride_n = t->c * t->h * t->w; }
}
size_t elem_size(int dtype) { return dtype == AA_U8 ? 1 : (dtype == AA_F32 ? 4 : 8); }

// Everything is validated BEFORE the first byte of the host buffers is touched.  -> memory format in *fmt
int host_validate(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int* fmt) {
  int rc;
  if ((rc = check_desc(in, "input")) != AA_OK) return rc;
  if ((rc = check_desc(out, "output")) != AA_OK) return rc;
  if ((rc = check_filter(filter)) != AA_OK) return rc;
  if (in->n != out->n || in->c != out->c) return fail(AA_ERR_INVALID, "input and output must agree in n and c");
  if (in->dtype > AA_F64) return fail(AA_ERR_INVALID, "input dtype must be u8, f32 or f64");
  if (out->dtype > AA_F64) return fail(AA_ERR_UNSUPPORTED, "host path: u8/f32/f64 outputs only");
  const int tdtype = in->dtype == AA_F64 ? AA_F64 : AA_F32;
  if (out->dtype != tdtype && !(out->dtype == AA_U8 && tdtype == AA_F32))
    return fail(AA_ERR_INVALID, "output dtype must be f32 (or u8) for u8/f32 inputs and f64 for f64 inputs");
  int ifmt = 0, ofmt = 0;
  if (dense_format(in, &ifmt) != AA_OK || dense_format(out, &ofmt) != AA_OK)
    return fail(AA_ERR_UNSUPPORTED, "host path needs fully dense NCHW or NHWC buffers (no padded rows, slices or views)");
  if (ifmt >= 0 && ofmt >= 0 && ifmt != ofmt) return fail(AA_ERR_UNSUPPORTED, "input and output must use the same memory format");
  *fmt = ifmt >= 0 ? ifmt : (ofmt >= 0 ? ofmt : 0);
  return AA_OK;
}

// Enqueues images [n0, n1) of the (validated) host batch on device `dev`'s rotating streams.  Caller holds C.mu and has
// made `dev` current.  Nothing is synchronised here.
int host_enqueue(const aa_tensor_desc* in, const aa_tensor_desc* out, int64_t n0, int64_t n1, int filter, int align, uint32_t flags,
                 int fmt, int dev, HostCtx& C) {
  const size_t ies = elem_size(in->dtype), oes = elem_size(out->dtype);
  const size_t img_in = (size_t)in->c * in->h * in->w, img_out = (size_t)out->c * out->h * out->w;
  if (!C.init) {
    for (int i = 0; i < HostCtx::NS; i++) AA_CUDA_TRY(cudaStreamCreateWithFlags(&C.streams[i], cudaStreamNonBlocking));
    C.init = true;
  }
  const int64_t n = n1 - n0;
  // chunk = as many images as fit ~96 MiB of input, at least 1, at most n/NS rounded up
  int64_t per = (int64_t)((96ull << 20) / (img_in * ies));
  if (per < 1) per = 1;
  const int64_t even = (n + HostCtx::NS - 1) / HostCtx::NS;
  if (per > even) per = even;
  const size_t need_in = (size_t)per * img_in * ies, need_out = (size_t)per * img_out * oes;
  if (need_in > C.cap_in || need_out > C.cap_out) {
    for (int i = 0; i < HostCtx::NS; i++) {
      AA_CUDA_TRY(cudaStreamSynchronize(C.streams[i]));
      if (C.din[i]) cudaFree(C.din[i]);
      if (C.dout[i]) cudaFree(C.dout[i]);
      C.din[i] = C.dout[i] = nullptr;
    }
    C.cap_in = C.cap_out = 0;
    for (int i = 0; i < HostCtx::NS; i++) {
      AA_CUDA_TRY(cudaMalloc(&C.din[i], need_in));
      AA_CUDA_TRY(cudaMalloc(&C.dout[i], need_out));
    }
    C.cap_in = need_in;
    C.cap_out = need_out;
  }
  // the staging buffers are dense by construction: their descs are rebuilt, never copied from the caller's strides
  aa_tensor_desc di = *in, dd_out = *out;
  di.device = dd_out.device = dev;
  dense_strides(&di, fmt);
  dense_strides(&dd_out, fmt);
  int64_t done = n0;
  for (int i = 0; done < n1; i++) {
    const int s = i % HostCtx::NS;
    const int64_t nb = std::min<int64_t>(per, n1 - done);
    di.data = C.din[s]; di.n = nb;
    dd_out.data = C.dout[s]; dd_out.n = nb;
    AA_CUDA_TRY(cudaMemcpyAsync(C.din[s], (const char*)in->data + (size_t)done * img_in * ies, (size_t)nb * img_in * ies,
                                cudaMemcpyHostToDevice, C.streams[s]));
    int rc = forward_impl(&di, &dd_out, filter, align, flags, C.streams[s]);
    if (rc != AA_OK) return rc;
    AA_CUDA_TRY(cudaMemcpyAsync((char*)out->data + (size_t)done * img_out * oes, C.dout[s], (size_t)nb * img_out * oes,
                                cudaMemcpyDeviceToHost, C.streams[s]));
    done += nb;
  }
  return AA_OK;
}

// Success or failure: nothing of the call may still be writing `out` (or reading `in`) when it returns.
int host_drain(int dev, HostCtx& C, int rc) {
  const std::string err = rc != AA_OK ? g_err : std::string();
  for (int i = 0; i < HostCtx::NS; i++) {
    if (!C.streams[i]) continue;
    const cudaError_t e = cudaStreamSynchronize(C.streams[i]);
    if (e != cudaSuccess && rc == AA_OK) rc = cuda_fail(e, "cudaStreamSynchronize");
  }
  if (rc != AA_OK) {
    if (!err.empty()) g_err = err;
    return rc;
  }
  return vmma_check_watchdog(dev);
}
}  // namespace

int aa_resize_forward_host(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align_corners,
                           uint32_t flags) {
  int rc, fmt = 0;
  if ((rc = host_validate(in, out, filter, &fmt)) != AA_OK) return rc;
  if (in->n == 0) return AA_OK;
  const int dev = in->device;
  if (dev < 0 || dev >= 64) return fail(AA_ERR_INVALID, "bad device ordinal");
  DeviceGuard g(dev);
  if (!g.ok) return cuda_fail(g.err, "cudaSetDevice");
  HostCtx& C = g_host_ctx[dev];
  std::lock_guard<std::mutex> lock(C.mu);
  rc = host_enqueue(in, out, 0, in->n, filter, align_corners, flags, fmt, dev, C);
  return host_drain(dev, C, rc);
}

int aa_resize_forward_host_multi(const aa_tensor_desc* in, const aa_tensor_desc* out, int filter, int align_corners,
                                 uint32_t flags, const int32_t* devices, int32_t n_devices) {
  int rc, fmt = 0;
  if ((rc = host_validate(in, out, filter, &fmt)) != AA_OK) return rc;
  int devs[64];
  int nd = 0;
  if (!devices || n_devices <= 0) {
    int cnt = 0;
    AA_CUDA_TRY(cudaGetDeviceCount(&cnt));
    for (int i = 0; i < cnt && i < 64; i++) devs[nd++] = i;
  } else {
    if (n_devices > 64) return fail(AA_ERR_INVALID, "too many devices");
    for (int i = 0; i < n_devices; i++) {
      if (devices[i] < 0 || devices[i] >= 64) return fail(AA_ERR_INVALID, "bad device ordinal");
      for (int j = 0; j < i; j++) if (devices[j] == devices[i]) return fail(AA_ERR_INVALID, "duplicate device ordinal");
      devs[nd++] = devices[i];
    }
  }
  if (nd == 0) return fail(AA_ERR_CUDA, "no CUDA device");
  if (in->n == 0) return AA_OK;
  // contiguous shards of ceil(n / devices) images (SURVEY 8(e)); every device gets its own stream set, staging buffers
  // and table cache entries; all devices are enqueued first, then all are drained
  const int64_t per = (in->n + nd - 1) / nd;
  int prev = -1;
  cudaGetDevice(&prev);
  int first_rc = AA_OK;
  std::string first_err;
  int locked = 0;
  for (int k = 0; k < nd; k++, locked++) {
    g_host_ctx[devs[k]].mu.lock();
    const int64_t n0 = std::min<int64_t>(in->n, per * k), n1 = std::min<int64_t>(in->n, per * (k + 1));
    if (first_rc != AA_OK || n0 >= n1) continue;
    cudaError_t e = cudaSetDevice(devs[k]);
    rc = e == cudaSuccess ? host_enqueue(in, out, n0, n1, filter, align_corners, flags, fmt, devs[k], g_host_ctx[devs[k]])
                          : cuda_fail(e, "cudaSetDevice");
    if (rc != AA_OK) { first_rc = rc; first_err = g_err; }
  }
  for (int k = 0; k < locked; k++) {
    if (cudaSetDevice(devs[k]) == cudaSuccess) {
      rc = host_drain(devs[k], g_host_ctx[devs[k]], AA_OK);
      if (rc != AA_OK && first_rc == AA_OK) { first_rc = rc; first_err = g_err; }
    }
    g_host_ctx[devs[k]].mu.unlock();
  }
  if (prev >= 0) cudaSetDevice(prev);
  if (first_rc != AA_OK) g_err = first_err;
  return first_rc;
}

}  // extern "C"

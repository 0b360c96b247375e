// aa_common.cuh -- shared declarations of the sm_100a anti-aliased resize library.
// Internal header: nothing here crosses the C ABI (include/aa_resize.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/aa_resize.h"

namespace aa {

// ---- error plumbing (thread-local message, negative status codes) --------------------------
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);
void count_launch(int n = 1);

#define AA_CUDA_TRY(expr)                                        \
  do {                                                           \
    cudaError_t _e = (expr);                                     \
    if (_e != cudaSuccess) return ::aa::cuda_fail(_e, #expr);    \
  } while (0)

#define AA_LAUNCH_CHECK(what)                                    \
  do {                                                           \
    ::aa::count_launch();                                        \
    cudaError_t _e = cudaGetLastError();                         \
    if (_e != cudaSuccess) return ::aa::cuda_fail(_e, what);     \
  } while (0)

// ---- per-axis tables -------------------------------------------------------------------------
// Forward tables follow HelperInterpBase::_compute_indices_weights_aa
// (/root/reference/step_two_dot_two/aa_interpolation_impl.h:194-281): for output index o the window
// is input [xmin[o], xmin[o]+xsize[o]) with weights w[o*K + j].
// Adjoint tables are the transpose: for input index x the outputs whose window covers x are the
// contiguous range [omin[x], omin[x]+osize[x]) (xmin and xmin+xsize are non-decreasing in o) and
// wT[x*KT + k] = w[(omin[x]+k)*K + (x - xmin[omin[x]+k])].
struct AxisTables {
  // key
  int device = 0;
  int64_t in = 0, out = 0;
  int filter = 0, align = 0;
  int dtype = AA_F32;  // AA_F32 or AA_F64: scalar_t of the table arithmetic
  double user_scale = 0.0;  // caller-provided scale factor (0 = none: scale = in/out)
  // cache bookkeeping
  uint64_t id = 0;        // unique per built table: launch-plan caches key on it (never on the address)
  uint64_t last_use = 0;  // LRU clock
  cudaEvent_t ready = nullptr;        // recorded after the table kernels; null once known complete
  cudaStream_t build_stream = nullptr;
  std::mutex mu;          // guards the lazily built derived tables below (slot, slot_adj, vq)
  // host-side scalars (computed with the same IEEE operations as the device kernel)
  float scale_f = 0.f, support_f = 0.f;
  double scale_d = 0.0, support_d = 0.0;
  int K = 0;         // padded taps per output (:210)
  int KT = 0;        // adjoint row pitch (>= kt_max)
  int kt_max = 0;    // max number of outputs covering one input index
  int xsize_max = 0; // max window length
  int monotone = 1;  // verified: xmin and xmin+xsize non-decreasing
  // device buffers (one allocation, `block`)
  void* block = nullptr;
  int32_t* xmin = nullptr;   // [out]
  int32_t* xsize = nullptr;  // [out]
  void* w = nullptr;         // [out*K]  float | double
  int32_t* omin = nullptr;   // [in]
  int32_t* osize = nullptr;  // [in]
  void* wT = nullptr;        // [in*KT]  float | double
  // per-input-row records of the streaming kernel's vertical pass (float only; built on first use)
  int slot_A = 0;            // accumulators per element = max(3, kt_max)
  int slot_RS = 0;           // record stride in 32-bit words = roundup4(A+1)
  float* slot = nullptr;     // [in][RS]: wT[y][0..A) ordered by age (k-th oldest open output row), then
                             //           (first_flush_o | nflush<<24)
  // the same records for the ADJOINT direction (grad_out rows streamed, grad_in rows produced): per
  // forward-output row o, the forward weights w[o][0..A) belong to the open grad_in rows xmin[o]+k
  int slot_adj_A = 0, slot_adj_RS = 0;
  float* slot_adj = nullptr;  // [out][RS]
  // tensor-core vertical pass (aa_vmma.cu): the forward weights of each block of `oyb` output rows as a
  // [ksteps*32 input rows][128] int8 matrix (3 balanced base-256 digits per weight, 128-byte-swizzled rows)
  int8_t* vq = nullptr;       // [vq_noyb][vq_ksteps*32][128]
  float* vq_meta = nullptr;   // {c0, c1, c2, K0, (int) s}
  int vq_ksteps = 0, vq_noyb = 0, vq_oyb = 0;  // K steps per block, number of blocks, output rows per block (32 or 16)
  // host mirrors of the integer tables (for launch planning)
  std::vector<int32_t> h_xmin, h_xsize, h_omin, h_osize;
  ~AxisTables();
};

// Returns the cached tables, building them on `stream` on a miss (stream-ordered, no synchronisation; users on
// other streams are made to wait on the build's event).  The cache is an LRU of AA_TABLE_CACHE_MAX (256) entries.
int get_axis_tables(int device, int64_t in, int64_t out, int filter, int align, int dtype, double user_scale,
                    cudaStream_t stream, std::shared_ptr<AxisTables>* result);
void table_cache_stats(int64_t* entries, int64_t* hits, int64_t* misses, int64_t* evictions);
void host_int_tables(int64_t in, int64_t out, int filter, int align, int dtype, double user_scale, int32_t* xmin_o,
                     int32_t* xsize_o);
void tile_plan_clear();
// Makes sure t->slot exists for `A` accumulators (A in 3..6); launches one tiny kernel on first use.
int ensure_slot_tables(AxisTables* t, int A, cudaStream_t stream);
int ensure_slot_tables_adj(AxisTables* t, int A, cudaStream_t stream);
// Quantised weight matrices of the tensor-core vertical pass; AA_ERR_UNSUPPORTED when a block of `oyb` output rows
// spans more than max_ksteps*kstep input rows.
int ensure_vq_tables(AxisTables* t, int oyb_max, int kstep, int max_ksteps, cudaStream_t stream);
int clear_table_cache();
// Host-only K computation (no device), same arithmetic as the table kernel.
int host_interp_size(int64_t in, int64_t out, int filter, int align, int dtype, double user_scale = 0.0);
// The fp32 table scale of an axis without a caller scale factor (area_pixel_compute_scale<float>), as the table kernel gets it.
float host_scale_f32(int64_t in, int64_t out, int align);

// ---- layout --------------------------------------------------------------------------------
// Both supported memory formats are expressed as `planes` independent 2-D images whose rows are
// flat arrays of W*Ci elements with the channel interleaved at stride 1:
//   channels_first: planes = N*C, Ci = 1;   channels_last: planes = N, Ci = C.
struct Layout {
  int64_t planes = 0;  // number of independent 2-D planes
  int Cp = 1;          // planes per batch element (C for channels_first, 1 for channels_last)
  int Ci = 1;          // interleave factor along the flat row
  int64_t stride_n = 0, stride_p = 0;  // element strides: plane p -> (p / Cp)*stride_n + (p % Cp)*stride_p
  int64_t stride_h = 0;                // element stride between rows
};
// Classifies a tensor desc; returns AA_ERR_UNSUPPORTED for anything but dense-row NCHW/NHWC.
int classify_layout(const aa_tensor_desc& t, bool prefer_channels_last, Layout* out, bool* is_channels_last);

// ---- fused output epilogue --------------------------------------------------------------------
// kind 1 (uint8): clamp to [0,255] then truncate (what the reference's caller does: torch.clamp + .byte(),
// /root/reference/test.py:71-75) or, with AA_FLAG_ROUND_NEAREST, add 0.5 first (PIL's rounding).
// kinds 2/3 (fp16/bf16), `norm` (v*scale[c] + bias[c]) and `planar` (channels_first output from a
// channels_last input) make up the decode-adjacent epilogue of aa_resize_forward_ex (SURVEY 8(f) row 4).
struct OutEpi {
  int kind = 0;    // 0: float32, 1: uint8, 2: float16, 3: bfloat16
  int round = 0;   // uint8: round to nearest instead of truncating
  int planar = 0;  // 1: write channel planes (offset c*stride_c + ox) although rows are processed interleaved
  int norm = 0;    // 1: v = v*scale[c] + bias[c]
  int stride_c = 0;  // planar: elements between channel planes
  float scale[4] = {1.f, 1.f, 1.f, 1.f};
  float bias[4] = {0.f, 0.f, 0.f, 0.f};
  // offset of output column (ox, c) inside one output row / plane set, and the step to (ox+1, c)
  __host__ __device__ int coloff(int ox, int c, int Ci) const { return planar ? c * stride_c + ox : ox * Ci + c; }
  __host__ __device__ int colstep(int Ci) const { return planar ? 1 : Ci; }
  __host__ __device__ bool plain() const { return kind == 0 && !planar && !norm; }
  // the decode-adjacent features need the GEN=true kernel instantiations (kept out of the default kernels so
  // their register budgets are untouched)
  __host__ __device__ bool generic() const { return planar || norm || kind >= 2; }
};
}  // namespace aa
#ifdef __CUDACC__
#include <cuda_bf16.h>
#include <cuda_fp16.h>
namespace aa {
// Horizontal pass of the few-tap kernels (aa_tile.cu, aa_band.cu): n patch rows -> n rows of T for one flat
// output column.  pb points at the column's first tap in patch row 0, taps are CI elements apart (CI = 0:
// runtime interleave `ci`).  With a compile-time interleave the taps are immediate offsets of one row pointer,
// so a row costs KW x (LDS + FFMA) + one address update instead of KW address updates.
template <int KW, int CI, bool CHK>
__device__ __forceinline__ void aa_hpass_rows(const float* pb, int pcp, int ci, const float (&w)[KW], float* dst, int tpitch, int n, float2& chk) {
  const int step = CI ? CI : ci;
  int r = 0;
  // two rows per step: packed FFMA2 (two fp32 FMAs per issue slot, the column's weight as the scalar operand)
#pragma unroll 2
  for (; r + 2 <= n; r += 2) {
    const float* p = pb + r * pcp;
    float2 a = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < KW; k++) a = __ffma2_rn(make_float2(w[k], w[k]), make_float2(p[k * step], p[pcp + k * step]), a);
    if constexpr (CHK) chk = __ffma2_rn(a, make_float2(0.f, 0.f), chk);  // 0 * a stays 0 unless a holds a NaN/Inf
    dst[r * tpitch] = a.x;
    dst[(r + 1) * tpitch] = a.y;
  }
  if (r < n) {
    const float* p = pb + r * pcp;
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < KW; k++) a = fmaf(p[k * step], w[k], a);
    if constexpr (CHK) chk.x = fmaf(a, 0.f, chk.x);
    dst[r * tpitch] = a;
  }
}
// uint8 -> float without the conversion unit (I2F runs on the 16-lane XU pipe): PRMT drops the byte
// into the mantissa of 2^23 (0x4B0000bb == 8388608 + b exactly) and a packed FADD2 removes the bias of two
// elements at once (the pairs are the ones the FFMA2 of the vertical pass consumes).
__device__ __forceinline__ void aa_unpack4(uint32_t w, float* v) {
  const float2 nb = make_float2(-8388608.0f, -8388608.0f);
  const float2 lo = __fadd2_rn(make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540)),
                                           __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7541))), nb);
  const float2 hi = __fadd2_rn(make_float2(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7542)),
                                           __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7543))), nb);
  v[0] = lo.x; v[1] = lo.y; v[2] = hi.x; v[3] = hi.y;
}
// Vertical taps of the few-tap kernels: a += w * v for 4 adjacent columns (two FFMA2)
__device__ __forceinline__ void aa_fma4(float4& a, const float4& v, float w) {
  const float2 w2 = make_float2(w, w);
  const float2 lo = __ffma2_rn(w2, make_float2(v.x, v.y), make_float2(a.x, a.y));
  const float2 hi = __ffma2_rn(w2, make_float2(v.z, v.w), make_float2(a.z, a.w));
  a = make_float4(lo.x, lo.y, hi.x, hi.y);
}
// CHK: `chk` collects 0 * (every value written to T): non-zero (NaN) iff one of them was NaN/Inf.  Every output of the
// vertical pass is a finite combination of T values, so this is where the tile kernel looks for non-finite data: the
// horizontal pass writes fewer values than the vertical pass stores whenever the gather upsamples.
template <int KW, bool CHK = false>
__device__ __forceinline__ void aa_hpass(const float* pb, int pcp, int ci, const float (&w)[KW], float* dst, int tpitch, int n, float2& chk) {
  switch (ci) {  // warp-uniform
    case 1: aa_hpass_rows<KW, 1, CHK>(pb, pcp, ci, w, dst, tpitch, n, chk); break;
    case 3: aa_hpass_rows<KW, 3, CHK>(pb, pcp, ci, w, dst, tpitch, n, chk); break;
    case 4: aa_hpass_rows<KW, 4, CHK>(pb, pcp, ci, w, dst, tpitch, n, chk); break;
    default: aa_hpass_rows<KW, 0, CHK>(pb, pcp, ci, w, dst, tpitch, n, chk); break;
  }
}
template <int KW>
__device__ __forceinline__ void aa_hpass(const float* pb, int pcp, int ci, const float (&w)[KW], float* dst, int tpitch, int n) {
  float2 none = make_float2(0.f, 0.f);
  aa_hpass<KW, false>(pb, pcp, ci, w, dst, tpitch, n, none);
}
// exact unsigned division by a runtime constant (Granlund-Montgomery, branch-free): n / d for all n < 2^32
struct FastDiv {
  uint32_t mul, sh1, sh2, d;
  static FastDiv make(uint32_t d) {
    uint32_t l = 0;
    while ((1ull << l) < d) l++;
    FastDiv f;
    f.mul = (uint32_t)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
    f.sh1 = l < 1 ? l : 1;
    f.sh2 = l > 0 ? l - 1 : 0;
    f.d = d;
    return f;
  }
  __device__ __forceinline__ uint32_t div(uint32_t n) const {
    const uint32_t t = __umulhi(n, mul);
    return (t + ((n - t) >> sh1)) >> sh2;
  }
};

__device__ __forceinline__ unsigned int aa_to_u8(float v, int round) {
  v = fminf(fmaxf(v, 0.f), 255.f);
  return (unsigned int)(round ? v + 0.5f : v);
}
// element store through a base pointer whose element type depends on the epilogue; c = channel of the element.
// GEN=false knows only float32 / uint8 (the reference-facing surface); GEN=true adds normalisation and halves.
template <bool GEN>
__device__ __forceinline__ void aa_store(void* base, int64_t idx, float v, int c, const OutEpi& e) {
  if constexpr (!GEN) {
    if (e.kind == 1) reinterpret_cast<uint8_t*>(base)[idx] = (uint8_t)aa_to_u8(v, e.round);
    else reinterpret_cast<float*>(base)[idx] = v;
  } else {
    if (e.norm) v = fmaf(v, e.scale[c & 3], e.bias[c & 3]);
    switch (e.kind) {
      case 0: reinterpret_cast<float*>(base)[idx] = v; break;
      case 1: reinterpret_cast<uint8_t*>(base)[idx] = (uint8_t)aa_to_u8(v, e.round); break;
      case 2: reinterpret_cast<__half*>(base)[idx] = __float2half_rn(v); break;
      default: reinterpret_cast<__nv_bfloat16*>(base)[idx] = __float2bfloat16_rn(v); break;
    }
  }
}

// ---- non-finite inputs: exact re-evaluation of an output region ---------------------------------------------
// The reference touches the taps j < xsize of a window and nothing else (aa_interpolation_impl.h:73-85), so an
// output is NaN/Inf iff one of ITS taps is.  The fast float kernels also multiply a few zero-weight neighbours
// (unrolled tap loops, accumulators that are not open yet, the union window of a column pair): 0 * Inf = NaN would
// leak into outputs whose own window is finite.  Every fast kernel therefore checks what it stores, and a CTA that
// stored anything non-finite appends its region to a small per-stream list (RedoList).  A second, tiny kernel
// (aa_redo.cu) follows every such launch: it reads the list's counter and exits -- about a microsecond -- unless
// there are entries, which it re-evaluates with aa_exact_region: in-window taps only, horizontal then vertical like
// the reference, straight from global memory.  (The redo used to live at the end of the fast kernels themselves:
// even there, inlined or called, it cost the streaming kernel its load hoisting -- cfg2 0.88 -> 0.74 of peak -- and
// the few-tap kernels registers.)  Finite images pay the check and the empty launch; an image with a NaN pays for the
// regions that contain one.  uint8 inputs cannot be non-finite: no check, no second launch.
struct ExactTabs {
  const int32_t *h_start, *h_size, *w_start, *w_size;
  const float *h_w, *w_w;
  int h_pitch, w_pitch;
};
// first instruction of the fast float kernels: lets the drain kernel behind them (launched with programmatic stream
// serialization, aa_redo.cu) become resident early; it still waits for this grid to complete before it reads anything
__device__ __forceinline__ void aa_trigger_drain() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ bool aa_nonfinite(float v) { return !(fabsf(v) <= 3.402823466e38f); }
template <bool GEN, typename in_t>
__device__ __forceinline__ void aa_exact_region(const in_t* __restrict__ ip, int64_t in_sh, int Ci, ExactTabs T, void* out,
                                             int64_t op, int64_t out_sh, const OutEpi& epi, int oy0, int oy1, int of0, int of1,
                                             int tid, int nt) {
  const int nf = of1 - of0;
  const int total = (oy1 - oy0) * nf;
  for (int i = tid; i < total; i += nt) {
    const int r = i / nf, of = of0 + (i - r * nf), oy = oy0 + r;
    const int ox = of / Ci, c = of - ox * Ci;
    const int ys = T.h_start[oy], yn = T.h_size[oy], xs = T.w_start[ox], xn = T.w_size[ox];
    const float* wy = T.h_w + (int64_t)oy * T.h_pitch;
    const float* wx = T.w_w + (int64_t)ox * T.w_pitch;
    const in_t* p = ip + (int64_t)ys * in_sh + (int64_t)xs * Ci + c;
    float acc = 0.f;
    for (int ky = 0; ky < yn; ky++, p += in_sh) {
      float h = 0.f;
      for (int kx = 0; kx < xn; kx++) h = fmaf((float)p[kx * Ci], wx[kx], h);
      acc = fmaf(h, wy[ky], acc);
    }
    aa_store<GEN>(out, op + (int64_t)oy * out_sh + epi.coloff(ox, c, Ci), acc, c, epi);
  }
}
// The per-(device, stream) list the fast kernels append to and the redo kernel drains (aa_redo.cu).
constexpr int kRedoCap = 2040;  // 64 KB per list
struct RedoEntry {
  int64_t a, b;            // b < 0: rows [oy0, oy1) x flat columns [of0, of1) of plane a; else the streaming kernel's units [a, b)
  int oy0, oy1, of0, of1;
};
struct RedoList {
  unsigned int count, overflow, done, pad;  // overflow: more dirty regions than entries -> the whole output is redone
  RedoEntry e[kRedoCap];
};
__device__ __forceinline__ void redo_push(RedoList* L, int64_t a, int64_t b, int oy0, int oy1, int of0, int of1) {
  const unsigned int i = atomicAdd(&L->count, 1u);
  if (i < (unsigned int)kRedoCap) L->e[i] = RedoEntry{a, b, oy0, oy1, of0, of1};
  else L->overflow = 1u;
}
struct RedoParams {
  const void* in;  // float
  void* out;
  OutEpi epi;
  Layout lin, lout;
  int Ci;
  ExactTabs T;
  int out_h, out_wf;      // output rows, flat output columns
  int n_strips, strip_ox; // streaming kernel's unit decode (units entries only)
  RedoList* list;
};
// the calling stream's list (host bookkeeping once the device has a chunk of lists: aa_redo.cu)
int redo_list(int device, cudaStream_t stream, RedoList** out);
// the drain kernel, right behind the fast kernel on the same stream
int launch_redo(const RedoParams& R, int device, cudaStream_t stream);
void redo_clear();  // frees every list (aa_clear_table_cache)
bool redo_set_enabled(bool on);  // this thread's launches: returns the previous setting
struct RedoScope {                // AA_FLAG_ASSUME_FINITE: no drain launch for the calls made inside the scope
  bool was;
  explicit RedoScope(bool on) : was(redo_set_enabled(on)) {}
  ~RedoScope() { redo_set_enabled(was); }
};
}  // namespace aa
#endif
namespace aa {

// ---- kernels' host launchers ---------------------------------------------------------------
struct BandedAxis {  // one axis of a banded separable apply: out index i reads in [start[i], start[i]+size[i])
  const int32_t* start;
  const int32_t* size;
  const void* w;  // [n_out * pitch]
  int pitch;
  int64_t n_in, n_out;
  const int32_t* h_start;  // host mirrors of start/size (launch planning)
  const int32_t* h_size;
  uint64_t id;             // identity of the tables for the launch-plan caches (AxisTables::id * 2 + direction)
  int device;
};

// Launch-geometry cache of the few-tap kernels (aa_tile.cu, aa_band.cu): what the host derives by scanning the table
// mirrors (patch sizes, tile height, shared memory) is kept per (tables, interleave, kernel family), so a steady-state
// call is a map lookup + one launch, like the streaming kernel's plan cache.
struct GeomKey {
  uint64_t ah, aw;
  int tag;  // family | Ci << 8 | input dtype << 24 | generic epilogue << 28
  bool operator<(const GeomKey& o) const {
    if (ah != o.ah) return ah < o.ah;
    if (aw != o.aw) return aw < o.aw;
    return tag < o.tag;
  }
};
struct GeomPlan {
  int nc = 0;       // widest input patch (flat elements)
  int vr4 = 0;      // tile: 4-rows-per-step variant
  int ty = 0;       // chosen tile / chunk height (0: not eligible)
  int nr = 0;       // patch rows for that height
  size_t smem = 0;
};
bool geom_lookup(const GeomKey& k, GeomPlan* p);
void geom_store(const GeomKey& k, const GeomPlan& p);
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device) instead of per call
cudaError_t ensure_smem_attr_impl(const void* kern, int device, size_t smem);
template <typename K>
inline cudaError_t ensure_smem_attr(K kern, int device, size_t smem) {
  return ensure_smem_attr_impl(reinterpret_cast<const void*>(kern), device, smem);
}

// General gather-form tile kernel: out = Ah * in * Aw^T per plane, horizontal pass first.
// exact=true: separate multiply and add (bit-identical to the reference's C++), else FMA.
int launch_general(const void* in, int in_dtype, const Layout& lin, void* out, int out_dtype,
                   const Layout& lout, const BandedAxis& ah, const BandedAxis& aw, bool exact,
                   OutEpi epi, cudaStream_t stream);

// Tile kernel for gathers with few taps (backward of downsampling, forward upsampling): input patch
// in shared memory -> horizontal pass -> shared memory -> vertical pass -> 128-bit stores.  f32 out,
// f32/u8 in.  Returns AA_ERR_UNSUPPORTED when the patch would not fit so the caller can fall back.
// few taps, scale about 0.6x..1x (aa_band.cu): same contract as launch_tile
int launch_band(const void* in, int in_dtype, const Layout& lin, void* out, const Layout& lout,
                const BandedAxis& ah, const BandedAxis& aw, int kh_max, int kw_max, OutEpi epi, cudaStream_t stream);
int launch_tile(const void* in, int in_dtype, const Layout& lin, void* out, const Layout& lout,
                const BandedAxis& ah, const BandedAxis& aw, int kh_max, int kw_max, OutEpi epi, cudaStream_t stream);

// Streaming fused kernel (downsampling in H, any scale in W; f32/u8 in, f32/u8 out).  Returns
// AA_ERR_UNSUPPORTED when not eligible so the caller can fall back to launch_general.
int launch_stream(const void* in, int in_dtype, const Layout& lin, void* out, const Layout& lout,
                  AxisTables* th, AxisTables* tw, int64_t H, int64_t W, int64_t oH, int64_t oW,
                  uint32_t flags, OutEpi epi, cudaStream_t stream);

// The adjoint (grad_in = Wh^T g Ww) on the same streaming kernel: used when the FORWARD was an upsampling,
// i.e. the backward is the many-taps, input-bound direction.  AA_ERR_UNSUPPORTED when not eligible.
int launch_stream_adjoint(const void* gout, const Layout& lo, void* gin, const Layout& li, AxisTables* th, AxisTables* tw,
                          cudaStream_t stream);

// uint8 input, downsampling in H: vertical pass on the tensor cores (tcgen05 kind::i8 + TMA), horizontal pass as a gather
// (aa_vmma.cu).  AA_ERR_UNSUPPORTED when not eligible.
int launch_vmma(const void* in, const Layout& lin, void* out, const Layout& lout, AxisTables* th, AxisTables* tw, int64_t H,
                int64_t W, int64_t oH, int64_t oW, OutEpi epi, cudaStream_t stream);
int vmma_check_watchdog(int device);
int vmma_read_counters(int device, unsigned long long* out, int reset);
int vmma_warm(AxisTables* th, cudaStream_t stream);  // everything a later launch_vmma would allocate or synchronise for
void vmma_plan_clear();

// Batched resized crops (aa_crops.cu): arguments validated by aa_resize_crops / aa_resize_crops_ex / aa_resize_crops_pad
// (`name` prefixes the messages); ceil(count / kCropsPerLaunch) launches, counted into *launches.  The per-crop descriptors
// travel in the kernel parameters (56 bytes each).  `fill` NULL or AA_FILL_NONE: windows inside the resized images;
// otherwise the padded kernel variant.
constexpr int kCropsPerLaunch = 512;
constexpr int kCropMaxTaps = 65;  // largest interp_size (2*ceil(support)+1) of a crop axis: shared weight rows
int launch_crops(const char* name, const aa_image_desc* images, const aa_crop_ex* crops, int32_t count, int32_t dtype,
                 int64_t channels, int32_t channels_last, const aa_tensor_desc* out, int filter, int align, const OutEpi& epi,
                 const aa_fill* fill, cudaStream_t stream, int32_t* launches);

int launch_backward_nonaa(const void* gout, void* gin, int dtype, const Layout& lout, const Layout& lin,
                          int64_t oH, int64_t oW, int64_t H, int64_t W, int align, cudaStream_t stream);

}  // namespace aa

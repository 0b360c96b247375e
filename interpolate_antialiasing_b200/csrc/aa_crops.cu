// aa_crops.cu -- batched resized crops (aa_resize_crops, aa_resize_crops_ex, aa_resize_crops_pad): one box per crop, any
// box size, resized to its own size, one (oH, oW) window of that resized image stored per crop, one launch.
//
//   out[n, c, oy', ox'] = sum_y sum_x Wh_n[y0_n + oy, y] * Ww_n[x0_n + ox, x] * image_n[top_n + y, left_n + x, c]
//   oy' = vflip ? oH-1-oy : oy,  ox' = hflip ? oW-1-ox : ox
//
// Wh_n, Ww_n: the tables of box -> resized size; (y0_n, x0_n): the window origin in the resized image.  aa_resize_crops is
// the case resized = (oH, oW), origin 0, no vertical flip.  aa_resize_crops_pad with a fill runs the padded variant
// (aa_crops_pad_kernel): the window may reach past the resized image, and its outputs there store the fill value.
//
// Random boxes almost never share a size, so table caches and per-size launch plans do not pay here: every CTA computes
// the tables of its own tile (xmin, xsize and weights of its output rows and of its tile's pixel columns) into shared
// memory with aa_window_f32, the same device function as the K1 table kernel, and the per-crop parameters travel in the
// kernel parameters.  No allocation, no copy, no synchronisation: the call is CUDA-graph capturable as it stands.
//
// Arithmetic: the EXACT order of aa_general_kernel -- horizontal pass into shared T rounded to fp32, then the vertical
// pass with ascending taps, separate multiply and add -- so every output is bit-identical to aa_resize_forward_ex on the
// crop's view with AA_FLAG_FORCE_GENERAL (to the resized size, then sliced to the window).  Only the in-window taps inside
// the box are read, so NaN/Inf land exactly where the reference puts them without the drain kernel behind the fast float
// paths.
#include <algorithm>
#include <type_traits>

#include "aa_common.cuh"
#include "aa_window.cuh"

namespace aa {
namespace {

constexpr int TW = 64;           // flat output columns per tile
constexpr int TH = 32;           // output rows per tile
constexpr int NTY = 4;           // thread rows
constexpr int RPT = TH / NTY;    // output rows per thread
constexpr int RC = 32;           // input rows per chunk
constexpr int HPT = RC / NTY;    // horizontal-pass rows per thread per chunk
constexpr int KP = kCropMaxTaps; // weight row pitch in shared memory (odd: the columns of a warp hit distinct banks)

// One crop, 56 bytes.  src already points at the box's first element (top, left) of channel 0, offset in 64 bits.
struct CropDesc {
  const void* src;
  int64_t stride_h, stride_c;  // elements; stride_c: between channel planes (planar input)
  int32_t h, w;                // box size
  int32_t y0, x0;              // origin of the stored window in the resized image
  float scale_h, scale_w;      // fp32 table scales of the two axes (h_scale_f32 of box -> resized size)
  int16_t kh, kw;              // interp_size of the two axes (<= kCropMaxTaps)
  int32_t flip;                // bit 0: horizontal, bit 1: vertical
};
static_assert(sizeof(CropDesc) == 56, "CropDesc layout");

struct CropParams {
  void* out;
  OutEpi epi;
  int64_t out_sn, out_sc, out_sh, out_sw;  // output element strides
  int64_t first;                           // output slot of c[0]
  int oH, oW, Ci, filter, tiles_x;
  CropDesc c[kCropsPerLaunch];
};
// sm_100 takes up to 32764 bytes of kernel parameters (512 x 56 bytes of descriptors + the header)
static_assert(sizeof(CropParams) <= 32764, "kCropsPerLaunch too large for the kernel parameter space");

// One crop of the padded variant, also 56 bytes: it needs the resized size to tell which outputs lie inside the resized
// image, so the table scales make room for it and the kernel computes them from the box and resized sizes (the same single
// IEEE division as h_scale_f32); interp sizes (<= 65) and flip bits fit in a byte each.
struct PadDesc {
  const void* src;
  int64_t stride_h, stride_c;
  int32_t h, w;        // box size
  int32_t y0, x0;      // origin of the stored window in the resized image; may be negative or past its end
  int32_t rh, rw;      // resized size
  uint8_t kh, kw;      // interp_size of the two axes
  uint8_t flip;
};
static_assert(sizeof(PadDesc) == 56, "PadDesc layout");

struct PadParams {
  void* out;
  OutEpi epi;
  int64_t out_sn, out_sc, out_sh, out_sw;
  int64_t first;
  int oH, oW, Ci, filter, tiles_x;
  int align;
  OutEpi fill_epi;  // the store of the fill: epi (AA_FILL_INPUT) or epi without the affine map (AA_FILL_OUTPUT)
  float fill[4];    // per channel
  PadDesc c[kCropsPerLaunch];
};
static_assert(sizeof(PadParams) <= 32764, "kCropsPerLaunch too large for the kernel parameter space");

template <typename in_t>
__device__ __forceinline__ float ld_in(const in_t* p) { return (float)__ldg(p); }

// h_scale_f32 (aa_tables.cu) on the device: both conversions and the division round to nearest, as on the host
__device__ __forceinline__ float crop_scale_f32(int in, int out, int align) {
  if (align) return out > 1 ? __fdiv_rn((float)(in - 1), (float)(out - 1)) : 0.0f;
  return __fdiv_rn((float)in, (float)out);
}

// One CTA: a TH x TW tile of the flat output (pixel columns x interleaved channels) of one plane of one crop.
// PAD: only the tile's rows and pixel columns inside the resized image get tables and sums; every other output stores
// the fill, and a tile with none inside stores only the fill (no tables, no loads).
template <typename in_t, bool PAD, typename Params>
__device__ __forceinline__ void crops_tile(const Params& P) {
  __shared__ float Ts[RC][TW + 1];
  __shared__ float sWh[TH][KP];
  __shared__ float sWw[TW][KP];
  __shared__ int32_t sHs[TH], sHn[TH], sWs[TW], sWn[TW];
  const auto& D = P.c[blockIdx.z];
  const int tid = threadIdx.x, tx = tid % TW, ty = tid / TW;
  const int Ci = P.Ci;
  const int owf = P.oW * Ci;
  const int tile_x = (int)(blockIdx.x % (unsigned)P.tiles_x), tile_y = (int)(blockIdx.x / (unsigned)P.tiles_x);
  const int plane = blockIdx.y;  // channel plane of a planar input; 0 for an interleaved (HWC) one
  const int oy0 = tile_y * TH, of0 = tile_x * TW;
  const int nrows = min(TH, P.oH - oy0);
  const int px0 = of0 / Ci;
  const int npx = (min(of0 + TW, owf) - 1) / Ci - px0 + 1;

  // PAD: tile rows [lr0, lr1) and tile pixel columns [lc0, lc1) lie inside the resized image; both empty when either is
  int lr0 = 0, lr1 = nrows, lc0 = 0, lc1 = npx;
  if constexpr (PAD) {
    const long long ry = (long long)D.y0 + oy0, rx = (long long)D.x0 + px0;  // resized-image index of row / column 0
    lr0 = (int)min((long long)nrows, max(0ll, -ry));
    lr1 = (int)max((long long)lr0, min((long long)nrows, D.rh - ry));
    lc0 = (int)min((long long)npx, max(0ll, -rx));
    lc1 = (int)max((long long)lc0, min((long long)npx, D.rw - rx));
    if (lr0 == lr1 || lc0 == lc1) lr1 = lr0, lc1 = lc0;
    // ---- the tables of the rows and columns inside
    if (lr0 < lr1) {
      const float scale_h = crop_scale_f32(D.h, D.rh, P.align), scale_w = crop_scale_f32(D.w, D.rw, P.align);
      for (int k = tid; k < TH + TW; k += TW * NTY) {
        if (k < TH) {
          if (k >= lr0 && k < lr1) aa_window_f32(D.h, P.filter, scale_h, D.kh, D.y0 + oy0 + k, &sHs[k], &sHn[k], sWh[k]);
        } else if (k - TH >= lc0 && k - TH < lc1) {
          const int j = k - TH;
          aa_window_f32(D.w, P.filter, scale_w, D.kw, D.x0 + px0 + j, &sWs[j], &sWn[j], sWw[j]);
        }
      }
      __syncthreads();
    }
  } else {
    // ---- the tile's tables, K1 arithmetic, at the tile's indices in the resized image
    for (int k = tid; k < TH + TW; k += TW * NTY) {
      if (k < TH) {
        if (k < nrows) aa_window_f32(D.h, P.filter, D.scale_h, D.kh, D.y0 + oy0 + k, &sHs[k], &sHn[k], sWh[k]);
      } else if (k - TH < npx) {
        const int j = k - TH;
        aa_window_f32(D.w, P.filter, D.scale_w, D.kw, D.x0 + px0 + j, &sWs[j], &sWn[j], sWw[j]);
      }
    }
    __syncthreads();
  }

  const int of = of0 + tx;
  const bool col_ok = of < owf;
  int px = px0, c = 0, wst = 0, wsz = 0;
  bool col_in = col_ok;  // a column inside the resized image
  if (col_ok) {
    px = of / Ci;
    c = of - px * Ci;
    if constexpr (PAD) col_in = px - px0 >= lc0 && px - px0 < lc1;
    if (col_in) {
      wst = sWs[px - px0];
      wsz = sWn[px - px0];
    }
  }
  const float* wrow = sWw[px - px0];
  const in_t* icol = (const in_t*)D.src + plane * D.stride_c + (int64_t)wst * Ci + c;
  int hst[RPT], hsz[RPT];
  float acc[RPT];
#pragma unroll
  for (int r = 0; r < RPT; r++) {
    const int oyl = ty + r * NTY;
    acc[r] = 0.f;
    if (PAD ? oyl >= lr0 && oyl < lr1 : oyl < nrows) { hst[r] = sHs[oyl]; hsz[r] = sHn[oyl]; }
    else { hst[r] = 0; hsz[r] = 0; }
  }
  // box rows the tile needs (window starts and ends are non-decreasing in the output index)
  const int row_begin = PAD ? (lr0 < lr1 ? sHs[lr0] : 0) : sHs[0];
  const int row_end = PAD ? (lr0 < lr1 ? sHs[lr1 - 1] + sHn[lr1 - 1] : 0) : sHs[nrows - 1] + sHn[nrows - 1];

  for (int r0 = row_begin; r0 < row_end; r0 += RC) {
    // ---- horizontal pass of box rows [r0, r0+RC) for this tile's columns -> Ts (ascending taps, multiply then add)
    float t[HPT];
#pragma unroll
    for (int i = 0; i < HPT; i++) t[i] = 0.f;
    if (col_in) {
      for (int k = 0; k < wsz; k++) {
        const float wk = wrow[k];
        const in_t* src = icol + (int64_t)k * Ci;
#pragma unroll
        for (int i = 0; i < HPT; i++) {
          const int row = r0 + ty + i * NTY;
          if (row < row_end) t[i] = __fadd_rn(t[i], __fmul_rn(ld_in(src + (int64_t)row * D.stride_h), wk));
        }
      }
    }
#pragma unroll
    for (int i = 0; i < HPT; i++) Ts[ty + i * NTY][tx] = t[i];
    __syncthreads();
    // ---- vertical accumulation over this chunk, ascending rows
#pragma unroll
    for (int r = 0; r < RPT; r++) {
      const int a = hst[r] > r0 ? hst[r] : r0;
      const int e = min(hst[r] + hsz[r], r0 + RC);
      const float* hrow = sWh[ty + r * NTY];
      for (int row = a; row < e; row++) acc[r] = __fadd_rn(acc[r], __fmul_rn(Ts[row - r0][tx], hrow[row - hst[r]]));
    }
    __syncthreads();
  }
  if (col_ok) {
    const int ch = plane + c;  // one of the two is 0
    const int oxs = (D.flip & 1) ? P.oW - 1 - px : px;
    const bool vflip = D.flip & 2;
    const int64_t sh = vflip ? -P.out_sh : P.out_sh;
    const int64_t base = (P.first + blockIdx.z) * P.out_sn + ch * P.out_sc + oxs * P.out_sw +
                         (int64_t)(vflip ? P.oH - 1 - oy0 : oy0) * P.out_sh;
#pragma unroll
    for (int r = 0; r < RPT; r++) {
      const int oyl = ty + r * NTY;
      if (oyl < nrows) {
        if constexpr (PAD) {
          if (!col_in || oyl < lr0 || oyl >= lr1) {
            aa_store<true>(P.out, base + (int64_t)oyl * sh, P.fill[ch & 3], ch, P.fill_epi);
            continue;
          }
        }
        aa_store<true>(P.out, base + (int64_t)oyl * sh, acc[r], ch, P.epi);
      }
    }
  }
}

// 4 CTAs per SM (64 registers, 4 x 34 KB of shared memory): with no minimum given, ptxas still allocates 64 registers for
// the uint8 instantiation but spills; with the minimum it fits them without spilling.
template <typename in_t>
__global__ void __launch_bounds__(TW* NTY, 4) aa_crops_kernel(const __grid_constant__ CropParams P) {
  crops_tile<in_t, false>(P);
}
template <typename in_t>
__global__ void __launch_bounds__(TW* NTY, 4) aa_crops_pad_kernel(const __grid_constant__ PadParams P) {
  crops_tile<in_t, true>(P);
}

template <bool PAD>
int launch(const char* name, const aa_image_desc* images, const aa_crop_ex* crops, int32_t count, int32_t dtype,
           int64_t channels, int32_t channels_last, const aa_tensor_desc* out, int filter, int align, const OutEpi& epi,
           const aa_fill* fill, cudaStream_t stream, int32_t* launches) {
  using Params = std::conditional_t<PAD, PadParams, CropParams>;
  const int64_t es = dtype == AA_U8 ? 1 : 4;
  const int Ci = channels_last ? (int)channels : 1;
  const int64_t owf = out->w * Ci;
  const int64_t tiles_x = (owf + TW - 1) / TW, tiles_y = (out->h + TH - 1) / TH;
  if (tiles_x * tiles_y >= (1ll << 31)) return fail(AA_ERR_UNSUPPORTED, std::string(name) + ": output too large for one launch");
  std::unique_ptr<Params> hold(new Params);  // ~28 KB, kept off the stack; each launch copies it
  Params& P = *hold;
  P.out = out->data;
  P.epi = epi;
  P.out_sn = out->stride_n; P.out_sc = out->stride_c; P.out_sh = out->stride_h; P.out_sw = out->stride_w;
  P.oH = (int)out->h; P.oW = (int)out->w; P.Ci = Ci; P.filter = filter; P.tiles_x = (int)tiles_x;
  if constexpr (PAD) {
    P.align = align;
    P.fill_epi = epi;
    if (fill->mode == AA_FILL_OUTPUT) P.fill_epi.norm = 0;
    // 0 + v: the sum of the 1x1 resize that defines the fill's outputs, which stores -0.0 as +0.0
    for (int k = 0; k < 4; k++) P.fill[k] = 0.0f + fill->value[k];
  }
  for (int32_t first = 0; first < count; first += kCropsPerLaunch) {
    const int n = (int)std::min<int64_t>(kCropsPerLaunch, (int64_t)count - first);
    P.first = first;
    for (int k = 0; k < n; k++) {
      const aa_image_desc& m = images[first + k];
      const aa_crop_ex& b = crops[first + k];
      auto& d = P.c[k];
      d.src = (const char*)m.data + (b.top * m.stride_h + b.left * Ci) * es;
      d.stride_h = m.stride_h;
      d.stride_c = channels_last ? 0 : m.stride_c;
      d.h = (int32_t)b.height; d.w = (int32_t)b.width;
      d.y0 = (int32_t)b.crop_top; d.x0 = (int32_t)b.crop_left;
      if constexpr (PAD) {
        d.rh = (int32_t)b.resized_h; d.rw = (int32_t)b.resized_w;
        d.kh = (uint8_t)host_interp_size(b.height, b.resized_h, filter, align, AA_F32);
        d.kw = (uint8_t)host_interp_size(b.width, b.resized_w, filter, align, AA_F32);
        d.flip = (uint8_t)b.flip;
      } else {
        d.scale_h = host_scale_f32(b.height, b.resized_h, align);
        d.scale_w = host_scale_f32(b.width, b.resized_w, align);
        d.kh = (int16_t)host_interp_size(b.height, b.resized_h, filter, align, AA_F32);
        d.kw = (int16_t)host_interp_size(b.width, b.resized_w, filter, align, AA_F32);
        d.flip = b.flip;
      }
    }
    const dim3 grid((unsigned)(tiles_x * tiles_y), (unsigned)(channels_last ? 1 : channels), (unsigned)n);
    if constexpr (PAD) {
      if (dtype == AA_U8) aa_crops_pad_kernel<uint8_t><<<grid, TW * NTY, 0, stream>>>(P);
      else aa_crops_pad_kernel<float><<<grid, TW * NTY, 0, stream>>>(P);
      AA_LAUNCH_CHECK("aa_crops_pad_kernel");
    } else {
      if (dtype == AA_U8) aa_crops_kernel<uint8_t><<<grid, TW * NTY, 0, stream>>>(P);
      else aa_crops_kernel<float><<<grid, TW * NTY, 0, stream>>>(P);
      AA_LAUNCH_CHECK("aa_crops_kernel");
    }
    (*launches)++;
  }
  return AA_OK;
}

}  // namespace

int launch_crops(const char* name, const aa_image_desc* images, const aa_crop_ex* crops, int32_t count, int32_t dtype,
                 int64_t channels, int32_t channels_last, const aa_tensor_desc* out, int filter, int align, const OutEpi& epi,
                 const aa_fill* fill, cudaStream_t stream, int32_t* launches) {
  // the padded variant only when a window leaves its resized image: inside it the two give the same bits, and the
  // unpadded one spends no instructions on the edges
  bool padded = false;
  for (int32_t i = 0; fill && fill->mode != AA_FILL_NONE && i < count && !padded; i++) {
    const aa_crop_ex& b = crops[i];
    padded = b.crop_top < 0 || b.crop_left < 0 || b.crop_top + out->h > b.resized_h || b.crop_left + out->w > b.resized_w;
  }
  if (padded)
    return launch<true>(name, images, crops, count, dtype, channels, channels_last, out, filter, align, epi, fill, stream,
                        launches);
  return launch<false>(name, images, crops, count, dtype, channels, channels_last, out, filter, align, epi, fill, stream,
                       launches);
}

}  // namespace aa

// clip_transform.cu — sm_100a kernels + C ABI of libnexar_clip_b200.so.
//
// Path (reference file:line in include/nexar_clip_transform.h):
//   K1 resize   : uint8 THWC frames -> antialiased separable resample -> either the
//                 final normalised tensor (no augmentation) or a brightness-adjusted
//                 8-byte intermediate pixel + per-band gray sums (augmentation).
//   K2 colour   : contrast (needs the frame's gray mean) -> saturation -> hue, in place; a programmatic dependent
//                 launch of K1 that starts in K1's last wave and waits per frame on a publication flag.
//   K3 geometry : affine gather with the fill=0 mask quirk, effects, normalise, store (a kernel specialised for the
//                 production letterboxes, a general one for everything else).
//   K4 blur     : only when blur_sigma > 0 (reflect-padded gaussian, then the rest of the chain).
//   YUV 4:2:0 -> RGB : decoder surfaces (NV12 / I420 with 8- or 16-bit samples, BT.601 / BT.709, limited / full range) converted in front of K1; window gather for inference.
// The /255 decision of VideoTransform.forward is clip-global and data dependent
// (nexar_video_aug.py:814): K1 runs assuming "max > 1", records the clip maximum, and
// a second, normally empty, launch (fixup_frame_kernel) redoes the clips whose maximum was <= 1.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <type_traits>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "nexar_clip_transform.h"

// ---------------------------------------------------------------------------------
// host-side error plumbing
// ---------------------------------------------------------------------------------
static thread_local std::string g_err;
static thread_local int g_launches = 0;
static thread_local int32_t g_resize_instance[5] = {0, 0, 0, 0, 0};  // nexar_last_resize_kernel: {fast, KX, NT, RS, AL4}
// experiment knobs and the optional kernel timing are per calling thread (the library keeps no process-global mutable state)
// 0 auto, 1 force the general fp32 kernels, 2 no programmatic overlap (K1 -> K2 and K3 -> fix-up serialised by the stream);
// nexar_set_resize_kernel refuses anything else.  tests/test_launch_paths.py pins
// every launch sequence these select (fast / general letterbox, resize-crop, fix-up, blur) against the oracle, and variant
// 2 against the overlapped default bit for bit.
static thread_local int g_resize_variant = 0;
static thread_local int g_fast_bands = 0;      // 0 auto
static thread_local int g_chunk_clips = 0;     // clips per chunk of an augmented batch (0: the whole batch at once)
static thread_local int g_geo_variant = 0;     // 0 auto (specialised geometry kernel when the shape allows it), 1 force the general one

static thread_local std::vector<cudaEvent_t> g_prof_ev;
static thread_local int g_prof_n = 0;

static inline int imin_host(int a, int b) { return a < b ? a : b; }

static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                  \
  do {                                                                                  \
    cudaError_t e__ = (expr);                                                           \
    if (e__ != cudaSuccess)                                                             \
      return fail(NEXAR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)

// ---------------------------------------------------------------------------------
// plan
// ---------------------------------------------------------------------------------
struct DevPlan {
  int src_h, src_w, cs, rh, rw, off_y, off_x, ky, kx;
  const int* ystart;
  const int* ycount;
  const float* ywt;
  const int* xstart;
  const int* xcount;
  const float* xwt;
  // fast (fixed-point, input-stationary) resize tables; pairs == nullptr when not applicable
  const uint4* pairs;      // [n_pairs] {w slot0, w slot1, w slot2 (u16x2: row 2p | row 2p+1 << 16), emit (count | first_row << 2)}
  int n_pairs, shift;      // weights are round(w * 2^shift), every row sums to exactly 2^shift
  const int* xstart_al;    // [rw] even-aligned first tap
  const unsigned* xw16;    // [rw][kx_al / 2] the same taps in 15-bit fixed point, two per word: lo bytes | hi bytes << 16 (dp2a operand)
  int kx_al;
  int x_align4;            // the horizontal windows start at multiples of four pixels (8-byte aligned: LDS.64, no bank conflicts at 4:1)
};

// Integer YUV -> RGB coefficients (include/nexar_clip_transform.h): round(256 * c) of the standard's float values.
struct YuvCoef { int yo, ys, rv, gu, gv, bu; };
static const YuvCoef kYuvCoef[2][2] = {        // [matrix][range]
    {{16, 298, 409, 100, 208, 516}, {0, 256, 359, 88, 183, 454}},    // BT.601 limited, full
    {{16, 298, 459, 55, 136, 541}, {0, 256, 403, 48, 120, 475}}};    // BT.709 limited, full

struct NexarPlan {
  NexarGeometry g;
  int src_dtype;               // NEXAR_SRC_NV12 stands for every YUV 4:2:0 source; yuv_* below say which
  int yuv_layout = NEXAR_YUV_NV12;
  int yuv_luma_rows = 0;
  bool yuv_16bit = false;      // 2-byte samples (nexar_plan_create_yuv16), aligned to the word's top by yuv_shift
  int yuv_shift = 0;
  YuvCoef yuv_coef = kYuvCoef[NEXAR_YUV_BT601][NEXAR_YUV_LIMITED];
  DevPlan d;
  void* dev_tables;
  std::vector<int> ystart, ycount, xstart, xcount;
  std::vector<float> ywt, xwt;
  bool fast_ok = false;
  int x_align = 2;
  std::vector<uint4> pairs;
  std::vector<int> xstart_al;
  std::vector<float> xwt_al;
  std::vector<unsigned> xw16;
};

// Fixed-point vertical taps for the input-stationary kernel.  The triangle filter of a >= 2x
// down-scale keeps at most two output rows alive at any source row (ymin[i+2] >= ymax[i]), so two
// rotating accumulator slots suffice (out row i lives in slot i % 2).  The kernel consumes source rows
// in PAIRS through dp2a; table entry p = {w slot0, w slot1, w post, emit} with w = u16x2 (row 2p | row
// 2p+1 << 16), z = bit0 (an output row's last tap lies in this pair) | slot << 1 | begin0 << 2 |
// begin1 << 3 (the slot's accumulators restart at this pair) | out_row << 4 | post tap << 16, and "w post" the first tap of the NEXT row of that slot when it falls in the same pair (it is
// accumulated after the finished row has been flushed).  Returns false when the geometry does not fit.
static const int kMaxPairs = 1024;
// Fixed-point taps of one row that sum to exactly 2^15 (constant images stay constant): every tap is the floor of
// w * 2^15, and the taps with the largest remainders (the first of equal ones) get one more until the row sums to 2^15,
// so no tap is a unit or more from its exact value.  (Rounding each tap and putting the whole residual on the largest
// one, up to 4 units, let 0/255 content aligned with the rounding reach 1.05e-3 after normalisation at 540x960 -> 224,
// above the 1e-3 gate; this way every letterbox stays below 7.1e-4, see tests/fast_resize_model.py.)
static bool quantise_taps(const float* w, int n, int shift, std::vector<long>& q) {
  std::vector<double> rem(n);
  std::vector<int> order(n);
  q.assign(n, 0);
  long sum = 0;
  for (int k = 0; k < n; ++k) {
    const double x = std::ldexp((double)w[k], shift);
    q[k] = (long)std::floor(x);
    rem[k] = x - (double)q[k];
    sum += q[k];
    order[k] = k;
  }
  const long deficit = (1L << shift) - sum;
  if (deficit < 0 || deficit > n) return false;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rem[a] > rem[b]; });
  for (long k = 0; k < deficit; ++k) ++q[order[k]];
  for (int k = 0; k < n; ++k)
    if (q[k] < 0 || q[k] > 65535) return false;
  return true;
}
static bool build_fast_tables(NexarPlan* p, int ky, int kx, int& shift, int& kx_al) {
  const NexarGeometry& g = p->g;
  if (p->src_dtype != NEXAR_SRC_U8 && p->src_dtype != NEXAR_SRC_NV12) return false;
  if ((g.src_w * 3) % 16 != 0 || g.src_w * 3 / 16 > 384 || (g.src_h & 1)) return false;  // rows are consumed in pairs
  if (g.src_h < 2 * g.resize_h || g.src_w < g.resize_w) return false;  // vertical down-scale by >= 2
  if (imin_host(g.resize_w, g.canvas) > 384) return false;
  kx_al = kx + 1;
  kx_al = kx_al <= 10 ? 10 : kx_al <= 14 ? 14 : kx_al <= 20 ? 20 : 0;
  if (!kx_al) return false;
  // Windows aligned to FOUR pixels (24 bytes of the staged row) when that still fits the tap budget: the horizontal pass
  // then reads its window with 8-byte loads, and at an exact 4:1 scale (720p -> 320: lanes 6 words apart) those are
  // conflict-free where the 4-byte loads of the 2-pixel alignment collide two ways on every access.
  int align = 4;
  for (int j = 0; j < g.resize_w; ++j)
    if (p->xcount[j] + (p->xstart[j] & 3) > kx_al) align = 2;
  if (kx_al != 10) align = 2;   // only the 10-tap kernels are instantiated with the 8-byte path
  p->x_align = align;
  float wmax = 0.f;
  for (float w : p->ywt) wmax = w > wmax ? w : wmax;
  if (!(wmax > 0.f)) return false;
  // 15 fractional bits: the finished sums are < 2^23, so "value * 128" (the 15-bit staging format) is simply
  // bytes 1..2 of the accumulator and two of them pack with ONE PRMT.  Measured against an exact evaluation on
  // 720p -> 224 noise: max error 2.2e-5 of full scale (1.3e-5 with 18 bits: the staging rounding dominates).
  shift = 15;
  if (std::ldexp((double)wmax, shift) > 65535.0) return false;
  const int n_pairs = (g.src_h + 1) / 2;
  if (n_pairs > kMaxPairs) return false;
  p->pairs.assign(n_pairs + 1, make_uint4(0, 0, 0, 0));  // + one spare entry: the kernel reads one pair ahead
  for (int i = 0; i < g.resize_h; ++i) {
    const int ys = p->ystart[i], yc = p->ycount[i];
    if (yc <= 0) return false;
    if (i + 2 < g.resize_h && p->ystart[i + 2] < ys + yc) return false;  // three rows alive at once
    if (i + 1 < g.resize_h && p->ystart[i + 1] + p->ycount[i + 1] <= ys + yc) return false;  // must finish in order
    std::vector<long> q;
    if (!quantise_taps(&p->ywt[(size_t)i * ky], yc, shift, q)) return false;
    const int slot = i % 2;
    const int prev_last = i >= 2 ? p->ystart[i - 2] + p->ycount[i - 2] - 1 : -1;  // last tap of the slot's previous row
    bool begun = false;
    for (int k = 0; k < yc; ++k) {
      const int y = ys + k;
      uint4& e = p->pairs[y / 2];
      if (prev_last >= 0 && prev_last / 2 == y / 2) {
        if (!(y & 1) || e.w) return false;
        e.w = (unsigned)q[k] << 16;  // accumulated with "begin" semantics after the flush (temporarily in .w)
        if (q[k]) begun = true;
      } else {
        unsigned& ws = slot ? e.y : e.x;
        if (!begun && q[k]) {  // first non-zero tap of the row: the accumulators restart from the rounding constant
          if (ws) return false;
          e.z |= slot ? 8u : 4u;
          begun = true;
        }
        ws |= (unsigned)q[k] << (16 * (y & 1));
      }
    }
    unsigned& em = p->pairs[(ys + yc - 1) / 2].z;
    if (em & 1u) return false;  // one flush per pair
    if (i >= 4096) return false;
    em |= 1u | ((unsigned)slot << 1) | ((unsigned)i << 4);
  }
  for (uint4& e : p->pairs) {  // final packing (the spare entry stays zero): z = post tap << 16 | out_row << 4 | flags, w unused
    if (e.w && !(e.z & 1u)) return false;
    e.z = (e.z & 0xFFFFu) | e.w;
    e.w = 0u;
  }
  p->xstart_al.assign(g.resize_w, 0);
  p->xwt_al.assign((size_t)g.resize_w * kx_al, 0.f);
  for (int j = 0; j < g.resize_w; ++j) {
    const int xs = p->xstart[j], al = xs & ~(align - 1), sh = xs - al;
    p->xstart_al[j] = al;
    for (int k = 0; k < p->xcount[j]; ++k) p->xwt_al[(size_t)j * kx_al + k + sh] = p->xwt[(size_t)j * kx + k];
  }
  // The horizontal pass runs on dp2a too: 15-bit taps (rows sum to exactly 2^15) split into low and high bytes,
  // two taps per word: byte0/1 = low bytes of the even/odd tap, byte2/3 = their high bytes.
  p->xw16.assign((size_t)g.resize_w * (kx_al / 2), 0u);
  for (int j = 0; j < g.resize_w; ++j) {
    std::vector<long> q;
    if (!quantise_taps(&p->xwt_al[(size_t)j * kx_al], kx_al, 15, q)) return false;
    for (int m = 0; m < kx_al / 2; ++m) {
      const unsigned e = (unsigned)q[2 * m], o = (unsigned)q[2 * m + 1];
      p->xw16[(size_t)j * (kx_al / 2) + m] = (e & 255u) | ((o & 255u) << 8) | ((e >> 8) << 16) | ((o >> 8) << 24);
    }
  }
  return true;
}

// ATen UpSampleKernel.cpp _compute_indices_min_size_weights_aa, float opmath.
static void aa_taps_host(int in_size, int out_size, std::vector<int>& start, std::vector<int>& count,
                         std::vector<float>& wts, int& kmax) {
  const float scale = (float)in_size / (float)out_size;
  const float support = scale >= 1.0f ? scale : 1.0f;
  const float invscale = scale >= 1.0f ? 1.0f / scale : 1.0f;
  kmax = (int)std::ceil(support) * 2 + 1;
  start.assign(out_size, 0);
  count.assign(out_size, 0);
  wts.assign((size_t)out_size * kmax, 0.0f);
  for (int i = 0; i < out_size; ++i) {
    const float center = scale * ((float)i + 0.5f);
    int lo = (int)(center - support + 0.5f);
    if (lo < 0) lo = 0;
    int hi = (int)(center + support + 0.5f);
    if (hi > in_size) hi = in_size;
    int n = hi - lo;
    if (n < 0) n = 0;
    if (n > kmax) n = kmax;
    float total = 0.0f;
    float* w = &wts[(size_t)i * kmax];
    for (int j = 0; j < n; ++j) {
      float x = ((float)(j + lo) - center + 0.5f) * invscale;
      x = std::fabs(x);
      w[j] = x < 1.0f ? 1.0f - x : 0.0f;
      total += w[j];
    }
    if (total != 0.0f)
      for (int j = 0; j < n; ++j) w[j] /= total;
    start[i] = lo;
    count[i] = n;
  }
}

extern "C" int nexar_abi_version(void) { return NEXAR_ABI_VERSION; }
extern "C" size_t nexar_sizeof_clip_params(void) { return sizeof(NexarClipParams); }
extern "C" size_t nexar_sizeof_transform_args(void) { return sizeof(NexarTransformArgs); }
extern "C" const char* nexar_last_error(void) { return g_err.c_str(); }
extern "C" int nexar_last_launch_count(void) { return g_launches; }
extern "C" int nexar_last_resize_kernel(int32_t out[5]) {
  if (!out) return fail(NEXAR_ERR_INVALID, "last_resize_kernel: null argument");
  memcpy(out, g_resize_instance, sizeof(g_resize_instance));
  return NEXAR_OK;
}
static void record_resize_instance(int fast, int kx, int nt, int rs, int al4) {
  const int32_t v[5] = {fast, kx, nt, rs, al4};
  memcpy(g_resize_instance, v, sizeof(v));
}
extern "C" int nexar_set_resize_kernel(int32_t v) {
  if (v == 4) return fail(NEXAR_ERR_UNSUPPORTED, "set_resize_kernel: variant 4 (the fused cluster kernel) was removed");
  if (v != 0 && v != 1 && v != 2)
    return fail(NEXAR_ERR_INVALID, "set_resize_kernel: variant must be 0 (auto), 1 (general) or 2 (no overlap)");
  g_resize_variant = v;
  return NEXAR_OK;
}
extern "C" int nexar_set_fast_bands(int32_t n) {
  g_fast_bands = n;
  return NEXAR_OK;
}
extern "C" int nexar_set_chunk_clips(int32_t n) {
  g_chunk_clips = n;
  return NEXAR_OK;
}
extern "C" int nexar_set_geometry_kernel(int32_t v) {
  g_geo_variant = v;
  return NEXAR_OK;
}

extern "C" int nexar_profile_begin(int32_t max_calls) {
  for (cudaEvent_t e : g_prof_ev) cudaEventDestroy(e);
  g_prof_ev.clear();
  g_prof_n = 0;
  for (int i = 0; i < 2 * max_calls; ++i) {
    cudaEvent_t e;
    CUDA_TRY(cudaEventCreate(&e));
    g_prof_ev.push_back(e);
  }
  return NEXAR_OK;
}
extern "C" int nexar_profile_end(float* ms_out, int32_t cap) {
  int n = 0;
  for (int i = 0; i < g_prof_n && n < cap; ++i) {
    if (cudaEventSynchronize(g_prof_ev[2 * i + 1]) != cudaSuccess) break;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g_prof_ev[2 * i], g_prof_ev[2 * i + 1]) != cudaSuccess) break;
    ms_out[n++] = ms;
  }
  for (cudaEvent_t e : g_prof_ev) cudaEventDestroy(e);
  g_prof_ev.clear();
  g_prof_n = 0;
  return n;
}

extern "C" int nexar_letterbox_geometry(int32_t h, int32_t w, int32_t cs, NexarGeometry* out) {
  if (!out || h <= 0 || w <= 0 || cs <= 0) return fail(NEXAR_ERR_INVALID, "letterbox_geometry: bad size");
  const double sh = (double)cs / (double)h, sw = (double)cs / (double)w;
  const double scale = sh < sw ? sh : sw;
  out->src_h = h;
  out->src_w = w;
  out->canvas = cs;
  out->resize_h = (int32_t)((double)h * scale);  // python int(): truncation of the float64 product
  out->resize_w = (int32_t)((double)w * scale);
  out->off_y = (cs - out->resize_h) / 2;         // both non-negative here, so / == python //
  out->off_x = (cs - out->resize_w) / 2;
  if (out->resize_h <= 0 || out->resize_w <= 0)
    return fail(NEXAR_ERR_INVALID, "letterbox_geometry: resized size is zero (torch would raise)");
  return NEXAR_OK;
}

static int floordiv(int a, int b) {  // python // for b > 0
  int q = a / b;
  if ((a % b != 0) && (a < 0)) --q;
  return q;
}

extern "C" int nexar_resize_crop_geometry(int32_t h, int32_t w, int32_t size, int32_t cs, NexarGeometry* out) {
  if (!out || h <= 0 || w <= 0 || cs <= 0 || size <= 0) return fail(NEXAR_ERR_INVALID, "resize_crop_geometry: bad size");
  out->src_h = h;
  out->src_w = w;
  out->canvas = cs;
  if (h > w) {
    out->resize_h = (int32_t)((int64_t)size * h / w);
    out->resize_w = size;
  } else {
    out->resize_h = size;
    out->resize_w = (int32_t)((int64_t)size * w / h);
  }
  if (out->resize_h < cs || out->resize_w < cs)
    return fail(NEXAR_ERR_INVALID, "resize_crop_geometry: resized frame smaller than crop_size");
  out->off_y = -floordiv(out->resize_h - cs, 2);
  out->off_x = -floordiv(out->resize_w - cs, 2);
  return NEXAR_OK;
}

extern "C" int nexar_aa_taps(int32_t in_size, int32_t out_size, int32_t* start, int32_t* count, float* weights,
                             int32_t cap, int32_t* kmax) {
  if (in_size <= 0 || out_size <= 0 || !start || !count || !weights || !kmax)
    return fail(NEXAR_ERR_INVALID, "aa_taps: bad argument");
  std::vector<int> s, c;
  std::vector<float> w;
  int k = 0;
  aa_taps_host(in_size, out_size, s, c, w, k);
  if (k > cap) return fail(NEXAR_ERR_INVALID, "aa_taps: kmax_capacity too small");
  *kmax = k;
  for (int i = 0; i < out_size; ++i) {
    start[i] = s[i];
    count[i] = c[i];
    for (int j = 0; j < cap; ++j) weights[(size_t)i * cap + j] = j < k ? w[(size_t)i * k + j] : 0.0f;
  }
  return NEXAR_OK;
}

static int plan_create(const NexarGeometry* g, int32_t src_dtype, const NexarYuvFormat* yuv, NexarPlan** out);

extern "C" int nexar_plan_create(const NexarGeometry* g, int32_t src_dtype, NexarPlan** out) {
  return plan_create(g, src_dtype, nullptr, out);
}

extern "C" size_t nexar_sizeof_yuv_format(void) { return sizeof(NexarYuvFormat); }

extern "C" int nexar_yuv_coefficients(int32_t matrix, int32_t range, int32_t out[6]) {
  if (!out) return fail(NEXAR_ERR_INVALID, "yuv_coefficients: null argument");
  if ((matrix != NEXAR_YUV_BT601 && matrix != NEXAR_YUV_BT709) || (range != NEXAR_YUV_LIMITED && range != NEXAR_YUV_FULL))
    return fail(NEXAR_ERR_INVALID, "yuv_coefficients: unknown matrix or range");
  const YuvCoef& k = kYuvCoef[matrix][range];
  const int32_t v[6] = {k.yo, k.ys, k.rv, k.gu, k.gv, k.bu};
  memcpy(out, v, sizeof(v));
  return NEXAR_OK;
}

extern "C" int nexar_plan_create_yuv(const NexarGeometry* g, const NexarYuvFormat* f, NexarPlan** out) {
  if (!f) return fail(NEXAR_ERR_INVALID, "plan_create_yuv: null argument");
  if (f->struct_size != sizeof(NexarYuvFormat)) return fail(NEXAR_ERR_INVALID, "plan_create_yuv: NexarYuvFormat size mismatch (ABI)");
  if (f->layout != NEXAR_YUV_NV12 && f->layout != NEXAR_YUV_I420) return fail(NEXAR_ERR_INVALID, "plan_create_yuv: unknown layout");
  if (f->matrix != NEXAR_YUV_BT601 && f->matrix != NEXAR_YUV_BT709) return fail(NEXAR_ERR_INVALID, "plan_create_yuv: unknown matrix");
  if (f->range != NEXAR_YUV_LIMITED && f->range != NEXAR_YUV_FULL) return fail(NEXAR_ERR_INVALID, "plan_create_yuv: unknown range");
  return plan_create(g, NEXAR_SRC_NV12, f, out);
}

extern "C" int nexar_plan_create_yuv16(const NexarGeometry* g, const NexarYuvFormat* f, int32_t sample_shift, NexarPlan** out) {
  if (!out) return fail(NEXAR_ERR_INVALID, "plan_create_yuv16: null argument");
  if (sample_shift != 0 && sample_shift != 4 && sample_shift != 6)
    return fail(NEXAR_ERR_INVALID, "plan_create_yuv16: sample_shift must be 0, 4 or 6");
  NexarPlan* p = nullptr;
  const int rc = nexar_plan_create_yuv(g, f, &p);
  if (rc != NEXAR_OK) return rc;
  p->yuv_16bit = true;
  p->yuv_shift = sample_shift;
  *out = p;
  return NEXAR_OK;
}

static int plan_create(const NexarGeometry* g, int32_t src_dtype, const NexarYuvFormat* yuv, NexarPlan** out) {
  if (!g || !out) return fail(NEXAR_ERR_INVALID, "plan_create: null argument");
  if (src_dtype != NEXAR_SRC_U8 && src_dtype != NEXAR_SRC_F32 && src_dtype != NEXAR_SRC_NV12)
    return fail(NEXAR_ERR_INVALID, "plan_create: bad src_dtype");
  if (src_dtype == NEXAR_SRC_NV12 && ((g->src_h | g->src_w) & 1))
    return fail(NEXAR_ERR_INVALID, "plan_create: NV12 frames need an even height and width");
  if (g->src_h <= 0 || g->src_w <= 0 || g->canvas <= 0 || g->resize_h <= 0 || g->resize_w <= 0)
    return fail(NEXAR_ERR_INVALID, "plan_create: bad geometry");
  const int luma_rows = yuv && yuv->luma_rows ? yuv->luma_rows : g->src_h;
  if (src_dtype == NEXAR_SRC_NV12 && (luma_rows < g->src_h || (luma_rows & 1)))
    return fail(NEXAR_ERR_INVALID, "plan_create_yuv: luma_rows must be even and >= src_h");
  NexarPlan* p = new NexarPlan();
  p->g = *g;
  p->src_dtype = src_dtype;
  p->yuv_luma_rows = luma_rows;
  if (yuv) {
    p->yuv_layout = yuv->layout;
    p->yuv_coef = kYuvCoef[yuv->matrix][yuv->range];
  }
  int ky = 0, kx = 0;
  aa_taps_host(g->src_h, g->resize_h, p->ystart, p->ycount, p->ywt, ky);
  aa_taps_host(g->src_w, g->resize_w, p->xstart, p->xcount, p->xwt, kx);
  int shift = 0, kx_al = 0;
  p->fast_ok = build_fast_tables(p, ky, kx, shift, kx_al);
  // one device allocation: [pairs (16B aligned)] [ints] [floats]
  const size_t n_pairs_b = p->fast_ok ? p->pairs.size() * sizeof(uint4) : 0;
  const size_t ni = ((size_t)(g->resize_h + g->resize_w) * 2 + (p->fast_ok ? g->resize_w : 0)) * sizeof(int);
  const size_t nf = ((size_t)g->resize_h * ky + (size_t)g->resize_w * kx + (p->fast_ok ? p->xw16.size() : 0)) * sizeof(float);
  p->dev_tables = nullptr;
  cudaError_t e = cudaMalloc(&p->dev_tables, n_pairs_b + ni + nf);
  if (e != cudaSuccess) {
    delete p;
    return fail(NEXAR_ERR_CUDA, std::string("plan_create: cudaMalloc: ") + cudaGetErrorString(e));
  }
  std::vector<char> host(n_pairs_b + ni + nf);
  if (n_pairs_b) memcpy(host.data(), p->pairs.data(), n_pairs_b);
  int* hi = (int*)(host.data() + n_pairs_b);
  memcpy(hi, p->ystart.data(), g->resize_h * sizeof(int));
  memcpy(hi + g->resize_h, p->ycount.data(), g->resize_h * sizeof(int));
  memcpy(hi + 2 * g->resize_h, p->xstart.data(), g->resize_w * sizeof(int));
  memcpy(hi + 2 * g->resize_h + g->resize_w, p->xcount.data(), g->resize_w * sizeof(int));
  if (p->fast_ok) memcpy(hi + 2 * g->resize_h + 2 * g->resize_w, p->xstart_al.data(), g->resize_w * sizeof(int));
  float* hf = (float*)(host.data() + n_pairs_b + ni);
  memcpy(hf, p->ywt.data(), p->ywt.size() * sizeof(float));
  memcpy(hf + p->ywt.size(), p->xwt.data(), p->xwt.size() * sizeof(float));
  if (p->fast_ok) memcpy(hf + p->ywt.size() + p->xwt.size(), p->xw16.data(), p->xw16.size() * sizeof(unsigned));
  e = cudaMemcpy(p->dev_tables, host.data(), host.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(p->dev_tables);
    delete p;
    return fail(NEXAR_ERR_CUDA, std::string("plan_create: cudaMemcpy: ") + cudaGetErrorString(e));
  }
  int* di = (int*)((char*)p->dev_tables + n_pairs_b);
  float* df = (float*)((char*)p->dev_tables + n_pairs_b + ni);
  DevPlan& d = p->d;
  d.src_h = g->src_h;
  d.src_w = g->src_w;
  d.cs = g->canvas;
  d.rh = g->resize_h;
  d.rw = g->resize_w;
  d.off_y = g->off_y;
  d.off_x = g->off_x;
  d.ky = ky;
  d.kx = kx;
  d.ystart = di;
  d.ycount = di + g->resize_h;
  d.xstart = di + 2 * g->resize_h;
  d.xcount = di + 2 * g->resize_h + g->resize_w;
  d.ywt = df;
  d.xwt = df + p->ywt.size();
  d.pairs = p->fast_ok ? (const uint4*)p->dev_tables : nullptr;
  d.n_pairs = (int)p->pairs.size() - (p->fast_ok ? 1 : 0);
  d.shift = shift;
  d.xstart_al = p->fast_ok ? di + 2 * g->resize_h + 2 * g->resize_w : nullptr;
  d.xw16 = p->fast_ok ? (const unsigned*)(df + p->ywt.size() + p->xwt.size()) : nullptr;
  d.kx_al = kx_al;
  d.x_align4 = p->fast_ok && p->x_align == 4;
  *out = p;
  return NEXAR_OK;
}

extern "C" void nexar_plan_destroy(NexarPlan* p) {
  if (!p) return;
  if (p->dev_tables) cudaFree(p->dev_tables);
  delete p;
}

extern "C" int nexar_plan_geometry(const NexarPlan* p, NexarGeometry* out) {
  if (!p || !out) return fail(NEXAR_ERR_INVALID, "plan_geometry: null argument");
  *out = p->g;
  return NEXAR_OK;
}

// ---------------------------------------------------------------------------------
// workspace layout
// ---------------------------------------------------------------------------------
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
static inline int imin(int a, int b) { return a < b ? a : b; }
static inline int imax(int a, int b) { return a > b ? a : b; }

static const int kMaxBands = 16;
constexpr unsigned kFrameReady = 0x80000000u;   // frame_done value once the frame's FrameInfo has been published


// Per-frame constants computed once by K1.5 (frame_stats_kernel) so that K2/K3 start with a few 16-byte loads
// instead of re-deriving the content box, the colour parameters and the pad colour in every thread.
struct alignas(16) FrameInfo {
  float padr, padg, padb, cmean;          // colour of a zero (pad) pixel after the colour chain; contrast_q * gray mean
  int by0, by1, bx0, bx1;                 // content box on the canvas (x already mirrored for flipped clips)
  float grid[6];                          // affine grid coefficients
  unsigned flags;
  float contrast;
  float saturation, saturation_q, hue;
  int reserved;
};
static_assert(sizeof(FrameInfo) == 80, "FrameInfo is five 16-byte words");


struct Workspace {
  unsigned* clip_max;   // [n_clips] non-zero iff some source value of the clip is > 1 (nexar_video_aug.py:814)
  unsigned* frame_done; // [n_frames] bands of the frame that have finished K1 (the last one publishes the FrameInfo); follows clip_max
  unsigned long long* gray_partial;  // [2][n_frames][kMaxBands] fixed-point (2^-22) gray sums: exact, order-independent
  FrameInfo* finfo;     // [n_frames] per-frame constants for K2/K3, written by K1.5
  uint2* inter;         // [n_frames][bh][bw]   q15 RGBX pixels (8 bytes), brightness-adjusted, then colour-adjusted in place
  float* canvas;        // [n_frames][3][cs][cs] pre-blur canvas (blur path only)
  int64_t* rgb_offsets; // [n_frames] YUV sources: byte offsets of the converted frames in `rgb`
  unsigned char* rgb;   // [n_frames][src_h][src_w][3] YUV sources: packed RGB produced by yuv420_to_rgb_*_kernel
  size_t total;
};

static Workspace carve(const NexarPlan* p, int n_clips, int T, void* base, unsigned any_flags) {
  Workspace w;
  const size_t nf = (size_t)n_clips * T;
  const int bh = imin(p->g.resize_h, p->g.canvas), bw = imin(p->g.resize_w, p->g.canvas);
  size_t off = 0;
  char* b = (char*)base;
  w.clip_max = (unsigned*)(b + off);
  w.frame_done = w.clip_max + n_clips;  // one memset clears both
  off = align_up(off + ((size_t)n_clips + nf) * sizeof(unsigned), 256);
  w.gray_partial = (unsigned long long*)(b + off);
  off = align_up(off + 2 * nf * kMaxBands * sizeof(unsigned long long), 256);
  w.finfo = (FrameInfo*)(b + off);
  off = align_up(off + nf * sizeof(FrameInfo), 256);
  w.inter = (uint2*)(b + off);  // only augmented clips use it
  if (any_flags & NEXAR_AUG) off = align_up(off + nf * bh * bw * sizeof(uint2), 256);
  w.canvas = (float*)(b + off);  // only the blur path uses it
  if (any_flags & NEXAR_BLUR) off = align_up(off + nf * 3 * (size_t)p->g.canvas * p->g.canvas * sizeof(float), 256);
  w.rgb_offsets = (int64_t*)(b + off);
  w.rgb = nullptr;
  if (p->src_dtype == NEXAR_SRC_NV12) {
    off = align_up(off + nf * sizeof(int64_t), 256);
    w.rgb = (unsigned char*)(b + off);
    off = align_up(off + nf * (size_t)p->g.src_h * p->g.src_w * 3, 256);
  }
  w.total = off;
  return w;
}

extern "C" size_t nexar_workspace_bytes(const NexarPlan* p, int32_t n_clips, int32_t T) {
  if (!p || n_clips <= 0 || T <= 0) return 0;
  return carve(p, n_clips, T, nullptr, ~0u).total;
}
extern "C" size_t nexar_workspace_bytes_for(const NexarPlan* p, int32_t n_clips, int32_t T, uint32_t any_flags) {
  if (!p || n_clips <= 0 || T <= 0) return 0;
  return carve(p, n_clips, T, nullptr, any_flags).total;
}

// ---------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------
struct KArgs {
  const void* src;
  const int64_t* frame_offsets;
  int64_t src_row_stride;
  const NexarClipParams* params;
  void* dst;
  int64_t sb, sc, st, sy, sx;
  int T;
  int normalize;
  float nscale[3], nbias[3];  // out = v * nscale + nbias  ((v - mean) / std)
  unsigned* clip_max;
  unsigned* frame_done;
  int finfo_by_k1;  // the fast resize kernel publishes the FrameInfo of every frame itself (K1.5 folded into K1)
  int overlap;      // the colour kernel was launched as a programmatic dependent of the resize kernel: it polls frame_done
  unsigned long long* gray_partial;
  FrameInfo* finfo;
  uint2* inter;
  float* canvas;
  int n_frames;
  int bh, bw;  // allocation dims of one intermediate frame
  int pass;    // 0: assume /255 and record max; 1: redo clips whose max <= 1 without scaling; 2: max already known
};

__device__ __forceinline__ float clamp01(float x) { return fminf(fmaxf(x, 0.0f), 1.0f); }
// tv rgb_to_grayscale: (0.2989 r + 0.587 g) + 0.114 b, every product rounded (no fma contraction)
__device__ __forceinline__ float gray_of(float r, float g, float b) {
  return __fadd_rn(__fadd_rn(__fmul_rn(0.2989f, r), __fmul_rn(0.587f, g)), __fmul_rn(0.114f, b));
}
// tv _blend: (ratio*a + q*b).clamp(0,1)
__device__ __forceinline__ float blend(float a, float b, float r, float q) {
  return clamp01(__fadd_rn(__fmul_rn(r, a), __fmul_rn(q, b)));
}

template <typename T>
__device__ __forceinline__ void store_out(void* dst, int64_t idx, float v);
template <>
__device__ __forceinline__ void store_out<float>(void* dst, int64_t idx, float v) {
  ((float*)dst)[idx] = v;
}
template <>
__device__ __forceinline__ void store_out<__nv_bfloat16>(void* dst, int64_t idx, float v) {
  ((__nv_bfloat16*)dst)[idx] = __float2bfloat16_rn(v);
}
template <>
__device__ __forceinline__ void store_out<__half>(void* dst, int64_t idx, float v) {
  ((__half*)dst)[idx] = __float2half_rn(v);
}

// same, through an explicit st.global (for pointers whose provenance the compiler cannot see)
template <typename T>
__device__ __forceinline__ void store_out_global(T* p, float v);
template <>
__device__ __forceinline__ void store_out_global<float>(float* p, float v) {
  asm volatile("st.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
template <>
__device__ __forceinline__ void store_out_global<__nv_bfloat16>(__nv_bfloat16* p, float v) {
  const unsigned short h = __bfloat16_as_ushort(__float2bfloat16_rn(v));
  asm volatile("st.global.u16 [%0], %1;" ::"l"(p), "h"(h) : "memory");
}
template <>
__device__ __forceinline__ void store_out_global<__half>(__half* p, float v) {
  const unsigned short h = __half_as_ushort(__float2half_rn(v));
  asm volatile("st.global.u16 [%0], %1;" ::"l"(p), "h"(h) : "memory");
}

// The frame's gray mean (torchvision's contrast blend) is accumulated in 2^-22 fixed point: integer sums are exact,
// so the mean does not depend on the band count, the thread mapping or which resize kernel produced the pixels.
constexpr float kGrayFix = 4194304.0f;  // 2^22: a thread sums <= 1023 pixels in 32 bits
__device__ __forceinline__ unsigned gray_fix(float r, float g, float b) { return __float2uint_rn(gray_of(r, g, b) * kGrayFix); }
__device__ __forceinline__ unsigned long long block_sum(unsigned long long v, unsigned long long* red /*[32]*/) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  unsigned long long t = 0ull;
  if (wid == 0) {
    t = lane < nw ? red[lane] : 0ull;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  }
  return t;  // valid in warp 0
}

// Visible box of one clip: canvas rows [by0,by1) x cols [bx0,bx1) hold resized rows
// [i_lo,i_hi) x cols [j_lo,j_hi) (mirrored in x when the clip is flipped).
struct Box {
  int oy, ox, i_lo, i_hi, j_lo, j_hi, by0, by1, bx0, bx1;
};
__device__ __forceinline__ Box clip_box(const DevPlan& P, int crop_dy, int crop_dx, bool flip) {
  Box b;
  b.oy = P.off_y + crop_dy;
  b.ox = P.off_x + crop_dx;
  b.i_lo = max(0, -b.oy);
  b.i_hi = max(b.i_lo, min(P.rh, P.cs - b.oy));
  b.j_lo = max(0, -b.ox);
  b.j_hi = max(b.j_lo, min(P.rw, P.cs - b.ox));
  b.by0 = b.i_lo + b.oy;
  b.by1 = b.i_hi + b.oy;
  if (!flip) {
    b.bx0 = b.j_lo + b.ox;
    b.bx1 = b.j_hi + b.ox;
  } else {
    b.bx0 = P.cs - (b.j_hi + b.ox);
    b.bx1 = P.cs - (b.j_lo + b.ox);
  }
  return b;
}


// Constant fill of the canvas rows/columns outside a band's content box (the normalised value of a
// zero pixel).  Runs of whole pad rows of a planar, row-contiguous layout go out as flat 16-byte stores.
template <typename DstT, int NT>
__device__ __forceinline__ void fill_pads(const DevPlan& P, const KArgs& A, const Box& B, int64_t dbase, int band, int nb,
                                          int i0, int i1, int tid) {
  const int cy0 = i0 + B.oy, cy1 = i1 + B.oy;            // content rows of this band
  const int Y0 = band == 0 ? 0 : cy0;
  const int Y1 = band == nb - 1 ? P.cs : cy1;
  float nbi[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) nbi[c] = A.normalize ? A.nbias[c] : 0.0f;
  constexpr int EPV = 16 / (int)sizeof(DstT);  // elements per 16-byte store
  const bool vec_ok = A.sx == 1 && A.sy == P.cs && (P.cs % EPV) == 0 && (A.sc % EPV) == 0 && (A.st % EPV) == 0 &&
                      (A.sb % EPV) == 0 && (((uintptr_t)A.dst) & 15) == 0;
#pragma unroll
  for (int part = 0; part < 2; ++part) {                 // pad rows above / below the band's content
    const int ya = part == 0 ? Y0 : cy1, yb = part == 0 ? cy0 : Y1;
    if (yb <= ya) continue;
    if (vec_ok) {
      const int nvec = (yb - ya) * (P.cs / EPV);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        DstT tmp[EPV];
#pragma unroll
        for (int k = 0; k < EPV; ++k) store_out<DstT>(tmp, k, nbi[c]);
        const uint4 val = *(const uint4*)tmp;
        uint4* d = (uint4*)((DstT*)A.dst + dbase + (int64_t)ya * A.sy + (int64_t)c * A.sc);
        for (int v = tid; v < nvec; v += NT) d[v] = val;
      }
    } else {
      for (int y = ya; y < yb; ++y)
        for (int x = tid; x < P.cs; x += NT) {
          const int64_t o = dbase + (int64_t)y * A.sy + (int64_t)x * A.sx;
#pragma unroll
          for (int c = 0; c < 3; ++c) store_out<DstT>(A.dst, o + c * A.sc, nbi[c]);
        }
    }
  }
  if (B.bx0 > 0 || B.bx1 < P.cs) {                       // pad columns beside the content (portrait sources)
    const int npad = B.bx0 + (P.cs - B.bx1);
    for (int y = cy0; y < cy1; ++y)
      for (int k = tid; k < npad; k += NT) {
        const int x = k < B.bx0 ? k : B.bx1 + (k - B.bx0);
        const int64_t o = dbase + (int64_t)y * A.sy + (int64_t)x * A.sx;
#pragma unroll
        for (int c = 0; c < 3; ++c) store_out<DstT>(A.dst, o + c * A.sc, nbi[c]);
      }
  }
}

// ---------------------------------------------------------------------------------
// K0: clip maximum (only for crop geometries, where K1 does not read every source pixel)
// ---------------------------------------------------------------------------------
template <typename SrcT>
__global__ void clip_max_kernel(DevPlan P, KArgs A) {
  const int frame = blockIdx.y;
  const int clip = frame / A.T;
  if (A.params[clip].flags & NEXAR_RANGE_255) {  // byte-range values: divided by 255 whatever the maximum
    if (threadIdx.x == 0) atomicOr(&A.clip_max[clip], 1u);
    return;
  }
  const char* base = (const char*)A.src + A.frame_offsets[frame];
  const int n = P.src_w * 3;
  float m = -INFINITY;
  for (int y = blockIdx.x; y < P.src_h; y += gridDim.x) {
    const SrcT* row = (const SrcT*)(base + (int64_t)y * A.src_row_stride);
    for (int e = threadIdx.x; e < n; e += blockDim.x) m = fmaxf(m, (float)row[e]);
  }
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 1.0f) atomicOr(&A.clip_max[clip], 1u);
}

// ---------------------------------------------------------------------------------
// K1 (general variant): output-stationary separable resample.  Any geometry
// (down- or up-scale, any width), uint8 or float32 source.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ uint2 pack_q21(float r, float g, float b);

template <typename SrcT, typename DstT>
__device__ __forceinline__ void resize_general_body(const DevPlan& P, const KArgs& A, int frame, int band, int nb, float* vbuf,
                                                    unsigned long long* red) {
  const int clip = frame / A.T;
  const int t = frame - clip * A.T;
  const NexarClipParams* cp = A.params + clip;
  const unsigned flags = cp->flags;
  float scale;
  if (A.pass == 0) {
    scale = 1.0f / 255.0f;
  } else {
    const bool big = A.clip_max[clip] != 0u;
    if (A.pass == 1 && big) return;
    scale = big ? 1.0f / 255.0f : 1.0f;
  }
  const bool flip = flags & NEXAR_FLIP, aug = flags & NEXAR_AUG;
  const Box B = clip_box(P, cp->crop_dy, cp->crop_dx, flip);
  const int per = (B.i_hi - B.i_lo + nb - 1) / nb;
  const int i0 = min(B.i_hi, B.i_lo + band * per), i1 = min(B.i_hi, i0 + per);
  const char* fbase = (const char*)A.src + A.frame_offsets[frame];
  const int W3 = P.src_w * 3;
  const float bright = cp->brightness;
  float nsc[3], nbi[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    nsc[c] = A.normalize ? A.nscale[c] : 1.0f;
    nbi[c] = A.normalize ? A.nbias[c] : 0.0f;
  }
  const int64_t dbase = (int64_t)clip * A.sb + (int64_t)t * A.st;
  float vmax = (flags & NEXAR_RANGE_255) ? INFINITY : -INFINITY;  // byte-range clips count as "max > 1" from the start
  unsigned long long gsum = 0ull;  // one thread may cover many pixels here

  for (int i = i0; i < i1; ++i) {
    const int ys = P.ystart[i], yc = P.ycount[i];
    const float* wy = P.ywt + (size_t)i * P.ky;
    for (int e = threadIdx.x; e < W3; e += blockDim.x) {
      float acc = 0.0f;
      for (int k = 0; k < yc; ++k) {
        const float v = (float)((const SrcT*)(fbase + (int64_t)(ys + k) * A.src_row_stride))[e];
        vmax = fmaxf(vmax, v);
        acc = fmaf(wy[k], v, acc);
      }
      vbuf[e] = acc;
    }
    __syncthreads();
    const int y = i + B.oy;
    for (int j = B.j_lo + threadIdx.x; j < B.j_hi; j += blockDim.x) {
      const int xs = P.xstart[j], xc = P.xcount[j];
      const float* wx = P.xwt + (size_t)j * P.kx;
      float r = 0.0f, g = 0.0f, b = 0.0f;
      for (int k = 0; k < xc; ++k) {
        const float w = wx[k];
        const float* p = vbuf + (xs + k) * 3;
        r = fmaf(w, p[0], r);
        g = fmaf(w, p[1], g);
        b = fmaf(w, p[2], b);
      }
      r *= scale;
      g *= scale;
      b *= scale;
      int x = j + B.ox;
      if (flip) x = P.cs - 1 - x;
      if (aug) {
        r = clamp01(__fmul_rn(bright, r));
        g = clamp01(__fmul_rn(bright, g));
        b = clamp01(__fmul_rn(bright, b));
        gsum += gray_fix(r, g, b);
        A.inter[((size_t)frame * A.bh + (y - B.by0)) * A.bw + (x - B.bx0)] = pack_q21(r, g, b);
      } else {
        const int64_t o = dbase + (int64_t)y * A.sy + (int64_t)x * A.sx;
        store_out<DstT>(A.dst, o, fmaf(r, nsc[0], nbi[0]));
        store_out<DstT>(A.dst, o + A.sc, fmaf(g, nsc[1], nbi[1]));
        store_out<DstT>(A.dst, o + 2 * A.sc, fmaf(b, nsc[2], nbi[2]));
      }
    }
    __syncthreads();
  }

  if (!aug) {
    // zero-padded canvas outside the box -> normalised pad value
    const int Y0 = band == 0 ? 0 : i0 + B.oy;
    const int Y1 = band == nb - 1 ? P.cs : i1 + B.oy;
    const int cy0 = i0 + B.oy, cy1 = i1 + B.oy;  // content rows of this band
    for (int y = Y0; y < Y1; ++y) {
      const bool content_row = (y >= cy0 && y < cy1);
      for (int x = threadIdx.x; x < P.cs; x += blockDim.x) {
        if (content_row && x >= B.bx0 && x < B.bx1) continue;
        const int64_t o = dbase + (int64_t)y * A.sy + (int64_t)x * A.sx;
#pragma unroll
        for (int c = 0; c < 3; ++c) store_out<DstT>(A.dst, o + c * A.sc, nbi[c]);
      }
    }
  }

  if (A.pass == 0) {
    for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    if ((threadIdx.x & 31) == 0 && vmax > 1.0f) atomicOr(&A.clip_max[clip], 1u);
  }
  if (aug) {
    const unsigned long long s = block_sum(gsum, red);
    if (threadIdx.x == 0) A.gray_partial[((size_t)(scale == 1.0f) * A.n_frames + frame) * kMaxBands + band] = s;
  }
}

template <typename SrcT, typename DstT>
__global__ void __launch_bounds__(256) resize_general_kernel(DevPlan P, KArgs A) {
  extern __shared__ float vbuf[];  // [src_w*3] vertical-pass result of the current resized row
  __shared__ unsigned long long red[32];
  resize_general_body<SrcT, DstT>(P, A, blockIdx.y, blockIdx.x, gridDim.x, vbuf, red);
}


// ---------------------------------------------------------------------------------
// K1 (fast variant): input-stationary fixed-point vertical pass + fixed-point horizontal pass, both on dp2a.
//
// Down-scaling (>= 2x vertically) uint8 frames whose rows are a multiple of 16 bytes.  A CTA owns
// one band of resized rows of one frame and streams the source rows it needs exactly once, two rows
// per step.  Every thread keeps one 16-byte column chunk: 128-bit coalesced streaming loads through a running
// pointer ([pointer + immediate] when the row stride is a compile-time constant), two pairs ahead in registers
// (ping-pong), while thread 0 pushes the rows LOOKAHEAD pairs ahead into L2 through the bulk-copy engine
// (cp.async.bulk.prefetch.L2).  The two rows' bytes are interleaved with PRMT and fed to dp2a against the
// 15-bit fixed-point taps of the (at most two) output rows alive at that height.  The per-pair control words
// (taps, begin/flush flags) sit in shared memory and are read one pair ahead with a uniform address, so no
// branch waits on its own load.  A finished row is rounded to 15-bit fixed point (value * 128) and staged in
// shared memory (double buffered); every warp then arrives on an mbarrier and goes on with the NEXT row pair,
// and only after that waits (by then for free) and resamples the staged row horizontally, one output pixel per
// thread: the staged (R0 G0)(B0 R1)(G1 B1) words are regrouped per channel with PRMT and dp2a'd against the
// horizontal taps, which are 15-bit too and stored as byte pairs (low bytes | high bytes, see build_fast_tables):
// value * 2^15 * sum(taps) = hi * 256 + lo.  Error of the fixed-point steps against an exact evaluation (720p -> 224
// noise): max < 3e-5 of full scale (bound: 2 x weights 2^-16 * 255 * taps/2 + staging 2^-8 in 0..255 units;
// gate: 1/255 before, 1e-3 after normalisation).
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void l2_prefetch_bulk(const void* p, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
// streaming 128-bit load of source bytes (evict-first: every byte is used once)
__device__ __forceinline__ uint4 ld_stream(const char* base, unsigned off) { return __ldcs((const uint4*)(base + off)); }

constexpr int kFastMinB = 3;    // CTAs per SM of the 256-thread instances (the wider ones take 2)
constexpr int kLookahead = 4;   // row pairs ahead pushed into L2 by the bulk-prefetch engine (multiple of 4)

// table entry .w bits
#define NEXAR_E_EMIT 1u
#define NEXAR_E_SLOT 2u
#define NEXAR_E_BEGIN0 4u
#define NEXAR_E_BEGIN1 8u
#define NEXAR_E_ROWSHIFT 4

// ---- mbarrier primitives ------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
               :: "r"(bar), "r"(parity) : "memory");
}

// ---- the 8-byte intermediate pixel of augmented clips -----------------------------------------------------------
// Stage 1 (K1 -> K2, brightness-adjusted): three 21-bit fixed-point channels packed into 64 bits (step 4.8e-7).
// Stage 2 (K2 -> K3, colour-adjusted, "q15"): four uint16 (R, G, B, spare), each 0x8000 | round(v * 32767): with that
// top bit set, ONE byte permute turns a stored value into the float 1 + q / 32768 (bits 0x3F800000 | q << 8), so the
// affine gather pays one PRMT per sample instead of an integer-to-float conversion, and the constant 1 is taken out
// once per pixel (see geometry_kernel).  Quantisation step 3.05e-5 of full scale (gate: 2.25e-4 after the division by std).
// (Measured: plain uint16 unpacked by I2F.U16 makes the geometry kernel 20 % slower; the conversion pipe runs at a
// quarter of the ALU rate.)
constexpr float kQ21 = 2097151.0f;                  // 2^21 - 1
constexpr float kQ21Inv = 1.0f / 2097151.0f;
__device__ __forceinline__ uint2 pack_q21(float r, float g, float b) {
  // float_bits(v * (2^21 - 1) + 2^23) = 0x4B000000 + round(v * (2^21 - 1))
  const unsigned qr = __float_as_uint(fmaf(r, kQ21, 8388608.0f)) & 0x1FFFFFu;
  const unsigned qg = __float_as_uint(fmaf(g, kQ21, 8388608.0f)) & 0x1FFFFFu;
  const unsigned qb = __float_as_uint(fmaf(b, kQ21, 8388608.0f)) & 0x1FFFFFu;
  return make_uint2(qr | (qg << 21), (qg >> 11) | (qb << 10));
}
constexpr float kQ15 = 32767.0f;
constexpr float kQ15Magic = 8388608.0f + 32768.0f;  // low 16 bits of float_bits(v * 32767 + magic) = 0x8000 | round(v * 32767)
constexpr float kS2Inv = 32768.0f / 32767.0f;       // v = (F - 1) * kS2Inv: sum_content(w * v) = kS2Inv * sum(w * F) + kS2Off * sum(w)
constexpr float kS2Off = -kS2Inv;
__device__ __forceinline__ float q15_r(uint2 v) { return __uint_as_float(__byte_perm(v.x, 0x3F000000u, 0x7104)); }
__device__ __forceinline__ float q15_g(uint2 v) { return __uint_as_float(__byte_perm(v.x, 0x3F000000u, 0x7324)); }
__device__ __forceinline__ float q15_b(uint2 v) { return __uint_as_float(__byte_perm(v.y, 0x3F000000u, 0x7104)); }
__device__ __forceinline__ uint2 pack_q15(float r, float g, float b) {
  const unsigned qr = __float_as_uint(fmaf(r, kQ15, kQ15Magic));
  const unsigned qg = __float_as_uint(fmaf(g, kQ15, kQ15Magic));
  const unsigned qb = __float_as_uint(fmaf(b, kQ15, kQ15Magic));
  return make_uint2(__byte_perm(qr, qg, 0x5410), qb & 0xFFFFu);
}

__device__ __forceinline__ void write_frame_info(const DevPlan& P, const KArgs& A, int frame, int slot, int nbands);

template <int KX, int NT, int MINB, int RS, typename DstT, bool AL4>
__global__ void __launch_bounds__(NT, MINB)
resize_fast_kernel(const __grid_constant__ DevPlan P, const __grid_constant__ KArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ unsigned long long red[32];
  __shared__ __align__(8) unsigned long long rowbar;  // "row staged" barrier: one arrival per warp, waited on one pair later
  constexpr int LA = kLookahead;
  const int tid = threadIdx.x;
  // Programmatic dependent launch: the colour kernel's CTAs may be scheduled as soon as every CTA of this grid has
  // started, i.e. into the SM slots this grid's last wave leaves empty; they synchronise per frame through frame_done.
  asm volatile("griddepcontrol.launch_dependents;");
  const int frame = blockIdx.y;
  const int clip = frame / A.T;
  const int t = frame - clip * A.T;
  const NexarClipParams* cp = A.params + clip;
  const unsigned flags = cp->flags;
  float scale;
  if (A.pass == 0) {
    scale = 1.0f / 255.0f;
  } else {
    const bool big = A.clip_max[clip] != 0u;
    if (A.pass == 1 && big) return;
    scale = big ? 1.0f / 255.0f : 1.0f;
  }
  const bool flip = flags & NEXAR_FLIP, aug = flags & NEXAR_AUG;
  const Box B = clip_box(P, cp->crop_dy, cp->crop_dx, flip);
  const int nb = gridDim.x, band = blockIdx.x;
  const int per = (B.i_hi - B.i_lo + nb - 1) / nb;
  const int i0 = min(B.i_hi, B.i_lo + band * per), i1 = min(B.i_hi, i0 + per);
  const int W3 = P.src_w * 3;
  const int nchunks = W3 >> 4;
  const int vstride = (W3 + KX * 3 + 15) & ~7;  // uint16 elements per staging buffer (16-byte multiple)
  unsigned short* vb = (unsigned short*)smem_raw;
  for (int e = W3 + tid; e < vstride; e += NT) vb[e] = vb[vstride + e] = 0;  // zero tail read by the padded taps

  const int64_t dbase = (int64_t)clip * A.sb + (int64_t)t * A.st;
  unsigned gsum = 0u;
  unsigned orv = 0u;

  if (i0 < i1) {
    // ---- horizontal taps of this thread's output pixel (registers) ----
    const int nj = B.j_hi - B.j_lo;
    const bool hth = tid < nj;
    const int j = B.j_lo + (hth ? tid : 0);
    // The taps live in shared memory as dp2a operands (two 15-bit taps per word, see build_fast_tables), NG uint4
    // groups per thread laid out group-major so that a warp's LDS.128 is conflict-free.
    constexpr int NW = KX / 2, NG = (NW + 3) / 4;
    uint4* const wsm = (uint4*)(smem_raw + 2u * (unsigned)vstride * 2u);
    {
      unsigned wtmp[4 * NG];
#pragma unroll
      for (int k = 0; k < 4 * NG; ++k) wtmp[k] = (k < NW && hth) ? P.xw16[(size_t)j * NW + k] : 0u;
#pragma unroll
      for (int g = 0; g < NG; ++g) wsm[g * NT + tid] = make_uint4(wtmp[4 * g], wtmp[4 * g + 1], wtmp[4 * g + 2], wtmp[4 * g + 3]);
    }
    const unsigned hbyte = (unsigned)(P.xstart_al[j] * 3) * 2u;  // byte offset of the first tap in a staging row
    int xo = j + B.ox;
    if (flip) xo = P.cs - 1 - xo;
    const float post = scale * (1.0f / (128.0f * 32768.0f));
    // where this frame's pixels go (uniform base; the per-thread column and the row are added per output row)
    uint2* const ibase = A.inter + ((int64_t)frame * A.bh - B.by0) * A.bw - B.bx0;  // 8-byte q15 pixels
    DstT* const obase = (DstT*)A.dst + dbase;

    // ---- vertical pass state ----
    const unsigned rnd = 1u << 7;  // P.shift == 15: staging value = (acc + 128) >> 8
    unsigned acc0[16], acc1[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) acc0[q] = acc1[q] = rnd;
    const int p0 = P.ystart[i0] >> 1;
    const int plast = (P.ystart[i1 - 1] + P.ycount[i1 - 1] - 1) >> 1;  // inclusive
    const int chunk = min(tid, nchunks - 1);  // surplus threads shadow the last chunk (no divergence); they never stage
    const bool vstore = tid < nchunks;
    const char* frame_base = (const char*)A.src + A.frame_offsets[frame];
    // RS > 0: the row stride is a compile-time constant, so every load below is [pointer + immediate]
    const unsigned rs = RS > 0 ? (unsigned)RS : (unsigned)A.src_row_stride;
    const unsigned vbytes = (unsigned)vstride * 2u;
    unsigned bufoff = 0u;  // byte offset of the current staging buffer (uniform)

    // this thread's 16 bytes of row 2p (running pointer, advanced once per two pairs); pairs p+2 / p+3 are
    // fetched at fixed row offsets from it, and nothing is fetched past the band's last pair
    const char* ptr = frame_base + (size_t)chunk * 16u + (size_t)(2 * p0) * rs;
    uint4 a0 = ld_stream(ptr, 0u), b0 = ld_stream(ptr, rs);
    uint4 a1 = a0, b1 = b0;
    if (p0 + 1 <= plast) {
      a1 = ld_stream(ptr, 2u * rs);
      b1 = ld_stream(ptr, 3u * rs);
    }
    // the band's control words, staged in shared memory: the loop reads them with a uniform address, one pair ahead
    uint4* const ctl = (uint4*)(wsm + NG * NT);
    for (int e = tid; e <= plast - p0 + 1; e += NT) ctl[e] = __ldg(P.pairs + p0 + e);  // table has a spare entry
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&rowbar);
    if (tid == 0) {
      mbar_init(bar, NT / 32);
      mbar_fence_init();
    }
    __syncthreads();
    unsigned phase = 0u;  // parity of the barrier phase the next wait is for
    int pend = -1;        // output row staged but not yet resampled horizontally (-1: none)
    unsigned pbuf = 0u;   // its staging buffer
    uint4 e_nx = ctl[0];
    const uint4* tp = ctl + 1;
    if (tid < 32) {
      const int q0 = p0 + 2, q1 = min(p0 + LA + 3, plast);
      if (tid == 0 && q1 >= q0)
        l2_prefetch_bulk(frame_base + (size_t)(2 * q0) * rs, (unsigned)min((int64_t)(2 * (q1 - q0 + 1)) * rs, (int64_t)P.src_h * rs - (int64_t)(2 * q0) * rs));
    }

#define NEXAR_ACCUM(ACC, WV)                                 \
  {                                                          \
    _Pragma("unroll") for (int q = 0; q < 4; ++q) {          \
      ACC[4 * q + 0] = __dp2a_lo(WV, lo[q], ACC[4 * q + 0]); \
      ACC[4 * q + 1] = __dp2a_hi(WV, lo[q], ACC[4 * q + 1]); \
      ACC[4 * q + 2] = __dp2a_lo(WV, hi[q], ACC[4 * q + 2]); \
      ACC[4 * q + 3] = __dp2a_hi(WV, hi[q], ACC[4 * q + 3]); \
    }                                                        \
  }
#define NEXAR_ACCUM_BEGIN(ACC, WV)                                                   \
  {                                                                                  \
    unsigned wv_; /* pin the tap pair in ONE vector register (else it is re-materialised per accumulator) */ \
    asm volatile("mov.b32 %0, %1;" : "=r"(wv_) : "r"(WV));                           \
    _Pragma("unroll") for (int q = 0; q < 4; ++q) {                                  \
      ACC[4 * q + 0] = __dp2a_lo(wv_, lo[q], rnd);                                   \
      ACC[4 * q + 1] = __dp2a_hi(wv_, lo[q], rnd);                                   \
      ACC[4 * q + 2] = __dp2a_lo(wv_, hi[q], rnd);                                   \
      ACC[4 * q + 3] = __dp2a_hi(wv_, hi[q], rnd);                                   \
    }                                                                                \
  }
#define NEXAR_STAGE(ACC)                                                                      \
  {                                                                                           \
    unsigned w_[8];                                                                           \
    _Pragma("unroll") for (int q = 0; q < 8; ++q)                                             \
        w_[q] = __byte_perm(ACC[2 * q], ACC[2 * q + 1], 0x6521); /* (a >> 8) | (b >> 8) << 16 */ \
    if (vstore) {                                                                             \
      uint4* d_ = (uint4*)(smem_raw + bufoff + (unsigned)tid * 32u);                          \
      d_[0] = make_uint4(w_[0], w_[1], w_[2], w_[3]);                                         \
      d_[1] = make_uint4(w_[4], w_[5], w_[6], w_[7]);                                         \
    }                                                                                         \
  }
// horizontal pass of one staged row (thread = output pixel, three channels)
#define NEXAR_HORIZ(ROW, BUF)                                                                              \
  {                                                                                                        \
    if (hth) {                                                                                         \
      const unsigned* src = (const unsigned*)(smem_raw + (BUF) + hbyte);                              \
      /* two taps per step: regroup (R0 G0)(B0 R1)(G1 B1) into per-channel pairs, dp2a against the low and */ \
      /* the high tap bytes; value * 2^15 * sum(taps) = hi * 256 + lo (< 2^31) */                     \
      unsigned rl = 0u, rh = 0u, gl = 0u, gh = 0u, bl_ = 0u, bh = 0u;                                  \
      uint4 wq = wsm[tid];                                                                             \
      unsigned wv[AL4 ? 3 * NW + 1 : 1]; /* AL4: the whole window, fetched with 8-byte loads */        \
      if constexpr (AL4) {                                                                             \
        _Pragma("unroll") for (int k = 0; k < (3 * NW + 1) / 2; ++k) {                                 \
          const uint2 t_ = ((const uint2*)src)[k];                                                     \
          wv[2 * k] = t_.x; wv[2 * k + 1] = t_.y;                                                      \
        }                                                                                              \
      }                                                                                                \
      _Pragma("unroll") for (int m = 0; m < NW; ++m) {                                                 \
        const unsigned w0 = AL4 ? wv[3 * m] : src[3 * m], w1 = AL4 ? wv[3 * m + 1] : src[3 * m + 1],   \
                       w2 = AL4 ? wv[3 * m + 2] : src[3 * m + 2];                                      \
        const unsigned ww = (m & 3) == 0 ? wq.x : (m & 3) == 1 ? wq.y : (m & 3) == 2 ? wq.z : wq.w;    \
        const unsigned rr = __byte_perm(w0, w1, 0x7610), gg = __byte_perm(w0, w2, 0x5432),             \
                       bb = __byte_perm(w1, w2, 0x7610);                                               \
        rl = __dp2a_lo(rr, ww, rl); rh = __dp2a_hi(rr, ww, rh);                                        \
        gl = __dp2a_lo(gg, ww, gl); gh = __dp2a_hi(gg, ww, gh);                                        \
        bl_ = __dp2a_lo(bb, ww, bl_); bh = __dp2a_hi(bb, ww, bh);                                      \
        if ((m & 3) == 3 && (m + 1) / 4 < NG) wq = wsm[((m + 1) / 4) * NT + tid];                      \
      }                                                                                                \
      float r = (float)(int)(rh * 256u + rl) * post;                                                   \
      float g = (float)(int)(gh * 256u + gl) * post;                                                   \
      float bl = (float)(int)(bh * 256u + bl_) * post;                                                 \
      const int y = (ROW) + B.oy;                                                                        \
      if (aug) {                                                                                       \
        const float bright = cp->brightness;                                                           \
        r = clamp01(__fmul_rn(bright, r));                                                             \
        g = clamp01(__fmul_rn(bright, g));                                                             \
        bl = clamp01(__fmul_rn(bright, bl));                                                           \
        gsum += gray_fix(r, g, bl);                                                                     \
        ibase[y * A.bw + xo] = pack_q21(r, g, bl);                                                      \
      } else {                                                                                         \
        DstT* const o = obase + ((int64_t)y * A.sy + (int64_t)xo * A.sx);                              \
        if (A.normalize) {                                                                             \
          r = fmaf(r, A.nscale[0], A.nbias[0]);                                                        \
          g = fmaf(g, A.nscale[1], A.nbias[1]);                                                        \
          bl = fmaf(bl, A.nscale[2], A.nbias[2]);                                                      \
        }                                                                                              \
        store_out<DstT>(o, 0, r);                                                                      \
        store_out<DstT>(o, A.sc, g);                                                                   \
        store_out<DstT>(o, 2 * A.sc, bl);                                                              \
      }                                                                                                \
    }                                                                                                  \
  }
// One row pair: CA/CB hold rows 2p / 2p+1 of this thread's chunk.  As soon as their bytes have been
// interleaved into lo/hi the same registers are refilled with pair p+2 (two register sets ping-pong, so
// every load has almost two iterations to land).
#define NEXAR_PAIR(CA, CB, ROFF)                                                                               \
  {                                                                                                        \
    const unsigned ex = e_nx.x, ey = e_nx.y, ez = e_nx.z;                                                  \
    e_nx = *tp; /* control words of the next pair, one iteration ahead (table has a spare entry) */        \
    ++tp;                                                                                                  \
    orv |= (CA.x | CA.y) | (CA.z | CA.w) | (CB.x | CB.y) | (CB.z | CB.w);                                  \
    unsigned lo[4], hi[4];                                                                                 \
    lo[0] = __byte_perm(CA.x, CB.x, 0x5140); hi[0] = __byte_perm(CA.x, CB.x, 0x7362);                      \
    lo[1] = __byte_perm(CA.y, CB.y, 0x5140); hi[1] = __byte_perm(CA.y, CB.y, 0x7362);                      \
    lo[2] = __byte_perm(CA.z, CB.z, 0x5140); hi[2] = __byte_perm(CA.z, CB.z, 0x7362);                      \
    lo[3] = __byte_perm(CA.w, CB.w, 0x5140); hi[3] = __byte_perm(CA.w, CB.w, 0x7362);                      \
    if (p + 2 <= plast) { /* refill with pair p+2 */                                                      \
      CA = ld_stream(ptr, (unsigned)(ROFF) * rs);                                                          \
      CB = ld_stream(ptr, (unsigned)(ROFF + 1) * rs);                                                      \
    }                                                                                                      \
    /* both slots accumulate unconditionally (both are live in > 99 % of the pairs; an idle slot has zero taps): a   */ \
    /* slot restarts from the rounding constant when its row is flushed below, so no begin / idle tests are needed    */ \
    NEXAR_ACCUM(acc0, ex)                                                                                  \
    NEXAR_ACCUM(acc1, ey)                                                                                  \
    if (pend >= 0) { /* the row staged by an earlier pair: by now every warp has arrived, the wait is free */ \
      mbar_wait(bar, phase);                                                                               \
      phase ^= 1u;                                                                                         \
      NEXAR_HORIZ(pend, pbuf)                                                                              \
      pend = -1;                                                                                           \
    }                                                                                                      \
    if (ez & NEXAR_E_EMIT) { /* an output row finished with this pair */                                  \
      const int row = (int)((ez >> NEXAR_E_ROWSHIFT) & 0xFFFu);                                            \
      const bool s1 = (ez & NEXAR_E_SLOT) != 0u;                                                          \
      if (row >= i0 && row < i1) {                                                                         \
        if (s1) NEXAR_STAGE(acc1) else NEXAR_STAGE(acc0)                                                   \
        if (tid == 0) { /* once per output row (~S/2 pairs): push the next 4 pairs, LA ahead, into L2 */    \
          const int q0 = p + 1 + LA;                                                                       \
          if (q0 <= plast) {                                                                               \
            const int64_t o0 = (int64_t)(2 * q0) * rs;                                                     \
            l2_prefetch_bulk(frame_base + o0, (unsigned)min((int64_t)8 * rs, (int64_t)P.src_h * rs - o0)); \
          }                                                                                                \
        }                                                                                                  \
        __syncwarp();                                                                                      \
        if ((tid & 31) == 0) mbar_arrive(bar); /* release: this warp's part of the row is staged */        \
        pend = row;                                                                                        \
        pbuf = bufoff;                                                                                     \
        bufoff = vbytes - bufoff; /* other staging buffer */                                               \
      }                                                                                                    \
      /* the flushed slot restarts: rounding constant + the first tap of its next row when that shares this pair */ \
      const unsigned wpost = ez & 0xFFFF0000u;                                                             \
      if (s1) NEXAR_ACCUM_BEGIN(acc1, wpost) else NEXAR_ACCUM_BEGIN(acc0, wpost)                           \
    }                                                                                                      \
  }

    for (int p = p0; p <= plast; ++p) {
      NEXAR_PAIR(a0, b0, 4)
      if (++p > plast) break;
      NEXAR_PAIR(a1, b1, 6)
      ptr += 4u * rs;
    }
    if (pend >= 0) {
      mbar_wait(bar, phase);
      NEXAR_HORIZ(pend, pbuf)
    }
#undef NEXAR_HORIZ
#undef NEXAR_PAIR
#undef NEXAR_ACCUM
#undef NEXAR_ACCUM_BEGIN
#undef NEXAR_STAGE
  }

  if (!aug) fill_pads<DstT, NT>(P, A, B, dbase, band, nb, i0, i1, tid);
  if (A.pass == 0) {
    const bool big = (orv & 0xFEFEFEFEu) != 0u || (flags & NEXAR_RANGE_255) != 0u;
    if (__any_sync(0xffffffffu, big) && (tid & 31) == 0) atomicOr(&A.clip_max[clip], 1u);
  }
  if (aug) {
    const unsigned long long s = block_sum((unsigned long long)gsum, red);
    if (tid == 0) A.gray_partial[((size_t)(scale == 1.0f) * A.n_frames + frame) * kMaxBands + band] = s;
  }
  // K1.5 folded in: the last band of the frame to get here publishes the frame's constants for K2 / K3 (gray mean of
  // the "divided by 255" pass; clips whose maximum turns out to be <= 1 are redone by fixup_frame_kernel anyway)
  if (A.finfo_by_k1 && tid == 0) {
    __threadfence();
    if (atomicAdd(&A.frame_done[frame], 1u) == (unsigned)nb - 1u) {
      __threadfence();
      write_frame_info(P, A, frame, 0, nb);
      __threadfence();
      atomicExch(&A.frame_done[frame], kFrameReady);   // published: intermediate rows, clip flag and FrameInfo are visible
    }
  }
}

// ---------------------------------------------------------------------------------
// colour chain on one pixel: contrast -> saturation -> hue  (tv:_functional_tensor.py:181-321)
// ---------------------------------------------------------------------------------
struct ColourParams {
  float cmean, contrast, saturation, saturation_q, hue6;  // cmean = contrast_q * frame mean; hue6 = 6 * hue factor
};
// torchvision's formulas written for the instruction count: multiply-adds are contracted (1 ulp against tv's separately
// rounded _blend), and the hue rotation works in sextant units without the HSV detour:
//   H = (h6 + 6 * hue) mod 6 with h6 torchvision's un-normalised hue, and for every channel
//   out = minc + cr * f(H),  f_r = sat(|H - 3| - 1), f_g = sat(2 - |H - 2|), f_b = sat(2 - |H - 4|)
// which is _hsv2rgb's (v, q, p, p, t, v) table with v * s = cr = maxc - minc (tv:_functional_tensor.py:258-321).
// hue == 0: torchvision still runs RGB -> HSV -> RGB, which is the identity up to a few ulp; it is skipped (uniform per
// frame).  Measured against the oracle, which always runs it: < 1e-6.
__device__ __forceinline__ void colour_chain_tail(float& r, float& g, float& b, const ColourParams& c);
__device__ __forceinline__ void colour_chain(float& r, float& g, float& b, const ColourParams& c) {
  r = __saturatef(fmaf(c.contrast, r, c.cmean));
  g = __saturatef(fmaf(c.contrast, g, c.cmean));
  b = __saturatef(fmaf(c.contrast, b, c.cmean));
  colour_chain_tail(r, g, b, c);
}
// The same chain on a packed stage-1 pixel.  The three 21-bit fields are OR-ed into the mantissa of 2^23 (one logic
// operation each, no integer-to-float conversion): F = 2^23 + q, and the contrast blend absorbs both the scale and the
// offset: contrast * q / (2^21 - 1) + cmean = F * cq + (cmean - cq * 2^23), cq = contrast / (2^21 - 1).
__device__ __forceinline__ void colour_chain_q21(uint2 v, float& r, float& g, float& b, const ColourParams& c) {
  const float fr = __uint_as_float((v.x & 0x1FFFFFu) | 0x4B000000u);
  const float fg = __uint_as_float((__funnelshift_r(v.x, v.y, 21) & 0x1FFFFFu) | 0x4B000000u);
  const float fb = __uint_as_float((v.y >> 10) | 0x4B000000u);   // bit 31 of a stage-1 pixel is zero
  const float cq = c.contrast * kQ21Inv, c0 = fmaf(-cq, 8388608.0f, c.cmean);
  r = __saturatef(fmaf(fr, cq, c0));
  g = __saturatef(fmaf(fg, cq, c0));
  b = __saturatef(fmaf(fb, cq, c0));
  colour_chain_tail(r, g, b, c);
}
__device__ __forceinline__ void colour_chain_tail(float& r, float& g, float& b, const ColourParams& c) {
  const float gq = c.saturation_q * fmaf(0.114f, b, fmaf(0.587f, g, 0.2989f * r));
  r = __saturatef(fmaf(c.saturation, r, gq));
  g = __saturatef(fmaf(c.saturation, g, gq));
  b = __saturatef(fmaf(c.saturation, b, gq));
  if (c.hue6 != 0.0f) {
    const float maxc = fmaxf(r, fmaxf(g, b)), minc = fminf(r, fminf(g, b));
    const float cr = maxc - minc;
    const float inv = cr > 0.0f ? __fdividef(1.0f, cr) : 0.0f;
    const float mi = maxc * inv;
    const float rc = fmaf(-r, inv, mi), gc = fmaf(-g, inv, mi), bc = fmaf(-b, inv, mi);
    const float h6 = (maxc == r) ? (bc - gc) : (maxc == g) ? (2.0f + rc - bc) : (4.0f + gc - rc);
    float H = h6 + c.hue6;                     // in (-7, 11): fold into [0, 6)
    H -= 6.0f * floorf(H * (1.0f / 6.0f));
    r = fmaf(cr, __saturatef(fabsf(H - 3.0f) - 1.0f), minc);
    g = fmaf(cr, __saturatef(2.0f - fabsf(H - 2.0f)), minc);
    b = fmaf(cr, __saturatef(2.0f - fabsf(H - 4.0f)), minc);
  }
}

__device__ __forceinline__ float frame_mean(const KArgs& A, const DevPlan& P, int frame, int slot, int nbands) {
  const unsigned long long* gp = A.gray_partial + ((size_t)slot * A.n_frames + frame) * kMaxBands;
  unsigned long long s = 0ull;
  for (int b = 0; b < nbands; ++b) s += gp[b];
  return (float)((double)s / ((double)kGrayFix * (double)(P.cs * P.cs)));
}

// K1.5: the per-frame constants of K2 / K3.  Reduces the band partial sums to the frame's gray mean (fixed order:
// deterministic) and evaluates the colour a zero pad pixel takes after the colour chain.  One thread per frame: either
// the last band of the frame to finish the fast resize kernel, or frame_stats_kernel after the general one.
__device__ __forceinline__ void write_frame_info(const DevPlan& P, const KArgs& A, int frame, int slot, int nbands) {
  const int clip = frame / A.T;
  const NexarClipParams* cp = A.params + clip;
  FrameInfo fi;
  fi.flags = cp->flags;
  fi.reserved = 0;
  if (!(fi.flags & NEXAR_AUG)) {
    A.finfo[frame].flags = 0u;
    return;
  }
  ColourParams c;
  c.cmean = __fmul_rn(cp->contrast_q, frame_mean(A, P, frame, slot, nbands));
  c.contrast = cp->contrast;
  c.saturation = cp->saturation;
  c.saturation_q = cp->saturation_q;
  c.hue6 = 6.0f * cp->hue;
  float r = 0.0f, g = 0.0f, b = 0.0f;
  colour_chain(r, g, b, c);
  const Box B = clip_box(P, cp->crop_dy, cp->crop_dx, fi.flags & NEXAR_FLIP);
  fi.padr = r; fi.padg = g; fi.padb = b; fi.cmean = c.cmean;
  fi.by0 = B.by0; fi.by1 = B.by1; fi.bx0 = B.bx0; fi.bx1 = B.bx1;
#pragma unroll
  for (int k = 0; k < 6; ++k) fi.grid[k] = cp->grid[k];
  fi.contrast = c.contrast; fi.saturation = c.saturation; fi.saturation_q = c.saturation_q; fi.hue = c.hue6;
  A.finfo[frame] = fi;
}
__global__ void __launch_bounds__(128) frame_stats_kernel(const __grid_constant__ DevPlan P, const __grid_constant__ KArgs A, int nbands) {
  const int frame = blockIdx.x * blockDim.x + threadIdx.x;
  if (frame >= A.n_frames) return;
  write_frame_info(P, A, frame, A.clip_max[frame / A.T] != 0u ? 0 : 1, nbands);
}

// K2: contrast/saturation/hue in place on the frame's content box (which always fills the
// [bh][bw] allocation: letterbox shows every resized row, a crop shows exactly cs x cs of them), 8-byte q15 pixels.
constexpr int kColourPerThread = 8;
constexpr int kColMinB = 6;   // CTAs per SM (8 measured: no change)
// Wait until the resize kernel has published a frame (overlapped launch only).  Bounded: a stuck wait traps instead of
// hanging the device.
__device__ __forceinline__ void wait_frame_ready(const unsigned* flag) {
  unsigned v;
  unsigned long long t0 = 0ull;
  for (unsigned spins = 0;; ++spins) {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if (v == kFrameReady) return;
    __nanosleep(256);
    if ((spins & 4095u) == 4095u) {   // about once a millisecond: give up after 30 s of wall time (the producer is resident
      unsigned long long now;        // and running whenever a consumer CTA exists, so this only fires on a broken device)
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
      if (t0 == 0ull) t0 = now;
      else if (now - t0 > 30000000000ull) __trap();
    }
  }
}

__global__ void __launch_bounds__(256, kColMinB) colour_kernel(const __grid_constant__ DevPlan P, const __grid_constant__ KArgs A) {
  __shared__ unsigned go;
  int frame;
  if (A.overlap) {
    // Launched as a programmatic dependent of the resize kernel: these CTAs fill the SM slots its last wave leaves
    // empty, oldest frames first (almost always published already), and wait per frame for the publication.
    frame = (int)blockIdx.y;
    if (threadIdx.x == 0) {
      const int clip = frame / A.T;
      wait_frame_ready(A.frame_done + frame);
      unsigned run = 1u;
      if (A.pass == 4 && __ldcg(A.clip_max + clip) == 0u) {  // the clip flag is final only once all its frames are in
        for (int f = clip * A.T; f < (clip + 1) * A.T; ++f) wait_frame_ready(A.frame_done + f);
        run = __ldcg(A.clip_max + clip) != 0u;               // still 0: fixup_frame_kernel finishes that clip on its own
      }
      go = run;
    }
    __syncthreads();
    if (!go) return;
  } else {
    // K1 wrote the frames in ascending order, so the LAST ones are still in L2: walk them in descending order (and
    // K3 then starts with frame 0, which this kernel wrote last)
    frame = (int)(gridDim.y - 1u - blockIdx.y);
  }
  const float4* fi4 = (const float4*)(A.finfo + frame);
  // coherent loads (L2): in the overlapped launch the producer may still be running on other SMs
  const float4 st = __ldcg(fi4), q3 = __ldcg(fi4 + 3), q4 = __ldcg(fi4 + 4);   // pad colour + cmean | g4, g5, flags, contrast | sat, sat_q, 6 * hue, -
  if (!(__float_as_uint(q3.z) & NEXAR_AUG)) return;
  if (!A.overlap && A.pass == 4 && A.clip_max[frame / A.T] == 0u) return;  // fixup_frame_kernel finishes those clips on its own
  ColourParams c;
  c.cmean = st.w;
  c.contrast = q3.w;
  c.saturation = q4.x;
  c.saturation_q = q4.y;
  c.hue6 = q4.z;
  const int n = A.bh * A.bw;
  uint2* base = A.inter + (size_t)frame * n;
  const int i0 = blockIdx.x * (256 * kColourPerThread) + threadIdx.x;
  uint2 v[kColourPerThread];
#pragma unroll
  for (int k = 0; k < kColourPerThread; ++k)
    if (i0 + k * 256 < n) v[k] = __ldcg(base + i0 + k * 256);
#pragma unroll
  for (int k = 0; k < kColourPerThread; ++k)
    if (i0 + k * 256 < n) {
      float r, g, b;
      colour_chain_q21(v[k], r, g, b, c);
      base[i0 + k * 256] = pack_q15(r, g, b);
    }
}

// ---------------------------------------------------------------------------------
// K3: affine gather + effects + normalise + store
// ---------------------------------------------------------------------------------
__device__ __forceinline__ unsigned hash_u32(unsigned x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
// counter-based standard normal (statistical stand-in for torch.randn_like, nexar_video_aug.py:245)
__device__ __forceinline__ float gauss_noise(unsigned s0, unsigned s1, unsigned idx) {
  const unsigned a = hash_u32(idx * 2u + s0), b = hash_u32((idx * 2u + 1u) ^ s1);
  const float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);
  const float u2 = (float)(b >> 8) * (1.0f / 16777216.0f);
  return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

__device__ __forceinline__ void point_effects(float& r, float& g, float& b, const NexarClipParams* cp, unsigned flags,
                                              int y, int x) {
  if (flags & NEXAR_POSTERIZE) {
    const unsigned mask = (0xFFu << (8 - cp->posterize_bits)) & 0xFFu;
    r = __fdiv_rn((float)((unsigned)__fmul_rn(r, 255.0f) & mask), 255.0f);
    g = __fdiv_rn((float)((unsigned)__fmul_rn(g, 255.0f) & mask), 255.0f);
    b = __fdiv_rn((float)((unsigned)__fmul_rn(b, 255.0f) & mask), 255.0f);
  }
  if (flags & NEXAR_SOLARIZE) {
    const float th = cp->solarize_threshold;
    r = r >= th ? __fsub_rn(1.0f, r) : r;
    g = g >= th ? __fsub_rn(1.0f, g) : g;
    b = b >= th ? __fsub_rn(1.0f, b) : b;
  }
  if (flags & NEXAR_INVERT) {
    r = __fsub_rn(1.0f, r);
    g = __fsub_rn(1.0f, g);
    b = __fsub_rn(1.0f, b);
  }
  if (flags & NEXAR_CUTOUT) {
    for (int k = 0; k < cp->n_cutout; ++k) {
      const int top = cp->cutout[k][0], left = cp->cutout[k][1];
      if (y >= top && y < top + cp->cutout[k][2] && x >= left && x < left + cp->cutout[k][3]) r = g = b = 0.0f;
    }
  }
}

enum { GEO_GENERAL = 0, GEO_FILL = 1, GEO_INTERIOR = 2 };
constexpr unsigned kTailFlags = NEXAR_GRAYSCALE | NEXAR_NOISE | NEXAR_BLUR | NEXAR_POSTERIZE | NEXAR_SOLARIZE | NEXAR_INVERT | NEXAR_CUTOUT;

struct GeoPx {
  int o00, o01, o10, o11;                     // pixel offsets from the frame's canvas origin
  float w00, w01, w10, w11, m, wc;
};
constexpr int kMaxTileClasses = 1536;         // tiles per CTA whose class is kept in shared memory (more are classified on the fly)

// grayscale / noise of the augmentation tail (rare: kept out of line)
__device__ __noinline__ float3 tail_pre_effects(float r, float g, float b, const NexarClipParams* cp, unsigned flags, int frame,
                                                int idx, int cs) {
  if (flags & NEXAR_GRAYSCALE) r = g = b = gray_of(r, g, b);
  if (flags & NEXAR_NOISE) {
    const unsigned base = (unsigned)((frame * 3) * cs * cs + idx);
    r = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base), cp->noise_level, r));
    g = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base + cs * cs), cp->noise_level, g));
    b = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base + 2 * cs * cs), cp->noise_level, b));
  }
  return make_float3(r, g, b);
}
__device__ __noinline__ float3 tail_point_effects(float r, float g, float b, const NexarClipParams* cp, unsigned flags, int y, int x) {
  point_effects(r, g, b, cp, flags, y, x);
  return make_float3(r, g, b);
}

template <typename T>
__device__ __forceinline__ void store_pair(T* p, float a, float b);
template <>
__device__ __forceinline__ void store_pair<float>(float* p, float a, float b) {
  asm volatile("st.global.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}
template <>
__device__ __forceinline__ void store_pair<__nv_bfloat16>(__nv_bfloat16* p, float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  asm volatile("st.global.b32 [%0], %1;" ::"l"(p), "r"(*(const unsigned*)&h) : "memory");
}
template <>
__device__ __forceinline__ void store_pair<__half>(__half* p, float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  asm volatile("st.global.b32 [%0], %1;" ::"l"(p), "r"(*(const unsigned*)&h) : "memory");
}

// ---------------------------------------------------------------------------------
// Augmentation tail of fixup_frame_kernel: K1.5 + K2 + K3 of one frame inside the CTA of 256 threads that has just
// resampled all of it (rows B.i_lo .. B.i_hi, gray sum in slot 1).
//   phase B  contrast -> saturation -> hue in place on the frame's rows of the intermediate;
//   phase C  the OUTPUT in tiles of 32 x 4 pixels pulled from a shared counter: a warp owns one tile at a time, two
//            horizontally adjacent pixels per lane (one 32-bit bf16x2 / f16x2 / 64-bit float2 store per channel), classified
//            FILL / INTERIOR / general exactly like geometry_kernel; the four neighbours are 8-byte loads of the q15
//            intermediate (L2 / L1 hits: this CTA wrote them microseconds ago), unpacked with one PRMT per sample:
//              sum_canvas(w * img) = pad * (m - wc) + k * sum_content(w * F) - k * wc,   F = 1 + q / 32768, k = 32768 / 32767
//            with m the interpolated ones-mask and wc the total weight of the content neighbours; out = m * that (tv fill = 0).
// ---------------------------------------------------------------------------------
template <typename DstT>
__device__ __forceinline__ void fixup_colour_geometry(const DevPlan& P, const KArgs& A, const NexarClipParams* cp,
                                                      unsigned flags, int frame, int clip, int t, const Box& B) {
  constexpr int NT = 256;
  __shared__ float fconst[4];  // pad colour after the colour chain, contrast_q * gray mean
  __shared__ unsigned char tile_cls[kMaxTileClasses];
  __shared__ int tile_next[1];
  const int tid = threadIdx.x;
  __threadfence_block();       // the frame's gray sum is in global memory
  __syncthreads();
  ColourParams c;
  c.contrast = cp->contrast; c.saturation = cp->saturation; c.saturation_q = cp->saturation_q; c.hue6 = 6.0f * cp->hue;
  if (tid == 0) {
    c.cmean = __fmul_rn(cp->contrast_q, frame_mean(A, P, frame, 1, 1));
    float r = 0.0f, g = 0.0f, b = 0.0f;
    colour_chain(r, g, b, c);
    fconst[0] = r; fconst[1] = g; fconst[2] = b; fconst[3] = c.cmean;
  }
  __syncthreads();
  const float padr = fconst[0], padg = fconst[1], padb = fconst[2];
  c.cmean = fconst[3];
  // ---- phase B: colour chain in place on the frame's rows -------------------------------------------------------
  const int nrows = B.i_hi - B.i_lo, bwid = B.bx1 - B.bx0;
  uint2* const rows = A.inter + ((int64_t)frame * A.bh + (B.i_lo + B.oy - B.by0)) * A.bw;
  if (bwid == A.bw) {  // the content box fills the allocation (always, for a letterbox): one flat, coalesced sweep
    const int n = nrows * A.bw;
    constexpr int U = 4;
    for (int e0 = tid; e0 < n; e0 += U * NT) {
      uint2 v[U];
#pragma unroll
      for (int k = 0; k < U; ++k)
        if (e0 + k * NT < n) v[k] = rows[e0 + k * NT];
#pragma unroll
      for (int k = 0; k < U; ++k)
        if (e0 + k * NT < n) {
          float r, g, b;
          colour_chain_q21(v[k], r, g, b, c);
          rows[e0 + k * NT] = pack_q15(r, g, b);
        }
    }
  } else {
    for (int row = tid >> 5; row < nrows; row += NT / 32)
      for (int col = tid & 31; col < bwid; col += 32) {
        uint2* q = rows + row * A.bw + col;
        const uint2 v = *q;
        float r, g, b;
        colour_chain_q21(v, r, g, b, c);
        *q = pack_q15(r, g, b);
      }
  }
  // ---- tile classes of phase C (geometry only: done before the barrier so that it overlaps the wait) -------------------
  const int ngroups = (P.cs + 3) >> 2, tiles_x = (P.cs + 31) >> 5;
  const int ntiles = max(ngroups, 0) * tiles_x;
  auto classify = [&](int tx, int ty0) -> int {
    if (!(flags & NEXAR_AFFINE)) return GEO_GENERAL;
    const float fcs = (float)P.cs, half = 0.5f * fcs;
    const float g0 = cp->grid[0], g1 = cp->grid[1], g2 = cp->grid[2], g3 = cp->grid[3], g4 = cp->grid[4], g5 = cp->grid[5];
    // image of the tile centre +- the half extents of the tile under the linear part (a superset for tiles that stick
    // out of the canvas); 0.01 px of slack for rounding differences against the per-pixel evaluation
    const float ex = (15.5f * fabsf(g0) + 1.5f * fabsf(g1)) * half + 0.01f;
    const float ey = (15.5f * fabsf(g3) + 1.5f * fabsf(g4)) * half + 0.01f;
    const float xc = (float)(tx * 32 + 16) - half, yc = (float)(ty0 + 2) - half;
    const float sxc = fmaf(fmaf(yc, g1, xc * g0) + g2 + 1.0f, fcs, -1.0f) * 0.5f;
    const float syc = fmaf(fmaf(yc, g4, xc * g3) + g5 + 1.0f, fcs, -1.0f) * 0.5f;
    const float xmin = sxc - ex, xmax = sxc + ex, ymin = syc - ey, ymax = syc + ey;
    const float fby0 = (float)B.by0, fby1 = (float)B.by1, fbx0 = (float)B.bx0, fbx1 = (float)B.bx1;
    const bool inside = xmin >= 0.0f && xmax <= fcs - 1.0f && ymin >= 0.0f && ymax <= fcs - 1.0f;
    const bool outside_box = ymax + 1.0f < fby0 || ymin >= fby1 || xmax + 1.0f < fbx0 || xmin >= fbx1;
    const bool interior = xmin >= fbx0 && xmax <= fbx1 - 1.0f && ymin >= fby0 && ymax <= fby1 - 1.0f;
    return (inside && outside_box) ? GEO_FILL : interior ? GEO_INTERIOR : GEO_GENERAL;
  };
  for (int tile = tid; tile < min(ntiles, kMaxTileClasses); tile += NT) {
    const int gk = tile / tiles_x, tx = tile - gk * tiles_x;
    tile_cls[tile] = (unsigned char)classify(tx, gk * 4);
  }
  if (tid == 0) *tile_next = 0;
  __threadfence_block();       // the whole frame is colour-adjusted
  __syncthreads();
  // ---- phase C: affine gather + effects + normalise + store -------------------------------------------------------
  // Warp tile = 32 x 4 output pixels: lane -> (x pair = lane & 15, row = lane >> 4), two passes two rows apart.  The
  // frame's tiles (its row groups x the tile columns) were classified once, into shared memory, before the barrier above;
  // the warps then pull tiles from a shared counter (FILL tiles cost a few stores, general ones about 700 instructions).
  const int cs = P.cs;
  const int lane = tid & 31;
  const float half = (float)cs * 0.5f, fcs = (float)cs;
  const bool affine = (flags & NEXAR_AFFINE) != 0u;
  const float g0 = cp->grid[0], g1 = cp->grid[1], g2 = cp->grid[2], g3 = cp->grid[3], g4 = cp->grid[4], g5 = cp->grid[5];
  const int bw = A.bw;
  const uint2* const fr = A.inter + ((int64_t)frame * (A.bh * bw) - (B.by0 * bw + B.bx0));  // indexed by canvas (y, x)
  DstT* const ob = (DstT*)A.dst + ((int64_t)clip * A.sb + (int64_t)t * A.st);
  const int osy = (int)A.sy, osc = (int)A.sc, osx = (int)A.sx;
  const bool vec2 = A.sx == 1 && ((A.sy | A.sc | A.sb | A.st) & 1) == 0 && (((uintptr_t)A.dst) & (2 * sizeof(DstT) - 1)) == 0;
  const bool tail_fx = (flags & kTailFlags) != 0u;
  const int lx = (lane & 15) * 2, ly = lane >> 4;
  const float nsr = A.nscale[0], nsg = A.nscale[1], nsb = A.nscale[2], nbr = A.nbias[0], nbg = A.nbias[1], nbb = A.nbias[2];

  auto geo = [&](GeoPx& q, float xg0, float xg3, float yb, int x, int y, int cls) {
    q.m = 1.0f;
    if (affine) {
      // tv _gen_affine_grid + grid_sample(bilinear, zeros, align_corners=False) on [img | ones], img * mask
      const float gx = fmaf(yb, g1, xg0) + g2;
      const float gy = fmaf(yb, g4, xg3) + g5;
      const float ix = fmaf(gx + 1.0f, fcs, -1.0f) * 0.5f;
      const float iy = fmaf(gy + 1.0f, fcs, -1.0f) * 0.5f;
      const float x0f = floorf(ix), y0f = floorf(iy);
      const float wx1 = ix - x0f, wy1 = iy - y0f;
      const float wx0 = 1.0f - wx1, wy0 = 1.0f - wy1;
      if (cls == GEO_INTERIOR) {
        q.o00 = (int)y0f * bw + (int)x0f;   // the other three neighbours sit at +1, +bw, +bw+1
        q.w00 = wx0 * wy0; q.w01 = wx1 * wy0; q.w10 = wx0 * wy1; q.w11 = wx1 * wy1;
        q.wc = 1.0f;
      } else {
        // clamp before the int cast so wild matrices cannot overflow
        const int x0 = (int)fminf(fmaxf(x0f, -2.0f), fcs + 1.0f);
        const int yq = (int)fminf(fmaxf(y0f, -2.0f), fcs + 1.0f);
        const bool inx0 = (unsigned)x0 < (unsigned)cs, inx1 = (unsigned)(x0 + 1) < (unsigned)cs;
        const bool iny0 = (unsigned)yq < (unsigned)cs, iny1 = (unsigned)(yq + 1) < (unsigned)cs;
        const float ax0 = inx0 ? wx0 : 0.0f, ax1 = inx1 ? wx1 : 0.0f, ay0 = iny0 ? wy0 : 0.0f, ay1 = iny1 ? wy1 : 0.0f;
        q.m = (ax0 + ax1) * (ay0 + ay1);                      // interpolated ones-mask
        const bool cx0 = x0 >= B.bx0 && x0 < B.bx1, cx1 = x0 + 1 >= B.bx0 && x0 + 1 < B.bx1;
        const bool cy0 = yq >= B.by0 && yq < B.by1, cy1 = yq + 1 >= B.by0 && yq + 1 < B.by1;
        const float bx0w = cx0 ? wx0 : 0.0f, bx1w = cx1 ? wx1 : 0.0f, by0w = cy0 ? wy0 : 0.0f, by1w = cy1 ? wy1 : 0.0f;
        const int xc0 = min(max(x0, B.bx0), B.bx1 - 1), xc1 = min(max(x0 + 1, B.bx0), B.bx1 - 1);
        const int yc0 = min(max(yq, B.by0), B.by1 - 1) * bw, yc1 = min(max(yq + 1, B.by0), B.by1 - 1) * bw;
        q.o00 = yc0 + xc0; q.o01 = yc0 + xc1; q.o10 = yc1 + xc0; q.o11 = yc1 + xc1;
        q.w00 = bx0w * by0w; q.w01 = bx1w * by0w; q.w10 = bx0w * by1w; q.w11 = bx1w * by1w;
        q.wc = (bx0w + bx1w) * (by0w + by1w);
      }
    } else {
      // no affine: the pixel itself when it is content, the pad colour otherwise
      const bool in = y >= B.by0 && y < B.by1 && x >= B.bx0 && x < B.bx1;
      q.o00 = q.o01 = q.o10 = q.o11 = min(max(y, B.by0), B.by1 - 1) * bw + min(max(x, B.bx0), B.bx1 - 1);
      q.w00 = q.wc = in ? 1.0f : 0.0f;
      q.w01 = q.w10 = q.w11 = 0.0f;
    }
  };
  auto gather = [&](const GeoPx& q, int cls, uint2& v00, uint2& v01, uint2& v10, uint2& v11) {
    if (cls == GEO_INTERIOR) {  // one address, immediate offsets
      const uint2* p0 = fr + q.o00;
      const uint2* p1 = p0 + bw;
      v00 = p0[0]; v01 = p0[1]; v10 = p1[0]; v11 = p1[1];
    } else {
      v00 = fr[q.o00]; v01 = fr[q.o01]; v10 = fr[q.o10]; v11 = fr[q.o11];
    }
  };
  auto blend = [&](const GeoPx& q, const uint2& v00, const uint2& v01, const uint2& v10, const uint2& v11, int cls, float& r,
                   float& g, float& b) {
    const float sr = fmaf(q15_r(v11), q.w11, fmaf(q15_r(v10), q.w10, fmaf(q15_r(v01), q.w01, q15_r(v00) * q.w00)));
    const float sg = fmaf(q15_g(v11), q.w11, fmaf(q15_g(v10), q.w10, fmaf(q15_g(v01), q.w01, q15_g(v00) * q.w00)));
    const float sb = fmaf(q15_b(v11), q.w11, fmaf(q15_b(v10), q.w10, fmaf(q15_b(v01), q.w01, q15_b(v00) * q.w00)));
    if (cls == GEO_INTERIOR) {  // m = wc = 1
      r = fmaf(sr, kS2Inv, kS2Off);
      g = fmaf(sg, kS2Inv, kS2Off);
      b = fmaf(sb, kS2Inv, kS2Off);
    } else {
      const float t0 = kS2Off * q.wc, pm = q.m - q.wc;
      r = q.m * fmaf(sr, kS2Inv, fmaf(padr, pm, t0));
      g = q.m * fmaf(sg, kS2Inv, fmaf(padg, pm, t0));
      b = q.m * fmaf(sb, kS2Inv, fmaf(padb, pm, t0));
    }
  };

#pragma unroll 1
  for (;;) {
    int tile = 0;
    if (lane == 0) tile = atomicAdd(tile_next, 1);
    tile = __shfl_sync(0xffffffffu, tile, 0);
    if (tile >= ntiles) break;
    const int gk = tile / tiles_x, tx = tile - gk * tiles_x;
    const int ty0 = gk * 4;
    const int cls = tile < kMaxTileClasses ? (int)tile_cls[tile] : classify(tx, ty0);
    const int x = tx * 32 + lx;
    const bool has2 = x + 1 < cs;
    const float xb = (float)x - half + 0.5f;
    const float xg0a = xb * g0, xg3a = xb * g3, xg0b = (xb + 1.0f) * g0, xg3b = (xb + 1.0f) * g3;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int y = ty0 + ly + 2 * pass;
      if (y >= cs || x >= cs) break;  // lanes past the canvas idle until the warp pulls its next tile
      float ra = padr, ga = padg, ba = padb, rb = padr, gb = padg, bb = padb;
      if (cls != GEO_FILL) {
        const float yb = (float)y - half + 0.5f;
        GeoPx qa, qb;
        geo(qa, xg0a, xg3a, yb, x, y, cls);
        geo(qb, has2 ? xg0b : xg0a, has2 ? xg3b : xg3a, yb, has2 ? x + 1 : x, y, cls);
        uint2 a00, a01, a10, a11, b00, b01, b10, b11;
        gather(qa, cls, a00, a01, a10, a11);
        gather(qb, cls, b00, b01, b10, b11);
        blend(qa, a00, a01, a10, a11, cls, ra, ga, ba);
        blend(qb, b00, b01, b10, b11, cls, rb, gb, bb);
      }
      if (tail_fx) {
        const int idx = y * cs + x;
        float3 pa = tail_pre_effects(ra, ga, ba, cp, flags, frame, idx, cs);
        float3 pb = has2 ? tail_pre_effects(rb, gb, bb, cp, flags, frame, idx + 1, cs) : pa;
        if (flags & NEXAR_BLUR) {  // the blur kernel finishes the chain from the planar canvas
          float* cv = A.canvas + (size_t)frame * 3 * cs * cs;
          cv[idx] = pa.x; cv[cs * cs + idx] = pa.y; cv[2 * cs * cs + idx] = pa.z;
          if (has2) { cv[idx + 1] = pb.x; cv[cs * cs + idx + 1] = pb.y; cv[2 * cs * cs + idx + 1] = pb.z; }
          continue;
        }
        pa = tail_point_effects(pa.x, pa.y, pa.z, cp, flags, y, x);
        if (has2) pb = tail_point_effects(pb.x, pb.y, pb.z, cp, flags, y, x + 1);
        ra = pa.x; ga = pa.y; ba = pa.z; rb = pb.x; gb = pb.y; bb = pb.z;
      }
      // nscale / nbias are 1 / 0 when the output is not normalised
      ra = fmaf(ra, nsr, nbr); rb = fmaf(rb, nsr, nbr);
      ga = fmaf(ga, nsg, nbg); gb = fmaf(gb, nsg, nbg);
      ba = fmaf(ba, nsb, nbb); bb = fmaf(bb, nsb, nbb);
      const int off = y * osy + x * osx;
      if (vec2 && has2) {
        store_pair<DstT>(ob + off, ra, rb);
        store_pair<DstT>(ob + (off + osc), ga, gb);
        store_pair<DstT>(ob + (off + 2 * osc), ba, bb);
      } else {
        store_out_global<DstT>(ob + off, ra);
        store_out_global<DstT>(ob + (off + osc), ga);
        store_out_global<DstT>(ob + (off + 2 * osc), ba);
        if (has2) {
          store_out_global<DstT>(ob + (off + osx), rb);
          store_out_global<DstT>(ob + (off + osx + osc), gb);
          store_out_global<DstT>(ob + (off + osx + 2 * osc), bb);
        }
      }
    }
  }
}

// Second pass of the fast path: the clips whose maximum was <= 1 are NOT divided by 255 (nexar_video_aug.py:814).  Rare, so
// it is ONE launch of one CTA per frame that exits at once for every other clip: the general fp32 resample of the whole
// frame (values in [0,1] are below the resolution of the fixed-point staging) and, for augmented clips, fixup_colour_geometry.
template <typename SrcT, typename DstT>
__global__ void __launch_bounds__(256) fixup_frame_kernel(const __grid_constant__ DevPlan P, const __grid_constant__ KArgs A) {
  extern __shared__ float vbuf[];  // [src_w*3]
  __shared__ unsigned long long red[32];
  const int frame = blockIdx.x;
  const int clip = frame / A.T;
  // launched as a programmatic dependent of the resize kernel itself (batches without augmentation): the clip flags are
  // final only when that grid has completed
  if (A.overlap) asm volatile("griddepcontrol.wait;" ::: "memory");
  if (A.clip_max[clip] != 0u) return;
  resize_general_body<SrcT, DstT>(P, A, frame, 0, 1, vbuf, red);  // A.pass == 1: unscaled, gray sum in slot 1
  const NexarClipParams* cp = A.params + clip;
  const unsigned flags = cp->flags;
  if (flags & NEXAR_AUG) {
    const Box B = clip_box(P, cp->crop_dy, cp->crop_dx, (flags & NEXAR_FLIP) != 0u);
    fixup_colour_geometry<DstT>(P, A, cp, flags, frame, clip, frame - clip * A.T, B);
  }
}

// K3.  Every frame of a clip shares the clip's affine map, content box and flags, so the per-pixel geometry (source
// position, the four neighbour offsets, their weights, the interpolated ones-mask m and the content weight wc) is
// computed ONCE and reused for kGeoFrames consecutive frames of the clip; per frame only the pad colour changes.
// CTA = 8 warps, a warp owns a tile of 32 x 4 output pixels (lane -> x pair = lane & 15, row = lane >> 4, two passes two
// rows apart) x kGeoFrames frames: two horizontally adjacent pixels per lane, so every channel goes out as one 32-bit
// bf16x2 / f16x2 / 64-bit float2 store.  The tile is classified once, by every lane identically, from the image of its centre
// and the half extents of the affine map: FILL — maps strictly inside the canvas and entirely into the pad band beside
// the content: constant pad colour, no loads; INTERIOR — every bilinear neighbour is a content pixel (one address,
// weights as they are, m = wc = 1); otherwise the four addresses are clamped into the content box and the weights of
// neighbours that are pad or outside the canvas are zeroed.  The neighbours are 8-byte q15 pixels, one PRMT per sample:
//   sum_canvas(w * img) = pad * (m - wc) + k * sum_content(w * F) - k * wc,   F = 1 + q / 32768, k = 32768 / 32767
// and out = m * that (torchvision's fill = 0 multiplies the zero-padded sample by the interpolated mask once more).
// Offsets inside one clip of the intermediate and one frame of the destination are 32-bit (checked on the host).
constexpr int kGeoFrames = 4;   // frames of one clip per CTA
constexpr int kGeoMinB = 4;     // CTAs per SM
constexpr int kGeoPasses = 2;   // row passes per warp: the warp tile is 32 x (2 * passes) pixels
template <typename DstT, bool TAIL>
__global__ void __launch_bounds__(256, kGeoMinB) geometry_kernel(const __grid_constant__ DevPlan P, const __grid_constant__ KArgs A) {
  asm volatile("griddepcontrol.launch_dependents;");   // the fix-up launch may drain through this grid's last wave
  const int nchunk = (A.T + kGeoFrames - 1) / kGeoFrames;
  const int clip = blockIdx.z / nchunk;
  const int t0 = (blockIdx.z - clip * nchunk) * kGeoFrames, t1 = min(A.T, t0 + kGeoFrames);
  const int frame0 = clip * A.T + t0;
  const float4* fi4 = (const float4*)(A.finfo + frame0);
  const float4 q3 = __ldg(fi4 + 3);
  const unsigned flags = __float_as_uint(q3.z);
  if (!(flags & NEXAR_AUG)) return;
  if (A.pass == 4 && A.clip_max[clip] == 0u) return;  // fixup_frame_kernel finishes those clips on its own
  const int cs = P.cs;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tx0 = blockIdx.x * 32, ty0 = (blockIdx.y * 8 + warp) * (2 * kGeoPasses);
  const int x = tx0 + (lane & 15) * 2, ly = lane >> 4;
  if (ty0 >= cs) return;
  const float4 q2 = __ldg(fi4 + 2);
  const int4 bx = __ldg((const int4*)fi4 + 1);
  const NexarClipParams* cp = A.params + clip;   // only the rare tail effects read it
  struct { int by0, by1, bx0, bx1; } B = {bx.x, bx.y, bx.z, bx.w};
  const float half = (float)cs * 0.5f, fcs = (float)cs;
  const bool affine = (flags & NEXAR_AFFINE) != 0u;
  const float g0 = q2.x, g1 = q2.y, g2 = q2.z, g3 = q2.w, g4 = q3.x, g5 = q3.y;
  int cls = GEO_GENERAL;
  if (affine) {
    // image of the tile centre +- the half extents of the tile under the linear part (a superset for tiles that stick
    // out of the canvas); 0.01 px of slack for rounding differences against the per-pixel evaluation
    constexpr float hr = (float)kGeoPasses - 0.5f;  // half the tile's row extent, centre to centre
    const float xc = (float)(tx0 + 16) - half, yc = (float)(ty0 + kGeoPasses) - half;
    const float sxc = fmaf(fmaf(yc, g1, xc * g0) + g2 + 1.0f, fcs, -1.0f) * 0.5f;
    const float syc = fmaf(fmaf(yc, g4, xc * g3) + g5 + 1.0f, fcs, -1.0f) * 0.5f;
    const float ex = (15.5f * fabsf(g0) + hr * fabsf(g1)) * half + 0.01f;
    const float ey = (15.5f * fabsf(g3) + hr * fabsf(g4)) * half + 0.01f;
    const float xmin = sxc - ex, xmax = sxc + ex, ymin = syc - ey, ymax = syc + ey;
    const float fby0 = (float)B.by0, fby1 = (float)B.by1, fbx0 = (float)B.bx0, fbx1 = (float)B.bx1;
    const bool inside = xmin >= 0.0f && xmax <= fcs - 1.0f && ymin >= 0.0f && ymax <= fcs - 1.0f;
    const bool outside_box = ymax + 1.0f < fby0 || ymin >= fby1 || xmax + 1.0f < fbx0 || xmin >= fbx1;
    const bool interior = xmin >= fbx0 && xmax <= fbx1 - 1.0f && ymin >= fby0 && ymax <= fby1 - 1.0f;
    cls = (inside && outside_box) ? GEO_FILL : interior ? GEO_INTERIOR : GEO_GENERAL;
  }
  if (x >= cs) return;
  const bool has2 = x + 1 < cs;
  const int bw = A.bw;
  const int fstride = A.bh * bw;  // pixels per intermediate frame
  const uint2* const fr0 = A.inter + ((int64_t)frame0 * fstride - (B.by0 * bw + B.bx0));  // frame t0, indexed by canvas (y, x)
  DstT* const obase0 = (DstT*)A.dst + ((int64_t)clip * A.sb + (int64_t)t0 * A.st);
  const int osy = (int)A.sy, osc = (int)A.sc, osx = (int)A.sx;
  const bool vec2 = A.sx == 1 && ((A.sy | A.sc | A.sb | A.st) & 1) == 0 && (((uintptr_t)A.dst) & (2 * sizeof(DstT) - 1)) == 0;
  // TAIL: some clip of the batch has an effect after the affine step (grayscale .. cutout); the common case compiles without them
  const bool tail_fx = TAIL && (flags & kTailFlags) != 0u;
  const float nsr = A.nscale[0], nsg = A.nscale[1], nsb = A.nscale[2], nbr = A.nbias[0], nbg = A.nbias[1], nbb = A.nbias[2];
  const float xb = (float)x - half + 0.5f;
  const float xg0[2] = {xb * g0, has2 ? (xb + 1.0f) * g0 : xb * g0}, xg3[2] = {xb * g3, has2 ? (xb + 1.0f) * g3 : xb * g3};
  const int64_t fbytes = (int64_t)fstride * 8, stbytes = A.st * (int64_t)sizeof(DstT);

#pragma unroll 1
  for (int pass = 0; pass < kGeoPasses; ++pass) {
    const int y = ty0 + ly + 2 * pass;
    if (y >= cs) break;
    // ---- geometry of this lane's two pixels, shared by the frames of the clip ----
    GeoPx q[2];
    float t0q[2], pmq[2];
    if (cls != GEO_FILL) {
      const float yb = (float)y - half + 0.5f;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        GeoPx& g = q[e];
        const int xe = has2 ? x + e : x;
        g.m = 1.0f;
        if (affine) {
          // tv _gen_affine_grid + grid_sample(bilinear, zeros, align_corners=False) on [img | ones], img * mask
          const float gx = fmaf(yb, g1, xg0[e]) + g2;
          const float gy = fmaf(yb, g4, xg3[e]) + g5;
          const float ix = fmaf(gx + 1.0f, fcs, -1.0f) * 0.5f;
          const float iy = fmaf(gy + 1.0f, fcs, -1.0f) * 0.5f;
          const float x0f = floorf(ix), y0f = floorf(iy);
          const float wx1 = ix - x0f, wy1 = iy - y0f;
          const float wx0 = 1.0f - wx1, wy0 = 1.0f - wy1;
          if (cls == GEO_INTERIOR) {
            g.o00 = (int)y0f * bw + (int)x0f;
            g.o01 = g.o00 + 1; g.o10 = g.o00 + bw; g.o11 = g.o10 + 1;
            g.w00 = wx0 * wy0; g.w01 = wx1 * wy0; g.w10 = wx0 * wy1; g.w11 = wx1 * wy1;
            g.wc = 1.0f;
          } else {
            // clamp before the int cast so wild matrices cannot overflow
            const int x0 = (int)fminf(fmaxf(x0f, -2.0f), fcs + 1.0f);
            const int yq = (int)fminf(fmaxf(y0f, -2.0f), fcs + 1.0f);
            const bool inx0 = (unsigned)x0 < (unsigned)cs, inx1 = (unsigned)(x0 + 1) < (unsigned)cs;
            const bool iny0 = (unsigned)yq < (unsigned)cs, iny1 = (unsigned)(yq + 1) < (unsigned)cs;
            const float ax0 = inx0 ? wx0 : 0.0f, ax1 = inx1 ? wx1 : 0.0f, ay0 = iny0 ? wy0 : 0.0f, ay1 = iny1 ? wy1 : 0.0f;
            g.m = (ax0 + ax1) * (ay0 + ay1);                      // interpolated ones-mask
            const bool cx0 = x0 >= B.bx0 && x0 < B.bx1, cx1 = x0 + 1 >= B.bx0 && x0 + 1 < B.bx1;
            const bool cy0 = yq >= B.by0 && yq < B.by1, cy1 = yq + 1 >= B.by0 && yq + 1 < B.by1;
            const float bx0w = cx0 ? wx0 : 0.0f, bx1w = cx1 ? wx1 : 0.0f, by0w = cy0 ? wy0 : 0.0f, by1w = cy1 ? wy1 : 0.0f;
            const int xc0 = min(max(x0, B.bx0), B.bx1 - 1), xc1 = min(max(x0 + 1, B.bx0), B.bx1 - 1);
            const int yc0 = min(max(yq, B.by0), B.by1 - 1) * bw, yc1 = min(max(yq + 1, B.by0), B.by1 - 1) * bw;
            g.o00 = yc0 + xc0; g.o01 = yc0 + xc1; g.o10 = yc1 + xc0; g.o11 = yc1 + xc1;
            g.w00 = bx0w * by0w; g.w01 = bx1w * by0w; g.w10 = bx0w * by1w; g.w11 = bx1w * by1w;
            g.wc = (bx0w + bx1w) * (by0w + by1w);
          }
        } else {
          // no affine: the pixel itself when it is content, the pad colour otherwise
          const bool in = y >= B.by0 && y < B.by1 && xe >= B.bx0 && xe < B.bx1;
          g.o00 = g.o01 = g.o10 = g.o11 = min(max(y, B.by0), B.by1 - 1) * bw + min(max(xe, B.bx0), B.bx1 - 1);
          g.w00 = g.wc = in ? 1.0f : 0.0f;
          g.w01 = g.w10 = g.w11 = 0.0f;
        }
        t0q[e] = kS2Off * g.wc;
        pmq[e] = g.m - g.wc;
      }
    }
    const int off = y * osy + x * osx;
    // ---- the frames (fully unrolled).  The per-frame base pointers are made opaque so that every address below
    // is ONE multiply-add (IMAD.WIDE index * size + base) instead of a 64-bit add chain ----
#pragma unroll
    for (int f = 0; f < kGeoFrames; ++f) {
      if (t0 + f >= t1) break;
      const float4 padv = __ldg(fi4 + 5 * f);  // FrameInfo is five float4; the pad colour comes first
      const uint2* fr = (const uint2*)((const char*)fr0 + f * fbytes);
      DstT* ob = (DstT*)((char*)obase0 + f * stbytes);
      asm volatile("" : "+l"(fr));
      asm volatile("" : "+l"(ob));
      float rr[2] = {padv.x, padv.x}, gg[2] = {padv.y, padv.y}, bb[2] = {padv.z, padv.z};
      if (cls != GEO_FILL) {
        uint2 v[2][4];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          v[e][0] = fr[q[e].o00]; v[e][1] = fr[q[e].o01]; v[e][2] = fr[q[e].o10]; v[e][3] = fr[q[e].o11];
        }
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const GeoPx& g = q[e];
          const float sr = fmaf(q15_r(v[e][3]), g.w11, fmaf(q15_r(v[e][2]), g.w10, fmaf(q15_r(v[e][1]), g.w01, q15_r(v[e][0]) * g.w00)));
          const float sg = fmaf(q15_g(v[e][3]), g.w11, fmaf(q15_g(v[e][2]), g.w10, fmaf(q15_g(v[e][1]), g.w01, q15_g(v[e][0]) * g.w00)));
          const float sb = fmaf(q15_b(v[e][3]), g.w11, fmaf(q15_b(v[e][2]), g.w10, fmaf(q15_b(v[e][1]), g.w01, q15_b(v[e][0]) * g.w00)));
          if (cls == GEO_INTERIOR) {  // m = wc = 1
            rr[e] = fmaf(sr, kS2Inv, kS2Off);
            gg[e] = fmaf(sg, kS2Inv, kS2Off);
            bb[e] = fmaf(sb, kS2Inv, kS2Off);
          } else {
            rr[e] = g.m * fmaf(sr, kS2Inv, fmaf(padv.x, pmq[e], t0q[e]));
            gg[e] = g.m * fmaf(sg, kS2Inv, fmaf(padv.y, pmq[e], t0q[e]));
            bb[e] = g.m * fmaf(sb, kS2Inv, fmaf(padv.z, pmq[e], t0q[e]));
          }
        }
      }
      if (tail_fx) {
        const int frame = frame0 + f;
        const int idx = y * cs + x;
        bool to_canvas = false;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          if (e == 1 && !has2) break;
          float r = rr[e], g = gg[e], b = bb[e];
          if (flags & NEXAR_GRAYSCALE) r = g = b = gray_of(r, g, b);
          if (flags & NEXAR_NOISE) {
            const unsigned base = (unsigned)((frame * 3) * cs * cs + idx + e);
            r = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base), cp->noise_level, r));
            g = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base + cs * cs), cp->noise_level, g));
            b = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base + 2 * cs * cs), cp->noise_level, b));
          }
          if (flags & NEXAR_BLUR) {  // the blur kernel finishes the chain from the planar canvas
            float* cv = A.canvas + (size_t)frame * 3 * cs * cs;
            cv[idx + e] = r;
            cv[cs * cs + idx + e] = g;
            cv[2 * cs * cs + idx + e] = b;
            to_canvas = true;
            continue;
          }
          point_effects(r, g, b, cp, flags, y, x + e);
          rr[e] = r; gg[e] = g; bb[e] = b;
        }
        if (to_canvas) continue;
      }
      // nscale / nbias are 1 / 0 when the output is not normalised
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        rr[e] = fmaf(rr[e], nsr, nbr); gg[e] = fmaf(gg[e], nsg, nbg); bb[e] = fmaf(bb[e], nsb, nbb);
      }
      if (vec2 && has2) {
        store_pair<DstT>(ob + off, rr[0], rr[1]);
        store_pair<DstT>(ob + (off + osc), gg[0], gg[1]);
        store_pair<DstT>(ob + (off + 2 * osc), bb[0], bb[1]);
      } else {
        store_out_global<DstT>(ob + off, rr[0]);
        store_out_global<DstT>(ob + (off + osc), gg[0]);
        store_out_global<DstT>(ob + (off + 2 * osc), bb[0]);
        if (has2) {
          store_out_global<DstT>(ob + (off + osx), rr[1]);
          store_out_global<DstT>(ob + (off + osx + osc), gg[1]);
          store_out_global<DstT>(ob + (off + osx + 2 * osc), bb[1]);
        }
      }
    }
  }
}

// K3, specialised.  The intermediate frame size (BH x BW), the canvas (CS) and a planar, row-contiguous destination
// (x stride 1, y stride CS, frame stride CS * CS) are compile-time constants, so that
//   * a pixel needs ONE 64-bit source pointer per lane pixel: its four bilinear neighbours sit at the immediate offsets
//     {0, 1, BW, BW + 1} pixels and frame f of the group at f * BH * BW pixels (every load is [pointer + immediate]);
//     at the edges of the content box the base is clamped into the box and the weights are re-assigned to the two
//     loaded columns / rows (a neighbour that is pad or outside the canvas keeps weight zero), so the boundary tiles
//     use the same addressing as the interior ones;
//   * a channel of the output needs one pointer too (frame f at f * CS * CS elements);
//   * the geometry of a pixel is shared by NF (8) frames of the clip instead of 4;
//   * the blend runs on packed fp32 pairs (FFMA2: the two pixels of a lane, channel by channel) and the interior
//     class folds the q15 scale and the normalisation into one multiply-add per channel.
// Same formulas and the same per-pixel operation order as geometry_kernel, which stays the general fallback.
constexpr int kGeo2Frames = 8;   // frames of one clip per CTA
constexpr int kGeo2MinB = 6;     // CTAs per SM (5 / 6 / 7 measured: 6 is best, 0.393 vs 0.399 / 0.399 ms)
constexpr int kGeo2Warps = 4;    // warps per CTA: the CTA tile is 32 x (4 * warps) pixels (3 / 4 / 5 / 8 measured: 4 is best by 1 %)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ void l2_prefetch_line(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

template <typename DstT, bool TAIL, int BH, int BW, int CS>
__global__ void __launch_bounds__(32 * kGeo2Warps, kGeo2MinB) geometry_spec_kernel(const __grid_constant__ DevPlan P, const __grid_constant__ KArgs A) {
  static_assert(BH >= 2 && BW >= 2, "the clamped 2 x 2 window needs a 2 x 2 box");
  constexpr int NF = kGeo2Frames;
  constexpr int FPX = BH * BW;   // pixels of one intermediate frame
  constexpr int OPX = CS * CS;   // elements of one output plane
  asm volatile("griddepcontrol.launch_dependents;");   // the fix-up launch may drain through this grid's last wave
  const int ngroup = (A.T + NF - 1) / NF;
  // last frame groups first: the colour kernel wrote them last (L2).  Measured: 0.3952 -> 0.3935 ms at cfg2
  const int bz = (int)(gridDim.z - 1u - blockIdx.z);
  const int clip = bz / ngroup;
  const int t0 = (bz - clip * ngroup) * NF;
  const int nfr = min(NF, A.T - t0);
  const int frame0 = clip * A.T + t0;
  const float4* fi4 = (const float4*)(A.finfo + frame0);
  const float4 q3 = __ldg(fi4 + 3);
  const unsigned flags = __float_as_uint(q3.z);
  if (!(flags & NEXAR_AUG)) return;
  if (A.pass == 4 && A.clip_max[clip] == 0u) return;  // fixup_frame_kernel finishes those clips on its own
  // Warp tile = 32 x 4 output pixels.  A lane owns ONE column and two vertically adjacent pixels per pass (two passes):
  // the 32 lanes of a load read 32 consecutive 8-byte pixels of one source row (two or three 128-byte lines) and the
  // 32 lanes of a store write 32 consecutive elements, which halves the L1 wavefronts of a two-pixels-per-lane row layout.
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tx0 = blockIdx.x * 32, ty0 = (blockIdx.y * kGeo2Warps + warp) * 4;
  const int x = tx0 + lane;
  if (ty0 >= CS) return;
  const float4 q2 = __ldg(fi4 + 2);
  const int4 bx = __ldg((const int4*)fi4 + 1);
  const NexarClipParams* cp = A.params + clip;   // only the rare tail effects read it
  const int by0 = bx.x, by1 = bx.y, bx0 = bx.z, bx1 = bx.w;
  constexpr float half = (float)CS * 0.5f, fcs = (float)CS;
  const bool affine = (flags & NEXAR_AFFINE) != 0u;
  const float g0 = q2.x, g1 = q2.y, g2 = q2.z, g3 = q2.w, g4 = q3.x, g5 = q3.y;
  int cls = GEO_GENERAL;
  if (affine) {  // tile class, as in geometry_kernel (tile = 32 x 4 pixels)
    const float xc = (float)(tx0 + 16) - half, yc = (float)(ty0 + 2) - half;
    const float sxc = fmaf(fmaf(yc, g1, xc * g0) + g2 + 1.0f, fcs, -1.0f) * 0.5f;
    const float syc = fmaf(fmaf(yc, g4, xc * g3) + g5 + 1.0f, fcs, -1.0f) * 0.5f;
    const float ex = (15.5f * fabsf(g0) + 1.5f * fabsf(g1)) * half + 0.01f;
    const float ey = (15.5f * fabsf(g3) + 1.5f * fabsf(g4)) * half + 0.01f;
    const float xmin = sxc - ex, xmax = sxc + ex, ymin = syc - ey, ymax = syc + ey;
    const float fby0 = (float)by0, fby1 = (float)by1, fbx0 = (float)bx0, fbx1 = (float)bx1;
    const bool inside = xmin >= 0.0f && xmax <= fcs - 1.0f && ymin >= 0.0f && ymax <= fcs - 1.0f;
    const bool outside_box = ymax + 1.0f < fby0 || ymin >= fby1 || xmax + 1.0f < fbx0 || xmin >= fbx1;
    const bool interior = xmin >= fbx0 && xmax <= fbx1 - 1.0f && ymin >= fby0 && ymax <= fby1 - 1.0f;
    cls = (inside && outside_box) ? GEO_FILL : interior ? GEO_INTERIOR : GEO_GENERAL;
  }
  if (x >= CS) return;
  const uint2* const fr0 = A.inter + ((int64_t)frame0 * FPX - (by0 * BW + bx0));  // frame t0, indexed by canvas (y, x)
  DstT* const ob0 = (DstT*)A.dst + ((int64_t)clip * A.sb + (int64_t)t0 * OPX);
  const int64_t osc = A.sc;
  const bool tail_fx = TAIL && (flags & kTailFlags) != 0u;
  const float nsr = A.nscale[0], nsg = A.nscale[1], nsb = A.nscale[2], nbr = A.nbias[0], nbg = A.nbias[1], nbb = A.nbias[2];
  // Unpacking: a byte permute per sample (ALU pipe, which bounds this kernel).  Measured: sending the B channel through
  // I2F.U16 on the conversion pipe instead changes nothing, the G and B channels lose 2 %.
  // interior class: out = s * (k * ns) + (nb - k * ns), s = sum(w * F), F = 1 + q / 32768, k = 32768 / 32767
  const float kir = kS2Inv * nsr, kig = kS2Inv * nsg, kib = kS2Inv * nsb;
  const float cir = fmaf(kS2Off, nsr, nbr), cig = fmaf(kS2Off, nsg, nbg), cib = fmaf(kS2Off, nsb, nbb);
  const float xb = (float)x - half + 0.5f;
  const float xg0 = xb * g0, xg3 = xb * g3;

#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    const int y = ty0 + 2 * pass;        // this lane's pixels: (x, y) and (x, y + 1)
    if (y >= CS) break;
    const bool has2 = y + 1 < CS;
    // ---- geometry of this lane's two pixels, shared by the frames of the group ----
    int o[2] = {0, 0};
    float2 w00 = {0.f, 0.f}, w01 = {0.f, 0.f}, w10 = {0.f, 0.f}, w11 = {0.f, 0.f};
    float mq[2] = {1.0f, 1.0f}, t0q[2] = {0.f, 0.f}, pmq[2] = {0.f, 0.f};
    if (cls != GEO_FILL) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ye = has2 ? y + e : y;
        const float yb = (float)ye - half + 0.5f;
        float wx0, wx1, wy0, wy1, x0f, y0f;
        if (affine) {
          // tv _gen_affine_grid + grid_sample(bilinear, zeros, align_corners=False) on [img | ones], img * mask
          const float gx = fmaf(yb, g1, xg0) + g2;
          const float gy = fmaf(yb, g4, xg3) + g5;
          const float ix = fmaf(gx + 1.0f, fcs, -1.0f) * 0.5f;
          const float iy = fmaf(gy + 1.0f, fcs, -1.0f) * 0.5f;
          x0f = floorf(ix); y0f = floorf(iy);
          wx1 = ix - x0f; wy1 = iy - y0f;
          wx0 = 1.0f - wx1; wy0 = 1.0f - wy1;
        } else {  // no affine: the pixel itself
          x0f = (float)x; y0f = (float)ye;
          wx1 = wy1 = 0.0f; wx0 = wy0 = 1.0f;
        }
        float a00, a01, a10, a11;
        if (cls == GEO_INTERIOR) {
          o[e] = (int)y0f * BW + (int)x0f;
          a00 = wx0 * wy0; a01 = wx1 * wy0; a10 = wx0 * wy1; a11 = wx1 * wy1;
        } else {
          // clamp before the int cast so wild matrices cannot overflow
          const int x0 = (int)fminf(fmaxf(x0f, -2.0f), fcs + 1.0f);
          const int yq = (int)fminf(fmaxf(y0f, -2.0f), fcs + 1.0f);
          const bool inx0 = (unsigned)x0 < (unsigned)CS, inx1 = (unsigned)(x0 + 1) < (unsigned)CS;
          const bool iny0 = (unsigned)yq < (unsigned)CS, iny1 = (unsigned)(yq + 1) < (unsigned)CS;
          const float ax0 = inx0 ? wx0 : 0.0f, ax1 = inx1 ? wx1 : 0.0f, ay0 = iny0 ? wy0 : 0.0f, ay1 = iny1 ? wy1 : 0.0f;
          const float m = (ax0 + ax1) * (ay0 + ay1);               // interpolated ones-mask
          const bool cx0 = x0 >= bx0 && x0 < bx1, cx1 = x0 + 1 >= bx0 && x0 + 1 < bx1;
          const bool cy0 = yq >= by0 && yq < by1, cy1 = yq + 1 >= by0 && yq + 1 < by1;
          const float bx0w = cx0 ? wx0 : 0.0f, bx1w = cx1 ? wx1 : 0.0f, by0w = cy0 ? wy0 : 0.0f, by1w = cy1 ? wy1 : 0.0f;
          // the loaded 2 x 2 window starts at (xc, yc), clamped into the box; each loaded column / row takes the weight
          // of the neighbour it coincides with (none: zero)
          const int xc = min(max(x0, bx0), bx1 - 2), yc = min(max(yq, by0), by1 - 2);
          const int dx = xc - x0, dy = yc - yq;
          const float wA = dx == 0 ? bx0w : dx == 1 ? bx1w : 0.0f, wB = dx == 0 ? bx1w : dx == -1 ? bx0w : 0.0f;
          const float hA = dy == 0 ? by0w : dy == 1 ? by1w : 0.0f, hB = dy == 0 ? by1w : dy == -1 ? by0w : 0.0f;
          o[e] = yc * BW + xc;
          a00 = wA * hA; a01 = wB * hA; a10 = wA * hB; a11 = wB * hB;
          const float wc = (bx0w + bx1w) * (by0w + by1w);
          mq[e] = m;
          t0q[e] = kS2Off * wc;
          pmq[e] = m - wc;
        }
        if (e == 0) { w00.x = a00; w01.x = a01; w10.x = a10; w11.x = a11; }
        else        { w00.y = a00; w01.y = a01; w10.y = a10; w11.y = a11; }
      }
    }
    const uint2* const pa = fr0 + o[0];
    const uint2* const pb = fr0 + o[1];
    DstT* const por = ob0 + (y * CS + x);
    DstT* const pog = por + osc;
    DstT* const pob = pog + osc;
    auto put = [&](DstT* p, int f, float va, float vb) {   // one channel of the lane's two pixels, frame f of the group
      store_out_global<DstT>(p + f * OPX, va);
      if (has2) store_out_global<DstT>(p + (f * OPX + CS), vb);
    };
    // ---- the frames of the group (fully unrolled: every address below is [pointer + immediate]); the eight neighbour
    // loads of frame f + 1 are issued before frame f is blended ----
    uint2 va[2][4], vb[2][4];
    if (cls != GEO_FILL) {
      // pull the three source rows this lane needs from the LATER frames of the group into L2 now (the intermediate of a
      // whole batch does not stay L2-resident behind the 1.4 GB source stream): their loads then find an L2 hit
#pragma unroll
      for (int f = 1; f < NF; ++f)
        if (f < nfr) {
          l2_prefetch_line(pa + f * FPX);
          l2_prefetch_line(pa + f * FPX + BW);
          l2_prefetch_line(pb + f * FPX + BW);
        }
      va[0][0] = __ldg(pa); va[0][1] = __ldg(pa + 1); va[0][2] = __ldg(pa + BW); va[0][3] = __ldg(pa + BW + 1);
      vb[0][0] = __ldg(pb); vb[0][1] = __ldg(pb + 1); vb[0][2] = __ldg(pb + BW); vb[0][3] = __ldg(pb + BW + 1);
    }
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      if (f >= nfr) break;
      const float4 padv = __ldg(fi4 + 5 * f);  // FrameInfo is five float4; the pad colour comes first
      float2 rr = {padv.x, padv.x}, gg = {padv.y, padv.y}, bb = {padv.z, padv.z};
      if (cls != GEO_FILL) {
        if (f + 1 < NF && f + 1 < nfr) {
          const uint2* qa = pa + (f + 1) * FPX;
          const uint2* qb = pb + (f + 1) * FPX;
          uint2* na = va[(f + 1) & 1];
          uint2* nb = vb[(f + 1) & 1];
          na[0] = __ldg(qa); na[1] = __ldg(qa + 1); na[2] = __ldg(qa + BW); na[3] = __ldg(qa + BW + 1);
          nb[0] = __ldg(qb); nb[1] = __ldg(qb + 1); nb[2] = __ldg(qb + BW); nb[3] = __ldg(qb + BW + 1);
        }
        const uint2* ca = va[f & 1];
        const uint2* cb = vb[f & 1];
        float2 sr = fmul2(make_float2(q15_r(ca[0]), q15_r(cb[0])), w00);
        float2 sg = fmul2(make_float2(q15_g(ca[0]), q15_g(cb[0])), w00);
        float2 sb = fmul2(make_float2(q15_b(ca[0]), q15_b(cb[0])), w00);
        sr = ffma2(make_float2(q15_r(ca[1]), q15_r(cb[1])), w01, sr);
        sg = ffma2(make_float2(q15_g(ca[1]), q15_g(cb[1])), w01, sg);
        sb = ffma2(make_float2(q15_b(ca[1]), q15_b(cb[1])), w01, sb);
        sr = ffma2(make_float2(q15_r(ca[2]), q15_r(cb[2])), w10, sr);
        sg = ffma2(make_float2(q15_g(ca[2]), q15_g(cb[2])), w10, sg);
        sb = ffma2(make_float2(q15_b(ca[2]), q15_b(cb[2])), w10, sb);
        sr = ffma2(make_float2(q15_r(ca[3]), q15_r(cb[3])), w11, sr);
        sg = ffma2(make_float2(q15_g(ca[3]), q15_g(cb[3])), w11, sg);
        sb = ffma2(make_float2(q15_b(ca[3]), q15_b(cb[3])), w11, sb);
        if (cls == GEO_INTERIOR) {  // m = wc = 1
          if (!tail_fx) {           // scale and normalisation in one multiply-add
            put(por, f, fmaf(sr.x, kir, cir), fmaf(sr.y, kir, cir));
            put(pog, f, fmaf(sg.x, kig, cig), fmaf(sg.y, kig, cig));
            put(pob, f, fmaf(sb.x, kib, cib), fmaf(sb.y, kib, cib));
            continue;
          }
          rr = make_float2(fmaf(sr.x, kS2Inv, kS2Off), fmaf(sr.y, kS2Inv, kS2Off));
          gg = make_float2(fmaf(sg.x, kS2Inv, kS2Off), fmaf(sg.y, kS2Inv, kS2Off));
          bb = make_float2(fmaf(sb.x, kS2Inv, kS2Off), fmaf(sb.y, kS2Inv, kS2Off));
        } else {
          rr = make_float2(mq[0] * fmaf(sr.x, kS2Inv, fmaf(padv.x, pmq[0], t0q[0])), mq[1] * fmaf(sr.y, kS2Inv, fmaf(padv.x, pmq[1], t0q[1])));
          gg = make_float2(mq[0] * fmaf(sg.x, kS2Inv, fmaf(padv.y, pmq[0], t0q[0])), mq[1] * fmaf(sg.y, kS2Inv, fmaf(padv.y, pmq[1], t0q[1])));
          bb = make_float2(mq[0] * fmaf(sb.x, kS2Inv, fmaf(padv.z, pmq[0], t0q[0])), mq[1] * fmaf(sb.y, kS2Inv, fmaf(padv.z, pmq[1], t0q[1])));
        }
      }
      if (tail_fx) {
        const int frame = frame0 + f;
        float rv[2] = {rr.x, rr.y}, gv[2] = {gg.x, gg.y}, bv[2] = {bb.x, bb.y};
        bool to_canvas = false;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          if (e == 1 && !has2) break;
          const int idx = (y + e) * CS + x;
          float r = rv[e], g = gv[e], b = bv[e];
          if (flags & NEXAR_GRAYSCALE) r = g = b = gray_of(r, g, b);
          if (flags & NEXAR_NOISE) {
            const unsigned base = (unsigned)((frame * 3) * CS * CS + idx);
            r = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base), cp->noise_level, r));
            g = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base + CS * CS), cp->noise_level, g));
            b = clamp01(fmaf(gauss_noise(cp->noise_seed[0], cp->noise_seed[1], base + 2 * CS * CS), cp->noise_level, b));
          }
          if (flags & NEXAR_BLUR) {  // the blur kernel finishes the chain from the planar canvas
            float* cv = A.canvas + (size_t)frame * 3 * CS * CS;
            cv[idx] = r;
            cv[CS * CS + idx] = g;
            cv[2 * CS * CS + idx] = b;
            to_canvas = true;
            continue;
          }
          point_effects(r, g, b, cp, flags, y + e, x);
          rv[e] = r; gv[e] = g; bv[e] = b;
        }
        if (to_canvas) continue;
        rr = make_float2(rv[0], rv[1]); gg = make_float2(gv[0], gv[1]); bb = make_float2(bv[0], bv[1]);
      }
      // nscale / nbias are 1 / 0 when the output is not normalised
      put(por, f, fmaf(rr.x, nsr, nbr), fmaf(rr.y, nsr, nbr));
      put(pog, f, fmaf(gg.x, nsg, nbg), fmaf(gg.y, nsg, nbg));
      put(pob, f, fmaf(bb.x, nsb, nbb), fmaf(bb.y, nsb, nbb));
    }
  }
}

// K4: gaussian blur (tv gaussian_blur: reflect pad, outer-product kernel) + rest of the chain.
template <typename DstT>
__global__ void __launch_bounds__(256) blur_kernel(DevPlan P, KArgs A) {
  const int frame = blockIdx.y;
  const int clip = frame / A.T;
  const int t = frame - clip * A.T;
  const NexarClipParams* cp = A.params + clip;
  const unsigned flags = cp->flags;
  if (!(flags & NEXAR_AUG) || !(flags & NEXAR_BLUR)) return;
  const int cs = P.cs;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= cs * cs) return;
  const int y = idx / cs, x = idx - y * cs;
  const int k = cp->blur_ksize, h = k / 2;
  const float* cv = A.canvas + (size_t)frame * 3 * cs * cs;
  float acc[3] = {0.0f, 0.0f, 0.0f};
  for (int dy = 0; dy < k; ++dy) {
    int yy = y + dy - h;
    yy = yy < 0 ? -yy : (yy >= cs ? 2 * cs - 2 - yy : yy);
    const float wyv = cp->blur_taps[dy];
    for (int dx = 0; dx < k; ++dx) {
      int xx = x + dx - h;
      xx = xx < 0 ? -xx : (xx >= cs ? 2 * cs - 2 - xx : xx);
      const float w = __fmul_rn(wyv, cp->blur_taps[dx]);
#pragma unroll
      for (int c = 0; c < 3; ++c) acc[c] = fmaf(cv[(size_t)c * cs * cs + yy * cs + xx], w, acc[c]);
    }
  }
  float r = acc[0], g = acc[1], b = acc[2];
  point_effects(r, g, b, cp, flags, y, x);
  const int64_t o = (int64_t)clip * A.sb + (int64_t)t * A.st + (int64_t)y * A.sy + (int64_t)x * A.sx;
  if (A.normalize) {
    r = fmaf(r, A.nscale[0], A.nbias[0]);
    g = fmaf(g, A.nscale[1], A.nbias[1]);
    b = fmaf(b, A.nscale[2], A.nbias[2]);
  }
  store_out<DstT>(A.dst, o, r);
  store_out<DstT>(A.dst, o + A.sc, g);
  store_out<DstT>(A.dst, o + 2 * A.sc, b);
}

// ---------------------------------------------------------------------------------
// YUV 4:2:0 sources (what decoders produce: 1.5 bytes per pixel instead of 3).  Y plane [L][pitch], then either the
// interleaved chroma plane [L/2][pitch] (NV12: U0 V0 U1 V1 ...) or the U and V planes [L/2][pitch/2] each (I420), where
// L >= H is the surface's luma height (uoff = L * pitch, voff = uoff + L/2 * pitch/2); one chroma pair per 2 x 2 pixels
// (nearest neighbour).  Conversion = the classic 8-bit integer form with the coefficients of YuvCoef,
//   C = Y - Yo, D = U - 128, E = V - 128
//   R = clip((Ys C + Rv E + 128) >> 8)   G = clip((Ys C - Gu D - Gv E + 128) >> 8)   B = clip((Ys C + Bu D + 128) >> 8)
// (BT.601 limited range: 16, 298, 409, 100, 208, 516) to packed RGB bytes — exactly the uint8 frames the resize kernels
// take, so everything downstream (the /255 rule on the clip maximum included) is the RGB path bit for bit
// (oracle/yuv420_oracle.py states the same formula in numpy).
// clip(x >> 8) is evaluated as clamp(x, 0, 65535) >> 8, so the shift merges with the byte packing.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ int clamp_u16(int x) { return min(max(x, 0), 65535); }
struct ChromaTerms { int r, g, b; };
__device__ __forceinline__ ChromaTerms chroma_terms(int u, int v, const YuvCoef& k) {
  const int d = u - 128, e = v - 128;
  const int base = 128 - k.ys * k.yo;
  return {k.rv * e + base, -k.gu * d - k.gv * e + base, k.bu * d + base};
}

// 16 pixels of two rows per thread: two 16-byte luma loads, one 16-byte (NV12) or two 8-byte (I420) chroma loads,
// six 16-byte stores
template <int Layout>
__global__ void __launch_bounds__(256) yuv420_to_rgb_vec_kernel(const unsigned char* __restrict__ src, const int64_t* __restrict__ frame_offsets,
                                                                int64_t pitch, int64_t uoff, int64_t voff, YuvCoef kc, int H, int W,
                                                                unsigned char* __restrict__ rgb, int64_t* __restrict__ out_offsets) {
  const int frame = blockIdx.y;
  const int cols = W >> 4;
  const int unit = blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t fbytes = (int64_t)H * W * 3;
  if (unit == 0) out_offsets[frame] = (int64_t)frame * fbytes;
  if (unit >= cols * (H >> 1)) return;
  const int r2 = unit / cols, c = unit - r2 * cols;
  const unsigned char* f = src + frame_offsets[frame];
  const uint4 ya = __ldcs((const uint4*)(f + (int64_t)(2 * r2) * pitch + 16 * c));
  const uint4 yb = __ldcs((const uint4*)(f + (int64_t)(2 * r2 + 1) * pitch + 16 * c));
  unsigned uvw[4];   // U V U V bytes of pixels 4q .. 4q+3
  if (Layout == NEXAR_YUV_NV12) {
    const uint4 uv = __ldcs((const uint4*)(f + uoff + (int64_t)r2 * pitch + 16 * c));
    uvw[0] = uv.x, uvw[1] = uv.y, uvw[2] = uv.z, uvw[3] = uv.w;
  } else {
    const int64_t cp = pitch >> 1;
    const uint2 u = __ldcs((const uint2*)(f + uoff + (int64_t)r2 * cp + 8 * c));
    const uint2 v = __ldcs((const uint2*)(f + voff + (int64_t)r2 * cp + 8 * c));
    uvw[0] = __byte_perm(u.x, v.x, 0x5140), uvw[1] = __byte_perm(u.x, v.x, 0x7362);
    uvw[2] = __byte_perm(u.y, v.y, 0x5140), uvw[3] = __byte_perm(u.y, v.y, 0x7362);
  }
  const unsigned yaw[4] = {ya.x, ya.y, ya.z, ya.w}, ybw[4] = {yb.x, yb.y, yb.z, yb.w};
  unsigned oa[12], ob[12];   // 48 output bytes per row
#pragma unroll
  for (int q = 0; q < 4; ++q) {  // four pixels (two chroma pairs) per 32-bit word of luma
    const ChromaTerms t0 = chroma_terms(uvw[q] & 255u, (uvw[q] >> 8) & 255u, kc);
    const ChromaTerms t1 = chroma_terms((uvw[q] >> 16) & 255u, uvw[q] >> 24, kc);
    unsigned char* pa = (unsigned char*)oa + 12 * q;
    unsigned char* pb = (unsigned char*)ob + 12 * q;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const ChromaTerms& t = k < 2 ? t0 : t1;
      const int la = kc.ys * (int)((yaw[q] >> (8 * k)) & 255u), lb = kc.ys * (int)((ybw[q] >> (8 * k)) & 255u);
      pa[3 * k + 0] = (unsigned char)(clamp_u16(la + t.r) >> 8);
      pa[3 * k + 1] = (unsigned char)(clamp_u16(la + t.g) >> 8);
      pa[3 * k + 2] = (unsigned char)(clamp_u16(la + t.b) >> 8);
      pb[3 * k + 0] = (unsigned char)(clamp_u16(lb + t.r) >> 8);
      pb[3 * k + 1] = (unsigned char)(clamp_u16(lb + t.g) >> 8);
      pb[3 * k + 2] = (unsigned char)(clamp_u16(lb + t.b) >> 8);
    }
  }
  unsigned char* o = rgb + (int64_t)frame * fbytes + ((int64_t)(2 * r2) * W + 16 * c) * 3;
  uint4* da = (uint4*)o;
  uint4* db = (uint4*)(o + (int64_t)W * 3);
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    da[v] = make_uint4(oa[4 * v], oa[4 * v + 1], oa[4 * v + 2], oa[4 * v + 3]);
    db[v] = make_uint4(ob[4 * v], ob[4 * v + 1], ob[4 * v + 2], ob[4 * v + 3]);
  }
}

// any even size / pitch / alignment: one 2 x 2 block per thread
template <int Layout>
__global__ void __launch_bounds__(256) yuv420_to_rgb_any_kernel(const unsigned char* __restrict__ src, const int64_t* __restrict__ frame_offsets,
                                                                int64_t pitch, int64_t uoff, int64_t voff, YuvCoef kc, int H, int W,
                                                                unsigned char* __restrict__ rgb, int64_t* __restrict__ out_offsets) {
  const int frame = blockIdx.y;
  const int cols = W >> 1;
  const int unit = blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t fbytes = (int64_t)H * W * 3;
  if (unit == 0) out_offsets[frame] = (int64_t)frame * fbytes;
  if (unit >= cols * (H >> 1)) return;
  const int r2 = unit / cols, c = unit - r2 * cols;
  const unsigned char* f = src + frame_offsets[frame];
  int u, v;
  if (Layout == NEXAR_YUV_NV12) {
    const unsigned char* uvp = f + uoff + (int64_t)r2 * pitch + 2 * c;
    u = uvp[0], v = uvp[1];
  } else {
    const int64_t at = (int64_t)r2 * (pitch >> 1) + c;
    u = f[uoff + at], v = f[voff + at];
  }
  const ChromaTerms t = chroma_terms(u, v, kc);
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) {
    const unsigned char* yp = f + (int64_t)(2 * r2 + dy) * pitch + 2 * c;
    unsigned char* o = rgb + (int64_t)frame * fbytes + ((int64_t)(2 * r2 + dy) * W + 2 * c) * 3;
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int l = kc.ys * (int)yp[dx];
      o[3 * dx + 0] = (unsigned char)(clamp_u16(l + t.r) >> 8);
      o[3 * dx + 1] = (unsigned char)(clamp_u16(l + t.g) >> 8);
      o[3 * dx + 2] = (unsigned char)(clamp_u16(l + t.b) >> 8);
    }
  }
}

// ---------------------------------------------------------------------------------
// 16-bit samples (P010 / P012 / P016, yuv420p10le; nexar_plan_create_yuv16): the same surfaces with 2-byte little-endian
// samples (pitch, uoff and voff in bytes as above).  Every sample is read as the word w = (sample << shift) & 0xFFFF and
// converted with the same coefficients at 16 bits of precision,
//   C = w_Y - (Yo << 8), D = w_U - 32768, E = w_V - 32768
//   R = clip((Ys C + Rv E + 32768) >> 16)   G = clip((Ys C - Gu D - Gv E + 32768) >> 16)   B = clip((Ys C + Bu D + 32768) >> 16)
// so a word x << 8 gives exactly the 8-bit result of the code x, and 10-bit content is rounded once to bytes.  Every term
// fits int32 (298 * 65535 + 541 * 32768 < 2^31); clip(x >> 16) is evaluated as clamp(x, 0, 2^24 - 1) >> 16
// (tests/yuv16_oracle.py states the same formula in numpy).
// ---------------------------------------------------------------------------------
__device__ __forceinline__ int clamp_u24(int x) { return min(max(x, 0), (1 << 24) - 1); }
__device__ __forceinline__ ChromaTerms chroma_terms16(int u, int v, const YuvCoef& k) {
  const int d = u - 32768, e = v - 32768;
  const int base = 32768 - k.ys * (k.yo << 8);
  return {k.rv * e + base, -k.gu * d - k.gv * e + base, k.bu * d + base};
}
// the two samples of a 32-bit word, each moved to the top of its 16-bit half
__device__ __forceinline__ unsigned align_words(unsigned w, int shift) { return (w & ((0xFFFFu >> shift) * 0x10001u)) << shift; }
// one sample at any byte address (little-endian), moved to the top of the word
__device__ __forceinline__ int load_word(const unsigned char* p, int shift) { return ((p[0] | (p[1] << 8)) << shift) & 0xFFFF; }

// 16 pixels of two rows per thread: four 16-byte luma loads, two 16-byte chroma loads (NV12: the U V words of the 8
// chroma pairs; I420: 8 U words and 8 V words), six 16-byte stores
template <int Layout>
__global__ void __launch_bounds__(256) yuv420_16_to_rgb_vec_kernel(const unsigned char* __restrict__ src, const int64_t* __restrict__ frame_offsets,
                                                                   int64_t pitch, int64_t uoff, int64_t voff, YuvCoef kc, int shift, int H, int W,
                                                                   unsigned char* __restrict__ rgb, int64_t* __restrict__ out_offsets) {
  const int frame = blockIdx.y;
  const int cols = W >> 4;
  const int unit = blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t fbytes = (int64_t)H * W * 3;
  if (unit == 0) out_offsets[frame] = (int64_t)frame * fbytes;
  if (unit >= cols * (H >> 1)) return;
  const int r2 = unit / cols, c = unit - r2 * cols;
  const unsigned char* f = src + frame_offsets[frame];
  const unsigned char* ra = f + (int64_t)(2 * r2) * pitch + 32 * c;
  const uint4 ya0 = __ldcs((const uint4*)ra), ya1 = __ldcs((const uint4*)(ra + 16));
  const uint4 yb0 = __ldcs((const uint4*)(ra + pitch)), yb1 = __ldcs((const uint4*)(ra + pitch + 16));
  unsigned uvw[8];   // U | V << 16 of chroma pairs 0 .. 7
  if (Layout == NEXAR_YUV_NV12) {
    const unsigned char* q = f + uoff + (int64_t)r2 * pitch + 32 * c;
    const uint4 a = __ldcs((const uint4*)q), b = __ldcs((const uint4*)(q + 16));
    uvw[0] = a.x, uvw[1] = a.y, uvw[2] = a.z, uvw[3] = a.w, uvw[4] = b.x, uvw[5] = b.y, uvw[6] = b.z, uvw[7] = b.w;
  } else {
    const int64_t cp = pitch >> 1;
    const uint4 u = __ldcs((const uint4*)(f + uoff + (int64_t)r2 * cp + 16 * c));
    const uint4 v = __ldcs((const uint4*)(f + voff + (int64_t)r2 * cp + 16 * c));
    const unsigned uw[4] = {u.x, u.y, u.z, u.w}, vw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) uvw[2 * i] = __byte_perm(uw[i], vw[i], 0x5410), uvw[2 * i + 1] = __byte_perm(uw[i], vw[i], 0x7632);
  }
  const unsigned yaw[8] = {ya0.x, ya0.y, ya0.z, ya0.w, ya1.x, ya1.y, ya1.z, ya1.w};
  const unsigned ybw[8] = {yb0.x, yb0.y, yb0.z, yb0.w, yb1.x, yb1.y, yb1.z, yb1.w};
  unsigned oa[12], ob[12];   // 48 output bytes per row
#pragma unroll
  for (int q = 0; q < 8; ++q) {  // two pixels (one chroma pair) per 32-bit word of luma
    const unsigned cw = align_words(uvw[q], shift);
    const ChromaTerms t = chroma_terms16(cw & 0xFFFFu, cw >> 16, kc);
    const unsigned wa = align_words(yaw[q], shift), wb = align_words(ybw[q], shift);
    unsigned char* pa = (unsigned char*)oa + 6 * q;
    unsigned char* pb = (unsigned char*)ob + 6 * q;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int la = kc.ys * (int)((wa >> (16 * k)) & 0xFFFFu), lb = kc.ys * (int)((wb >> (16 * k)) & 0xFFFFu);
      pa[3 * k + 0] = (unsigned char)(clamp_u24(la + t.r) >> 16);
      pa[3 * k + 1] = (unsigned char)(clamp_u24(la + t.g) >> 16);
      pa[3 * k + 2] = (unsigned char)(clamp_u24(la + t.b) >> 16);
      pb[3 * k + 0] = (unsigned char)(clamp_u24(lb + t.r) >> 16);
      pb[3 * k + 1] = (unsigned char)(clamp_u24(lb + t.g) >> 16);
      pb[3 * k + 2] = (unsigned char)(clamp_u24(lb + t.b) >> 16);
    }
  }
  unsigned char* o = rgb + (int64_t)frame * fbytes + ((int64_t)(2 * r2) * W + 16 * c) * 3;
  uint4* da = (uint4*)o;
  uint4* db = (uint4*)(o + (int64_t)W * 3);
#pragma unroll
  for (int v = 0; v < 3; ++v) {
    da[v] = make_uint4(oa[4 * v], oa[4 * v + 1], oa[4 * v + 2], oa[4 * v + 3]);
    db[v] = make_uint4(ob[4 * v], ob[4 * v + 1], ob[4 * v + 2], ob[4 * v + 3]);
  }
}

// any even size / even pitch / alignment: one 2 x 2 block per thread, every sample read byte by byte
template <int Layout>
__global__ void __launch_bounds__(256) yuv420_16_to_rgb_any_kernel(const unsigned char* __restrict__ src, const int64_t* __restrict__ frame_offsets,
                                                                   int64_t pitch, int64_t uoff, int64_t voff, YuvCoef kc, int shift, int H, int W,
                                                                   unsigned char* __restrict__ rgb, int64_t* __restrict__ out_offsets) {
  const int frame = blockIdx.y;
  const int cols = W >> 1;
  const int unit = blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t fbytes = (int64_t)H * W * 3;
  if (unit == 0) out_offsets[frame] = (int64_t)frame * fbytes;
  if (unit >= cols * (H >> 1)) return;
  const int r2 = unit / cols, c = unit - r2 * cols;
  const unsigned char* f = src + frame_offsets[frame];
  int u, v;
  if (Layout == NEXAR_YUV_NV12) {
    const unsigned char* uvp = f + uoff + (int64_t)r2 * pitch + 4 * c;
    u = load_word(uvp, shift), v = load_word(uvp + 2, shift);
  } else {
    const int64_t at = (int64_t)r2 * (pitch >> 1) + 2 * c;
    u = load_word(f + uoff + at, shift), v = load_word(f + voff + at, shift);
  }
  const ChromaTerms t = chroma_terms16(u, v, kc);
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) {
    const unsigned char* yp = f + (int64_t)(2 * r2 + dy) * pitch + 4 * c;
    unsigned char* o = rgb + (int64_t)frame * fbytes + ((int64_t)(2 * r2 + dy) * W + 2 * c) * 3;
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int l = kc.ys * load_word(yp + 2 * dx, shift);
      o[3 * dx + 0] = (unsigned char)(clamp_u24(l + t.r) >> 16);
      o[3 * dx + 1] = (unsigned char)(clamp_u24(l + t.g) >> 16);
      o[3 * dx + 2] = (unsigned char)(clamp_u24(l + t.b) >> 16);
    }
  }
}

// ---------------------------------------------------------------------------------
// launcher
// ---------------------------------------------------------------------------------
static int sm_count() {  // of the current device (cached per device)
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (!cached[dev]) {
    int n = 0;
    cached[dev] = (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) ? n : 148;
  }
  return cached[dev];
}

// launch of the fast resize kernel
template <typename Kern>
static cudaError_t launch_fast(Kern kern, dim3 grid, int nt, size_t smem, cudaStream_t st, const DevPlan& P, const KArgs& K) {
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(nt);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  return cudaLaunchKernelEx(&cfg, kern, P, K);
}

template <typename SrcT, typename DstT>
static int launch_all(const NexarPlan* p, const NexarTransformArgs* a, KArgs& K, int n_clips, int aug_mode, int blur_mode) {
  cudaStream_t st = (cudaStream_t)a->stream;
  const int nf = K.n_frames;
  const DevPlan& P = p->d;
  const bool covers_source = (p->g.off_y >= 0 && p->g.off_x >= 0 && p->g.off_y + p->g.resize_h <= p->g.canvas &&
                              p->g.off_x + p->g.resize_w <= p->g.canvas);
  CUDA_TRY(cudaMemsetAsync(K.clip_max, 0, ((size_t)n_clips + nf) * sizeof(unsigned), st));
  const int vis_rows = imin(p->g.resize_h, p->g.canvas);
  const bool prof = (size_t)(2 * g_prof_n + 1) < g_prof_ev.size();
  const bool use_fast = std::is_same<SrcT, uint8_t>::value && p->fast_ok && covers_source && g_resize_variant != 1 &&
                        K.src_row_stride % 16 == 0 && ((uintptr_t)K.src % 16) == 0;
  bool tail_done = false;  // K2 / K3's work has already been enqueued
  int nbands = 1;
  cudaError_t tail_err = cudaSuccess;
  auto launch_tail = [&]() {  // K1.5 + K2 + K3 (K.pass == 4: only the clips whose maximum was > 1)
    const int cs = P.cs;
    if (!K.finfo_by_k1) {
      frame_stats_kernel<<<(nf + 127) / 128, 128, 0, st>>>(P, K, nbands);
      ++g_launches;
    }
    {
      const dim3 cgrid((K.bh * K.bw + 256 * kColourPerThread - 1) / (256 * kColourPerThread), nf);
      // Right behind the fast resize kernel the colour kernel is a PROGRAMMATIC DEPENDENT launch: its CTAs start in the
      // SM slots the resize grid's last wave leaves empty and wait per frame for that frame's publication.
      K.overlap = K.finfo_by_k1 && K.pass == 4 && g_resize_variant != 2;
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = cgrid;
      cfg.blockDim = dim3(256);
      cfg.stream = st;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = at;
      cfg.numAttrs = K.overlap ? 1 : 0;
      tail_err = cudaLaunchKernelEx(&cfg, colour_kernel, P, K);   // checked by the caller (this lambda returns nothing)
      K.overlap = 0;
    }
    // the two production geometries (720p -> 224 and 720p / 1080p -> 320 letterboxes) writing a planar row-contiguous
    // tensor take the specialised kernel; everything else the general one
    const bool planar = K.sx == 1 && K.sy == cs && K.st == (int64_t)cs * cs && g_geo_variant != 1;
    const bool tail = (a->any_flags & kTailFlags) != 0;
    const dim3 sgrid((cs + 31) / 32, (cs + 4 * kGeo2Warps - 1) / (4 * kGeo2Warps), n_clips * ((a->frames_per_clip + kGeo2Frames - 1) / kGeo2Frames));
#define NEXAR_GEO_SPEC(BHV, BWV, CSV)                                                   \
  {                                                                                     \
    if (tail) geometry_spec_kernel<DstT, true, BHV, BWV, CSV><<<sgrid, 32 * kGeo2Warps, 0, st>>>(P, K); \
    else geometry_spec_kernel<DstT, false, BHV, BWV, CSV><<<sgrid, 32 * kGeo2Warps, 0, st>>>(P, K);  \
  }
    if (planar && K.bh == 125 && K.bw == 224 && cs == 224) NEXAR_GEO_SPEC(125, 224, 224)
    else if (planar && K.bh == 180 && K.bw == 320 && cs == 320) NEXAR_GEO_SPEC(180, 320, 320)
    else {
      const dim3 ggrid((cs + 31) / 32, (cs + 16 * kGeoPasses - 1) / (16 * kGeoPasses), n_clips * ((a->frames_per_clip + kGeoFrames - 1) / kGeoFrames));
      if (tail)
        geometry_kernel<DstT, true><<<ggrid, 256, 0, st>>>(P, K);
      else
        geometry_kernel<DstT, false><<<ggrid, 256, 0, st>>>(P, K);
    }
#undef NEXAR_GEO_SPEC
    g_launches += 2;
  };
  if (use_fast) {
    const int need_threads = imax(P.src_w * 3 / 16, imin(P.rw, P.cs));
    // Bands per frame: every band re-reads the source rows it shares with its neighbour and pays the CTA prologue, so
    // fewer is better as long as the grid still fills the machine about 4.5 times over (measured on cfg2 / cfg3 /
    // 8-clip batches: 4 / 2 / 8 bands beat the old fixed 25-rows-per-band rule by 1-6 %).
    if (g_fast_bands > 0) {
      nbands = imin(g_fast_bands, kMaxBands);
    } else {
      const int slots = sm_count() * (need_threads <= 256 ? kFastMinB : 2);
      nbands = imin(8, ((9 * slots) / 2 + nf - 1) / nf);
    }
    nbands = imax(1, imin(nbands, imin(kMaxBands, vis_rows)));
    const int kx = P.kx_al;
    const size_t smem = 2 * (size_t)((P.src_w * 3 + kx * 3 + 15) & ~7) * sizeof(unsigned short);
    dim3 grid(nbands, nf);
    K.pass = 0;
    K.finfo_by_k1 = aug_mode;
    const int ng = (kx / 2 + 3) / 4;
    const int nt_fast = need_threads <= 256 ? 256 : need_threads <= 320 ? 320 : 384;
    const size_t smem_fast = smem + (size_t)ng * nt_fast * 16 + (size_t)(P.n_pairs + 1) * 16;
    if (prof) cudaEventRecord(g_prof_ev[2 * g_prof_n], st);
#define NEXAR_FAST_RS(KXV, NTV, MB, RSV)                                                                          \
  {                                                                                                               \
    constexpr bool kAl = (KXV) == 10;  /* 8-byte window loads exist for the 10-tap kernels only */                \
    record_resize_instance(1, KXV, NTV, RSV, kAl && P.x_align4);                                                  \
    if (kAl && P.x_align4)                                                                                        \
      CUDA_TRY(launch_fast(resize_fast_kernel<KXV, NTV, MB, RSV, DstT, kAl>, grid, NTV, smem_fast, st, P, K));    \
    else                                                                                                          \
      CUDA_TRY(launch_fast(resize_fast_kernel<KXV, NTV, MB, RSV, DstT, false>, grid, NTV, smem_fast, st, P, K));  \
  }
#define NEXAR_FAST(KXV, NTV, MB) NEXAR_FAST_RS(KXV, NTV, MB, 0)
// tightly packed 720p / 1080p rows get the row stride as a compile-time constant (immediate load offsets)
#define NEXAR_FAST_SPEC(KXV, NTV, MB, RSV) \
  if (K.src_row_stride == RSV) NEXAR_FAST_RS(KXV, NTV, MB, RSV) else NEXAR_FAST_RS(KXV, NTV, MB, 0)
    if (need_threads <= 256) {
      if (kx == 10) NEXAR_FAST(10, 256, kFastMinB) else if (kx == 14) NEXAR_FAST_SPEC(14, 256, kFastMinB, 3840) else NEXAR_FAST(20, 256, 2)
    } else if (need_threads <= 320) {
      if (kx == 10) NEXAR_FAST_SPEC(10, 320, 2, 3840) else if (kx == 14) NEXAR_FAST(14, 320, 2) else NEXAR_FAST(20, 320, 2)
    } else {
      if (kx == 10) NEXAR_FAST(10, 384, 2) else if (kx == 14) NEXAR_FAST(14, 384, 2) else NEXAR_FAST_SPEC(20, 384, 2, 5760)
    }
#undef NEXAR_FAST_SPEC
#undef NEXAR_FAST
#undef NEXAR_FAST_RS
    if (prof) cudaEventRecord(g_prof_ev[2 * g_prof_n++ + 1], st);
    // fix-up of clips whose maximum was <= 1 (not divided by 255): their values live in [0,1], below the
    // resolution of the 15-bit staging, so the rare second pass uses the fp32 resample.
    // K1.5 / K2 / K3 for the clips whose maximum was > 1 (pass 4: the others are skipped, see fixup_frame_kernel)
    if (aug_mode) {
      K.pass = 4;
      launch_tail();
    }
    // one launch that finishes the clips whose maximum was <= 1 completely (a no-op CTA per frame otherwise)
    K.pass = 1;
    const size_t gsm = (size_t)P.src_w * 3 * sizeof(float);
    if (gsm > 48 * 1024)
      CUDA_TRY(cudaFuncSetAttribute(fixup_frame_kernel<SrcT, DstT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm));
    {
      // Behind the geometry kernel the fix-up is a programmatic dependent launch too: it only needs the clip flags, which
      // are final before the geometry kernel starts, and the two kernels write disjoint clips, so its (normally empty) CTAs
      // drain through the geometry grid's last wave instead of costing a launch of their own.
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(nf);
      cfg.blockDim = dim3(256);
      cfg.dynamicSmemBytes = gsm;
      cfg.stream = st;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = at;
      cfg.numAttrs = g_resize_variant != 2 ? 1 : 0;
      K.overlap = cfg.numAttrs && !aug_mode;   // directly behind the resize kernel: wait for its completion on the device
      CUDA_TRY(cudaLaunchKernelEx(&cfg, fixup_frame_kernel<SrcT, DstT>, P, K));
      K.overlap = 0;
    }
    tail_done = true;
    g_launches += 2;
  } else {
    record_resize_instance(0, 0, 0, 0, 0);
    nbands = imax(1, imin(kMaxBands, vis_rows / 24));
    const size_t smem = (size_t)P.src_w * 3 * sizeof(float);
    if (smem > 48 * 1024)
      CUDA_TRY(cudaFuncSetAttribute(resize_general_kernel<SrcT, DstT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(nbands, nf);
    if (!covers_source) {
      clip_max_kernel<SrcT><<<dim3(8, nf), 256, 0, st>>>(P, K);
      ++g_launches;
      K.pass = 2;
      resize_general_kernel<SrcT, DstT><<<grid, 256, smem, st>>>(P, K);
      ++g_launches;
    } else {
      K.pass = 0;
      if (prof) cudaEventRecord(g_prof_ev[2 * g_prof_n], st);
      resize_general_kernel<SrcT, DstT><<<grid, 256, smem, st>>>(P, K);
      if (prof) cudaEventRecord(g_prof_ev[2 * g_prof_n++ + 1], st);
      K.pass = 1;
      resize_general_kernel<SrcT, DstT><<<grid, 256, smem, st>>>(P, K);
      g_launches += 2;
    }
  }
  if (aug_mode && !tail_done) {
    K.pass = 0;
    launch_tail();
  }
  if (aug_mode && blur_mode) {
    const int cs = P.cs;
    blur_kernel<DstT><<<dim3((cs * cs + 255) / 256, nf), 256, 0, st>>>(P, K);
    ++g_launches;
  }
  CUDA_TRY(tail_err);
  CUDA_TRY(cudaGetLastError());
  return NEXAR_OK;
}

// Optional chunking of a batch into groups of whole clips (K1, K2, K3 of a chunk back to back; every chunk has its own
// slice of the workspace; the result does not depend on it).  Measured on B200 it does NOT pay: at cfg2 (115 MB of
// intermediate) 3 chunks cost 0.488 ms against 0.429 ms unchunked, at cfg3 (3.8 GB) every chunk size from 3 to 8 clips is
// slower than one launch set (9.4 ms) — the smaller resize grids lose more to wave quantisation and launch gaps than the
// L2 hits of the colour / geometry kernels win.  So the default is one chunk; nexar_set_chunk_clips keeps the experiment.
template <typename SrcT, typename DstT>
static int launch_chunked(const NexarPlan* p, const NexarTransformArgs* a, const KArgs& K0, int aug_mode, int blur_mode) {
  const int n = a->n_clips, T = a->frames_per_clip;
  const int chunk = g_chunk_clips > 0 ? imin(n, g_chunk_clips) : n;
  for (int c0 = 0; c0 < n; c0 += chunk) {
    const int nc = imin(chunk, n - c0);
    const size_t f0 = (size_t)c0 * T;
    KArgs K = K0;
    K.frame_offsets = K0.frame_offsets + f0;
    K.params = K0.params + c0;
    K.dst = (DstT*)K0.dst + (int64_t)c0 * K0.sb;
    K.clip_max = K0.clip_max + c0 + f0;            // [nc clip flags | nc * T frame counters], one memset per chunk
    K.frame_done = K.clip_max + nc;
    K.gray_partial = K0.gray_partial + 2 * f0 * kMaxBands;
    K.finfo = K0.finfo + f0;
    K.inter = K0.inter + f0 * K0.bh * K0.bw;
    K.canvas = K0.canvas + f0 * 3 * (size_t)p->g.canvas * p->g.canvas;
    K.n_frames = nc * T;
    const int rc = launch_all<SrcT, DstT>(p, a, K, nc, aug_mode, blur_mode);
    if (rc != NEXAR_OK) return rc;
  }
  return NEXAR_OK;
}

// ---------------------------------------------------------------------------------
// Materialised sliding windows (BASELINE config 4): the val chain is per frame, so a video is transformed once into
// [3][cs][cs] planes per frame and window k = frames first + k*stride .. first + k*stride+window-1 (the last frame repeated
// past the end, nexar_videos.py:429-433).  The per-frame results live in a ring of ring_frames slots (video frame f in
// slot f % ring_frames; a whole video is the ring of n_frames slots):
// dst[k][c][t] = ring[min(first + k*stride + t, last) % ring_frames][c].  Whole-plane copies, 16 bytes per thread.
// kTable: the slot of every window frame comes from a device table instead (many streams sharing one pool of per-frame
// results): dst[k][c][t] = ring[slots[k*window + t]][c], or, with dst_slots (window 1), ring[dst_slots[k]][c].  Slots are
// clamped into [0, ring_frames): a bad table can never address outside the pool.
// ---------------------------------------------------------------------------------
template <bool kTable>
__global__ void __launch_bounds__(256) gather_windows_kernel(const unsigned char* __restrict__ ring, long long ring_frames,
                                                             long long plane_bytes, int window, int stride, long long first_frame,
                                                             long long last_frame, unsigned char* __restrict__ dst,
                                                             const int* __restrict__ slots, const int* __restrict__ dst_slots) {
  const long long plane = blockIdx.x;              // (k * 3 + c) * window + t
  const int t = (int)(plane % window);
  const long long kc = plane / window;
  const int c = (int)(kc % 3);
  const long long k = kc / 3;
  const unsigned char* s;
  unsigned char* d;
  if constexpr (kTable) {
    const long long f = min(max((long long)__ldg(slots + k * window + t), 0LL), ring_frames - 1);
    s = ring + (f * 3 + c) * plane_bytes;
    if (dst_slots) {
      const long long g = min(max((long long)__ldg(dst_slots + k), 0LL), ring_frames - 1);
      d = dst + (g * 3 + c) * plane_bytes;
    } else {
      d = dst + plane * plane_bytes;
    }
  } else {
    long long f = first_frame + k * stride + t;
    if (f > last_frame) f = last_frame;
    s = ring + ((f % ring_frames) * 3 + c) * plane_bytes;
    d = dst + plane * plane_bytes;
  }
  const long long lo = (long long)blockIdx.y * plane_bytes / gridDim.y, hi = (long long)(blockIdx.y + 1) * plane_bytes / gridDim.y;
  if ((plane_bytes & 15) == 0 && (lo & 15) == 0 && (hi & 15) == 0 && ((((uintptr_t)s) | ((uintptr_t)d)) & 15) == 0) {
    const uint4* s4 = (const uint4*)(s + lo);
    uint4* d4 = (uint4*)(d + lo);
    const long long n4 = (hi - lo) >> 4;
    for (long long i = threadIdx.x; i < n4; i += blockDim.x) __stcs(d4 + i, __ldg(s4 + i));   // the result is written once: streaming store
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) d[i] = s[i];
  }
}

// each plane is split over `split` CTAs so that short videos still fill the machine; splits fall on 16-byte boundaries
template <bool kTable>
static int launch_gather_windows(int64_t planes, const void* ring, int64_t ring_frames, int64_t plane_bytes, int32_t window,
                                 int32_t stride, int64_t first_frame, int64_t last_frame, void* dst, const int32_t* slots,
                                 const int32_t* dst_slots, void* stream) {
  int split = 1;
  while (split < 8 && planes * split < 4 * (int64_t)sm_count() && (plane_bytes / (2 * split)) % 16 == 0 && plane_bytes / (2 * split) >= 4096) split *= 2;
  gather_windows_kernel<kTable><<<dim3((unsigned)planes, split), 256, 0, (cudaStream_t)stream>>>(
      (const unsigned char*)ring, ring_frames, plane_bytes, window, stride, first_frame, last_frame, (unsigned char*)dst, slots,
      dst_slots);
  CUDA_TRY(cudaGetLastError());
  g_launches = 1;
  return NEXAR_OK;
}

static int gather_windows(const char* who, const void* ring, int64_t ring_frames, int64_t plane_bytes, int32_t window,
                          int32_t stride, int64_t first_frame, int64_t last_frame, int64_t n_windows, void* dst, void* stream) {
  if (!ring || !dst || ring_frames <= 0 || plane_bytes <= 0 || window <= 0 || stride <= 0 || n_windows <= 0 ||
      first_frame < 0 || last_frame < first_frame)
    return fail(NEXAR_ERR_INVALID, std::string(who) + ": bad argument");
  const int64_t planes = n_windows * 3 * window;
  if (n_windows > 2147483647LL || planes > 2147483647LL) return fail(NEXAR_ERR_UNSUPPORTED, std::string(who) + ": more than 2^31 planes");
  // the frames one call reads, first_frame .. min(first_frame + (n_windows-1)*stride + window-1, last_frame), must each
  // have a slot of their own: a wider span would read a slot that has been overwritten with a later frame
  const int64_t reach = (n_windows - 1) * stride + window - 1;
  if ((reach < last_frame - first_frame ? reach : last_frame - first_frame) >= ring_frames)
    return fail(NEXAR_ERR_INVALID, std::string(who) + ": the windows span more frames than the ring holds");
  return launch_gather_windows<false>(planes, ring, ring_frames, plane_bytes, window, stride, first_frame, last_frame, dst,
                                      nullptr, nullptr, stream);
}

extern "C" int nexar_gather_windows(const void* frames, int64_t n_frames, int64_t plane_bytes, int32_t window, int32_t stride,
                                    int64_t n_windows, void* dst, void* stream) {
  return gather_windows("gather_windows", frames, n_frames, plane_bytes, window, stride, 0, n_frames - 1, n_windows, dst, stream);
}

extern "C" int nexar_gather_windows_ring(const void* ring, int32_t ring_frames, int64_t plane_bytes, int32_t window, int32_t stride,
                                         int64_t first_frame, int64_t last_frame, int64_t n_windows, void* dst, void* stream) {
  return gather_windows("gather_windows_ring", ring, ring_frames, plane_bytes, window, stride, first_frame, last_frame,
                        n_windows, dst, stream);
}

extern "C" int nexar_gather_windows_table(const void* pool, int32_t pool_frames, int64_t plane_bytes, int32_t window,
                                          const int32_t* slots, int64_t n_windows, void* dst, const int32_t* dst_slots,
                                          void* stream) {
  if (!pool || !slots || (dst == nullptr) == (dst_slots == nullptr) || pool_frames <= 0 || plane_bytes <= 0 || window <= 0 ||
      n_windows <= 0 || (dst_slots && window != 1))
    return fail(NEXAR_ERR_INVALID, "gather_windows_table: bad argument");
  if (n_windows > 2147483647LL / (3LL * window)) return fail(NEXAR_ERR_INVALID, "gather_windows_table: more than 2^31 planes");
  return launch_gather_windows<true>(n_windows * 3 * window, pool, pool_frames, plane_bytes, window, 1, 0, 0,
                                     dst_slots ? const_cast<void*>(pool) : dst, slots, dst_slots, stream);
}

extern "C" int nexar_clip_transform(const NexarPlan* p, const NexarTransformArgs* a) {
  g_launches = 0;
  record_resize_instance(0, 0, 0, 0, 0);
  if (!p || !a) return fail(NEXAR_ERR_INVALID, "clip_transform: null argument");
  if (a->struct_size != sizeof(NexarTransformArgs)) return fail(NEXAR_ERR_INVALID, "clip_transform: NexarTransformArgs size mismatch (ABI)");
  if (a->n_clips <= 0 || a->frames_per_clip <= 0) return fail(NEXAR_ERR_INVALID, "clip_transform: empty batch");
  if ((int64_t)a->n_clips * a->frames_per_clip > 65535)  // frames are a grid dimension (y / z): split larger batches
    return fail(NEXAR_ERR_UNSUPPORTED, "clip_transform: more than 65535 frames in one call");
  if (!a->src || !a->frame_offsets || !a->params || !a->dst) return fail(NEXAR_ERR_INVALID, "clip_transform: null buffer");
  if (a->dst_dtype != NEXAR_DST_F32 && a->dst_dtype != NEXAR_DST_BF16 && a->dst_dtype != NEXAR_DST_F16)
    return fail(NEXAR_ERR_INVALID, "clip_transform: bad dst_dtype");
  const size_t need = nexar_workspace_bytes_for(p, a->n_clips, a->frames_per_clip, a->any_flags);
  if (!a->workspace || a->workspace_bytes < need) return fail(NEXAR_ERR_WORKSPACE, "clip_transform: workspace too small");
  for (int c = 0; c < 3; ++c)
    if (a->normalize && !(a->std[c] != 0.0f)) return fail(NEXAR_ERR_INVALID, "clip_transform: std must be non-zero");
  const bool nv12 = p->src_dtype == NEXAR_SRC_NV12;
  const size_t esz = p->src_dtype == NEXAR_SRC_F32 ? 4 : 1;
  const int64_t sample_bytes = nv12 && p->yuv_16bit ? 2 : 1;
  if (a->src_row_stride < (int64_t)(nv12 ? p->g.src_w * sample_bytes : p->g.src_w * 3 * esz))
    return fail(NEXAR_ERR_INVALID, "clip_transform: src_row_stride smaller than a row");
  if (nv12 && p->yuv_layout == NEXAR_YUV_I420 && (a->src_row_stride & 1))
    return fail(NEXAR_ERR_INVALID, "clip_transform: I420 surfaces need an even src_row_stride");
  if (nv12 && p->yuv_16bit && (a->src_row_stride & 1))
    return fail(NEXAR_ERR_INVALID, "clip_transform: 16-bit surfaces need an even src_row_stride");

  Workspace w = carve(p, a->n_clips, a->frames_per_clip, a->workspace, a->any_flags);
  KArgs K;
  K.src = a->src;
  K.frame_offsets = a->frame_offsets;
  K.src_row_stride = a->src_row_stride;
  if (nv12) {
    // decoder surfaces -> packed RGB bytes in the workspace (one launch), then the uint8 path on those
    const int H = p->g.src_h, W = p->g.src_w, nf = a->n_clips * a->frames_per_clip;
    cudaStream_t st = (cudaStream_t)a->stream;
    const int64_t pitch = a->src_row_stride, uoff = (int64_t)p->yuv_luma_rows * pitch;
    const int64_t voff = uoff + (int64_t)(p->yuv_luma_rows / 2) * (pitch / 2);
    const unsigned char* s = (const unsigned char*)a->src;
    // pitch % 16 == 0 with an even luma height also keeps the 8-byte I420 chroma loads aligned
    const bool vec = (W % 16) == 0 && (pitch % 16) == 0 && (((uintptr_t)a->src) & 15) == 0;
    const dim3 gv(((W / 16) * (H / 2) + 255) / 256, nf), ga(((W / 2) * (H / 2) + 255) / 256, nf);
    if (p->yuv_16bit) {
      // 32-byte luma / NV12 chroma and 16-byte I420 chroma loads per thread: the chroma rows stay 16-byte aligned
      const int sh = p->yuv_shift;
      const bool vec16 = (W % 16) == 0 && (pitch % (p->yuv_layout == NEXAR_YUV_I420 ? 32 : 16)) == 0 && (((uintptr_t)a->src) & 15) == 0;
      if (p->yuv_layout == NEXAR_YUV_I420) {
        if (vec16)
          yuv420_16_to_rgb_vec_kernel<NEXAR_YUV_I420><<<gv, 256, 0, st>>>(s, a->frame_offsets, pitch, uoff, voff, p->yuv_coef, sh, H, W, w.rgb, w.rgb_offsets);
        else
          yuv420_16_to_rgb_any_kernel<NEXAR_YUV_I420><<<ga, 256, 0, st>>>(s, a->frame_offsets, pitch, uoff, voff, p->yuv_coef, sh, H, W, w.rgb, w.rgb_offsets);
      } else {
        if (vec16)
          yuv420_16_to_rgb_vec_kernel<NEXAR_YUV_NV12><<<gv, 256, 0, st>>>(s, a->frame_offsets, pitch, uoff, voff, p->yuv_coef, sh, H, W, w.rgb, w.rgb_offsets);
        else
          yuv420_16_to_rgb_any_kernel<NEXAR_YUV_NV12><<<ga, 256, 0, st>>>(s, a->frame_offsets, pitch, uoff, voff, p->yuv_coef, sh, H, W, w.rgb, w.rgb_offsets);
      }
    } else if (p->yuv_layout == NEXAR_YUV_I420) {
      if (vec)
        yuv420_to_rgb_vec_kernel<NEXAR_YUV_I420><<<gv, 256, 0, st>>>(s, a->frame_offsets, pitch, uoff, voff, p->yuv_coef, H, W, w.rgb, w.rgb_offsets);
      else
        yuv420_to_rgb_any_kernel<NEXAR_YUV_I420><<<ga, 256, 0, st>>>(s, a->frame_offsets, pitch, uoff, voff, p->yuv_coef, H, W, w.rgb, w.rgb_offsets);
    } else {
      if (vec)
        yuv420_to_rgb_vec_kernel<NEXAR_YUV_NV12><<<gv, 256, 0, st>>>(s, a->frame_offsets, pitch, uoff, voff, p->yuv_coef, H, W, w.rgb, w.rgb_offsets);
      else
        yuv420_to_rgb_any_kernel<NEXAR_YUV_NV12><<<ga, 256, 0, st>>>(s, a->frame_offsets, pitch, uoff, voff, p->yuv_coef, H, W, w.rgb, w.rgb_offsets);
    }
    CUDA_TRY(cudaGetLastError());
    ++g_launches;
    K.src = w.rgb;
    K.frame_offsets = w.rgb_offsets;
    K.src_row_stride = (int64_t)W * 3;
  }
  K.params = a->params;
  K.dst = a->dst;
  K.sb = a->dst_stride[0];
  K.sc = a->dst_stride[1];
  K.st = a->dst_stride[2];
  K.sy = a->dst_stride[3];
  K.sx = a->dst_stride[4];
  K.T = a->frames_per_clip;
  K.normalize = a->normalize;
  for (int c = 0; c < 3; ++c) {
    const double inv = a->normalize ? 1.0 / (double)a->std[c] : 1.0;
    K.nscale[c] = (float)inv;
    K.nbias[c] = a->normalize ? (float)(-(double)a->mean[c] * inv) : 0.0f;
  }
  K.clip_max = w.clip_max;
  K.frame_done = w.frame_done;
  K.finfo_by_k1 = 0;
  K.overlap = 0;
  K.gray_partial = w.gray_partial;
  K.finfo = w.finfo;
  K.inter = w.inter;
  K.canvas = w.canvas;
  K.n_frames = a->n_clips * a->frames_per_clip;
  K.bh = imin(p->g.resize_h, p->g.canvas);
  K.bw = imin(p->g.resize_w, p->g.canvas);
  K.pass = 0;
  // stages no clip of the batch needs are not launched; within a launch, clips without the flag exit at once.
  const int aug_mode = (a->any_flags & NEXAR_AUG) != 0, blur_mode = (a->any_flags & NEXAR_BLUR) != 0;
  if (aug_mode) {  // K3 addresses one frame of the destination with 32-bit element offsets
    const double span = 2.0 * std::fabs((double)K.sc) + (double)(p->g.canvas - 1) * (std::fabs((double)K.sy) + std::fabs((double)K.sx));
    if (span >= 2147483647.0) return fail(NEXAR_ERR_UNSUPPORTED, "clip_transform: destination strides span more than 2^31 elements per frame");
  }
  if (p->src_dtype != NEXAR_SRC_F32) {
    if (a->dst_dtype == NEXAR_DST_F32) return launch_chunked<uint8_t, float>(p, a, K, aug_mode, blur_mode);
    if (a->dst_dtype == NEXAR_DST_F16) return launch_chunked<uint8_t, __half>(p, a, K, aug_mode, blur_mode);
    return launch_chunked<uint8_t, __nv_bfloat16>(p, a, K, aug_mode, blur_mode);
  }
  if (a->dst_dtype == NEXAR_DST_F32) return launch_chunked<float, float>(p, a, K, aug_mode, blur_mode);
  if (a->dst_dtype == NEXAR_DST_F16) return launch_chunked<float, __half>(p, a, K, aug_mode, blur_mode);
  return launch_chunked<float, __nv_bfloat16>(p, a, K, aug_mode, blur_mode);
}

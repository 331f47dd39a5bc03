// wind.cu -- hub-height extrapolation + power-curve interpolation, fused with
// the shape reduce.  Follows wind.py:75-112 (extrapolate_wind_speed) and
// convert.py:648-649 (np.interp(v_hub, V, POW / P)).
//
// Algorithmic traffic: 8 B per cell-timestep (wnd + roughness | shear
// exponent), 4 B in the wnd{hub}m fast lane (wind.py:75-78).
#include <cmath>
#include <cstring>
#include <vector>

#include "kernels.cuh"

// experiment knobs (tools/build_variants.sh)
#ifndef ATL_WIND_SAT_R
#define ATL_WIND_SAT_R 8  // replicas of the saturating table's 256 rows (8: 16 KB, 16: 32 KB)
#endif
#ifndef ATL_WIND_B
#define ATL_WIND_B 2
#define ATL_WIND_MINB 6
#endif
#ifndef ATL_WIND_PREFETCH
#define ATL_WIND_PREFETCH 1  // L2 prefetch distance in batches (0 = off); measured: big 0.868 -> 0.930, small 0.822 -> 0.816
#endif
#ifndef ATL_WIND_RESIDENT
#define ATL_WIND_RESIDENT 1
#endif

namespace atl {

// Power curve in shared memory.
//
// LUT mode (every shipped turbine; the host decides): a uniform grid of NB buckets on
// [V0, Vn-1], shifted by half a bucket, in which every bucket holds at most ONE
// distinct knot value, none within 1e-3 of a bucket edge.  One float4 per bucket,
//   {k, y(k), slope below k, slope from k on}
// k = the bucket's knot rounded UP to float (so `x >= k` is exactly the float64
// comparison `x >= V[j]` numpy's search does for a float x), or the bucket centre
// when it has no knot (both slopes equal).  The curve stored is the CONTINUOUS
// one: np.interp's jumps at duplicate knots (cut-in step, the appended cut-out) are
// taken out on the host and put back by two selects -- at most one interior jump
// plus the one at the last knot, else the fallback.  So a cell costs one 16-byte
// shared-memory load.  For NB <= 128 the table is replicated 8x, entry (b, lane%8),
// which makes the 128-bit loads bank-conflict free for arbitrary bucket patterns
// (a quarter-warp's 8 lanes hit 8 different 16-byte bank groups).
//
// Fallback (NK = power of two > n_knots):
//   xcmp[NK]   knot abscissae rounded UP to float, padded with +inf so a
//              branch-free binary search counts the knots <= x
//   seg[NK+1]  float4 {x0, f0, slope, -} indexed by that COUNT c: c = 0 -> left
//              clamp f[0]; 1 <= c < n -> segment [V[c-1], V[c]) with x0 = V[c-1]
//              (nearest float), slope = 0 on zero-width (duplicate-knot)
//              segments; c >= n -> right clamp f[n-1]      (np.interp semantics)

// One LUT lookup; the SAME function evaluates on the host for the CPU tests
// (atl_wind_curve_eval_host), with the PTX clamp / floor spelled out.
__host__ __device__ __forceinline__ float lut_interp(float x, const char* lut, int stride,
                                                     float x_lo, float x_hi, float inv_w, float c0,
                                                     float k_jump, float jump, float k_end,
                                                     float y_end) {
#ifdef __CUDA_ARCH__
  // NaN-propagating clamp: a NaN speed picks bucket 0 and comes out NaN
  const float xc = fmin_nan(fmax_nan(x, x_lo), x_hi);
  const int b = __float2int_rd(fmaf(xc, inv_w, c0));
#else
  const float xc = (x != x) ? x : std::fmin(std::fmax(x, x_lo), x_hi);
  const int b = (x != x) ? 0 : (int)std::floor(std::fmaf(xc, inv_w, c0));
#endif
  const float4 e = *reinterpret_cast<const float4*>(lut + b * stride);
  const float sl = (x >= e.x) ? e.w : e.z;
  float y = fmaf(sl, xc - e.x, e.y);
  y = (x >= k_jump) ? y + jump : y;
  return (x >= k_end) ? y_end : y;
}

// Lattice mode: all knots lie on lo + m*w, so every bucket [lo + b*w, lo + (b+1)*w)
// sits inside ONE segment of the (jump-free, hence continuous) curve and holds just
// {slope, intercept}: which bucket a speed within rounding of a knot lands in does
// not matter.  The steps come back through `nj` exact compares.  `lut` points one
// entry past a guard copy of bucket 0 (floor may give -1 at x_lo).
template <int NJ>  // number of steps to add back (compile time: each costs 3 instructions per cell)
__host__ __device__ __forceinline__ float lattice_interp(float x, const char* lut, int stride,
                                                         float x_lo, float x_hi, float inv_w,
                                                         float c0, float k1, float j1,
                                                         float k2, float j2) {
#ifdef __CUDA_ARCH__
  const float xc = fmin_nan(fmax_nan(x, x_lo), x_hi);
  const int b = __float2int_rd(fmaf(xc, inv_w, c0));
#else
  const float xc = (x != x) ? x : std::fmin(std::fmax(x, x_lo), x_hi);
  const int b = (x != x) ? 0 : (int)std::floor(std::fmaf(xc, inv_w, c0));
#endif
  const float2 e = *reinterpret_cast<const float2*>(lut + b * stride);
  float y = fmaf(e.x, xc, e.y);
  if (NJ > 0) y = (x >= k1) ? y + j1 : y;
  if (NJ > 1) y = (x >= k2) ? y + j2 : y;
  return y;
}

// Saturating lattice mode: 256 rows; row 0 = flat left end, rows 1..NB = the NB lattice buckets
// (steps folded in, see build_curve), rows NB+1..255 = flat right end.  The float -> u8
// conversion (one F2I.U8.FLOOR) saturates to [0, 255] and sends NaN to 0, so the speed needs no
// clamps: 5 instructions per cell (FFMA, F2I, IMAD, LDS.64, FFMA).  A flat row times an
// infinite speed is NaN -- CLAMPED = true (the kernels' cold exact path, taken when a fast
// result is not finite) evaluates the same table with the speed clamped to the knot range
// first, which is np.interp for +-inf and keeps NaN.
template <bool CLAMPED>
__host__ __device__ __forceinline__ float sat_interp(float x, const char* lut, int stride,
                                                     float x_lo, float x_hi, float inv_w, float c0) {
#ifdef __CUDA_ARCH__
  const float xc = CLAMPED ? fmin_nan(fmax_nan(x, x_lo), x_hi) : x;
  unsigned int b;
  asm("cvt.rmi.u8.f32 %0, %1;" : "=r"(b) : "f"(fmaf(xc, inv_w, c0)));
#else
  const float xc = (!CLAMPED || x != x) ? x : std::fmin(std::fmax(x, x_lo), x_hi);
  const float t = std::fmaf(xc, inv_w, c0);
  const unsigned int b = (t != t) ? 0u : (unsigned int)std::fmin(std::fmax(std::floor(t), 0.f), 255.f);
#endif
  const float2 e = *reinterpret_cast<const float2*>(lut + b * stride);
  return fmaf(e.x, xc, e.y);
}

// METHOD: ATL_WIND_NONE / _LOG / _POWER and LMODE (0: binary search or general LUT, chosen at
// run time; 1 + nj: lattice LUT with nj steps; 4: saturating lattice LUT) are compile time: no predicated duplicates of
// the loads, no uniform branches or re-loaded kernel parameters in the per-cell code.
template <bool VEC, int METHOD, int LMODE>
struct WindPhys {
  static constexpr bool kVec = VEC;
  using Geom = TileGeomT<VEC>;
  const float* wnd;
  const float* aux;
  const float* curve;  // device: the LUT, or xcmp | seg for the fallback
  int64_t S;
  int method;
  int n_knots, NK;
  float lg2_to, lg2_from, lg2_ratio;
  float neg_lg2_to, neg_lg2_from;
  float x_lo, x_hi;
  int use_lut, n_stage;   // use_lut: 0 binary search, 1 general LUT, 2 lattice LUT
  float inv_w, c0;        // bucket = floor(x * inv_w + c0)
  int lut_stride, rep_mask;  // bytes between buckets; lane & rep_mask picks the replica
  int lut_entry;          // bytes per entry (16 general, 8 lattice)
  int nj;                 // lattice: number of steps (0..2), at k_jump / k_end
  float k_jump, jump;     // general: interior jump, y += jump for x >= k_jump (+inf: none)
  float k_end, y_end;     // general: x >= k_end -> y_end (right clamp incl. cut-out step);
                          // lattice: second step, y += y_end for x >= k_end

  struct Cell {
    int rep_off;  // byte offset of this lane's replica inside a bucket's entries
  };
  struct Raw {
    float w[4], a[4];
  };
  // general LUT: <= 129 buckets x 8 replicas or <= 1025 x 1, 4 floats each; lattice:
  // <= 130 x 16 or <= 258 x 4 replicas, 2 floats each; fallback: 256 + 4*257
  static constexpr int kSmemFloats = 2 * 130 * 16 > 2 * 256 * ATL_WIND_SAT_R ? 2 * 130 * 16 : 2 * 256 * ATL_WIND_SAT_R;
  static constexpr int kBatch = ATL_WIND_B, kMinBlocks = ATL_WIND_MINB;  // (7 CTAs = 28 warps per SM measured the same)
  // NaN speeds / roughness propagate like np.interp's in every mode; the saturating table also
  // turns +-inf speeds into NaN and relies on the cold exact path for them
  static constexpr bool kHasExact = LMODE == 4;
  static constexpr bool kResidentWeights = ATL_WIND_RESIDENT != 0 && VEC;  // first slot group's weights in registers
  static constexpr int kL2Prefetch = VEC ? ATL_WIND_PREFETCH : 0;
  static constexpr bool kSplitMask = true;  // issue-bound: interior tiles skip the out-of-grid selects
  static constexpr bool kStaged = false;
  static constexpr int kStage = 8, kBatchStaged = 4, kMinBlocksStaged = 5;  // staged: 4 register sets, 5 CTAs (smem)

  __device__ void stage(float* smem) const {
    for (int i = threadIdx.x; i < n_stage; i += blockDim.x) smem[i] = curve[i];
    __syncthreads();
  }
  __device__ void init(Cell& c, const Geom&, const float*) const {
    c.rep_off = ((threadIdx.x & 31) & rep_mask) * lut_entry;
  }
  __device__ void load(const Cell&, const Geom& g, int64_t tb, Raw& r) const {
    load4(wnd, tb, g, r.w);
    if (METHOD != ATL_WIND_NONE) load4(aux, tb, g, r.a);
  }
  __device__ void prefetch(const Cell&, const Geom& g, int64_t tb) const {
    prefetch4_l2(wnd, tb, g);
    if (METHOD != ATL_WIND_NONE) prefetch4_l2(aux, tb, g);
  }
  // np.interp for the lane's 4 values at once.
  template <bool EXACT = false>
  __device__ __forceinline__ void interp4(const Cell& c, const float (&x)[4], float (&r)[4],
                                          const float* sm) const {
    if constexpr (LMODE == 4) {
      const char* lut = reinterpret_cast<const char*>(sm) + c.rep_off;
#pragma unroll
      for (int i = 0; i < 4; ++i) r[i] = sat_interp<EXACT>(x[i], lut, lut_stride, x_lo, x_hi, inv_w, c0);
      return;
    } else if constexpr (LMODE >= 1) {
      const char* lut = reinterpret_cast<const char*>(sm) + lut_stride + c.rep_off;  // skip the guard
#pragma unroll
      for (int i = 0; i < 4; ++i)
        r[i] = lattice_interp<LMODE - 1>(x[i], lut, lut_stride, x_lo, x_hi, inv_w, c0, k_jump, jump, k_end, y_end);
      return;
    }
    if (use_lut) {
      const char* lut = reinterpret_cast<const char*>(sm) + c.rep_off;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        r[i] = lut_interp(x[i], lut, lut_stride, x_lo, x_hi, inv_w, c0, k_jump, jump, k_end, y_end);
      return;
    }
    const float* xcmp = sm;
    const float4* seg = reinterpret_cast<const float4*>(sm + NK);
    int cnt[4] = {0, 0, 0, 0};  // number of knots <= x  (NaN compares false -> 0)
#pragma unroll 1
    for (int step = NK >> 1; step >= 1; step >>= 1) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (xcmp[cnt[i] + step - 1] <= x[i]) cnt[i] += step;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 s = seg[min(cnt[i], n_knots)];
      // clamp keeps inf * 0 out of the clamped ends; NaN is restored below
      const float xc = fminf(fmaxf(x[i], x_lo), x_hi);
      const float y = fmaf(s.z, xc - s.x, s.y);
      r[i] = (x[i] != x[i] && n_knots > 1) ? x[i] : y;  // np.interp: one knot -> constant, even for NaN
    }
  }
  __device__ __forceinline__ void compute(const Cell& c, const Geom&, int, const Raw& r, float (&v)[4],
                                          const float* sm) const {
    compute_impl<false>(c, r, v, sm);
  }
  // cold, out of line, arguments by value (see PvPhys::exact_by_value)
  static __device__ __noinline__ float4 exact_by_value(const WindPhys self, const Cell c, const Raw r,
                                                       const float* sm) {
    float v[4];
    self.template compute_impl<true>(c, r, v, sm);
    return make_float4(v[0], v[1], v[2], v[3]);
  }
  __device__ __forceinline__ void compute_exact(const Cell& c, const Geom&, int, const Raw& r,
                                                float (&v)[4], const float* sm) const {
    const float4 o = exact_by_value(*this, c, r, sm);
    v[0] = o.x; v[1] = o.y; v[2] = o.z; v[3] = o.w;
  }
  template <bool EXACT>
  __device__ __forceinline__ void compute_impl(const Cell& c, const Raw& r, float (&v)[4],
                                               const float* sm) const {
    float x[4];
    if (METHOD == ATL_WIND_LOG) {
      // v * ln(to/z0) / ln(from/z0) = v * (lg2 to - lg2 z0) / (lg2 from - lg2 z0)
      // (not rewritten as v + v*c/(..): z0 = 0 must give NaN = inf/inf like the reference).
      // The subtractions and products run on the packed FP32 pipe, two cells per instruction.
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        // (L - lg2 to) / (L - lg2 from): both signs flipped, so no negations
        const float2 L = make_float2(__log2f(r.a[2 * p]), __log2f(r.a[2 * p + 1]));
        const float2 num = __fadd2_rn(L, make_float2(neg_lg2_to, neg_lg2_to));
        const float2 den = __fadd2_rn(L, make_float2(neg_lg2_from, neg_lg2_from));
        const float2 q = __fmul2_rn(num, make_float2(rcp_approx(den.x), rcp_approx(den.y)));
        const float2 xv = __fmul2_rn(make_float2(r.w[2 * p], r.w[2 * p + 1]), q);
        x[2 * p] = xv.x;
        x[2 * p + 1] = xv.y;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        x[i] = r.w[i];
        if (METHOD == ATL_WIND_POWER) x[i] = x[i] * exp2f(r.a[i] * lg2_ratio);  // v * (to/from)^alpha
      }
    }
    interp4<EXACT>(c, x, v, sm);
  }
};

}  // namespace atl

using namespace atl;

struct AtlWindOp : AtlOpBase {
  int method;
  int n_knots, NK;
  float lg2_to, lg2_from, lg2_ratio;
  float x_lo, x_hi;
  int use_lut, n_stage;
  float inv_w, c0;
  int lut_stride, rep_mask, lut_entry, nj;
  float k_jump, jump, k_end, y_end;
  float* d_curve = nullptr;
};

template <bool VEC, int METHOD, int LMODE>
static WindPhys<VEC, METHOD, LMODE> make_phys(const AtlWindOp* op, const AtlWindFields* f) {
  WindPhys<VEC, METHOD, LMODE> p;
  p.wnd = f->wnd;
  p.aux = f->aux;
  p.curve = op->d_curve;
  p.S = op->grid.S;
  p.method = op->method;
  p.n_knots = op->n_knots;
  p.NK = op->NK;
  p.lg2_to = op->lg2_to;
  p.lg2_from = op->lg2_from;
  p.lg2_ratio = op->lg2_ratio;
  p.neg_lg2_to = -op->lg2_to;
  p.neg_lg2_from = -op->lg2_from;
  p.x_lo = op->x_lo;
  p.x_hi = op->x_hi;
  p.use_lut = op->use_lut;
  p.n_stage = op->n_stage;
  p.inv_w = op->inv_w;
  p.c0 = op->c0;
  p.lut_stride = op->lut_stride;
  p.rep_mask = op->rep_mask;
  p.lut_entry = op->lut_entry;
  p.nj = op->nj;
  p.k_jump = op->k_jump;
  p.jump = op->jump;
  p.k_end = op->k_end;
  p.y_end = op->y_end;
  return p;
}

// compile-time table mode of the operator: 0 generic (binary search / general LUT), 1 + nj lattice,
// 4 saturating lattice
static int lut_mode(const AtlWindOp* op) { return op->use_lut == 3 ? 4 : op->use_lut == 2 ? 1 + op->nj : 0; }

// The wind operator's part of the shared entry sequence (kernels.cuh: run_entry).  Wind has no
// time axis: t0 is ignored.
struct WindBinding {
  using Op = AtlWindOp;
  using Fields = AtlWindFields;
  static int check(const AtlWindOp* op, const AtlWindFields* f, int64_t, int64_t) {
    ATL_REQUIRE(op && f && f->wnd, "NULL argument");
    ATL_REQUIRE(op->method == ATL_WIND_NONE || f->aux,
                "roughness / wnd_shear_exp field missing for the chosen method");
    return ATL_OK;
  }
  template <class F, class Visit>
  static void each_field(const AtlWindOp*, F& f, Visit visit) {
    visit(f.wnd, 4);
    visit(f.aux, 4);
  }
  template <class Run>
  static int with_phys(const AtlWindOp* op, const AtlWindFields* f, int64_t, Run run) {
#define ATL_WIND_CASE(M, L) \
  case 8 * M + L:           \
    return run([&](auto vec) { return make_phys<decltype(vec)::value, M, L>(op, f); });
#define ATL_WIND_METHOD_CASES(M) \
  ATL_WIND_CASE(M, 0) ATL_WIND_CASE(M, 1) ATL_WIND_CASE(M, 2) ATL_WIND_CASE(M, 3) ATL_WIND_CASE(M, 4)
    switch (8 * op->method + lut_mode(op)) {
      ATL_WIND_METHOD_CASES(ATL_WIND_NONE) ATL_WIND_METHOD_CASES(ATL_WIND_LOG) ATL_WIND_METHOD_CASES(ATL_WIND_POWER)
    }
#undef ATL_WIND_METHOD_CASES
#undef ATL_WIND_CASE
    return ATL_ERR_INVALID;
  }
};

// Host-side tables of a power curve (shared by atl_wind_create and the host
// evaluator atl_wind_curve_eval_host the CPU tests use).
struct CurveTables {
  std::vector<float> curve;
  int n_knots = 0, NK = 0, use_lut = 0, lut_stride = 16, rep_mask = 0, lut_entry = 16, nj = 0;
  float x_lo = 0.f, x_hi = 0.f, inv_w = 0.f, c0 = 0.f;
  float k_jump = INFINITY, jump = 0.f, k_end = 0.f, y_end = 0.f;
};

// force_mode: -1 best available, 0 binary search, 1 general LUT, 2 lattice LUT with compares,
// 3 saturating lattice LUT
static int build_curve(const double* V, const double* POW, int n, CurveTables& T,
                       int force_mode = -1) {
  const bool force_fallback = force_mode == 0;
  ATL_REQUIRE(n >= 1 && n <= 255, "n_knots must be in [1, 255]");
  ATL_REQUIRE(V && POW, "power curve missing");
  for (int i = 1; i < n; ++i)
    ATL_REQUIRE(V[i] >= V[i - 1], "wind speed knots must be non-decreasing");
  int NK = 2;  // strictly more slots than knots: the search counts up to NK-1
  while (NK <= n) NK <<= 1;
  // xcmp[NK] followed by seg[NK + 1] (float4), see WindPhys; NK * 4 bytes keeps
  // the float4 part 16-byte aligned (NK >= 4)
  if (NK < 4) NK = 4;
  std::vector<float> curve((size_t)NK + 4 * ((size_t)NK + 1), 0.f);
  for (int j = 0; j < NK; ++j) {
    if (j < n) {
      const double x = V[j];
      float xc = (float)x;
      if ((double)xc < x) xc = nextafterf(xc, INFINITY);  // round up
      curve[j] = xc;
    } else {
      curve[j] = INFINITY;
    }
  }
  float* seg = curve.data() + NK;
  for (int c = 0; c <= NK; ++c) {
    float x0 = 0.f, f0 = 0.f, sl = 0.f;
    if (c == 0) {
      x0 = (float)V[0];
      f0 = (float)POW[0];
    } else if (c >= n) {
      x0 = (float)V[n - 1];
      f0 = (float)POW[n - 1];
    } else {
      const int j = c - 1;
      x0 = (float)V[j];
      f0 = (float)POW[j];
      if (V[j + 1] > V[j])
        sl = (float)((POW[j + 1] - POW[j]) / (V[j + 1] - V[j]));
    }
    seg[4 * c + 0] = x0;
    seg[4 * c + 1] = f0;
    seg[4 * c + 2] = sl;
    seg[4 * c + 3] = 0.f;
  }
  // ---- uniform-bucket LUT (see the comment above WindPhys)
  auto ceil_f = [](double v) {
    float f = (float)v;
    if ((double)f < v) f = nextafterf(f, INFINITY);
    return f;
  };
  int use_lut = 0, lut_stride = 16, rep_mask = 0, lut_entry = 16, nj = 0;
  float inv_w = 0.f, c0 = 0.f;
  float k_jump = INFINITY, jump = 0.f;
  float k_end = ceil_f(V[n - 1]), y_end = (float)POW[n - 1];
  // ---- lattice LUT: knots on lo + m*w, at most two steps
  if (n >= 2 && V[n - 1] > V[0] && (force_mode == -1 || force_mode >= 2)) {
    const double lo = V[0], hi = V[n - 1];
    struct Jump { double K, J; };
    std::vector<Jump> jumps;
    std::vector<int> last;  // last index of every run of equal knots
    for (int a = 0; a < n;) {
      int z = a;
      while (z + 1 < n && V[z + 1] == V[a]) ++z;
      if (POW[z] != POW[a]) jumps.push_back({V[a], POW[z] - POW[a]});
      last.push_back(z);
      a = z + 1;
    }
    double dmin = hi - lo;
    for (size_t k = 1; k < last.size(); ++k) dmin = std::min(dmin, V[last[k]] - V[last[k - 1]]);
    int NB = 0;
    double wdt = 0.0;
    for (int q = 1; q <= 8 && !NB; ++q) {
      const double w = dmin / q;
      const double nb = (hi - lo) / w;
      if (nb > 256.5) break;
      bool ok = std::fabs(nb - std::round(nb)) < 1e-6;
      for (size_t k = 0; k < last.size() && ok; ++k) {
        const double m = (V[last[k]] - lo) / w;
        ok = std::fabs(m - std::round(m)) < 1e-6;
      }
      if (ok) {
        NB = (int)std::round(nb);
        wdt = (hi - lo) / NB;
      }
    }
    if (NB) {
      const int R = NB <= 128 ? 16 : 4;
      std::vector<float> lut((size_t)(NB + 2) * R * 2);
      auto put = [&](int slot, double sl, double icpt) {
        const float e[2] = {(float)sl, (float)icpt};
        for (int r = 0; r < R; ++r) std::memcpy(&lut[((size_t)slot * R + r) * 2], e, 8);
      };
      // value of the continuous (steps removed) curve at the last knot of run k
      auto cont = [&](size_t k) {
        double y = POW[last[k]];
        for (const Jump& j : jumps)
          if (j.K <= V[last[k]]) y -= j.J;
        return y;
      };
      size_t k = 0;
      for (int b = 0; b < NB; ++b) {
        const double mid = lo + (b + 0.5) * wdt;
        while (k + 1 < last.size() && V[last[k + 1]] <= mid) ++k;
        const int z = last[k];  // segment [V[z], V[z+1])
        const double sl = (POW[z + 1] - POW[z]) / (V[z + 1] - V[z]);
        put(b + 1, sl, cont(k) - sl * V[z]);
        if (b == 0) put(0, sl, cont(k) - sl * V[z]);  // guard for floor(..) == -1
      }
      put(NB + 1, 0.0, cont(last.size() - 1));  // x == x_hi: right clamp of the continuous curve
      use_lut = 2;
      lut_entry = 8;
      lut_stride = 8 * R;
      rep_mask = R - 1;
      inv_w = (float)(1.0 / wdt);
      c0 = (float)(-lo / wdt);
      nj = (int)jumps.size();
      k_jump = k_end = INFINITY;
      jump = y_end = 0.f;
      // A step sits on a bucket boundary.  When the bucket function itself -- the kernel's
      // floor(fmaf(clamp(x), inv_w, c0)), monotone in x -- crosses that boundary EXACTLY at the
      // step's float threshold k (first float >= the knot), i.e. bucket(k) = m and
      // bucket(prev(k)) = m - 1, the table can hold the curve WITH its steps and the per-cell
      // compares go away (nj = 0).  True for the usual curves (knots and bucket widths that are
      // binary fractions); verified here in the kernel's own float arithmetic, a few ulps of
      // c0 / inv_w are tried otherwise.  A step at the first knot cannot fold (x < x_lo clamps
      // onto it).  `sat`: the saturating table's bucket function (no clamp of x, rows shifted by
      // one, floor saturated to [0, 255]).
      const float x_lo_f = (float)V[0], x_hi_f = (float)V[n - 1];
      auto bucket = [&](float x, float iw, float cc, bool sat) {
        if (sat) return (int)std::fmin(std::fmax(std::floor(std::fmaf(x, iw, cc)), 0.f), 255.f);
        const float xc = std::fmin(std::fmax(x, x_lo_f), x_hi_f);
        return (int)std::floor(std::fmaf(xc, iw, cc));
      };
      bool foldable = true;
      for (const Jump& j : jumps) foldable = foldable && j.K > lo && (double)ceil_f(j.K) <= (double)x_hi_f;
      auto search = [&](bool sat, float& iw_out, float& cc_out) {
        const float iw0 = (float)(1.0 / wdt), cc0 = (float)(-lo / wdt + (sat ? 1.0 : 0.0));
        const int sh = sat ? 1 : 0;
        for (int ti = 0; ti < 25 && foldable; ++ti) {
          float iw = iw0, cc = cc0;
          const int di = (ti % 5 + 2) % 5 - 2, dc = (ti / 5 + 2) % 5 - 2;  // 0, 1, 2, -2, -1: exact values first
          for (int a = 0; a < std::abs(di); ++a) iw = nextafterf(iw, di < 0 ? 0.f : INFINITY);
          for (int a = 0; a < std::abs(dc); ++a) cc = nextafterf(cc, dc < 0 ? -INFINITY : INFINITY);
          if (cc != 0.f && std::fabs(cc) < 1.2e-38f) continue;  // flushed to zero on the device
          bool ok = bucket(x_lo_f, iw, cc, sat) >= sh - 1 && bucket(x_lo_f, iw, cc, sat) <= sh &&
                    bucket(x_hi_f, iw, cc, sat) >= NB - 1 + sh && bucket(x_hi_f, iw, cc, sat) <= NB + sh;
          for (const Jump& j : jumps) {
            const float k = ceil_f(j.K);
            const int m = (int)std::lround((j.K - lo) / wdt) + sh;
            ok = ok && bucket(k, iw, cc, sat) == m && bucket(nextafterf(k, -INFINITY), iw, cc, sat) == m - 1;
          }
          if (ok) {
            iw_out = iw;
            cc_out = cc;
            return true;
          }
        }
        return false;
      };
      // rows of the curve WITH its steps: bucket b in segment [V[z], V[z+1])
      auto stepped_rows = [&](auto&& emit) {
        size_t kk = 0;
        for (int b = 0; b < NB; ++b) {
          const double mid = lo + (b + 0.5) * wdt;
          while (kk + 1 < last.size() && V[last[kk + 1]] <= mid) ++kk;
          const int z = last[kk];
          const double sl = (POW[z + 1] - POW[z]) / (V[z + 1] - V[z]);
          emit(b, sl, POW[z] - sl * V[z]);
        }
      };
      bool done = false;
      // measured slower than the clamped lattice table on B200 (profiles/r2_kernel_experiments.md:
      // 8 replicas of 256 rows conflict in the banks, 16 replicas cost the L1): only on request
      const bool sat_allowed = force_mode == 3;
      if (sat_allowed && NB + 2 <= 256) {  // ---- saturating lattice LUT
        float iw, cc;
        if (search(true, iw, cc)) {
          const int Rs = ATL_WIND_SAT_R;
          std::vector<float> ls((size_t)256 * Rs * 2);
          auto put_s = [&](int row, double sl, double icpt) {
            const float e[2] = {(float)sl, (float)icpt};
            for (int r = 0; r < Rs; ++r) std::memcpy(&ls[((size_t)row * Rs + r) * 2], e, 8);
          };
          put_s(0, 0.0, POW[0]);
          stepped_rows([&](int b, double sl, double icpt) { put_s(b + 1, sl, icpt); });
          for (int row = NB + 1; row < 256; ++row) put_s(row, 0.0, POW[n - 1]);
          use_lut = 3;
          lut_stride = 8 * Rs;
          rep_mask = Rs - 1;
          inv_w = iw;
          c0 = cc;
          nj = 0;
          lut.swap(ls);
          done = true;
        }
      }
      if (force_mode == 3 && !done) use_lut = 0;  // forced but not qualified: fall back to the search
      if (!done && nj > 0 && force_mode == -1) {
        float iw, cc;
        if (search(false, iw, cc)) {
          inv_w = iw;
          c0 = cc;
          stepped_rows([&](int b, double sl, double icpt) {
            put(b + 1, sl, icpt);
            if (b == 0) put(0, sl, icpt);
          });
          put(NB + 1, 0.0, POW[n - 1]);
          nj = 0;
        }
      }
      if (nj > 0 && nj <= 2) {
        k_jump = ceil_f(jumps[0].K);
        jump = (float)jumps[0].J;
      }
      if (nj == 2) {
        k_end = ceil_f(jumps[1].K);
        y_end = (float)jumps[1].J;
      }
      if (use_lut == 2 && nj > 2) use_lut = 0;  // more steps than compares and they do not fold
      if (use_lut) curve.swap(lut);
    }
  }
  if (!use_lut && force_mode != 2 && force_mode != 3) {
    const double lo = V[0], hi = V[n - 1];
    // jumps of np.interp: a run of equal knots a..z with POW[a] != POW[z]
    int n_interior = 0, jump_first = n;  // knots with index > jump_first sit above the jump
    double Kj = 0.0, J = 0.0;
    for (int a = 0; a < n;) {
      int z = a;
      while (z + 1 < n && V[z + 1] == V[a]) ++z;
      if (POW[z] != POW[a] && V[a] != hi) {
        ++n_interior;
        Kj = V[a];
        J = POW[z] - POW[a];
        jump_first = a;
      }
      a = z + 1;
    }
    auto adj = [&](int j) { return POW[j] - (j > jump_first ? J : 0.0); };
    auto slope = [&](int j) {  // of segment [V[j], V[j+1]); 0 on zero-width segments
      return (j + 1 < n && V[j + 1] > V[j])
                 ? (POW[j + 1] - POW[j]) / (V[j + 1] - V[j])
                 : 0.0;
    };
    for (int NB = 32; NB <= 1024 && !use_lut && hi > lo && n_interior <= 1 && !force_fallback;
         NB *= 2) {  // general LUT
      const double wdt = (hi - lo) / NB;
      std::vector<int> bucket_of(n);
      std::vector<double> knot_in((size_t)NB + 1, std::nan(""));
      bool ok = true;
      for (int j = 0; j < n && ok; ++j) {
        const double pos = (V[j] - lo) / wdt + 0.5;
        const int b = (int)std::floor(pos);
        const double frac = pos - b;
        if (b < 0 || b > NB || frac < 1e-3 || frac > 1.0 - 1e-3) ok = false;
        else if (!std::isnan(knot_in[b]) && knot_in[b] != V[j]) ok = false;  // 2 distinct knots
        else {
          knot_in[b] = V[j];
          bucket_of[j] = b;
        }
      }
      if (!ok) continue;
      const int R = NB <= 128 ? 8 : 1;
      std::vector<float> lut((size_t)(NB + 1) * R * 4);
      int c_lo = 0;  // knots in buckets < b  ==  the segment index left of this bucket's knot
      for (int b = 0; b <= NB; ++b) {
        int c_hi = c_lo;
        while (c_hi < n && bucket_of[c_hi] == b) ++c_hi;
        float e[4];
        if (c_hi > c_lo) {  // bucket with a knot K = V[c_lo] = ... = V[c_hi-1]
          const double K = V[c_lo];
          const double sA = c_lo == 0 ? 0.0 : slope(c_lo - 1);
          const double sB = c_hi >= n ? 0.0 : slope(c_hi - 1);
          e[0] = ceil_f(K);
          // the reference point is e[0], not K (up to one ulp apart when K is not a
          // float): split the difference between the two sides
          e[1] = (float)(adj(c_lo) + 0.5 * (sA + sB) * ((double)e[0] - K));
          e[2] = (float)sA;
          e[3] = (float)sB;
        } else {  // inside segment c_lo - 1 (1 <= c_lo <= n-1): expand about the bucket centre
          const int j = c_lo - 1;
          const double sl = slope(j);
          const float kc = (float)(lo + (b * wdt));
          e[0] = kc;
          e[1] = (float)(adj(j) + sl * ((double)kc - V[j]));
          e[2] = e[3] = (float)sl;
        }
        for (int r = 0; r < R; ++r) std::memcpy(&lut[((size_t)b * R + r) * 4], e, 16);
        c_lo = c_hi;
      }
      use_lut = 1;
      lut_stride = 16 * R;
      rep_mask = R - 1;
      inv_w = (float)(1.0 / wdt);
      c0 = (float)(0.5 - lo / wdt);
      if (n_interior) {
        k_jump = ceil_f(Kj);
        jump = (float)J;
      }
      curve.swap(lut);  // LUT mode stages the table only
    }
  }

  T.curve.swap(curve);
  T.n_knots = n;
  T.NK = NK;
  T.use_lut = use_lut;
  T.lut_stride = lut_stride;
  T.rep_mask = rep_mask;
  T.lut_entry = lut_entry;
  T.nj = nj;
  T.x_lo = (float)V[0];
  T.x_hi = (float)V[n - 1];
  T.inv_w = inv_w;
  T.c0 = c0;
  T.k_jump = k_jump;
  T.jump = jump;
  T.k_end = k_end;
  T.y_end = y_end;
  return ATL_OK;
}

extern "C" {

int atl_wind_create(int device, const AtlWindConfig* cfg, AtlWindOp** op_out) {
  ATL_REQUIRE(cfg && op_out, "NULL argument");
  *op_out = nullptr;
  ATL_REQUIRE(cfg->ny > 0 && cfg->nx > 0, "bad grid");
  ATL_REQUIRE(cfg->method >= ATL_WIND_NONE && cfg->method <= ATL_WIND_POWER, "bad method");
  if (cfg->method != ATL_WIND_NONE)
    ATL_REQUIRE(cfg->from_height > 0 && cfg->to_height > 0, "heights must be positive");

  CurveTables T;
  int table = -1;  // ATL_WIND_TABLE = 0..3 forces a table form (experiments, tests)
  if (const char* e = getenv("ATL_WIND_TABLE")) table = std::max(-1, std::min(3, atoi(e)));
  if (int rc = build_curve(cfg->V, cfg->POW_norm, cfg->n_knots, T, table)) return rc;
  const int n = T.n_knots;
  AtlWindOp* op = new AtlWindOp();
  op->device = device;
  ATL_REQUIRE(cfg->pitch == 0 || cfg->pitch >= cfg->nx, "pitch must be >= nx");
  op->grid = make_grid(cfg->ny, cfg->nx, cfg->pitch);
  op->method = cfg->method;
  op->n_knots = n;
  op->NK = T.NK;
  op->lg2_to = op->lg2_from = op->lg2_ratio = 0.f;
  op->x_lo = T.x_lo;
  op->x_hi = T.x_hi;
  op->use_lut = T.use_lut;
  op->n_stage = (int)T.curve.size();
  op->inv_w = T.inv_w;
  op->c0 = T.c0;
  op->lut_stride = T.lut_stride;
  op->rep_mask = T.rep_mask;
  op->lut_entry = T.lut_entry;
  op->nj = T.nj;
  op->k_jump = T.k_jump;
  op->jump = T.jump;
  op->k_end = T.k_end;
  op->y_end = T.y_end;
  if (cfg->method != ATL_WIND_NONE) {
    op->lg2_to = (float)std::log2(cfg->to_height);
    op->lg2_from = (float)std::log2(cfg->from_height);
    op->lg2_ratio = (float)std::log2(cfg->to_height / cfg->from_height);
  }
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaMalloc((void**)&op->d_curve, T.curve.size() * 4);
  if (e == cudaSuccess)
    e = cudaMemcpy(op->d_curve, T.curve.data(), T.curve.size() * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    atl_wind_destroy(op);
    return cuda_fail(e, "atl_wind_create");
  }
  *op_out = op;
  return ATL_OK;
}

void atl_wind_destroy(AtlWindOp* op) {
  if (!op) return;
  cudaSetDevice(op->device);
  cudaFree(op->d_curve);
  delete op;
}

int atl_wind_curve_eval_host(const double* V, const double* POW_norm, int32_t n_knots,
                             int32_t force_mode, const float* x, int64_t n, float* y_out,
                             int32_t* used_lut_out) {
  ATL_REQUIRE(x && y_out && n >= 0, "bad arguments");
  CurveTables T;
  ATL_REQUIRE(force_mode >= -1 && force_mode <= 3, "force_mode must be -1 .. 3");
  if (int rc = build_curve(V, POW_norm, n_knots, T, force_mode)) return rc;
  if (used_lut_out) *used_lut_out = T.use_lut;
  // replicas must be identical copies; evaluate through a different one per element
  for (int64_t i = 0; i < n; ++i) {
    if (T.use_lut == 3) {  // what the kernels return: the fast value, or the clamped one if that is not finite
      const char* lut = reinterpret_cast<const char*>(T.curve.data()) + ((int)i & T.rep_mask) * 8;
      float y = sat_interp<false>(x[i], lut, T.lut_stride, T.x_lo, T.x_hi, T.inv_w, T.c0);
      if (!(std::fabs(y) <= 3.0e38f)) y = sat_interp<true>(x[i], lut, T.lut_stride, T.x_lo, T.x_hi, T.inv_w, T.c0);
      y_out[i] = y;
      continue;
    }
    if (T.use_lut == 2) {
      const char* lut = reinterpret_cast<const char*>(T.curve.data()) + T.lut_stride + ((int)i & T.rep_mask) * 8;
      y_out[i] = T.nj == 0   ? lattice_interp<0>(x[i], lut, T.lut_stride, T.x_lo, T.x_hi, T.inv_w, T.c0,
                                                  T.k_jump, T.jump, T.k_end, T.y_end)
                 : T.nj == 1 ? lattice_interp<1>(x[i], lut, T.lut_stride, T.x_lo, T.x_hi, T.inv_w, T.c0,
                                                  T.k_jump, T.jump, T.k_end, T.y_end)
                             : lattice_interp<2>(x[i], lut, T.lut_stride, T.x_lo, T.x_hi, T.inv_w, T.c0,
                                                  T.k_jump, T.jump, T.k_end, T.y_end);
      continue;
    }
    if (T.use_lut) {
      const char* lut = reinterpret_cast<const char*>(T.curve.data()) + ((int)i & T.rep_mask) * 16;
      y_out[i] = lut_interp(x[i], lut, T.lut_stride, T.x_lo, T.x_hi, T.inv_w, T.c0, T.k_jump,
                            T.jump, T.k_end, T.y_end);
      continue;
    }
    const float* xcmp = T.curve.data();
    const float* seg = T.curve.data() + T.NK;
    int cnt = 0;
    for (int step = T.NK >> 1; step >= 1; step >>= 1)
      if (xcmp[cnt + step - 1] <= x[i]) cnt += step;
    const float* sg = seg + 4 * (cnt < T.n_knots ? cnt : T.n_knots);
    const float xc = std::fmin(std::fmax(x[i], T.x_lo), T.x_hi);
    y_out[i] = (x[i] != x[i] && T.n_knots > 1) ? x[i] : std::fmaf(sg[2], xc - sg[0], sg[1]);
  }
  return ATL_OK;
}

int atl_wind_curve_info_host(const double* V, const double* POW_norm, int32_t n_knots,
                             int32_t force_mode, int32_t info[4]) {
  ATL_REQUIRE(info, "NULL argument");
  ATL_REQUIRE(force_mode >= -1 && force_mode <= 3, "force_mode must be -1 .. 3");
  CurveTables T;
  if (int rc = build_curve(V, POW_norm, n_knots, T, force_mode)) return rc;
  int steps = 0;
  for (int a = 0; a < n_knots;) {
    int z = a;
    while (z + 1 < n_knots && V[z + 1] == V[a]) ++z;
    steps += POW_norm[z] != POW_norm[a];
    a = z + 1;
  }
  info[0] = T.use_lut;
  info[1] = T.use_lut >= 2 ? T.nj : (T.use_lut == 1 ? (T.k_jump < INFINITY) + 1 : 0);
  info[2] = steps;
  info[3] = (int32_t)(T.curve.size() * sizeof(float));
  return ATL_OK;
}

int atl_wind_op_info(const AtlWindOp* op, int32_t* device, int32_t* ny, int32_t* nx) {
  return op_info(op, device, ny, nx);
}

int atl_wind_reduce(const AtlWindOp* op, const AtlPlan* plan, const AtlWindFields* f,
                    int64_t nt, float* out_dev, void* stream) {
  return run_entry<WindBinding>(Entry::kReduce, op, plan, f, 0, nt, out_dev, nullptr, stream);
}

int atl_wind_cells(const AtlWindOp* op, const AtlWindFields* f, int64_t nt, float* out_dev,
                   void* stream) {
  return run_entry<WindBinding>(Entry::kCells, op, nullptr, f, 0, nt, out_dev, nullptr, stream);
}

int atl_wind_timesum(const AtlWindOp* op, const AtlWindFields* f, int64_t nt, float* out_dev,
                     float* count_dev, void* stream) {
  return run_entry<WindBinding>(Entry::kTimesum, op, nullptr, f, 0, nt, out_dev, count_dev, stream);
}

int atl_wind_reduce_host(const AtlWindOp* op, const AtlPlan* plan, const AtlWindFields* f,
                         int64_t nt, float* out_host, int64_t chunk_steps) {
  return run_reduce_host<WindBinding>(op, plan, f, 0, nt, out_host, chunk_steps);
}

}  // extern "C"

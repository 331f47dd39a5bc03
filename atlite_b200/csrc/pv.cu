// pv.cu -- fused PV conversion: SolarPosition -> SurfaceOrientation ->
// TiltedIrradiation -> SolarPanelModel -> shape reduce  (convert.py:840-854).
//
// Algorithmic traffic (ERA5 branch, solar position computed in-kernel):
// 5 float32 fields = 20 B per cell-timestep.
//
// Solar geometry is SEPARABLE (pv/solar_position.py:86-114): everything except
// cos/sin of the hour angle h = H0(t) + lon(x) depends on time only.  The host
// evaluates the almanac in float64 once per time step and ships
//     tt[t] = { sin dec, cos dec, cos H0, sin H0 }
// with H0 = radians(lmst without lon) - ra; per column xt[x] = {cos lon, sin lon};
// per row yt[y] = {sin lat, cos lat, cos slope, sin slope, cos saz, sin saz,
// sin^3(slope/2)}.  Per cell the kernel then needs NO transcendental for the
// geometry:
//     cos h = cH0 coslon - sH0 sinlon,  sin h = sH0 coslon + cH0 sinlon
//     sinalt            = sd sl + cd cl cos h                   (:103-105)
//     X = cosalt cos az = sd cl - cd sl cos h                   (:109-113)
//     Y = cosalt sin az = -cd sin h                             (:114, sign of h)
// and every orientation / tracking formula of pv/orientation.py:114-176 is a
// polynomial/sqrt expression in (sinalt, cosalt, X, Y) (derivations inline).
#include <cmath>
#include <vector>

#include "kernels.cuh"
#include "solar_host.cuh"

namespace atl {

enum {  // panel coefficient slots (float, device)
  PC_C_AMB = 0, PC_C_IRR, PC_R_TMOD, PC_INV_R_IRR, PC_K1, PC_K2, PC_K3, PC_K4, PC_K5, PC_K6,
  PC_INV_EFF,
  // bofinger
  PC_A = 0, PC_B, PC_C, PC_D, PC_FRACTION, PC_TSTD, PC_DEN, PC_SCALE, PC_THRESHOLD
};

// MODE: 0 = every switch at run time (Reindl split, outflux albedo, tracking modes, Hay-Davies,
// Bofinger, irradiation / solar-thermal outputs, per-cell orientation); 1 / 2 / 3 = the ERA5
// default configuration compiled to constants with the solar position computed in-kernel (1: the
// synthetic / pre-2023 cutouts) or read from the cutout as float64 (2: what real ERA5 cutouts
// store, datasets/era5.py:182-188) / float32 (3).
// FAST (MODE != 0) = the ERA5 default configuration compiled to constants: fixed panel
// (tracking None), solar position computed in-kernel, influx_direct +
// influx_diffuse + albedo variables, simple trigon model, Huld panel.
// FAST=false keeps every switch at run time (stored solar position, Reindl
// split, outflux albedo, tracking modes, Hay-Davies, Bofinger).
template <int MODE, bool VEC>
struct PvPhys {
  static constexpr bool FAST = MODE >= 1 && MODE <= 3;
  // MODE 4: ERA5 inputs (direct + diffuse influx, albedo variable) and the solar position computed
  // in-kernel are compiled in, tracking / trigon model / panel / output / per-cell orientation stay
  // run-time switches: only 5 fields are live per step, so two steps fit in flight
  static constexpr bool ERA5_INPUTS = FAST || MODE == 4;
  static constexpr bool kVec = VEC;
  using Geom = TileGeomT<VEC>;
  // cell i of a lane -> index into the per-column / per-row constant arrays: the
  // SCALAR layout has 1 column x 4 rows per lane, the VEC layout 4 columns x 1 row
  static constexpr int NXC = VEC ? 4 : 1, NYC = VEC ? 1 : 4;
  static __device__ __forceinline__ int ix(int i) { return VEC ? i : 0; }
  static __device__ __forceinline__ int iy(int i) { return VEC ? 0 : i; }
  const float *toa, *dir, *dif, *influx, *alb, *outflux, *temp, *hum;
  const void *salt, *saz;
  const float4* tt;  // per time step (absolute index t_off + t)
  const float2* xt;  // per column
  const float* yt;   // per row, 8 floats
  const float4* ot;  // per CELL orientation {cos b, sin b, cos phi, sin phi}, {sin^3(b/2), ..}: only when
                     // the orientation callback returned (y, x) arrays (pv/orientation.py:107), else NULL
  int64_t S;
  int nx, ny;
  int t_off;
  int tracking_, trigon_, clearsky, irr_branch_, albedo_src_, solar_src_, panel_model_, output_;
  float sin_thr, alt_thr;
  float pc[12];
  float th_c0, th_c1, th_tstore;  // solar thermal (convert.py:565-573), t_store in K

  __device__ __forceinline__ int tracking() const { return FAST ? ATL_TRACK_NONE : tracking_; }
  __device__ __forceinline__ int trigon() const { return FAST ? ATL_TRIGON_SIMPLE : trigon_; }
  __device__ __forceinline__ int panel_model() const { return FAST ? ATL_PANEL_HULD : panel_model_; }
  __device__ __forceinline__ int output() const { return FAST ? ATL_OUT_PANEL : output_; }
  __device__ __forceinline__ int irr_branch() const {
    return ERA5_INPUTS ? ATL_IRR_DIRECT_DIFFUSE : irr_branch_;
  }
  __device__ __forceinline__ int albedo_src() const { return ERA5_INPUTS ? ATL_ALBEDO_VAR : albedo_src_; }
  __device__ __forceinline__ int solar_src() const {
    return (MODE == 1 || MODE == 4) ? ATL_SOLAR_COMPUTED
           : MODE == 2 ? ATL_SOLAR_STORED_F64 : MODE == 3 ? ATL_SOLAR_STORED_F32 : solar_src_;
  }

  struct Cell {
    float clon[NXC], slon[NXC];
    float sl[NYC], cl[NYC], cs[NYC], u[NYC], v[NYC], ss[NYC], cph[NYC], sph[NYC], hd3[NYC];
    float e1[NYC], e2[NYC];  // u cl + cs sl,  cs cl - u sl  (fixed-panel incidence, see compute)
  };
  struct Raw {
    float toa[4], a[4], b[4], alb[4], temp[4], hum[4], salt[4], saz[4];
  };
  static constexpr int kSmemFloats = 0;
  // two steps in flight whenever the configuration is compiled in; the stored-solar modes carry
  // 7 fields per step (28 raw registers): 4 CTAs per SM
  static constexpr int kBatch = MODE != 0 ? 2 : 1, kMinBlocks = MODE == 1 ? 5 : 4;
  // compute() is the reference's arithmetic for finite inputs, straight-line code (no per-cell
  // branches: they would split the 4-cell basic block and cost ~7 % of PV's throughput);
  // NaN-preserving clips (pv/irradiation.py:198-200) make a NaN input always surface as a
  // non-finite result.  The kernels test the RESULTS of a step and only then call
  // compute_exact(), out of line, which adds the per-term fillna(0) of the simple trigon model
  // (:226) and keeps Bofinger / solar-thermal NaNs from being masked by their `where`s.
  static constexpr bool kHasExact = true;
  // measured (profiles/r2_variants.jsonl): the shuffle reduce streams PV at 0.98-1.03 of the
  // HBM peak, the staged reduce at 0.80-0.91 (fewer instructions, but its two-phase structure
  // exposes more latency at 20 warps per SM)
  static constexpr bool kStaged = false;
  static constexpr int kStage = 8, kBatchStaged = kBatch, kMinBlocksStaged = kMinBlocks;
  __device__ void stage(float*) const {}

  __device__ void init(Cell& c, const Geom& g, const float*) const {
#pragma unroll
    for (int a = 0; a < NXC; ++a) {
      const float2 xl = __ldg(xt + min(g.cell_x(VEC ? a : 0), nx - 1));
      c.clon[a] = xl.x;
      c.slon[a] = xl.y;
    }
#pragma unroll
    for (int b = 0; b < NYC; ++b) {
      const int y = min(g.cell_y(VEC ? 0 : b), ny - 1);
      const float4 p0 = __ldg(reinterpret_cast<const float4*>(yt) + 2 * y);
      const float4 p1 = __ldg(reinterpret_cast<const float4*>(yt) + 2 * y + 1);
      c.sl[b] = p0.x; c.cl[b] = p0.y; c.cs[b] = p0.z; c.ss[b] = p0.w;
      c.cph[b] = p1.x; c.sph[b] = p1.y; c.hd3[b] = p1.z;
      c.u[b] = p0.w * p1.x;  // sin(slope) cos(azimuth)
      c.v[b] = p0.w * p1.y;  // sin(slope) sin(azimuth)
      c.e1[b] = fmaf(c.u[b], c.cl[b], c.cs[b] * c.sl[b]);
      c.e2[b] = fmaf(c.cs[b], c.cl[b], -c.u[b] * c.sl[b]);
    }
  }

  __device__ void load(const Cell&, const Geom& g, int64_t tb, Raw& r) const {
    load4(toa, tb, g, r.toa);
    if (irr_branch() == ATL_IRR_DIRECT_DIFFUSE) {
      load4(dir, tb, g, r.a);
      load4(dif, tb, g, r.b);
    } else {
      load4(influx, tb, g, r.a);
      if (clearsky == ATL_CLEARSKY_ENHANCED) load4(hum, tb, g, r.hum);
    }
    load4(albedo_src() == ATL_ALBEDO_VAR ? alb : outflux, tb, g, r.alb);
    load4(temp, tb, g, r.temp);
    if (solar_src() == ATL_SOLAR_STORED_F32) {
      load4((const float*)salt, tb, g, r.salt);
      load4((const float*)saz, tb, g, r.saz);
    } else if (solar_src() == ATL_SOLAR_STORED_F64) {
      load4((const double*)salt, tb, g, r.salt);
      load4((const double*)saz, tb, g, r.saz);
    }
  }

  // pv/solar_panel_model.py:12-44 (huld), 47-74 (bofinger)
  __device__ __forceinline__ float panel(float G, float T) const {
    if (panel_model() == ATL_PANEL_HULD) {
      const float T_ = fmaf(pc[PC_C_AMB], T, fmaf(pc[PC_C_IRR], G, -pc[PC_R_TMOD]));
      const float G_ = G * pc[PC_INV_R_IRR];
      const float lg = __logf(G_);  // G_ <= 0 -> -inf/NaN -> eff NaN/-inf -> 0 below
      const float p1 = fmaf(fmaf(pc[PC_K2], lg, pc[PC_K1]), lg, 1.f);
      const float p2 = fmaf(fmaf(pc[PC_K5], lg, pc[PC_K4]), lg, pc[PC_K3]);
      float eff = fmaf(T_, fmaf(pc[PC_K6], T_, p2), p1);
      eff = (G_ > 0.f) ? fmaxf(eff, 0.f) : 0.f;  // .where(G_>0) .. fillna(0).clip(min=0)
      return G_ * eff * pc[PC_INV_EFF];
    } else {
      const float eta_ref = fmaf(pc[PC_B], G, fmaf(pc[PC_C], __logf(G), pc[PC_A]));
      float eta = eta_ref * fmaf(pc[PC_D], fmaf(pc[PC_FRACTION], G, T - pc[PC_TSTD]), 1.f) /
                  fmaf(pc[PC_DEN] * eta_ref, G, 1.f);
      eta = (G != 0.f && eta == eta) ? eta : 0.f;  // log(where(G != 0)) -> NaN -> fillna(0)
      const float power = G * eta * pc[PC_SCALE];
      return (G >= pc[PC_THRESHOLD]) ? power : 0.f;
    }
  }

  __device__ __forceinline__ void compute(const Cell& c, const Geom& g, int t, const Raw& r, float (&v)[4],
                                          const float* sm) const {
    if constexpr (FAST && VEC)
      compute_fast_packed(c, t, r, v);
    else
      compute_impl<false>(c, g, t, r, v, sm);
  }

  // ---- The ERA5-default configuration on Blackwell's packed FP32 pipe: the lane's cells (0,1)
  // and (2,3) -- neighbours in x that share every per-row constant -- are evaluated as float2
  // pairs with FFMA2 / FMUL2 / FADD2 (one issue slot for two FMAs; scalar operands broadcast for
  // free, `R.F32`).  26 of the ~65 instructions per cell are FMA-pipe arithmetic, so this removes
  // ~16 % of the kernel's instruction issues; clamps, MUFU and predicate logic stay scalar.
  // Same formulas, same operation order as compute_impl<false> (the reference arithmetic:
  // pv/solar_position.py:103-114, orientation.py:114-117, irradiation.py:198-226,252,
  // solar_panel_model.py:23-40).
  static __device__ __forceinline__ float2 bc(float s) { return make_float2(s, s); }
  __device__ __forceinline__ void compute_fast_packed(const Cell& c, int t, const Raw& r, float (&v)[4]) const {
    const float cs = c.cs[0];
    const float dfac = fmaf(0.5f, cs, 0.5f), gfac = fmaf(-0.5f, cs, 0.5f);  // (1 +- cos slope) / 2
    float2 sinalt[2], cosinc[2];
    if (MODE == 1) {  // solar position from the almanac: linear in (cos h, sin h)
      const float4 q = __ldg(tt + t_off + t);
      const float sd = q.x, cd = q.y;
      const float a1 = cd * c.cl[0], a0 = sd * c.sl[0];
      const float b2 = -(c.v[0] * cd), b1 = cd * c.e2[0], b0 = sd * c.e1[0];
      const float nqw = -q.w;
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        const float2 clon = make_float2(c.clon[2 * p], c.clon[2 * p + 1]);
        const float2 slon = make_float2(c.slon[2 * p], c.slon[2 * p + 1]);
        const float2 ch = __ffma2_rn(clon, bc(q.z), __fmul2_rn(slon, bc(nqw)));
        const float2 sh = __ffma2_rn(clon, bc(q.w), __fmul2_rn(slon, bc(q.z)));
        sinalt[p] = __ffma2_rn(ch, bc(a1), bc(a0));
        cosinc[p] = __ffma2_rn(sh, bc(b2), __ffma2_rn(ch, bc(b1), bc(b0)));
      }
    } else {  // stored altitude / azimuth: MUFU sine / cosine inside their accurate range
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        float sa[2], ca[2], ss[2], cc[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int i = 2 * p + e;
          const float az = r.saz[i] > 3.14159265f ? r.saz[i] - 6.28318531f : r.saz[i];
          sa[e] = __sinf(r.salt[i]);
          ca[e] = __cosf(r.salt[i]);
          ss[e] = __sinf(az);
          cc[e] = __cosf(az);
        }
        const float2 ca2 = make_float2(ca[0], ca[1]);
        const float2 X = __fmul2_rn(ca2, make_float2(cc[0], cc[1]));
        const float2 Y = __fmul2_rn(ca2, make_float2(ss[0], ss[1]));
        sinalt[p] = make_float2(sa[0], sa[1]);
        cosinc[p] = __ffma2_rn(X, bc(c.u[0]), __ffma2_rn(Y, bc(c.v[0]), __fmul2_rn(sinalt[p], bc(cs))));
      }
    }
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const int i0 = 2 * p, i1 = 2 * p + 1;
      const float2 ci = make_float2(fmaxf(cosinc[p].x, 0.f), fmaxf(cosinc[p].y, 0.f));  // :188
      // influx.clip(min=0, max=influx_toa): NaN-preserving (value or bound)
      const float2 toa2 = make_float2(r.toa[i0], r.toa[i1]);
      const float2 direct = make_float2(fmin_nan(fmax_nan(r.a[i0], 0.f), toa2.x),
                                        fmin_nan(fmax_nan(r.a[i1], 0.f), toa2.y));
      const float2 room = __fadd2_rn(toa2, make_float2(-direct.x, -direct.y));
      const float2 diffuse = make_float2(fmin_nan(fmax_nan(r.b[i0], 0.f), room.x),
                                         fmin_nan(fmax_nan(r.b[i1], 0.f), room.y));
      const float2 influx = __fadd2_rn(direct, diffuse);
      const float2 rcp = make_float2(rcp_approx(sinalt[p].x), rcp_approx(sinalt[p].y));
      const float2 Rb = __fmul2_rn(ci, rcp);
      const float2 ground = __fmul2_rn(__fmul2_rn(make_float2(r.alb[i0], r.alb[i1]), influx), bc(gfac));
      const float2 total = __ffma2_rn(Rb, direct, __ffma2_rn(diffuse, bc(dfac), ground));
      // result.where(~(alt < thr | direct + diffuse <= 0.01), 0): NaN compares false on both
      const bool low0 = (MODE == 1) ? (sinalt[p].x < sin_thr) : (r.salt[i0] < alt_thr);
      const bool low1 = (MODE == 1) ? (sinalt[p].y < sin_thr) : (r.salt[i1] < alt_thr);
      const float2 G = make_float2((!low0 & !(influx.x <= 0.01f)) ? total.x : 0.f,
                                   (!low1 & !(influx.y <= 0.01f)) ? total.y : 0.f);
      // Huld panel
      const float2 T_ = __ffma2_rn(make_float2(r.temp[i0], r.temp[i1]), bc(pc[PC_C_AMB]),
                                   __ffma2_rn(G, bc(pc[PC_C_IRR]), bc(-pc[PC_R_TMOD])));
      const float2 G_ = __fmul2_rn(G, bc(pc[PC_INV_R_IRR]));
      const float2 lg = __fmul2_rn(make_float2(__log2f(G_.x), __log2f(G_.y)), bc(0.693147181f));
      const float2 p1 = __ffma2_rn(__ffma2_rn(lg, bc(pc[PC_K2]), bc(pc[PC_K1])), lg, bc(1.f));
      const float2 p2 = __ffma2_rn(__ffma2_rn(lg, bc(pc[PC_K5]), bc(pc[PC_K4])), lg, bc(pc[PC_K3]));
      float2 eff = __ffma2_rn(T_, __ffma2_rn(T_, bc(pc[PC_K6]), p2), p1);
      eff.x = (G_.x > 0.f) ? fmaxf(eff.x, 0.f) : 0.f;  // .where(G_>0) .. fillna(0).clip(min=0)
      eff.y = (G_.y > 0.f) ? fmaxf(eff.y, 0.f) : 0.f;
      const float2 o = __fmul2_rn(__fmul2_rn(G_, eff), bc(pc[PC_INV_EFF]));
      v[i0] = o.x;
      v[i1] = o.y;
    }
  }
  // Out of line, and every argument BY VALUE (copied to the call's parameter area on the cold
  // path only): taking references here would pin Cell / Raw / the functor in local memory for
  // the whole kernel and halve the hot path's throughput (measured: profiles/r2_variants*.jsonl).
  static __device__ __noinline__ float4 exact_by_value(const PvPhys self, const Cell c, const Geom g, int t,
                                                       const Raw r) {
    float v[4];
    self.template compute_impl<true>(c, g, t, r, v, nullptr);
    return make_float4(v[0], v[1], v[2], v[3]);
  }
  __device__ __forceinline__ void compute_exact(const Cell& c, const Geom& g, int t, const Raw& r,
                                                float (&v)[4], const float*) const {
    const float4 o = exact_by_value(*this, c, g, t, r);
    v[0] = o.x; v[1] = o.y; v[2] = o.z; v[3] = o.w;
  }

  template <bool EXACT>
  __device__ __forceinline__ void compute_impl(const Cell& c, const Geom& g, int t, const Raw& r,
                                               float (&v)[4], const float*) const {
    float sd = 0.f, cd = 0.f, ch[NXC], sh[NXC];
    if (solar_src() == ATL_SOLAR_COMPUTED) {
      const float4 q = __ldg(tt + t_off + t);
      sd = q.x;
      cd = q.y;
#pragma unroll
      for (int a = 0; a < NXC; ++a) {
        ch[a] = q.z * c.clon[a] - q.w * c.slon[a];
        sh[a] = q.w * c.clon[a] + q.z * c.slon[a];
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int a = ix(i), b = iy(i);
      // ---- panel orientation: per row (tables in Cell) or per cell (orientation callback
      // returning (y, x) arrays)
      float cs = c.cs[b], ss = c.ss[b], cph = c.cph[b], sph = c.sph[b], hd3c = c.hd3[b];
      float ou = c.u[b], ov = c.v[b], e1 = c.e1[b], e2 = c.e2[b];
      if (!FAST && ot != nullptr) {
        const int cell = min(g.cell_y(i), ny - 1) * nx + min(g.cell_x(i), nx - 1);
        const float4 p0 = __ldg(ot + 2 * cell), p1 = __ldg(ot + 2 * cell + 1);
        cs = p0.x; ss = p0.y; cph = p0.z; sph = p0.w; hd3c = p1.x;
        ou = ss * cph;
        ov = ss * sph;
        e1 = fmaf(ou, c.cl[b], cs * c.sl[b]);
        e2 = fmaf(cs, c.cl[b], -ou * c.sl[b]);
      }
      // ---- solar position (pv/solar_position.py:103-114)
      float sinalt, cosalt, X, Y;
      if (solar_src() == ATL_SOLAR_COMPUTED) {
        sinalt = fmaf(cd * c.cl[b], ch[a], sd * c.sl[b]);  // no asin taken: the [-1,1] clip is moot
        X = fmaf(-(cd * c.sl[b]), ch[a], sd * c.cl[b]);
        Y = -cd * sh[a];
        cosalt = sqrtf(fmaxf(fmaf(-sinalt, sinalt, 1.f), 0.f));
      } else {
        float saz_s, saz_c;
        if (MODE != 1 && MODE != 4) {  // every stored-solar configuration
          // altitude in [-pi/2, pi/2], azimuth in [0, 2 pi) brought into (-pi, pi]: inside the range
          // where the MUFU sine / cosine are good to 2^-21 absolute (4e-7: 2e-5 of sin(1 deg), the
          // smallest unmasked sin(altitude)); sincosf's full range reduction costs ~100 instructions
          const float az = r.saz[i] > 3.14159265f ? r.saz[i] - 6.28318531f : r.saz[i];
          sinalt = __sinf(r.salt[i]);
          cosalt = __cosf(r.salt[i]);
          saz_s = __sinf(az);
          saz_c = __cosf(az);
        } else {  // (not reached: these modes compute the solar position)
          sincosf(r.salt[i], &sinalt, &cosalt);
          sincosf(r.saz[i], &saz_s, &saz_c);
        }
        X = cosalt * saz_c;
        Y = cosalt * saz_s;
      }
      // ---- surface orientation (pv/orientation.py:114-188)
      float cosinc, cslope;  // cos(incidence), cos(surface slope)
      const int trk = tracking();
      if (trk == ATL_TRACK_NONE) {
        // sin b cos a cos(phi - az) + cos b sin a, with cos a cos az = X, cos a sin az = Y
        if (solar_src() == ATL_SOLAR_COMPUTED) {
          // u X + v Y + cs sinalt is linear in (cos h, sin h):
          //   sd (u cl + cs sl) + cd (cs cl - u sl) cos h - v cd sin h
          cosinc = fmaf(-(ov * cd), sh[a], fmaf(cd * e2, ch[a], sd * e1));
        } else {
          cosinc = fmaf(ou, X, fmaf(ov, Y, cs * sinalt));
        }
        cslope = cs;
      } else if (trk == ATL_TRACK_VERTICAL) {
        cosinc = fmaf(ss, cosalt, cs * sinalt);
        cslope = cs;
      } else if (trk == ATL_TRACK_DUAL) {
        cosinc = 1.f;
        cslope = (trigon() == ATL_TRIGON_SIMPLE) ? sinalt : cs;  // irradiation.py:216-219
      } else {
        // q = cos a sin(az - phi), p = cos a cos(az - phi)
        const float q = fmaf(Y, cph, -X * sph);
        if (trk == ATL_TRACK_HORIZONTAL) {
          // rotation = atan(q / sinalt); slope = |rotation|; the panel azimuth is
          // phi + sign(rotation) pi/2, so cosinc = sign(sinalt) sqrt(sinalt^2 + q^2)
          const float D = sqrtf(fmaf(sinalt, sinalt, q * q));
          cosinc = sinalt > 0.f ? D : 0.f;
          cslope = __fdividef(fabsf(sinalt), D);
        } else {  // tilted_horizontal: rotation = atan2(q, den) after the +-pi fix-ups
          const float p = fmaf(X, cph, Y * sph);
          const float den = fmaf(p, ss, sinalt * cs);
          const float E = sqrtf(fmaf(q, q, den * den));
          cosinc = E;  // cos(rot) den + sin(rot) q
          cslope = __fdividef(fabsf(den) * cs, E);
        }
      }
      cosinc = fmaxf(cosinc, 0.f);  // :188

      // ---- irradiation split (pv/irradiation.py:198-208, 13-73)
      const float toa_ = r.toa[i];
      float direct, diffuse;
      if (irr_branch() == ATL_IRR_DIRECT_DIFFUSE) {
        // influx.clip(min=0, max=influx_toa): xarray's clip keeps NaN (in the value or the bound)
        direct = fmin_nan(fmax_nan(r.a[i], 0.f), toa_);
        diffuse = fmin_nan(fmax_nan(r.b[i], 0.f), toa_ - direct);
      } else {
        const float inf_ = fmin_nan(fmax_nan(r.a[i], 0.f), toa_);
        const float k = inf_ / toa_;  // 0/0 -> NaN -> fraction 0
        float fr = 0.f;
        if (clearsky == ATL_CLEARSKY_SIMPLE) {
          if (k > 0.f && k <= 0.3f)
            fr = fminf(1.f, 1.020f - 0.254f * k + 0.0123f * sinalt);
          else if (k > 0.3f && k < 0.78f)
            fr = fminf(0.97f, fmaxf(0.1f, 1.400f - 1.749f * k + 0.177f * sinalt));
          else if (k >= 0.78f)
            fr = fmaxf(0.1f, 0.486f * k - 0.182f * sinalt);
        } else {
          const float T = r.temp[i], rh = r.hum[i];
          if (k > 0.f && k <= 0.3f)
            fr = fminf(1.f, 1.000f - 0.232f * k + 0.0239f * sinalt - 0.000682f * T + 0.0195f * rh);
          else if (k > 0.3f && k < 0.78f)
            fr = fminf(0.97f, fmaxf(0.1f, 1.329f - 1.716f * k + 0.267f * sinalt - 0.00357f * T +
                                              0.106f * rh));
          else if (k >= 0.78f)
            fr = fmaxf(0.1f, 0.426f * k - 0.256f * sinalt + 0.00349f * T + 0.0734f * rh);
        }
        diffuse = inf_ * fr;
        direct = inf_ - diffuse;
      }
      const float influx_ = direct + diffuse;
      float albedo;
      if (albedo_src() == ATL_ALBEDO_VAR) {
        albedo = r.alb[i];
      } else {  // (outflux / influx.where(influx != 0)).fillna(0).clip(max=1)  :132
        const float a = r.alb[i] / influx_;
        albedo = (influx_ != 0.f && a == a) ? fminf(a, 1.f) : 0.f;
      }

      // ---- tilted irradiation (pv/irradiation.py:214-236, 76-125, 142-145)
      const float Rb = __fdividef(cosinc, sinalt);
      const float direct_t = Rb * direct;
      const float ground_t = albedo * influx_ * fmaf(-0.5f, cslope, 0.5f);
      float diffuse_t;
      if (trigon() == ATL_TRIGON_SIMPLE) {
        diffuse_t = fmaf(0.5f, cslope, 0.5f) * diffuse;
      } else {
        float hd3 = hd3c;
        if (trk == ATL_TRACK_HORIZONTAL || trk == ATL_TRACK_TILTED_HORIZONTAL) {
          const float s2 = sqrtf(fmaxf(fmaf(-0.5f, cslope, 0.5f), 0.f));  // sin(slope/2)
          hd3 = s2 * s2 * s2;
        }
        const float f = influx_ > 0.f ? sqrtf(__fdividef(direct, influx_)) : 0.f;
        const float A = direct / toa_;
        diffuse_t = fmaf(A, Rb, (1.f - A) * fmaf(0.5f, cslope, 0.5f) * fmaf(f, hd3, 1.f)) * diffuse;
        diffuse_t = fmaxf(diffuse_t, 0.f);  // clip(min=0).fillna(0): fmaxf drops NaN
      }
      const int out = output();
      float total;
      if (out == ATL_OUT_DIRECT) total = direct_t;  // pv/irradiation.py:238-245
      else if (out == ATL_OUT_DIFFUSE) total = diffuse_t;
      else if (out == ATL_OUT_GROUND) total = ground_t;
      else if (trigon() == ATL_TRIGON_SIMPLE) {
        if (EXACT) {  // direct_t.fillna(0) + diffuse_t.fillna(0) + ground_t.fillna(0)   (:226)
          total = ((direct_t == direct_t) ? direct_t : 0.f) + ((diffuse_t == diffuse_t) ? diffuse_t : 0.f) +
                  ((ground_t == ground_t) ? ground_t : 0.f);
        } else {  // one FMA chain on the hot path; NaN in any term -> NaN -> compute_exact
          total = fmaf(Rb, direct, fmaf(fmaf(0.5f, cslope, 0.5f), diffuse, ground_t));
        }
      } else
        total = fmaf(Rb, direct, diffuse_t) + ground_t;
      // computed mode: alt < thr  <=>  sin(alt) < sin(thr) on [-pi/2, pi/2];
      // stored mode compares the stored altitude itself, as the reference does
      // result.where(~(cap_alt | (direct + diffuse <= 0.01)), 0): keep iff NOT(alt < thr) AND
      // NOT(influx <= 0.01); NaN compares false on both, exactly as in the reference
      const bool low = (solar_src() == ATL_SOLAR_COMPUTED) ? (sinalt < sin_thr)
                                                           : (r.salt[i] < alt_thr);
      const bool keep_it = !low & !(influx_ <= 0.01f);
      const float G = keep_it ? total : 0.f;
      if (!EXACT && !FAST && G != G) {
        // a NaN irradiance must SURFACE (Bofinger's threshold and the solar-thermal `where`
        // would turn it into a finite 0): the kernels then re-evaluate with compute_exact
        v[i] = G;
      } else if (out == ATL_OUT_PANEL) {
        v[i] = panel(G, r.temp[i]);
      } else if (out == ATL_OUT_SOLAR_THERMAL) {
        // eta = c0 - c1 * ((t_store - T) / irr.where(irr != 0)).fillna(0); output.where(> 0, 0)
        const float q = (th_tstore - r.temp[i]) / G;
        const float eta = th_c0 - th_c1 * ((G != 0.f && q == q) ? q : 0.f);
        const float o = G * eta;
        v[i] = (o > 0.f) ? o : 0.f;
      } else {
        v[i] = G;
      }
    }
  }
};

}  // namespace atl

using namespace atl;

struct AtlPvOp : AtlOpBase {
  int64_t nt;
  int tracking, trigon, clearsky, irr_branch, albedo_src, solar_src, panel_model, output;
  float th_c0, th_c1, th_tstore;
  float sin_thr, alt_thr;
  float pc[12];
  float4* d_tt = nullptr;
  float2* d_xt = nullptr;
  float* d_yt = nullptr;
  float4* d_ot = nullptr;  // per-cell orientation table (orientation_2d)
  int mode;                // PvPhys MODE
};

template <int MODE, bool VEC>
static PvPhys<MODE, VEC> make_phys(const AtlPvOp* op, const AtlPvFields* f, int64_t t0) {
  PvPhys<MODE, VEC> p;
  p.toa = f->influx_toa;
  p.dir = f->influx_direct;
  p.dif = f->influx_diffuse;
  p.influx = f->influx;
  p.alb = f->albedo;
  p.outflux = f->outflux;
  p.temp = f->temperature;
  p.hum = f->humidity;
  p.salt = f->solar_altitude;
  p.saz = f->solar_azimuth;
  p.tt = op->d_tt;
  p.xt = op->d_xt;
  p.yt = op->d_yt;
  p.ot = op->d_ot;
  p.S = op->grid.S;
  p.nx = op->grid.nx;
  p.ny = op->grid.ny;
  p.t_off = (int)t0;
  p.tracking_ = op->tracking;
  p.trigon_ = op->trigon;
  p.clearsky = op->clearsky;
  p.irr_branch_ = op->irr_branch;
  p.albedo_src_ = op->albedo_src;
  p.solar_src_ = op->solar_src;
  p.panel_model_ = op->panel_model;
  p.output_ = op->output;
  p.th_c0 = op->th_c0;
  p.th_c1 = op->th_c1;
  p.th_tstore = op->th_tstore;
  p.sin_thr = op->sin_thr;
  p.alt_thr = op->alt_thr;
  for (int i = 0; i < 12; ++i) p.pc[i] = op->pc[i];
  return p;
}

// The PV operator's part of the shared entry sequence (kernels.cuh: run_entry).
struct PvBinding {
  using Op = AtlPvOp;
  using Fields = AtlPvFields;
  static int check(const AtlPvOp* op, const AtlPvFields* f, int64_t t0, int64_t nt) {
    ATL_REQUIRE(op && f, "NULL argument");
    ATL_REQUIRE(t0 >= 0 && nt >= 0 && t0 + nt <= op->nt, "slab outside the operator's time axis");
    ATL_REQUIRE(f->influx_toa && f->temperature, "influx_toa / temperature field missing");
    if (op->irr_branch == ATL_IRR_DIRECT_DIFFUSE)
      ATL_REQUIRE(f->influx_direct && f->influx_diffuse,
                  "Need either influx or influx_direct and influx_diffuse in the dataset.");
    else {
      ATL_REQUIRE(f->influx, "influx field missing");
      if (op->clearsky == ATL_CLEARSKY_ENHANCED) ATL_REQUIRE(f->humidity, "humidity field missing");
    }
    if (op->albedo_src == ATL_ALBEDO_VAR)
      ATL_REQUIRE(f->albedo, "Need either albedo or outflux as a variable in the dataset.");
    else
      ATL_REQUIRE(f->outflux, "outflux field missing");
    if (op->solar_src != ATL_SOLAR_COMPUTED)
      ATL_REQUIRE(f->solar_altitude && f->solar_azimuth, "stored solar position fields missing");
    return ATL_OK;
  }
  template <class Run>
  static int with_phys(const AtlPvOp* op, const AtlPvFields* f, int64_t t0, Run run) {
#define ATL_PV_MODE(M) \
  case M:              \
    return run([&](auto vec) { return make_phys<M, decltype(vec)::value>(op, f, t0); });
    switch (op->mode) { ATL_PV_MODE(0) ATL_PV_MODE(1) ATL_PV_MODE(2) ATL_PV_MODE(3) ATL_PV_MODE(4) }
#undef ATL_PV_MODE
    return ATL_ERR_INVALID;
  }
  template <class F, class Visit>
  static void each_field(const AtlPvOp* op, F& f, Visit visit) {
    const size_t sol = op->solar_src == ATL_SOLAR_STORED_F64 ? 8 : 4;
    visit(f.influx_toa, 4);
    visit(f.influx_direct, 4);
    visit(f.influx_diffuse, 4);
    visit(f.influx, 4);
    visit(f.albedo, 4);
    visit(f.outflux, 4);
    visit(f.temperature, 4);
    visit(f.humidity, 4);
    visit(f.solar_altitude, sol);
    visit(f.solar_azimuth, sol);
  }
};

extern "C" {

int atl_pv_create(int device, const AtlPvConfig* cfg, AtlPvOp** op_out) {
  ATL_REQUIRE(cfg && op_out, "NULL argument");
  *op_out = nullptr;
  ATL_REQUIRE(cfg->ny > 0 && cfg->nx > 0 && cfg->nt >= 0, "bad shape");
  ATL_REQUIRE(cfg->lon_deg && cfg->lat_deg && cfg->slope_rad && cfg->azimuth_rad,
              "coordinate / orientation tables missing");
  ATL_REQUIRE(cfg->solar_src != ATL_SOLAR_COMPUTED || cfg->time_ns || cfg->nt == 0,
              "time axis missing");
  ATL_REQUIRE(cfg->tracking >= 0 && cfg->tracking <= ATL_TRACK_DUAL, "bad tracking mode");
  ATL_REQUIRE(cfg->trigon_model >= 0 && cfg->trigon_model <= 1, "bad trigon model");
  ATL_REQUIRE(cfg->clearsky_model >= 0 && cfg->clearsky_model <= 1,
              "`clearsky model` must be chosen from 'simple' and 'enhanced'");
  ATL_REQUIRE(cfg->irr_branch >= 0 && cfg->irr_branch <= 1, "bad irradiation branch");
  ATL_REQUIRE(cfg->albedo_src >= 0 && cfg->albedo_src <= 1, "bad albedo source");
  ATL_REQUIRE(cfg->solar_src >= 0 && cfg->solar_src <= 2, "bad solar source");
  ATL_REQUIRE(cfg->panel_model >= 0 && cfg->panel_model <= 1, "Unknown panel model");
  ATL_REQUIRE(cfg->pitch == 0 || cfg->pitch >= cfg->nx, "pitch must be >= nx");
  ATL_REQUIRE(cfg->output >= ATL_OUT_PANEL && cfg->output <= ATL_OUT_SOLAR_THERMAL, "bad output kind");

  const double PI = 3.14159265358979323846;
  const double D2R = PI / 180.0;
  AtlPvOp* op = new AtlPvOp();
  op->device = device;
  op->grid = make_grid(cfg->ny, cfg->nx, cfg->pitch);
  op->nt = cfg->nt;
  op->tracking = cfg->tracking;
  op->trigon = cfg->trigon_model;
  op->clearsky = cfg->clearsky_model;
  op->irr_branch = cfg->irr_branch;
  op->albedo_src = cfg->albedo_src;
  op->solar_src = cfg->solar_src;
  op->panel_model = cfg->panel_model;
  op->output = cfg->output;
  op->th_c0 = (float)cfg->thermal[0];
  op->th_c1 = (float)cfg->thermal[1];
  op->th_tstore = (float)(cfg->thermal[2] + 273.15);
  op->sin_thr = (float)std::sin(cfg->altitude_threshold_deg * D2R);
  op->alt_thr = (float)(cfg->altitude_threshold_deg * D2R);
  const bool era5_default = cfg->tracking == ATL_TRACK_NONE && cfg->irr_branch == ATL_IRR_DIRECT_DIFFUSE &&
                            cfg->albedo_src == ATL_ALBEDO_VAR && cfg->trigon_model == ATL_TRIGON_SIMPLE &&
                            cfg->panel_model == ATL_PANEL_HULD && cfg->output == ATL_OUT_PANEL &&
                            !cfg->orientation_2d;
  const bool era5_inputs = cfg->irr_branch == ATL_IRR_DIRECT_DIFFUSE && cfg->albedo_src == ATL_ALBEDO_VAR;
  op->mode = era5_default ? (cfg->solar_src == ATL_SOLAR_COMPUTED ? 1 : cfg->solar_src == ATL_SOLAR_STORED_F64 ? 2 : 3)
             : (era5_inputs && cfg->solar_src == ATL_SOLAR_COMPUTED) ? 4 : 0;
  const double* P = cfg->panel;
  for (int i = 0; i < 12; ++i) op->pc[i] = 0.f;
  if (cfg->panel_model == ATL_PANEL_HULD) {
    op->pc[PC_C_AMB] = (float)P[0];
    op->pc[PC_C_IRR] = (float)P[1];
    op->pc[PC_R_TMOD] = (float)P[2];
    op->pc[PC_INV_R_IRR] = (float)(1.0 / P[3]);
    for (int k = 0; k < 6; ++k) op->pc[PC_K1 + k] = (float)P[4 + k];
    op->pc[PC_INV_EFF] = (float)P[10];
  } else {
    // A, B, C, D, NOCT, Tamb, Intc, Tstd, ta, threshold, inverter_efficiency
    const double A = P[0], B = P[1], C = P[2], D = P[3], NOCT = P[4], Tamb = P[5], Intc = P[6],
                 Tstd = P[7], ta = P[8], thr = P[9], inv = P[10];
    const double fraction = (NOCT - Tamb) / Intc;
    const double capacity = (A + B * 1000.0 + C * std::log(1000.0)) * 1e3;
    op->pc[PC_A] = (float)A;
    op->pc[PC_B] = (float)B;
    op->pc[PC_C] = (float)C;
    op->pc[PC_D] = (float)D;
    op->pc[PC_FRACTION] = (float)fraction;
    op->pc[PC_TSTD] = (float)Tstd;
    op->pc[PC_DEN] = (float)(D * fraction / ta);
    op->pc[PC_SCALE] = (float)(inv / capacity);
    op->pc[PC_THRESHOLD] = (float)thr;
  }

  // ---- per-time-step almanac (pv/solar_position.py:71-97), float64 on host
  std::vector<float4> tt;
  solar_almanac(cfg->time_ns, cfg->nt, cfg->time_shift_ns, tt);
  std::vector<float2> xt((size_t)cfg->nx);
  for (int i = 0; i < cfg->nx; ++i) {
    const double lon = cfg->lon_deg[i] * D2R;
    xt[(size_t)i] = make_float2((float)std::cos(lon), (float)std::sin(lon));
  }
  // orientation_2d: slope_rad / azimuth_rad hold ny * nx entries; the per-row table then only
  // serves the latitude terms (its orientation part is taken from the first column)
  const int ostride = cfg->orientation_2d ? cfg->nx : 1;
  std::vector<float4> ot;
  if (cfg->orientation_2d) {
    ot.resize((size_t)cfg->ny * cfg->nx * 2);
    for (size_t k = 0; k < (size_t)cfg->ny * cfg->nx; ++k) {
      const double sl = cfg->slope_rad[k], az = cfg->azimuth_rad[k];
      ot[2 * k] = make_float4((float)std::cos(sl), (float)std::sin(sl), (float)std::cos(az), (float)std::sin(az));
      ot[2 * k + 1] = make_float4((float)std::pow(std::sin(sl / 2.0), 3), 0.f, 0.f, 0.f);
    }
  }
  std::vector<float> yt((size_t)cfg->ny * 8);
  for (int j = 0; j < cfg->ny; ++j) {
    const double lat = cfg->lat_deg[j] * D2R, sl = cfg->slope_rad[(size_t)j * ostride],
                 az = cfg->azimuth_rad[(size_t)j * ostride];
    float* o = &yt[(size_t)j * 8];
    o[0] = (float)std::sin(lat);
    o[1] = (float)std::cos(lat);
    o[2] = (float)std::cos(sl);
    o[3] = (float)std::sin(sl);
    o[4] = (float)std::cos(az);
    o[5] = (float)std::sin(az);
    o[6] = (float)std::pow(std::sin(sl / 2.0), 3);
    o[7] = 0.f;
  }
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaMalloc((void**)&op->d_tt, tt.size() * sizeof(float4));
  if (e == cudaSuccess)
    e = cudaMemcpy(op->d_tt, tt.data(), tt.size() * sizeof(float4), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc((void**)&op->d_xt, xt.size() * sizeof(float2));
  if (e == cudaSuccess)
    e = cudaMemcpy(op->d_xt, xt.data(), xt.size() * sizeof(float2), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc((void**)&op->d_yt, yt.size() * sizeof(float));
  if (e == cudaSuccess)
    e = cudaMemcpy(op->d_yt, yt.data(), yt.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess && !ot.empty()) e = cudaMalloc((void**)&op->d_ot, ot.size() * sizeof(float4));
  if (e == cudaSuccess && !ot.empty())
    e = cudaMemcpy(op->d_ot, ot.data(), ot.size() * sizeof(float4), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    atl_pv_destroy(op);
    return cuda_fail(e, "atl_pv_create");
  }
  *op_out = op;
  return ATL_OK;
}

void atl_pv_destroy(AtlPvOp* op) {
  if (!op) return;
  cudaSetDevice(op->device);
  cudaFree(op->d_tt);
  cudaFree(op->d_xt);
  cudaFree(op->d_yt);
  cudaFree(op->d_ot);
  delete op;
}

int atl_pv_op_info(const AtlPvOp* op, int32_t* device, int32_t* ny, int32_t* nx,
                   int32_t* solar_src) {
  if (op && solar_src) *solar_src = op->solar_src;
  return op_info(op, device, ny, nx);
}

int atl_pv_reduce(const AtlPvOp* op, const AtlPlan* plan, const AtlPvFields* f, int64_t t0,
                  int64_t nt, float* out_dev, void* stream) {
  return run_entry<PvBinding>(Entry::kReduce, op, plan, f, t0, nt, out_dev, nullptr, stream);
}

int atl_pv_cells(const AtlPvOp* op, const AtlPvFields* f, int64_t t0, int64_t nt,
                 float* out_dev, void* stream) {
  return run_entry<PvBinding>(Entry::kCells, op, nullptr, f, t0, nt, out_dev, nullptr, stream);
}

int atl_pv_timesum(const AtlPvOp* op, const AtlPvFields* f, int64_t t0, int64_t nt,
                   float* out_dev, float* count_dev, void* stream) {
  return run_entry<PvBinding>(Entry::kTimesum, op, nullptr, f, t0, nt, out_dev, count_dev, stream);
}

int atl_pv_reduce_host(const AtlPvOp* op, const AtlPlan* plan, const AtlPvFields* f, int64_t t0,
                       int64_t nt, float* out_host, int64_t chunk_steps) {
  return run_reduce_host<PvBinding>(op, plan, f, t0, nt, out_host, chunk_steps);
}

}  // extern "C"

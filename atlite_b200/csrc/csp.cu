// csp.cu -- concentrated solar power fused with the shape reduce
// (convert.py:940-972, csp.py:18-58): solar position -> direct irradiation
// (horizontal for parabolic troughs, DNI = direct / sin(max(alt, 3.75 deg)) for
// solar towers) x solar-field efficiency, bilinearly interpolated from the
// installation's (altitude, azimuth) table (xarray .interp == scipy interpn,
// linear, NaN outside the table), / r_irradiance, clip(max=1), NaN -> 0.
//
// Algorithmic traffic: 4 B per cell-timestep (influx_direct; + 8/16 B when the
// cutout stores the solar position).
#include <cmath>
#include <vector>

#include "kernels.cuh"
#include "solar_host.cuh"

namespace atl {

template <bool VEC>
struct CspPhys {
  static constexpr bool kVec = VEC;
  using Geom = TileGeomT<VEC>;
  static constexpr int NXC = VEC ? 4 : 1, NYC = VEC ? 1 : 4;
  static __device__ __forceinline__ int ix(int i) { return VEC ? i : 0; }
  static __device__ __forceinline__ int iy(int i) { return VEC ? 0 : i; }

  const float* direct;
  const void *salt, *saz;
  const float4* tt;
  const float2* xt;
  const float2* yt;    // per row {sin lat, cos lat}
  const float* table;  // device: alt[n_alt] | az[n_az] | eff[n_alt * n_az]
  int nx, ny, t_off, solar_src, tower, n_alt, n_az;
  float inv_r, dni_thr;

  struct Cell {
    float clon[NXC], slon[NXC], sl[NYC], cl[NYC];
  };
  struct Raw {
    float d[4], salt[4], saz[4];
  };
  static constexpr int kSmemFloats = 128 + 128 + 8192;
  static constexpr int kBatch = 1, kMinBlocks = 4;
  static constexpr bool kHasExact = false;
  static constexpr bool kStaged = false;
  static constexpr int kStage = 8, kBatchStaged = kBatch, kMinBlocksStaged = kMinBlocks;

  __device__ void stage(float* smem) const {
    const int n = n_alt + n_az + n_alt * n_az;
    for (int i = threadIdx.x; i < n; i += blockDim.x) smem[i] = table[i];
    __syncthreads();
  }
  __device__ void init(Cell& c, const Geom& g, const float*) const {
#pragma unroll
    for (int a = 0; a < NXC; ++a) {
      const float2 xl = __ldg(xt + min(g.cell_x(VEC ? a : 0), nx - 1));
      c.clon[a] = xl.x;
      c.slon[a] = xl.y;
    }
#pragma unroll
    for (int b = 0; b < NYC; ++b) {
      const float2 yl = __ldg(yt + min(g.cell_y(VEC ? 0 : b), ny - 1));
      c.sl[b] = yl.x;
      c.cl[b] = yl.y;
    }
  }
  __device__ void load(const Cell&, const Geom& g, int64_t sb, Raw& r) const {
    load4(direct, sb, g, r.d);
    if (solar_src == ATL_SOLAR_STORED_F32) {
      load4((const float*)salt, sb, g, r.salt);
      load4((const float*)saz, sb, g, r.saz);
    } else if (solar_src == ATL_SOLAR_STORED_F64) {
      load4((const double*)salt, sb, g, r.salt);
      load4((const double*)saz, sb, g, r.saz);
    }
  }
  // scipy interpn index rule: i = clamp(#coords <= x  - 1, 0, n - 2)
  static __device__ __forceinline__ int interval(const float* c, int n, float x) {
    int lo = 0, hi = n;  // first index with c[idx] > x
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (c[mid] <= x) lo = mid + 1;
      else hi = mid;
    }
    return min(max(lo - 1, 0), n - 2);
  }
  __device__ void compute(const Cell& c, const Geom&, int t, const Raw& r, float (&v)[4],
                          const float* sm) const {
    const float* ac = sm;
    const float* zc = sm + n_alt;
    const float* ef = sm + n_alt + n_az;
    float sd = 0.f, cd = 0.f, ch[NXC], sh[NXC];
    if (solar_src == ATL_SOLAR_COMPUTED) {
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
      float alt, az;
      if (solar_src == ATL_SOLAR_COMPUTED) {
        const float sinalt = fminf(fmaxf(fmaf(cd * c.cl[b], ch[a], sd * c.sl[b]), -1.f), 1.f);
        const float X = fmaf(-(cd * c.sl[b]), ch[a], sd * c.cl[b]);  // cos alt cos az
        const float Y = -cd * sh[a];                                 // cos alt sin az
        alt = asinf(sinalt);                                         // solar_position.py:103-105
        az = atan2f(Y, X);                                           // :109-114 on [0, 2 pi)
        az = az < 0.f ? az + 6.283185307179586f : az;
      } else {
        alt = r.salt[i];
        az = r.saz[i];
      }
      float irr = r.d[i];
      if (tower) irr = irr / sinf(fmaxf(alt, dni_thr));  // csp.py:50-58 (NaN > thr is False -> thr)
      float eff = __int_as_float(0x7fc00000);  // NaN outside the table
      if (alt >= ac[0] && alt <= ac[n_alt - 1] && az >= zc[0] && az <= zc[n_az - 1]) {
        const int ia = interval(ac, n_alt, alt), iz = interval(zc, n_az, az);
        const float wa = (alt - ac[ia]) / (ac[ia + 1] - ac[ia]);
        const float wz = (az - zc[iz]) / (zc[iz + 1] - zc[iz]);
        const float* e0 = ef + ia * n_az + iz;
        const float e00 = e0[0], e01 = e0[1], e10 = e0[n_az], e11 = e0[n_az + 1];
        eff = (1.f - wa) * ((1.f - wz) * e00 + wz * e01) + wa * ((1.f - wz) * e10 + wz * e11);
      }
      float da = eff * irr * inv_r;
      da = fminf(da, 1.f);  // NaN stays NaN through the product; fminf(NaN, 1) = 1 -> fix below
      v[i] = (eff == eff && irr == irr) ? da : 0.f;  // .clip(max=1).fillna(0)
    }
  }
};

}  // namespace atl

using namespace atl;

struct AtlCspOp : AtlOpBase {
  int64_t nt;
  int solar_src, tower, n_alt, n_az;
  float inv_r, dni_thr;
  float4* d_tt = nullptr;
  float2* d_xt = nullptr;
  float2* d_yt = nullptr;
  float* d_table = nullptr;
};

template <bool VEC>
static CspPhys<VEC> make_phys(const AtlCspOp* op, const AtlCspFields* f, int64_t t0) {
  CspPhys<VEC> p;
  p.direct = f->influx_direct;
  p.salt = f->solar_altitude;
  p.saz = f->solar_azimuth;
  p.tt = op->d_tt;
  p.xt = op->d_xt;
  p.yt = op->d_yt;
  p.table = op->d_table;
  p.nx = op->grid.nx;
  p.ny = op->grid.ny;
  p.t_off = (int)t0;
  p.solar_src = op->solar_src;
  p.tower = op->tower;
  p.n_alt = op->n_alt;
  p.n_az = op->n_az;
  p.inv_r = op->inv_r;
  p.dni_thr = op->dni_thr;
  return p;
}

// The CSP operator's part of the shared entry sequence (kernels.cuh: run_entry).
struct CspBinding {
  using Op = AtlCspOp;
  using Fields = AtlCspFields;
  static int check(const AtlCspOp* op, const AtlCspFields* f, int64_t t0, int64_t nt) {
    ATL_REQUIRE(op && f && f->influx_direct, "NULL argument / influx_direct missing");
    ATL_REQUIRE(t0 >= 0 && nt >= 0 && t0 + nt <= op->nt, "slab outside the operator's time axis");
    if (op->solar_src != ATL_SOLAR_COMPUTED)
      ATL_REQUIRE(f->solar_altitude && f->solar_azimuth, "stored solar position fields missing");
    return ATL_OK;
  }
  template <class F, class Visit>
  static void each_field(const AtlCspOp* op, F& f, Visit visit) {
    const size_t sol = op->solar_src == ATL_SOLAR_STORED_F64 ? 8 : 4;
    visit(f.influx_direct, 4);
    visit(f.solar_altitude, sol);
    visit(f.solar_azimuth, sol);
  }
  template <class Run>
  static int with_phys(const AtlCspOp* op, const AtlCspFields* f, int64_t t0, Run run) {
    return run([&](auto vec) { return make_phys<decltype(vec)::value>(op, f, t0); });
  }
};

extern "C" {

int atl_csp_create(int device, const AtlCspConfig* cfg, AtlCspOp** op_out) {
  ATL_REQUIRE(cfg && op_out, "NULL argument");
  *op_out = nullptr;
  ATL_REQUIRE(cfg->ny > 0 && cfg->nx > 0 && cfg->nt >= 0, "bad shape");
  ATL_REQUIRE(cfg->lon_deg && cfg->lat_deg, "coordinate tables missing");
  ATL_REQUIRE(cfg->solar_src >= 0 && cfg->solar_src <= 2, "bad solar source");
  ATL_REQUIRE(cfg->solar_src != ATL_SOLAR_COMPUTED || cfg->time_ns || cfg->nt == 0, "time axis missing");
  ATL_REQUIRE(cfg->technology == 0 || cfg->technology == 1, "Unknown CSP technology option");
  ATL_REQUIRE(cfg->n_alt >= 2 && cfg->n_az >= 2 && cfg->n_alt <= 128 && cfg->n_az <= 128 &&
                  (int64_t)cfg->n_alt * cfg->n_az <= 8192,
              "efficiency table must be 2..128 x 2..128 with at most 8192 entries");
  ATL_REQUIRE(cfg->altitude_rad && cfg->azimuth_rad && cfg->efficiency, "efficiency table missing");
  for (int i = 1; i < cfg->n_alt; ++i)
    ATL_REQUIRE(cfg->altitude_rad[i] > cfg->altitude_rad[i - 1], "altitude coordinates must increase");
  for (int i = 1; i < cfg->n_az; ++i)
    ATL_REQUIRE(cfg->azimuth_rad[i] > cfg->azimuth_rad[i - 1], "azimuth coordinates must increase");
  ATL_REQUIRE(cfg->r_irradiance > 0, "r_irradiance must be positive");

  const double D2R = 3.14159265358979323846 / 180.0;
  AtlCspOp* op = new AtlCspOp();
  op->device = device;
  ATL_REQUIRE(cfg->pitch == 0 || cfg->pitch >= cfg->nx, "pitch must be >= nx");
  op->grid = make_grid(cfg->ny, cfg->nx, cfg->pitch);
  op->nt = cfg->nt;
  op->solar_src = cfg->solar_src;
  op->tower = cfg->technology;
  op->n_alt = cfg->n_alt;
  op->n_az = cfg->n_az;
  op->inv_r = (float)(1.0 / cfg->r_irradiance);
  op->dni_thr = (float)(cfg->dni_altitude_threshold_deg * D2R);

  std::vector<float4> tt;
  solar_almanac(cfg->time_ns, cfg->nt, cfg->time_shift_ns, tt);
  std::vector<float2> xt((size_t)cfg->nx), yt((size_t)cfg->ny);
  for (int i = 0; i < cfg->nx; ++i)
    xt[(size_t)i] = make_float2((float)std::cos(cfg->lon_deg[i] * D2R), (float)std::sin(cfg->lon_deg[i] * D2R));
  for (int j = 0; j < cfg->ny; ++j)
    yt[(size_t)j] = make_float2((float)std::sin(cfg->lat_deg[j] * D2R), (float)std::cos(cfg->lat_deg[j] * D2R));
  std::vector<float> table((size_t)cfg->n_alt + cfg->n_az + (size_t)cfg->n_alt * cfg->n_az);
  for (int i = 0; i < cfg->n_alt; ++i) table[(size_t)i] = (float)cfg->altitude_rad[i];
  for (int i = 0; i < cfg->n_az; ++i) table[(size_t)cfg->n_alt + i] = (float)cfg->azimuth_rad[i];
  for (int64_t i = 0; i < (int64_t)cfg->n_alt * cfg->n_az; ++i)
    table[(size_t)cfg->n_alt + cfg->n_az + (size_t)i] = (float)cfg->efficiency[i];

  cudaError_t e = cudaSetDevice(device);
  auto up = [&](void** d, const void* h, size_t bytes) {
    if (e == cudaSuccess) e = cudaMalloc(d, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(*d, h, bytes, cudaMemcpyHostToDevice);
  };
  up((void**)&op->d_tt, tt.data(), tt.size() * sizeof(float4));
  up((void**)&op->d_xt, xt.data(), xt.size() * sizeof(float2));
  up((void**)&op->d_yt, yt.data(), yt.size() * sizeof(float2));
  up((void**)&op->d_table, table.data(), table.size() * sizeof(float));
  if (e != cudaSuccess) {
    atl_csp_destroy(op);
    return cuda_fail(e, "atl_csp_create");
  }
  *op_out = op;
  return ATL_OK;
}

void atl_csp_destroy(AtlCspOp* op) {
  if (!op) return;
  cudaSetDevice(op->device);
  cudaFree(op->d_tt);
  cudaFree(op->d_xt);
  cudaFree(op->d_yt);
  cudaFree(op->d_table);
  delete op;
}

int atl_csp_op_info(const AtlCspOp* op, int32_t* device, int32_t* ny, int32_t* nx,
                    int32_t* solar_src) {
  if (op && solar_src) *solar_src = op->solar_src;
  return op_info(op, device, ny, nx);
}

int atl_csp_reduce(const AtlCspOp* op, const AtlPlan* plan, const AtlCspFields* f, int64_t t0,
                   int64_t nt, float* out_dev, void* stream) {
  return run_entry<CspBinding>(Entry::kReduce, op, plan, f, t0, nt, out_dev, nullptr, stream);
}

int atl_csp_cells(const AtlCspOp* op, const AtlCspFields* f, int64_t t0, int64_t nt,
                  float* out_dev, void* stream) {
  return run_entry<CspBinding>(Entry::kCells, op, nullptr, f, t0, nt, out_dev, nullptr, stream);
}

int atl_csp_timesum(const AtlCspOp* op, const AtlCspFields* f, int64_t t0, int64_t nt,
                    float* out_dev, float* count_dev, void* stream) {
  return run_entry<CspBinding>(Entry::kTimesum, op, nullptr, f, t0, nt, out_dev, count_dev, stream);
}

int atl_csp_reduce_host(const AtlCspOp* op, const AtlPlan* plan, const AtlCspFields* f, int64_t t0,
                        int64_t nt, float* out_host, int64_t chunk_steps) {
  return run_reduce_host<CspBinding>(op, plan, f, t0, nt, out_host, chunk_steps);
}

}  // extern "C"

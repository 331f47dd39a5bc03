// heat.cu -- degree-day heat demand fused with the shape reduce
// (convert.py:405-418): daily mean of `temperature` over calendar-day bins of
// (time + hour_shift), a * (threshold + 273.15 - Tmean), clip(min=0), + constant.
//
// Algorithmic traffic: 4 B per cell-timestep; output has one row per DAY.
#include <vector>

#include "kernels.cuh"

#ifndef ATL_HEAT_PREFETCH
#define ATL_HEAT_PREFETCH 0  // experiment knob (tools/build_variants.sh): L2 prefetch of the next day
#endif

namespace atl {

struct HeatParams {
  const float* temp;
  const int32_t* day_start;  // device, n_days + 1 step offsets
  int32_t base;              // subtracted from day_start[] -> offsets relative to `temp`
  int64_t S;
  int nx;
  float thr_k, a, constant;
  int cooling;  // 1: a * (Tmean - threshold)   (convert.py:475-491)
};

constexpr int HEAT_UNROLL = 6;
constexpr int HEAT_STAGE = 8;  // days a warp parks in shared memory before one reduce phase

// One chunk of up to HEAT_UNROLL consecutive time steps for the lane's 4 cells.
template <bool VEC>
__device__ __forceinline__ void heat_load_chunk(const HeatParams& hp, const TileGeomT<VEC>& g, int s,
                                                int s1, float (&x)[HEAT_UNROLL][4]) {
#pragma unroll
  for (int u = 0; u < HEAT_UNROLL; ++u) {
    if (s + u < s1) {
      load4(hp.temp, (int64_t)(s + u) * (hp.S * 4), g, x[u]);
    } else {
#pragma unroll
      for (int r = 0; r < 4; ++r) x[u][r] = __int_as_float(0x7fc00000);  // NaN: skipped
    }
  }
}

// daily mean + degree-day formula for the lane's 4 cells of day d.  The loads of
// chunk k+1 are issued before chunk k is accumulated (register double buffer).
// `s_last` = number of steps of the slab (L2 prefetch of the NEXT day's steps stops there).
template <bool VEC>
__device__ __forceinline__ void heat_day(const HeatParams& hp, const TileGeomT<VEC>& g, int d,
                                         float (&v)[4], int s_last) {
  const int s0 = __ldg(hp.day_start + d) - hp.base, s1 = __ldg(hp.day_start + d + 1) - hp.base;
  float sum[4] = {0.f, 0.f, 0.f, 0.f}, cnt[4] = {0.f, 0.f, 0.f, 0.f};
  float x[HEAT_UNROLL][4], y[HEAT_UNROLL][4];
  heat_load_chunk(hp, g, s0, s1, x);
#if ATL_HEAT_PREFETCH
  {  // the next day's slabs go to L2 while this day is summed (no registers: the kernel is latency-bound)
    const int e = min(s1 + (s1 - s0), s_last);
#pragma unroll 4
    for (int s = s1; s < e; ++s) prefetch4_l2(hp.temp, (int64_t)s * (hp.S * 4), g);
  }
#endif
#pragma unroll 1
  for (int s = s0; s < s1; s += HEAT_UNROLL) {
    const bool more = s + HEAT_UNROLL < s1;
    if (more) heat_load_chunk(hp, g, s + HEAT_UNROLL, s1, y);
#pragma unroll
    for (int u = 0; u < HEAT_UNROLL; ++u)
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const bool ok = x[u][r] == x[u][r];  // resample(...).mean() skips NaN
        sum[r] += ok ? x[u][r] : 0.f;
        cnt[r] += ok ? 1.f : 0.f;
      }
    if (more) {
#pragma unroll
      for (int u = 0; u < HEAT_UNROLL; ++u)
#pragma unroll
        for (int r = 0; r < 4; ++r) x[u][r] = y[u][r];
    }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const float mean = sum[r] / cnt[r];  // empty bin -> NaN, as xarray
    float h = hp.a * (hp.cooling ? (mean - hp.thr_k) : (hp.thr_k - mean));  // convert.py:413-414 / 484-485
    h = (h == h) ? fmaxf(h, 0.f) : h;    // .clip(min=0) keeps NaN  :416
    h = hp.constant + h;                 // :418
    v[r] = h;
  }
}

// MODE 0: fused reduce -> out (n_days, n_bus); 1: cells -> out (n_days, ny, nx);
// MODE 2: per-cell sum over days accumulated into out (ny, nx), and the number of non-NaN
// days into cnt_out (may be NULL)
template <int MODE, bool VEC>
__global__ void __launch_bounds__(CTA_THREADS, 6)  // latency-bound (ncu: long_scoreboard): 24 warps per SM
    k_heat(const HeatParams hp, const GridDev gd, const PlanDev plan, float* __restrict__ out,
           float* __restrict__ cnt_out, int n_days, int db) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ai = blockIdx.x * WARPS_PER_CTA + warp;
  int tile, s_beg = 0, s_end = 0;
  if (MODE == 0) {
    if (ai >= plan.n_active) return;
    tile = __ldg(plan.active_tiles + ai);
    s_beg = __ldg(plan.tile_slot_ptr + tile);
    s_end = __ldg(plan.tile_slot_ptr + tile + 1);
  } else {
    if (ai >= gd.n_tx * gd.n_ty) return;
    tile = ai;
  }
  const TileGeomT<VEC> g = make_geom<VEC>(tile, lane, gd);
  const int d0 = blockIdx.y * db, d1 = min(n_days, d0 + db);
  const int s_last = ATL_HEAT_PREFETCH ? __ldg(hp.day_start + n_days) - hp.base : 0;
  float acc[4] = {0.f, 0.f, 0.f, 0.f}, cnt[4] = {0.f, 0.f, 0.f, 0.f};
  float v[4];
  if (MODE == 0) {
    // daily values of HEAT_STAGE days are parked in shared memory, then reduced with the lanes
    // along the days (kernels.cuh: staged_reduce); NaN days poison exactly the buses whose
    // stored entries meet them
    extern __shared__ __align__(16) float smem[];
    char* const stage = reinterpret_cast<char*>(smem) + warp * StageT<HEAT_STAGE>::kWarpBytes;
    stage_init<HEAT_STAGE>(stage, lane);
    const bool cached = tile_cache_load<HEAT_STAGE>(stage, plan, s_beg, s_end, lane);
    for (int dc = d0; dc < d1; dc += HEAT_STAGE) {
      const int n = min(HEAT_STAGE, d1 - dc);
      for (int k = 0; k < n; ++k) {
        heat_day(hp, g, dc + k, v, s_last);
        zero_invalid(g, v);
        stage_store1<HEAT_STAGE>(stage, lane, k, v);
      }
      __syncwarp();
      staged_reduce<HEAT_STAGE>(stage, plan, s_beg, s_end, out, dc, n, lane, cached);
      __syncwarp();
    }
    return;
  }
  for (int d = d0; d < d1; ++d) {
    heat_day(hp, g, d, v, s_last);
    if (MODE == 1) {
      store4(out + (int64_t)d * gd.S_out, gd, g, v);
    } else {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const bool ok = v[r] == v[r];
        acc[r] += ok ? v[r] : 0.f;
        cnt[r] += ok ? 1.f : 0.f;
      }
    }
  }
  if (MODE == 2) {
    atomic_add4(out, gd, g, acc);
    if (cnt_out) atomic_add4(cnt_out, gd, g, cnt);
  }
}

}  // namespace atl

using namespace atl;

struct AtlHeatOp : AtlOpBase {
  float thr_k, a, constant;
  int cooling;  // 1: a * (Tmean - threshold)   (convert.py:475-491)
};

// Every argument check of a heat entry point, before any CUDA call.  The day table holds
// n_days + 1 step offsets, non-decreasing and below 2^31.
static int check_heat(Entry kind, const AtlHeatOp* op, const AtlPlan* plan, const float* temp,
                      const int64_t* day_start, int64_t n_days, const float* out) {
  ATL_REQUIRE(op && temp && day_start && out, "NULL argument");
  if (kind == Entry::kReduce) {
    ATL_REQUIRE(plan, "NULL plan");
    if (int rc = check_plan_grid(op, plan)) return rc;
  }
  ATL_REQUIRE(n_days < (1LL << 31), "bad day count");
  for (int64_t i = 0; i <= n_days; ++i) {
    ATL_REQUIRE(day_start[i] >= 0 && day_start[i] < (1LL << 31), "day offset out of range");
    ATL_REQUIRE(i == 0 || day_start[i] >= day_start[i - 1], "day offsets not monotone");
  }
  return ATL_OK;
}

// The checked day table as int32 in device memory.
static int upload_days(const int64_t* day_start, int64_t n_days, int32_t** d_out, cudaStream_t st) {
  const std::vector<int32_t> ds(day_start, day_start + n_days + 1);
  ATL_CUDA(cudaMallocAsync((void**)d_out, ds.size() * 4, st));
  // pageable source: the copy is staged before the call returns
  ATL_CUDA(cudaMemcpyAsync(*d_out, ds.data(), ds.size() * 4, cudaMemcpyHostToDevice, st));
  ATL_CUDA(cudaStreamSynchronize(st));
  return ATL_OK;
}

// Days [0, n) of the device table `d_days`; `base` is subtracted from its entries, so that a slab of
// the time axis can index into a table uploaded once for the whole axis (atl_heat_reduce_host).
static HeatParams heat_params(const AtlHeatOp* op, const float* temp, const int32_t* d_days, int32_t base) {
  HeatParams hp;
  hp.temp = temp;
  hp.day_start = d_days;
  hp.base = base;
  hp.S = op->grid.S;
  hp.nx = op->grid.nx;
  hp.thr_k = op->thr_k;
  hp.a = op->a;
  hp.constant = op->constant;
  hp.cooling = op->cooling;
  return hp;
}

// k_heat<MODE> over `n_days` days and `n_warps` warp tiles: MODE 0 reduces through `pd` (the
// plan's active tiles), 1 / 2 store the per-cell daily values / add their sum over all tiles.
static int launch_heat(int mode, bool vec, const HeatParams& hp, const GridDev& grid, const PlanDev& pd,
                       int n_warps, int64_t n_days, float* out, float* cnt_out, cudaStream_t st) {
  const int gx = (n_warps + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
  int db = (int)((n_days * gx + 148LL * 4 * 8 - 1) / (148LL * 4 * 8));
  db = db < 1 ? 1 : (db > 8 ? 8 : db);
  size_t smem = 0;
  if (mode == 0) {  // whole staging chunks per block
    db = HEAT_STAGE;
    smem = StageT<HEAT_STAGE>::kCtaBytes;
  }
  GridDev gdo = grid;
  gdo.out_vec = (mode == 1 && gdo.nx % 4 == 0 && aligned16(out)) ? 1 : 0;
  auto* kern = vec ? (mode == 0 ? k_heat<0, true> : mode == 1 ? k_heat<1, true> : k_heat<2, true>)
                   : (mode == 0 ? k_heat<0, false> : mode == 1 ? k_heat<1, false> : k_heat<2, false>);
  kern<<<dim3(gx, (unsigned)((n_days + db - 1) / db)), CTA_THREADS, smem, st>>>(hp, gdo, pd, out, cnt_out,
                                                                                 (int)n_days, db);
  ++g_launches;
  ATL_CUDA(cudaGetLastError());
  return ATL_OK;
}

// lane layout of the per-cell kernels: by grid width and alignment
static bool cells_vec(const AtlHeatOp* op, const float* temp) {
  return op->grid.pitch % 4 == 0 && aligned16(temp);
}

// (day, bus) sums of days [0, n_days) of the table (see heat_params).
static int heat_reduce(const AtlHeatOp* op, const AtlPlan* plan, const float* temp, const int32_t* d_days,
                       int32_t base, int64_t n_days, float* out, cudaStream_t st) {
  const int n_tiles = op->grid.n_tx * op->grid.n_ty;
  if (!plan->fused)
    return two_pass(plan, out, n_days, st, [&](float* scratch, int64_t d0, int64_t n) {
      return launch_heat(1, cells_vec(op, temp), heat_params(op, temp, d_days + d0, base), op->grid, PlanDev{},
                         n_tiles, n, scratch, nullptr, st);
    });
  ATL_REQUIRE(!plan->vec || aligned16(temp),
              "field pointers must be 16-byte aligned (pitch % 4 == 0 uses 128-bit loads)");
  return reduce_into(plan, out, n_days, st, [&](const PlanDev& pd, float* acc) {
    return launch_heat(0, plan->vec, heat_params(op, temp, d_days, base), op->grid, pd, plan->n_active, n_days,
                       acc, nullptr, st);
  });
}

// atl_heat_reduce / _cells / _timesum
static int heat_entry(Entry kind, const AtlHeatOp* op, const AtlPlan* plan, const float* temp,
                      const int64_t* day_start, int64_t n_days, float* out, float* cnt_out, void* stream) {
  if (int rc = check_heat(kind, op, plan, temp, day_start, n_days, out)) return rc;
  if (n_days <= 0) return ATL_OK;
  const cudaStream_t st = (cudaStream_t)stream;
  ATL_CUDA(cudaSetDevice(op->device));
  int32_t* d_days = nullptr;
  if (int rc = upload_days(day_start, n_days, &d_days, st)) return rc;
  int rc;
  if (kind == Entry::kReduce)
    rc = heat_reduce(op, plan, temp, d_days, 0, n_days, out, st);
  else
    rc = launch_heat(kind == Entry::kCells ? 1 : 2, cells_vec(op, temp), heat_params(op, temp, d_days, 0),
                     op->grid, PlanDev{}, op->grid.n_tx * op->grid.n_ty, n_days, out, cnt_out, st);
  cudaFreeAsync(d_days, st);
  return rc;
}

extern "C" {

int atl_heat_create(int device, const AtlHeatConfig* cfg, AtlHeatOp** op_out) {
  ATL_REQUIRE(cfg && op_out, "NULL argument");
  *op_out = nullptr;
  ATL_REQUIRE(cfg->ny > 0 && cfg->nx > 0, "bad grid");
  AtlHeatOp* op = new AtlHeatOp();
  op->device = device;
  ATL_REQUIRE(cfg->pitch == 0 || cfg->pitch >= cfg->nx, "pitch must be >= nx");
  op->grid = make_grid(cfg->ny, cfg->nx, cfg->pitch);
  // the reference adds 273.15 in float64 and then meets the float32 field
  // (weak python scalar -> float32): convert.py:413-414
  op->thr_k = (float)(cfg->threshold_c + 273.15);
  op->a = (float)cfg->a;
  op->constant = (float)cfg->constant;
  op->cooling = cfg->cooling ? 1 : 0;
  *op_out = op;
  return ATL_OK;
}

void atl_heat_destroy(AtlHeatOp* op) { delete op; }

int atl_heat_op_info(const AtlHeatOp* op, int32_t* device, int32_t* ny, int32_t* nx) {
  return op_info(op, device, ny, nx);
}

int atl_heat_reduce(const AtlHeatOp* op, const AtlPlan* plan, const float* temperature_dev,
                    const int64_t* day_start_host, int64_t n_days, float* out_dev,
                    void* stream) {
  return heat_entry(Entry::kReduce, op, plan, temperature_dev, day_start_host, n_days, out_dev, nullptr, stream);
}
int atl_heat_cells(const AtlHeatOp* op, const float* temperature_dev,
                   const int64_t* day_start_host, int64_t n_days, float* out_dev, void* stream) {
  return heat_entry(Entry::kCells, op, nullptr, temperature_dev, day_start_host, n_days, out_dev, nullptr, stream);
}
int atl_heat_timesum(const AtlHeatOp* op, const float* temperature_dev,
                     const int64_t* day_start_host, int64_t n_days, float* out_dev,
                     float* count_dev, void* stream) {
  return heat_entry(Entry::kTimesum, op, nullptr, temperature_dev, day_start_host, n_days, out_dev, count_dev,
                    stream);
}

// Host temperature: the day table is uploaded once, a slab of days [u0, u0 + n) indexes into it.
int atl_heat_reduce_host(const AtlHeatOp* op, const AtlPlan* plan, const float* temperature,
                         const int64_t* day_start, int64_t n_days, float* out_host,
                         int64_t chunk_days) {
  ATL_REQUIRE(op && plan && temperature && day_start, "NULL argument");
  if (int rc = check_host(op, plan, out_host)) return rc;
  if (int rc = check_heat(Entry::kReduce, op, plan, temperature, day_start, n_days, out_host)) return rc;
  if (n_days <= 0) return ATL_OK;
  ATL_CUDA(cudaSetDevice(op->device));
  int32_t* d_days = nullptr;
  if (int rc = upload_days(day_start, n_days, &d_days, 0)) return rc;
  auto launch = [&](const std::vector<void*>& dev, int64_t u0, int64_t n, float* out_dev, cudaStream_t st) {
    return heat_reduce(op, plan, (const float*)dev[0], d_days + u0, (int32_t)day_start[u0], n, out_dev, st);
  };
  const std::vector<SlabField> fields = {{(const char*)temperature, 4}};
  const int rc = stream_slabs(op, plan, fields, n_days, day_start, chunk_days, out_host, launch);
  cudaFree(d_days);
  return rc;
}

}  // extern "C"

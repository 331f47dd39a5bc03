// common.cuh -- shared device/host helpers for libatlite_b200 (sm_100a)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/atlite_b200.h"

namespace atl {

// ---------------------------------------------------------------- errors
void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);
extern int64_t g_launches;

#define ATL_CUDA(call)                                  \
  do {                                                  \
    cudaError_t _e = (call);                            \
    if (_e != cudaSuccess) return atl::cuda_fail(_e, #call); \
  } while (0)

#define ATL_REQUIRE(cond, msg)        \
  do {                                \
    if (!(cond)) {                    \
      atl::set_error(msg);            \
      return ATL_ERR_INVALID;         \
    }                                 \
  } while (0)

// ---------------------------------------------------------------- tiling
// The grid (ny, nx) is covered by warp tiles of 32 (x) x 4 (y) cells.  Lane l of
// the owning warp handles column x = 32*tx + l and the four rows 4*ty .. 4*ty+3,
// so every field load of a warp is one fully coalesced 128-byte row segment and
// needs no alignment of nx (works for any cutout width).  A CTA is 4 warps = 4
// consecutive tiles (adjacent in x: 512 contiguous bytes per row and field).
constexpr int TILE_X = 32;
constexpr int TILE_Y = 4;
constexpr int TILE_CELLS = TILE_X * TILE_Y;
constexpr int WARPS_PER_CTA = 4;
constexpr int CTA_THREADS = 32 * WARPS_PER_CTA;

struct GridDev {
  int nx, ny;
  int pitch;       // elements per stored row of the INPUT fields (>= nx).  Device-resident
                   // cutouts with nx % 4 != 0 are stored row-padded to a multiple of 4 so
                   // that the 128-bit VEC kernels apply (Cutout.to_device()).
  int n_tx, n_ty;  // tiles per row / column
  int64_t S;       // ny * pitch: elements per input time slab
  int64_t S_out;   // ny * nx:    elements per OUTPUT plane (per-cell results are never padded)
  int out_vec;     // per-cell outputs may use 128-bit stores (nx % 4 == 0, aligned base)
};

inline GridDev make_grid(int ny, int nx, int pitch = 0) {
  GridDev g;
  g.nx = nx;
  g.ny = ny;
  g.pitch = pitch > 0 ? pitch : nx;
  g.n_tx = (nx + TILE_X - 1) / TILE_X;
  g.n_ty = (ny + TILE_Y - 1) / TILE_Y;
  g.S = (int64_t)ny * g.pitch;
  g.S_out = (int64_t)ny * nx;
  g.out_vec = 0;
  return g;
}

// One stored matrix entry of a (tile, bus) slot, as the staged reduce consumes it:
// `off` = BYTE offset of the cell inside one row of the warp's staging area (stage
// index * 8, see stage_index below), `w` = the weight.
struct __align__(8) PairEnt {
  uint32_t off;
  float w;
};

// Device view of an aggregation plan (see plan.cu).
struct PlanDev {
  const int32_t* tile_slot_ptr;  // [n_tiles + 1]
  const int32_t* slot_row;       // [n_slots] bus index of each (tile, bus) slot
  const float4* slot_w4;         // [n_slots * 32] dense weights: lane l -> its 4 cells (layout per `vec`)
  const int2* slot_rec;          // [n_slots] {first entry, entry count / PAIR_PAD} into `pairs`
  const PairEnt* pairs;          // the STORED entries of every slot (CSR semantics: nothing else is
                                 // touched), each slot padded to a multiple of PAIR_PAD
  const int32_t* active_tiles;   // [n_active]
  int32_t n_active;
  int32_t n_bus;
};

// Two lane layouts over the same 32 x 4 tile:
//  * SCALAR (any nx): lane l owns column 32*tx + l and rows 4*ty .. 4*ty+3; four
//    scalar loads per field, each a coalesced 128-byte row segment.
//  * VEC (pitch % 4 == 0, 16-byte aligned fields): lane l owns row 4*ty + l/8 and the
//    four consecutive columns 32*tx + 4*(l%8) ..+3: ONE 16-byte load per field
//    (a warp still touches four full 128-byte lines), a quarter of the address
//    arithmetic.
// Cell i of a lane is (cell_y(i), cell_x(i)); `valid` has bit i set if it lies in
// the grid.  Load offsets are CLAMPED into the grid so loads never need a
// predicate; out-of-grid lanes read a border cell whose value is discarded.
template <bool VEC>
struct TileGeomT;

template <>
struct TileGeomT<false> {
  int x, y0;
  unsigned valid;
  int64_t boff[4];  // BYTE offset (float fields) of the lane's 4 cells inside a time slab
  __host__ __device__ int cell_x(int) const { return x; }
  __host__ __device__ int cell_y(int i) const { return y0 + i; }
};
template <>
struct TileGeomT<true> {
  int x0, y;
  unsigned valid;
  int64_t boff;  // BYTE offset (float fields) of the first of the 4 cells (16-byte multiple)
  __host__ __device__ int cell_x(int i) const { return x0 + i; }
  __host__ __device__ int cell_y(int) const { return y; }
};

// position of cell (iy, ix) inside its tile's 128-entry weight vector: 4 * lane + i
// (i = which of the lane's 4 cells), for either lane layout
__host__ __device__ inline int tile_local_index(bool vec, int iy, int ix) {
  const int lx = ix % TILE_X, ly = iy % TILE_Y;
  return vec ? ((ly * 8 + lx / 4) * 4 + (lx & 3)) : (lx * 4 + ly);
}
// position of the same cell in a row of the warp's staging area (staged reduce): value i
// of lane l sits at 32 * i + l, so the 32 lanes of a store hit 32 consecutive slots
__host__ __device__ inline int stage_index(int local) { return 32 * (local & 3) + (local >> 2); }
// The entry list of a slot is sorted by stage index and padded to a multiple of
// PAIR_PAD entries with {PAD_OFF, 0}: PAD_OFF addresses the padding bytes behind the 128
// cells of a staging row, which the kernel keeps at 0.0f, so a pad entry adds exactly 0
// whatever the cells hold (0 * NaN would not).
constexpr int PAIR_PAD = 8;
constexpr uint32_t PAD_OFF = TILE_CELLS * 8;

#ifdef __CUDACC__
template <bool VEC>
__device__ __forceinline__ TileGeomT<VEC> make_geom(int tile, int lane, const GridDev& gd);

template <>
__device__ __forceinline__ TileGeomT<false> make_geom<false>(int tile, int lane, const GridDev& gd) {
  TileGeomT<false> g;
  const int tx = tile % gd.n_tx, ty = tile / gd.n_tx;
  g.x = tx * TILE_X + lane;
  g.y0 = ty * TILE_Y;
  unsigned v = 0;
  if (g.x < gd.nx) {
#pragma unroll
    for (int r = 0; r < TILE_Y; ++r)
      if (g.y0 + r < gd.ny) v |= 1u << r;
  }
  g.valid = v;
  const int xc = min(g.x, gd.nx - 1);
#pragma unroll
  for (int r = 0; r < TILE_Y; ++r)
    g.boff[r] = 4 * (int64_t)(min(g.y0 + r, gd.ny - 1) * gd.pitch + xc);
  return g;
}
template <>
__device__ __forceinline__ TileGeomT<true> make_geom<true>(int tile, int lane, const GridDev& gd) {
  TileGeomT<true> g;
  const int tx = tile % gd.n_tx, ty = tile / gd.n_tx;
  g.x0 = tx * TILE_X + 4 * (lane & 7);
  g.y = ty * TILE_Y + (lane >> 3);
  unsigned v = 0;  // with a padded pitch a chunk may straddle the logical width nx
  if (g.y < gd.ny) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (g.x0 + i < gd.nx) v |= 1u << i;
  }
  g.valid = v;
  g.boff = 4 * (int64_t)(min(g.y, gd.ny - 1) * gd.pitch + min(g.x0, gd.pitch - 4));
  return g;
}

// NaN-propagating min / max (FMNMX.NAN): xarray's / numpy's clip keeps NaN, CUDA's
// fminf / fmaxf drop it
__device__ __forceinline__ float fmin_nan(float a, float b) {
  float d;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float d;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
  return d;
}

__device__ __forceinline__ float warp_sum(float p) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
  return p;
}

// Streaming (read-once) global load: bypass L1 allocation so the small, hot
// weight / table lines stay resident.
__device__ __forceinline__ float ld_stream(const float* p) {
  float v;
  asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ double ld_stream(const double* p) {
  double v;
  asm("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}

__device__ __forceinline__ float4 ld_stream4(const float* p) {
  float4 v;
  asm("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
      : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
      : "l"(p));
  return v;
}

// Load the lane's 4 cells of one field.  `tb` = BYTE offset of the time slab
// (t * S * 4 for float fields), kept as a running 64-bit value by the caller so a
// load costs one 64-bit add (uniform field base + per-lane offset) and no
// multiply.  float64 fields (stored solar position) scale the offset by 2.
__device__ __forceinline__ const float* at_bytes(const float* f, int64_t b) {
  return reinterpret_cast<const float*>(reinterpret_cast<const char*>(f) + b);
}
__device__ __forceinline__ const double* at_bytes(const double* f, int64_t b) {
  return reinterpret_cast<const double*>(reinterpret_cast<const char*>(f) + 2 * b);
}
// One MUFU.RCP (div.approx / __fdividef(1.f, x) add a canonicalising FADD behind it).
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ void load4(const float* __restrict__ f, int64_t tb,
                                      const TileGeomT<false>& g, float (&o)[4]) {
#pragma unroll
  for (int r = 0; r < TILE_Y; ++r) o[r] = ld_stream(at_bytes(f, tb + g.boff[r]));
}
__device__ __forceinline__ void load4(const float* __restrict__ f, int64_t tb,
                                      const TileGeomT<true>& g, float (&o)[4]) {
  const float4 v = ld_stream4(at_bytes(f, tb + g.boff));
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
__device__ __forceinline__ void load4(const double* __restrict__ f, int64_t tb,
                                      const TileGeomT<false>& g, float (&o)[4]) {
#pragma unroll
  for (int r = 0; r < TILE_Y; ++r) o[r] = (float)ld_stream(at_bytes(f, tb + g.boff[r]));
}
__device__ __forceinline__ void load4(const double* __restrict__ f, int64_t tb,
                                      const TileGeomT<true>& g, float (&o)[4]) {
  const double* p = at_bytes(f, tb + g.boff);
#pragma unroll
  for (int r = 0; r < 4; ++r) o[r] = (float)ld_stream(p + r);
}

// L2 prefetch of the lane's 4 cells of a later time slab (VEC layout: the warp's 32 x 16 B are the
// same four 128-byte lines the LDG.128 will read).  Costs no registers: this is how a kernel that
// is at its register budget gets more bytes in flight.
__device__ __forceinline__ void prefetch4_l2(const float* __restrict__ f, int64_t tb, const TileGeomT<true>& g) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(at_bytes(f, tb + g.boff)));
}
__device__ __forceinline__ void prefetch4_l2(const float* __restrict__, int64_t, const TileGeomT<false>&) {}

// Store the lane's 4 per-cell values into a (y, x) plane.
__device__ __forceinline__ void store4(float* __restrict__ plane, const GridDev& gd,
                                       const TileGeomT<false>& g, const float (&v)[4]) {
#pragma unroll
  for (int r = 0; r < TILE_Y; ++r)
    if ((g.valid >> r) & 1u) plane[(g.y0 + r) * gd.nx + g.x] = v[r];
}
__device__ __forceinline__ void store4(float* __restrict__ plane, const GridDev& gd,
                                       const TileGeomT<true>& g, const float (&v)[4]) {
  float* o = plane + g.y * gd.nx + g.x0;
  if (gd.out_vec) {
    if (g.valid) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if ((g.valid >> r) & 1u) o[r] = v[r];
  }
}
__device__ __forceinline__ void atomic_add4(float* __restrict__ plane, const GridDev& gd,
                                            const TileGeomT<false>& g, const float (&v)[4]) {
#pragma unroll
  for (int r = 0; r < TILE_Y; ++r)
    if ((g.valid >> r) & 1u) atomicAdd(plane + (g.y0 + r) * gd.nx + g.x, v[r]);
}
__device__ __forceinline__ void atomic_add4(float* __restrict__ plane, const GridDev& gd,
                                            const TileGeomT<true>& g, const float (&v)[4]) {
#pragma unroll
  for (int r = 0; r < 4; ++r)
    if ((g.valid >> r) & 1u) atomicAdd(plane + g.y * gd.nx + g.x0 + r, v[r]);
}

// Values of out-of-grid cells (row padding / tile overhang) are unspecified; zero
// them so that padding contents can never send a tile down the NaN path.
template <class Geom>
__device__ __forceinline__ void zero_invalid(const Geom& g, float (&v)[4]) {
  if (g.valid != 0xFu) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (!((g.valid >> i) & 1u)) v[i] = 0.f;
  }
}

// Exact path for tiles holding a NaN/Inf: zero weights must not touch the value
// (a sparse matrix never multiplies entries it does not store: aggregate.py:25 /
// scipy CSR product).  Kept out of line: it is cold.
static __device__ __noinline__ void reduce_slots_exact(float v0, float v1, float v2, float v3, int s_beg,
                                               int s_end, const PlanDev& plan,
                                               float* __restrict__ out_row, int lane) {
#pragma unroll 1
  for (int s = s_beg; s < s_end; ++s) {
    const float4 w = __ldg(plan.slot_w4 + (size_t)s * 32 + lane);
    float p = 0.f;
    if (w.x != 0.f) p += w.x * v0;
    if (w.y != 0.f) p += w.y * v1;
    if (w.z != 0.f) p += w.z * v2;
    if (w.w != 0.f) p += w.w * v3;
    p = warp_sum(p);
    if (lane == 0) atomicAdd(out_row + __ldg(plan.slot_row + s), p);
  }
}

// Reduce the 4 per-cell values of every lane into the tile's (tile, bus) slots
// and add the warp totals to out_row[bus].  Weight lines are L1-resident after
// the first time step.
__device__ __forceinline__ void reduce_slots(const float (&v)[4], int s_beg, int s_end,
                                             const PlanDev& plan, float* __restrict__ out_row,
                                             int lane) {
  const float chk = (v[0] + v[1]) + (v[2] + v[3]);
  const bool bad = !(fabsf(chk) <= 3.0e38f);
  if (__any_sync(0xffffffffu, bad)) {
    reduce_slots_exact(v[0], v[1], v[2], v[3], s_beg, s_end, plan, out_row, lane);
    return;
  }
#pragma unroll 1
  for (int s = s_beg; s < s_end; ++s) {
    const float4 w = __ldg(plan.slot_w4 + (size_t)s * 32 + lane);
    float p = fmaf(w.x, v[0], fmaf(w.y, v[1], fmaf(w.z, v[2], w.w * v[3])));
    p = warp_sum(p);
    if (lane == 0) atomicAdd(out_row + __ldg(plan.slot_row + s), p);
  }
}

// Two time steps at once: lanes 0-15 finish the butterfly for step t, lanes
// 16-31 for step t+1 (one exchange instead of a second full reduction), then
// lane 0 and lane 16 issue their atomics in the same instruction.
__device__ __forceinline__ void reduce_slots2(const float (&v0)[4], const float (&v1)[4],
                                              int s_beg, int s_end, const PlanDev& plan,
                                              float* __restrict__ out_row0, int lane) {
  const float chk = ((v0[0] + v0[1]) + (v0[2] + v0[3])) + ((v1[0] + v1[1]) + (v1[2] + v1[3]));
  const bool bad = !(fabsf(chk) <= 3.0e38f);
  if (__any_sync(0xffffffffu, bad)) {
    reduce_slots_exact(v0[0], v0[1], v0[2], v0[3], s_beg, s_end, plan, out_row0, lane);
    reduce_slots_exact(v1[0], v1[1], v1[2], v1[3], s_beg, s_end, plan, out_row0 + plan.n_bus,
                       lane);
    return;
  }
  const bool hi = lane >= 16;
  float* const my_row = out_row0 + (hi ? plan.n_bus : 0);
  // running pointers: one 64-bit add per slot instead of re-deriving the addresses
  const float4* wp = plan.slot_w4 + (size_t)s_beg * 32 + lane;
  const int32_t* rp = plan.slot_row + s_beg;
#pragma unroll 1
  for (int n = s_end - s_beg; n > 0; --n, wp += 32, ++rp) {
    const float4 w = __ldg(wp);
    const float p0 = fmaf(w.x, v0[0], fmaf(w.y, v0[1], fmaf(w.z, v0[2], w.w * v0[3])));
    const float p1 = fmaf(w.x, v1[0], fmaf(w.y, v1[1], fmaf(w.z, v1[2], w.w * v1[3])));
    float keep = hi ? p1 : p0;
    const float send = hi ? p0 : p1;
    keep += __shfl_xor_sync(0xffffffffu, send, 16);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    if ((lane & 15) == 0) atomicAdd(my_row + __ldg(rp), keep);
  }
}

// Four slots x two time steps in ONE transposed butterfly: 9 shuffles for 8 sums
// instead of 20, and one atomic instruction (8 active lanes) instead of four.
// Lane L ends up holding the sum of step (L >> 4) for slot f = (L >> 2) & 3 of the
// group.  It evaluates the group's slots in the order f, f^1, f^2, f^3, so at the
// xor-8 stage it keeps positions 0,1 and receives its partner's positions 2,3 (the
// partner's f differs in bit 1: those ARE slots f, f^1), at xor-4 it keeps
// position 0 and receives the partner's position 1 -- no selects anywhere.  The
// step split (xor 16) is folded into which of v0/v1 a lane treats as "keep".
// A group may run past the tile's last slot (2 or 3 left): those weight vectors
// belong to the next tile (or the zero padding of the array); their sums live in
// separate accumulators and are dropped.  A single left-over slot takes the
// pairwise path.
// PROBE = false: the caller has already established that no lane holds a NaN/Inf value.
template <bool PROBE = true>
__device__ __forceinline__ void reduce_slots2g(const float (&v0)[4], const float (&v1)[4],
                                               int s_beg, int s_end, const PlanDev& plan,
                                               float* __restrict__ out_row0, int lane) {
  const float chk = ((v0[0] + v0[1]) + (v0[2] + v0[3])) + ((v1[0] + v1[1]) + (v1[2] + v1[3]));
  const bool bad = !(fabsf(chk) <= 3.0e38f);
  if (PROBE && __any_sync(0xffffffffu, bad)) {
    reduce_slots_exact(v0[0], v0[1], v0[2], v0[3], s_beg, s_end, plan, out_row0, lane);
    reduce_slots_exact(v1[0], v1[1], v1[2], v1[3], s_beg, s_end, plan, out_row0 + plan.n_bus,
                       lane);
    return;
  }
  const bool hi = lane >= 16;
  float* const my_row = out_row0 + (hi ? plan.n_bus : 0);
  float vk[4], vs[4];  // the step this half-warp keeps / sends
  float2 ks[4];        // ... as {keep, send} pairs: both dot products of a slot share the weights, so
                       // one packed FFMA2 (weight broadcast) does what two FFMAs did
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    vk[i] = hi ? v1[i] : v0[i];
    vs[i] = hi ? v0[i] : v1[i];
    ks[i] = make_float2(vk[i], vs[i]);
  }
  const int f = (lane >> 2) & 3;
  int s = s_beg;
  const int32_t* rp = plan.slot_row + s_beg + f;  // running pointer: this lane's slot of the group
#pragma unroll 1
  for (; s_end - s >= 2; s += 4, rp += 4) {
    const float4* wp = plan.slot_w4 + (size_t)s * 32 + lane;
    float a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 w = __ldg(wp + (f ^ i) * 32);
      const float2 ab = __ffma2_rn(make_float2(w.x, w.x), ks[0],
                                   __ffma2_rn(make_float2(w.y, w.y), ks[1],
                                              __ffma2_rn(make_float2(w.z, w.z), ks[2],
                                                         __fmul2_rn(make_float2(w.w, w.w), ks[3]))));
      a[i] = ab.x;
      b[i] = ab.y;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] += __shfl_xor_sync(0xffffffffu, b[i], 16);
    a[0] += __shfl_xor_sync(0xffffffffu, a[2], 8);
    a[1] += __shfl_xor_sync(0xffffffffu, a[3], 8);
    a[0] += __shfl_xor_sync(0xffffffffu, a[1], 4);
    a[0] += __shfl_xor_sync(0xffffffffu, a[0], 2);
    a[0] += __shfl_xor_sync(0xffffffffu, a[0], 1);
    if ((lane & 3) == 0 && s + f < s_end) atomicAdd(my_row + __ldg(rp), a[0]);
  }
  if (s < s_end) {  // one slot left
    const float4 w = __ldg(plan.slot_w4 + (size_t)s * 32 + lane);
    float keep = fmaf(w.x, vk[0], fmaf(w.y, vk[1], fmaf(w.z, vk[2], w.w * vk[3])));
    const float send = fmaf(w.x, vs[0], fmaf(w.y, vs[1], fmaf(w.z, vs[2], w.w * vs[3])));
    keep += __shfl_xor_sync(0xffffffffu, send, 16);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    if ((lane & 15) == 0) atomicAdd(my_row + __ldg(plan.slot_row + s), keep);
  }
}

// reduce_slots2g with the FIRST group's weights resident in registers (`wres`, loaded once per
// tile walk by load_group_weights): the weights of a tile do not change along time, and
// re-reading them every two steps costs as many L1 wavefronts as the fields themselves (wind).
// Later groups (tiles with more than 4 slots, about a quarter) and the odd last slot load as before.
// `row_res`: the output column (bus) this lane adds the first group's sum to, -1 if none.
__device__ __forceinline__ void load_group_weights(float4 (&wres)[4], int& row_res, int s_beg, int s_end,
                                                   const PlanDev& plan, int lane) {
  const int f = (lane >> 2) & 3;
  const float4* wp = plan.slot_w4 + (size_t)s_beg * 32 + lane;
#pragma unroll
  for (int i = 0; i < 4; ++i) wres[i] = __ldg(wp + (f ^ i) * 32);
  row_res = ((lane & 3) == 0 && s_beg + f < s_end) ? __ldg(plan.slot_row + s_beg + f) : -1;
}
template <bool PROBE = true>
__device__ __forceinline__ void reduce_slots2g_res(const float (&v0)[4], const float (&v1)[4],
                                                   const float4 (&wres)[4], int row_res, int s_beg, int s_end,
                                                   const PlanDev& plan, float* __restrict__ out_row0,
                                                   int lane) {
  const float chk = ((v0[0] + v0[1]) + (v0[2] + v0[3])) + ((v1[0] + v1[1]) + (v1[2] + v1[3]));
  const bool bad = !(fabsf(chk) <= 3.0e38f);
  if (PROBE && __any_sync(0xffffffffu, bad)) {
    reduce_slots_exact(v0[0], v0[1], v0[2], v0[3], s_beg, s_end, plan, out_row0, lane);
    reduce_slots_exact(v1[0], v1[1], v1[2], v1[3], s_beg, s_end, plan, out_row0 + plan.n_bus,
                       lane);
    return;
  }
  const bool hi = lane >= 16;
  float* const my_row = out_row0 + (hi ? plan.n_bus : 0);
  float vk[4], vs[4];
  float2 ks[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    vk[i] = hi ? v1[i] : v0[i];
    vs[i] = hi ? v0[i] : v1[i];
    ks[i] = make_float2(vk[i], vs[i]);
  }
  const int f = (lane >> 2) & 3;
  int s = s_beg;
  const int32_t* rp = plan.slot_row + s_beg + f;
  auto group = [&](auto&& weight, auto&& add) {
    float a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 w = weight(i);
      const float2 ab = __ffma2_rn(make_float2(w.x, w.x), ks[0],
                                   __ffma2_rn(make_float2(w.y, w.y), ks[1],
                                              __ffma2_rn(make_float2(w.z, w.z), ks[2],
                                                         __fmul2_rn(make_float2(w.w, w.w), ks[3]))));
      a[i] = ab.x;
      b[i] = ab.y;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] += __shfl_xor_sync(0xffffffffu, b[i], 16);
    a[0] += __shfl_xor_sync(0xffffffffu, a[2], 8);
    a[1] += __shfl_xor_sync(0xffffffffu, a[3], 8);
    a[0] += __shfl_xor_sync(0xffffffffu, a[1], 4);
    a[0] += __shfl_xor_sync(0xffffffffu, a[0], 2);
    a[0] += __shfl_xor_sync(0xffffffffu, a[0], 1);
    add(a[0]);
  };
  // the resident group (also serves a 1-slot tile)
  group([&](int i) { return wres[i]; }, [&](float sum) { if (row_res >= 0) atomicAdd(my_row + row_res, sum); });
  s += 4;
  rp += 4;
#pragma unroll 1
  for (; s_end - s >= 2; s += 4, rp += 4) {
    const float4* wp = plan.slot_w4 + (size_t)s * 32 + lane;
    group([&](int i) { return __ldg(wp + (f ^ i) * 32); },
          [&](float sum) { if ((lane & 3) == 0 && s + f < s_end) atomicAdd(my_row + __ldg(rp), sum); });
  }
  if (s < s_end) {  // one slot left
    const float4 w = __ldg(plan.slot_w4 + (size_t)s * 32 + lane);
    float keep = fmaf(w.x, vk[0], fmaf(w.y, vk[1], fmaf(w.z, vk[2], w.w * vk[3])));
    const float send = fmaf(w.x, vs[0], fmaf(w.y, vs[1], fmaf(w.z, vs[2], w.w * vs[3])));
    keep += __shfl_xor_sync(0xffffffffu, send, 16);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    if ((lane & 15) == 0) atomicAdd(my_row + __ldg(plan.slot_row + s), keep);
  }
}
#endif  // __CUDACC__

}  // namespace atl

// Opaque handle definitions shared between translation units.

// Every operator handle (AtlPvOp, AtlWindOp, ...) starts with this: the device it lives on and
// the grid of its input fields.
struct AtlOpBase {
  int device;
  atl::GridDev grid;
};

namespace atl {
// what atl_<op>_op_info reports for every operator
inline int op_info(const AtlOpBase* op, int32_t* device, int32_t* ny, int32_t* nx) {
  ATL_REQUIRE(op, "NULL argument");
  if (device) *device = op->device;
  if (ny) *ny = op->grid.ny;
  if (nx) *nx = op->grid.nx;
  return ATL_OK;
}
}  // namespace atl

struct AtlPlan {
  int device;
  atl::GridDev grid;
  int32_t n_bus;
  int64_t nnz;
  int32_t n_tiles, n_active;
  int64_t n_slots;
  bool fused;
  bool vec;  // weight layout / kernels: VEC lane layout (grid.pitch % 4 == 0)
  // device arrays
  int32_t* d_tile_slot_ptr = nullptr;
  int32_t* d_slot_row = nullptr;
  float4* d_slot_w4 = nullptr;
  int2* d_slot_rec = nullptr;
  atl::PairEnt* d_pairs = nullptr;
  int64_t n_pairs = 0;
  int32_t* d_active = nullptr;
  // deterministic mode: identity slot index + (bus -> slots) lists
  int32_t* d_slot_ident = nullptr;
  int32_t* d_row_slot_ptr = nullptr;
  int32_t* d_row_slots = nullptr;
  // CSR copy for the two-pass fallback / generic SpMM
  int64_t* d_indptr = nullptr;
  int32_t* d_indices = nullptr;
  float* d_vals = nullptr;
  atl::PlanDev dev() const {
    atl::PlanDev p;
    p.tile_slot_ptr = d_tile_slot_ptr;
    p.slot_row = d_slot_row;
    p.slot_w4 = d_slot_w4;
    p.slot_rec = d_slot_rec;
    p.pairs = d_pairs;
    p.active_tiles = d_active;
    p.n_active = n_active;
    p.n_bus = n_bus;
    return p;
  }
  // Deterministic mode: every (slot, step) partial goes to its own address
  // (exactly one writer -> the float atomics become order-independent); a
  // second kernel sums each bus's slots in a fixed order.
  atl::PlanDev dev_partial() const {
    atl::PlanDev p = dev();
    p.slot_row = d_slot_ident;
    p.n_bus = (int32_t)n_slots;
    return p;
  }
};

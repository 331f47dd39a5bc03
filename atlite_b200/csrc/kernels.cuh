// kernels.cuh -- generic "per-cell physics -> {shape reduce | per-cell store |
// per-cell time sum}" kernels, templated on a physics functor.
//
// A physics functor `Phys` provides
//   static constexpr bool kVec;   lane layout (see common.cuh: TileGeomT<VEC>)
//   struct Cell;   per-thread constants (geometry of the lane's 4 cells)
//   struct Raw;    the raw field values of one time step (4 cells)
//   static constexpr int kSmemFloats;        CTA-shared lookup tables
//   static constexpr int kBatch, kMinBlocks; time steps per batch / CTAs per SM
//   __device__ void stage(float* smem) const;            (whole CTA, before use)
//   __device__ void init(Cell&, const Geom&, const float* smem) const;
//   __device__ void load(const Cell&, const Geom&, int64_t tb, Raw&) const;
//        tb = byte offset of the time slab (t * S * 4), maintained by the caller
//   __device__ void compute(const Cell&, const Geom&, int t, const Raw&,
//                           float (&v)[4], const float* smem) const;
//        values of out-of-grid lanes are unspecified (finite border copies): they
//        carry zero weight in every slot and are never stored
//   static constexpr bool kHasExact;  if true, compute() may differ from the reference
//        when an INPUT is NaN/Inf but then always yields a non-finite value, and
//        compute_exact(...) (same signature) reproduces the reference's NaN rules; the
//        kernels call it only for steps whose fast result came out non-finite
//   static constexpr bool kStaged; int kStage, kBatchStaged, kMinBlocksStaged;  which fused kernel
//        serves this physics by default (staged reduce or shuffle reduce), the chunk length and
//        batch / occupancy parameters of the staged kernel
// `t` is relative to the slab the functor's field pointers address.
//
// Loop structure: a warp owns one 32x4 tile and walks a block of `tb`
// consecutive time steps.  Memory latency is hidden by occupancy (PREFETCH=0:
// few registers, many resident warps) or additionally by a register double
// buffer (PREFETCH=1: the loads of step t+1 are issued before the arithmetic
// of step t).
#pragma once
#include <functional>
#include <type_traits>
#include <vector>

#include "common.cuh"

namespace atl {

// Physics that are issue-bound rather than HBM-bound opt into two copies of the time walk
// (`static constexpr bool kSplitMask = true`), see fused_v1_walk.
template <class P, class = void>
struct resident_weights : std::false_type {};
template <class P>
struct resident_weights<P, std::void_t<decltype(P::kResidentWeights)>> : std::bool_constant<P::kResidentWeights> {};
template <class P, class = void>
struct l2_prefetch : std::integral_constant<int, 0> {};
template <class P>
struct l2_prefetch<P, std::void_t<decltype(P::kL2Prefetch)>> : std::integral_constant<int, P::kL2Prefetch> {};
template <class P, class = void>
struct split_mask : std::false_type {};
template <class P>
struct split_mask<P, std::void_t<decltype(P::kSplitMask)>> : std::bool_constant<P::kSplitMask> {};

// The time walk of one warp tile.  MASK = the tile overhangs the grid (row padding / last tile
// column): only then are the values of out-of-grid lanes zeroed; interior tiles (the vast
// majority) run the copy of the loop without the selects (about one instruction in eight of
// the wind kernel).  The choice is warp-uniform, made once per tile.
template <class Phys, int B, int G, bool MASK, class Geom>
__device__ __forceinline__ void fused_v1_walk(const Phys& phys, const GridDev& gd, const PlanDev& plan,
                                              float* __restrict__ out, int nt, int tb, const Geom& g,
                                              int s_beg, int s_end, int lane, const float* smem) {
  const int t0 = blockIdx.y * tb;
  const int t1 = min(nt, t0 + tb);
  const int nb = plan.n_bus;

  typename Phys::Cell c;
  phys.init(c, g, smem);
  typename Phys::Raw r[B];
  float v[B][4];
  const int64_t S4 = gd.S * 4;
  int64_t sb = (int64_t)t0 * S4;  // byte offset of the next slab to LOAD
  const int nfull = (t1 - t0) / B;
  int t = t0;
  constexpr bool RES = resident_weights<Phys>::value && G == 1 && (B % 2 == 0);
  float4 wres[RES ? 4 : 1];
  int row_res = -1;
  if constexpr (RES) load_group_weights(wres, row_res, s_beg, s_end, plan, lane);
  if (nfull > 0) {
#pragma unroll
    for (int j = 0; j < B; ++j) phys.load(c, g, sb + j * S4, r[j]);
    sb += B * S4;
#pragma unroll 1
    for (int k = 0; k < nfull; ++k, t += B) {
#pragma unroll
      for (int j = 0; j < B; ++j) {
        phys.compute(c, g, t + j, r[j], v[j], smem);
        if (MASK) zero_invalid(g, v[j]);
      }
      bool bad = false;  // kHasExact: one probe serves the physics' NaN rules AND the reduce
      if constexpr (Phys::kHasExact) {
        float chk = 0.f;
#pragma unroll
        for (int j = 0; j < B; ++j) chk += (v[j][0] + v[j][1]) + (v[j][2] + v[j][3]);
        bad = __any_sync(0xffffffffu, !(fabsf(chk) <= 3.0e38f));
        if (bad) {  // cold: a NaN/Inf reached a result -> the reference's NaN rules
#pragma unroll
          for (int j = 0; j < B; ++j) {
            phys.compute_exact(c, g, t + j, r[j], v[j], smem);
            if (MASK) zero_invalid(g, v[j]);
          }
        }
      }
      if (k + 1 < nfull) {
#pragma unroll
        for (int j = 0; j < B; ++j) phys.load(c, g, sb + j * S4, r[j]);
        sb += B * S4;
        // kL2Prefetch = D > 0: the batch D batches past the one just requested goes to L2 now
        if constexpr (l2_prefetch<Phys>::value > 0) {
          constexpr int D = l2_prefetch<Phys>::value;
          if (k + 1 + D < nfull) {
#pragma unroll
            for (int j = 0; j < B; ++j) phys.prefetch(c, g, sb + ((D - 1) * B + j) * S4);
          }
        }
      }
#pragma unroll
      for (int j = 0; j + 1 < B; j += 2) {
        float* const o = out + (size_t)(t + j) * nb;
        if constexpr (Phys::kHasExact) {
          if (bad) {  // cold: what is left non-finite is meant to be; stored entries only
            reduce_slots_exact(v[j][0], v[j][1], v[j][2], v[j][3], s_beg, s_end, plan, o, lane);
            reduce_slots_exact(v[j + 1][0], v[j + 1][1], v[j + 1][2], v[j + 1][3], s_beg, s_end, plan, o + nb, lane);
          } else if constexpr (RES) {
            reduce_slots2g_res<false>(v[j], v[j + 1], wres, row_res, s_beg, s_end, plan, o, lane);
          } else {
            reduce_slots2g<false>(v[j], v[j + 1], s_beg, s_end, plan, o, lane);
          }
        } else if constexpr (RES) {
          reduce_slots2g_res(v[j], v[j + 1], wres, row_res, s_beg, s_end, plan, o, lane);
        } else if (G) {  // slots in groups of four (transposed butterfly)
          reduce_slots2g(v[j], v[j + 1], s_beg, s_end, plan, o, lane);
        } else {
          reduce_slots2(v[j], v[j + 1], s_beg, s_end, plan, o, lane);
        }
      }
      if (B & 1) reduce_slots(v[B - 1], s_beg, s_end, plan, out + (size_t)(t + B - 1) * nb, lane);
    }
  }
  // tail: fewer than B steps left
#pragma unroll 1
  for (; t < t1; ++t, sb += S4) {
    phys.load(c, g, sb, r[0]);
    phys.compute(c, g, t, r[0], v[0], smem);
    if (MASK) zero_invalid(g, v[0]);
    if constexpr (Phys::kHasExact) {
      if (__any_sync(0xffffffffu, !(fabsf((v[0][0] + v[0][1]) + (v[0][2] + v[0][3])) <= 3.0e38f))) {
        phys.compute_exact(c, g, t, r[0], v[0], smem);
        if (MASK) zero_invalid(g, v[0]);
      }
    }
    reduce_slots(v[0], s_beg, s_end, plan, out + (size_t)t * nb, lane);
  }
}

// A warp owns one 32x4 tile and walks `tb` consecutive time steps in batches of
// B.  Per batch: the arithmetic of the B resident steps runs first, then the
// loads of the NEXT batch are issued into the now-dead raw registers, and only
// then the shuffle-reduce + atomics of the current batch execute -- so B steps of
// loads are in flight across the whole reduce phase at no extra register cost.
// Steps are reduced two at a time, slots four at a time, in one transposed
// butterfly (reduce_slots2g; G = 0 selects the older pairwise reduce_slots2).  B is chosen per
// physics so that B x (#fields) 16-byte loads per lane cover the HBM latency
// (PV: 2 x 5, wind: 4 x 2, SpMM: 4 x 1).  MINB = CTAs/SM the register allocator
// must allow.
template <class Phys, int B, int MINB, int G = 0>
__global__ void __launch_bounds__(CTA_THREADS, MINB)
    k_fused_reduce_v1(const Phys phys, const GridDev gd, const PlanDev plan,
                      float* __restrict__ out, int nt, int tb) {
  extern __shared__ float smem[];
  phys.stage(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ai = blockIdx.x * WARPS_PER_CTA + warp;
  if (ai >= plan.n_active) return;
  const int tile = __ldg(plan.active_tiles + ai);
  const auto g = make_geom<Phys::kVec>(tile, lane, gd);
  const int s_beg = __ldg(plan.tile_slot_ptr + tile);
  const int s_end = __ldg(plan.tile_slot_ptr + tile + 1);
  if constexpr (split_mask<Phys>::value) {
    if (__any_sync(0xffffffffu, g.valid != 0xFu))
      fused_v1_walk<Phys, B, G, true>(phys, gd, plan, out, nt, tb, g, s_beg, s_end, lane, smem);
    else
      fused_v1_walk<Phys, B, G, false>(phys, gd, plan, out, nt, tb, g, s_beg, s_end, lane, smem);
  } else {
    fused_v1_walk<Phys, B, G, true>(phys, gd, plan, out, nt, tb, g, s_beg, s_end, lane, smem);
  }
}


// ---------------------------------------------------------------- staged reduce
// The round-2 kernel.  A warp still owns one 32x4 tile and walks `tb` consecutive
// time steps, but it no longer reduces every step with warp shuffles against DENSE
// 128-float weight vectors (4 FMAs + ~1.1 shuffles per slot and step whatever the
// slot's fill: 70 of wind's 213 warp-instructions per step).  Instead the per-cell
// values of TS steps are parked in shared memory, and the reduce runs with the lanes
// spanning TIME: lane (q, r) owns the step pair r of the chunk and walks a q-th of the
// slot's STORED matrix entries {cell, weight}; per entry it costs one broadcast 8-byte
// load of the entry, one conflict-light 8-byte shared load of the cell's two steps and
// two FMAs -- work proportional to the entries of the tile (~1.2 per cell for
// NUTS-like shapes), independent of how many buses touch the tile, ~12 instructions
// per step instead of ~70.  Entries a CSR matrix does not store are never multiplied,
// so NaN/Inf cells poison exactly the buses that contain them (scipy semantics) with no
// special path.
//
// Staging area of one warp: R = TS/2 rows (one per PAIR of consecutive steps); a row holds
// the tile's 128 cells as float2 {even step, odd step} in stage_index order, then 8 * 16/R
// bytes that stay 0.0f (the target of the plan's padding entries) and shift consecutive rows
// by 16/R eight-byte bank pairs.  In the reduce phase the R lanes of a group read R
// different rows at the same cell (bank pairs 16/R apart) and the 16/R groups that share a
// shared-memory pass read CONSECUTIVE entries of the slot's list, which is sorted by stage
// index -- neighbouring cells, i.e. the bank pairs in between: conflict-free for the usual
// contiguous slot, never worse than 2-way.
constexpr int ENT_CAP = 256;  // entries of the warp's tile kept in shared memory (8 B each)
constexpr int SLOT_CAP = 24;  // slot records of the warp's tile kept in shared memory (16 B each)
template <int TS>
struct StageT {
  static constexpr int kRows = TS / 2;
  static constexpr int kShift = 16 / kRows > 0 ? 16 / kRows : 1;
  static constexpr int kRowBytes = TILE_CELLS * 8 + 8 * kShift;
  static constexpr int kEntOff = kRows * kRowBytes;          // entry cache (16-byte aligned)
  static constexpr int kSlotOff = kEntOff + ENT_CAP * 8;     // slot-record cache
  static constexpr int kWarpBytes = kSlotOff + SLOT_CAP * 16;
  static constexpr int kCtaBytes = WARPS_PER_CTA * kWarpBytes;
  static_assert(kEntOff % 16 == 0, "entry cache must be 16-byte aligned");
};
__host__ __device__ constexpr int smem_table_bytes(int floats) { return (floats * 4 + 15) & ~15; }

// The bytes behind the 128 cells of every staging row hold 0.0f (the padding entries of the
// plan point there).
template <int TS>
__device__ __forceinline__ void stage_init(char* stage, int lane) {
  using Stage = StageT<TS>;
  if (lane < Stage::kRows) {
#pragma unroll
    for (int k = 0; k < Stage::kShift; ++k)
      *reinterpret_cast<float2*>(stage + lane * Stage::kRowBytes + PAD_OFF + 8 * k) = make_float2(0.f, 0.f);
  }
}

// Park the lane's 4 values of one step (row = step pair, half = parity) / of a step pair.
template <int TS>
__device__ __forceinline__ void stage_store1(char* stage, int lane, int k, const float (&v)[4]) {
  char* const w = stage + lane * 8 + (k >> 1) * StageT<TS>::kRowBytes + (k & 1) * 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) *reinterpret_cast<float*>(w + 256 * i) = v[i];
}
template <int TS>
__device__ __forceinline__ void stage_store2(char* stage, int lane, int k_even, const float (&v0)[4],
                                             const float (&v1)[4]) {
  char* const w = stage + lane * 8 + (k_even >> 1) * StageT<TS>::kRowBytes;
#pragma unroll
  for (int i = 0; i < 4; ++i) *reinterpret_cast<float2*>(w + 256 * i) = make_float2(v0[i], v1[i]);
}

// A warp keeps its tile for many chunks, so the tile's slot records {first entry, entry count /
// PAIR_PAD, bus} and entry lists are copied into shared memory once (they are contiguous in the
// plan): the reduce phase then depends on shared-memory latency only, not on whether L1 / L2
// still hold the lists.  Tiles with more than SLOT_CAP slots or ENT_CAP entries (rare: the
// average is 4 slots / 160 entries) keep reading the plan from global memory.
template <int TS>
__device__ __forceinline__ bool tile_cache_load(char* stage, const PlanDev& plan, int s_beg, int s_end,
                                                int lane) {
  using Stage = StageT<TS>;
  const int K = s_end - s_beg;
  if (K <= 0 || K > SLOT_CAP) return false;
  const int base = __ldg(plan.slot_rec + s_beg).x;
  const int2 last = __ldg(plan.slot_rec + s_end - 1);
  const int total = last.x + last.y * PAIR_PAD - base;
  if (total > ENT_CAP) return false;
  int4* const slots = reinterpret_cast<int4*>(stage + Stage::kSlotOff);
  uint2* const ent = reinterpret_cast<uint2*>(stage + Stage::kEntOff);
  if (lane < K) {
    const int2 r = __ldg(plan.slot_rec + s_beg + lane);
    slots[lane] = make_int4(r.x - base, r.y, __ldg(plan.slot_row + s_beg + lane), 0);
  }
  const uint2* const src = reinterpret_cast<const uint2*>(plan.pairs) + base;
  for (int i = lane; i < total; i += 32) ent[i] = __ldg(src + i);
  return true;
}

// The reduce phase of one chunk: rows [row0, row0 + nvalid) of `out` receive the sums of the
// staged steps.  Lane = group * R + row: lane (q, r) owns the step pair r and walks the
// entries q, q + NQ, q + 2 NQ, ... of every slot's list; one butterfly over the groups, then
// group 0 adds the even step and group 1 the odd one in ONE atomic instruction.
// (__syncwarp() before -- the stores of all lanes must be visible -- and after.)
template <int TS>
__device__ __forceinline__ void staged_reduce(const char* stage, const PlanDev& plan, int s_beg, int s_end,
                                              float* __restrict__ out, int row0, int nvalid, int lane,
                                              bool cached) {
  static_assert(TS == 8 || TS == 16 || TS == 32, "TS/2 rows must divide the warp");
  using Stage = StageT<TS>;
  constexpr int R = TS / 2;   // rows = lanes along time
  constexpr int NQ = 32 / R;  // lanes sharing a row split a slot's entries NQ ways
  constexpr int U = PAIR_PAD / NQ;  // entries per group and padding unit
  static_assert(U >= 1 && U * NQ == PAIR_PAD, "PAIR_PAD must be a multiple of the group count");
  const int rp = lane & (R - 1), q = lane / R;
  const char* const rd_row = stage + rp * Stage::kRowBytes;
  const int nb = plan.n_bus;
  const int odd = lane >= R ? 1 : 0;
  float* const o_mine = out + (size_t)(row0 + 2 * rp + odd) * nb;
  const bool w_mine = lane < 2 * R && 2 * rp + odd < nvalid;
  auto finish = [&](float a0, float a1, int row) {
#pragma unroll
    for (int o = R; o < 32; o <<= 1) {
      a0 += __shfl_xor_sync(0xffffffffu, a0, o);
      a1 += __shfl_xor_sync(0xffffffffu, a1, o);
    }
    if (w_mine) atomicAdd(o_mine + row, odd ? a1 : a0);
  };
  if (cached) {
    const int4* const slots = reinterpret_cast<const int4*>(stage + Stage::kSlotOff);
    const uint2* const ent_q = reinterpret_cast<const uint2*>(stage + Stage::kEntOff) + q;
    const int K = s_end - s_beg;
    // two slots at a time: their load -> load -> FMA chains are independent, which halves the
    // latency a warp spends in this phase (the phase is latency-, not issue-bound)
    int k = 0;
#pragma unroll 1
    for (; k + 1 < K; k += 2) {
      const int4 sa = slots[k], sb = slots[k + 1];
      const uint2 *pa = ent_q + sa.x, *pb = ent_q + sb.x;
      float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
      const int nmin = min(sa.y, sb.y);
      int it = 0;
#pragma unroll 2
      for (; it < nmin; ++it, pa += PAIR_PAD, pb += PAIR_PAD) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint2 wa = pa[u * NQ], wb = pb[u * NQ];
          const float2 xa = *reinterpret_cast<const float2*>(rd_row + wa.x);
          const float2 xb = *reinterpret_cast<const float2*>(rd_row + wb.x);
          a0 = fmaf(__uint_as_float(wa.y), xa.x, a0);
          a1 = fmaf(__uint_as_float(wa.y), xa.y, a1);
          b0 = fmaf(__uint_as_float(wb.y), xb.x, b0);
          b1 = fmaf(__uint_as_float(wb.y), xb.y, b1);
        }
      }
#pragma unroll 2
      for (int ia = it; ia < sa.y; ++ia, pa += PAIR_PAD) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint2 wa = pa[u * NQ];
          const float2 xa = *reinterpret_cast<const float2*>(rd_row + wa.x);
          a0 = fmaf(__uint_as_float(wa.y), xa.x, a0);
          a1 = fmaf(__uint_as_float(wa.y), xa.y, a1);
        }
      }
#pragma unroll 2
      for (int ib = it; ib < sb.y; ++ib, pb += PAIR_PAD) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint2 wb = pb[u * NQ];
          const float2 xb = *reinterpret_cast<const float2*>(rd_row + wb.x);
          b0 = fmaf(__uint_as_float(wb.y), xb.x, b0);
          b1 = fmaf(__uint_as_float(wb.y), xb.y, b1);
        }
      }
#pragma unroll
      for (int o = R; o < 32; o <<= 1) {  // both butterflies interleaved
        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        a1 += __shfl_xor_sync(0xffffffffu, a1, o);
        b0 += __shfl_xor_sync(0xffffffffu, b0, o);
        b1 += __shfl_xor_sync(0xffffffffu, b1, o);
      }
      if (w_mine) {
        atomicAdd(o_mine + sa.z, odd ? a1 : a0);
        atomicAdd(o_mine + sb.z, odd ? b1 : b0);
      }
    }
    if (k < K) {
      const int4 sr = slots[k];
      const uint2* p = ent_q + sr.x;
      float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
      for (int it = 0; it < sr.y; ++it, p += PAIR_PAD) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint2 pw = p[u * NQ];
          const float2 x = *reinterpret_cast<const float2*>(rd_row + pw.x);
          const float w = __uint_as_float(pw.y);
          a0 = fmaf(w, x.x, a0);
          a1 = fmaf(w, x.y, a1);
        }
      }
      finish(a0, a1, sr.z);
    }
    return;
  }
  const uint2* const pairs_q = reinterpret_cast<const uint2*>(plan.pairs) + q;
#pragma unroll 1
  for (int s = s_beg; s < s_end; ++s) {
    const int2 rec = __ldg(plan.slot_rec + s);
    const uint2* p = pairs_q + rec.x;
    float a0 = 0.f, a1 = 0.f;
#pragma unroll 2
    for (int it = 0; it < rec.y; ++it, p += PAIR_PAD) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint2 pw = __ldg(p + u * NQ);
        const float2 x = *reinterpret_cast<const float2*>(rd_row + pw.x);
        const float w = __uint_as_float(pw.y);
        a0 = fmaf(w, x.x, a0);
        a1 = fmaf(w, x.y, a1);
      }
    }
    finish(a0, a1, __ldg(plan.slot_row + s));
  }
}

template <class Phys, int B, int MINB, int TS>
__global__ void __launch_bounds__(CTA_THREADS, MINB)
    k_fused_reduce(const Phys phys, const GridDev gd, const PlanDev plan,
                   float* __restrict__ out, int nt, int tb) {
  static_assert(B == 1 || B % 2 == 0, "steps are staged in pairs");
  static_assert(TS % B == 0, "a chunk is a whole number of batches");
  using Stage = StageT<TS>;
  extern __shared__ __align__(16) float smem[];
  phys.stage(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ai = blockIdx.x * WARPS_PER_CTA + warp;
  if (ai >= plan.n_active) return;
  char* const stage = reinterpret_cast<char*>(smem) + smem_table_bytes(Phys::kSmemFloats) +
                      warp * Stage::kWarpBytes;
  const int tile = __ldg(plan.active_tiles + ai);
  const auto g = make_geom<Phys::kVec>(tile, lane, gd);
  const int s_beg = __ldg(plan.tile_slot_ptr + tile);
  const int s_end = __ldg(plan.tile_slot_ptr + tile + 1);
  const int t0 = blockIdx.y * tb;
  const int t1 = min(nt, t0 + tb);
  if (t0 >= t1) return;
  const int tlast = t1 - 1;

  typename Phys::Cell c;
  phys.init(c, g, smem);
  typename Phys::Raw r[B];
  float v[B][4];
  const int64_t S4 = gd.S * 4;
  // Load indices are clamped to the block's last step instead of predicated: at most
  // B - 1 redundant loads / evaluations per time block, their results never written.
#pragma unroll
  for (int j = 0; j < B; ++j) phys.load(c, g, (int64_t)min(t0 + j, tlast) * S4, r[j]);
  stage_init<TS>(stage, lane);
  const bool cached = tile_cache_load<TS>(stage, plan, s_beg, s_end, lane);

#pragma unroll 1
  for (int tc = t0; tc < t1; tc += TS) {
    // ---- physics of up to TS steps -> staging area (registers only in between)
#pragma unroll 1
    for (int k = 0; k < TS; k += B) {
      const int t = tc + k;
      if (t >= t1) break;
      // rolling pipeline over the B register sets: as soon as a step has been evaluated, its raw
      // registers are re-loaded with step t + B, so every load has B - 1 steps of arithmetic (and
      // the other warps) between issue and first use; across a chunk boundary it additionally
      // flies through the whole reduce phase
#pragma unroll
      for (int j = 0; j < B; ++j) {
        phys.compute(c, g, min(t + j, tlast), r[j], v[j], smem);
        zero_invalid(g, v[j]);
        if constexpr (Phys::kHasExact) {
          const float chk = (v[j][0] + v[j][1]) + (v[j][2] + v[j][3]);
          if (__any_sync(0xffffffffu, !(fabsf(chk) <= 3.0e38f))) {  // cold: a NaN/Inf reached a result
            phys.compute_exact(c, g, min(t + j, tlast), r[j], v[j], smem);
            zero_invalid(g, v[j]);
          }
        }
        phys.load(c, g, (int64_t)min(t + B + j, tlast) * S4, r[j]);
      }
      if (B == 1) {
        stage_store1<TS>(stage, lane, k, v[0]);
      } else {
#pragma unroll
        for (int j = 0; j + 1 < B; j += 2) stage_store2<TS>(stage, lane, k + j, v[j], v[j + 1]);
      }
    }
    __syncwarp();
    staged_reduce<TS>(stage, plan, s_beg, s_end, out, tc, min(TS, t1 - tc), lane, cached);
    __syncwarp();  // the next chunk's stores must not overtake this chunk's reads
  }
}

// MODE 0: store per-cell values out[(t - t_begin), y, x]
// MODE 1: accumulate the (NaN-skipping) time sum into out[y, x]
// Rolling software pipeline over B register sets: as soon as step t has been
// evaluated from set j its registers are reloaded with step t + B, so B - 1 steps
// of arithmetic (and the other warps) cover every load.  Load indices are clamped
// to the block's last step instead of predicated (at most B - 1 redundant loads
// and evaluations per time block, their results discarded).
// MODE 1 also counts the valid (non-NaN) steps per cell into `cnt_out` (may be NULL): the
// reference's per-cell mean skips NaN steps (convert.py:51-56).
template <class Phys, int MODE, int B, int MINB>
__global__ void __launch_bounds__(CTA_THREADS, MINB)
    k_cells(const Phys phys, const GridDev gd, float* __restrict__ out,
            float* __restrict__ cnt_out, int t_begin, int t_end, int tb) {
  extern __shared__ float smem[];
  phys.stage(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x * WARPS_PER_CTA + warp;
  if (tile >= gd.n_tx * gd.n_ty) return;
  const auto g = make_geom<Phys::kVec>(tile, lane, gd);
  const int t0 = t_begin + blockIdx.y * tb;
  const int t1 = min(t_end, t0 + tb);
  if (t0 >= t1) return;

  typename Phys::Cell c;
  phys.init(c, g, smem);
  typename Phys::Raw r[B];
  float v[4];
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  int n_nan[4] = {0, 0, 0, 0};
  const int64_t S4 = gd.S * 4;
  const int tl = t1 - 1;
#pragma unroll
  for (int j = 0; j < B; ++j) phys.load(c, g, (int64_t)min(t0 + j, tl) * S4, r[j]);
#pragma unroll 1
  for (int t = t0; t < t1; t += B) {
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const bool live = t + j < t1;
      phys.compute(c, g, min(t + j, tl), r[j], v, smem);
      if constexpr (Phys::kHasExact) {  // cold, warp-uniform: a NaN/Inf reached a result
        if (__any_sync(0xffffffffu, !(fabsf((v[0] + v[1]) + (v[2] + v[3])) <= 3.0e38f)))
          phys.compute_exact(c, g, min(t + j, tl), r[j], v, smem);
      }
      phys.load(c, g, (int64_t)min(t + j + B, tl) * S4, r[j]);
      if (MODE == 0) {
        if (live) store4(out + (int64_t)(t + j - t_begin) * gd.S_out, gd, g, v);
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {  // NaN steps are skipped and counted (one predicated add)
          const bool ok = v[q] == v[q];
          acc[q] += (live && ok) ? v[q] : 0.f;
          if (live && !ok) ++n_nan[q];
        }
      }
    }
  }
  if (MODE == 1) {
    atomic_add4(out, gd, g, acc);
    if (cnt_out) {  // valid steps of this block = its steps minus the NaN ones
      float cnt[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) cnt[q] = (float)(t1 - t0 - n_nan[q]);
      atomic_add4(cnt_out, gd, g, cnt);
    }
  }
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Deterministic reduce mode (atl_set_deterministic): bitwise-repeatable results.
bool deterministic();

// Generic CSR gather SpMM: out[t, row] = sum_k val[k] * dense[t, col[k]]
// (aggregate.py:24-32 on an already materialised field).  One warp per
// (row, t); used for plans that do not tile well and as second pass of the
// two-pass fallback.
__global__ void k_csr_spmm(const int64_t* __restrict__ indptr, const int32_t* __restrict__ idx,
                           const float* __restrict__ val, const float* __restrict__ dense,
                           int64_t S, float* __restrict__ out, int n_bus, int nt);

// Run-time tuning knobs (environment: ATL_VARIANT, ATL_TB), for experiments.
struct Tuning {
  int variant = 0;
  int tb = 0;
};
const Tuning& tuning();

__global__ void k_gather_slots(const float* __restrict__ partial, const int32_t* __restrict__ row_slot_ptr,
                               const int32_t* __restrict__ row_slots, float* __restrict__ out,
                               int n_bus, int64_t n_slots, int nt);
int launch_gather_slots(const AtlPlan* plan, const float* partial, int64_t nt, float* out,
                        cudaStream_t st);

inline int pick_tb(int n_cta_x, int64_t nt) {
  // time steps per CTA: aim for ~24 CTAs per resident slot (148 SMs x 5 CTAs) so
  // the tail wave is small, but keep the per-CTA prologue (geometry, slot setup)
  // amortised over >= 16 steps.  Measured optimum 32..128 (profiles/r1_tb_sweep.log).
  const int64_t want = 148LL * 5 * 24;
  int64_t tb = (nt * n_cta_x + want - 1) / want;
  if (tb < 16) tb = 16;
  if (tb > 128) tb = 128;
  tb += tb & 1;
  if (tb > nt) tb = nt > 0 ? nt : 1;
  return (int)tb;
}

template <class Phys>
int launch_cells(const Phys& phys, const GridDev& gd, float* out, int64_t t_begin,
                 int64_t t_end, bool timesum, cudaStream_t st, float* cnt_out = nullptr) {
  if (t_end <= t_begin) return ATL_OK;
  const int n_tiles = gd.n_tx * gd.n_ty;
  const int gx = (n_tiles + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
  // deterministic time sums: one time block, so every cell receives exactly one add
  const int tb = (timesum && deterministic()) ? (int)(t_end - t_begin) : pick_tb(gx, t_end - t_begin);
  const int gy = (int)((t_end - t_begin + tb - 1) / tb);
  dim3 grid(gx, gy);
  const size_t smem = Phys::kSmemFloats * sizeof(float);
  GridDev go = gd;
  go.out_vec = (gd.nx % 4 == 0 && aligned16(out)) ? 1 : 0;
  if (timesum)
    k_cells<Phys, 1, Phys::kBatch, Phys::kMinBlocks>
        <<<grid, CTA_THREADS, smem, st>>>(phys, go, out, cnt_out, (int)t_begin, (int)t_end, tb);
  else
    k_cells<Phys, 0, Phys::kBatch, Phys::kMinBlocks>
        <<<grid, CTA_THREADS, smem, st>>>(phys, go, out, nullptr, (int)t_begin, (int)t_end, tb);
  ++g_launches;
  ATL_CUDA(cudaGetLastError());
  return ATL_OK;
}

int launch_csr_spmm(const AtlPlan* plan, const float* dense, int64_t nt, float* out,
                    cudaStream_t st);

template <class Phys, int TS>
int launch_staged(const Phys& phys, const AtlPlan* plan, const GridDev& gd, const PlanDev& pd, float* acc,
                  int64_t nt, int tb, int gx, cudaStream_t st) {
  tb = ((tb + TS - 1) / TS) * TS;  // whole chunks per time block
  dim3 grid(gx, (unsigned)((nt + tb - 1) / tb));
  const size_t smem = smem_table_bytes(Phys::kSmemFloats) + StageT<TS>::kCtaBytes;
  auto kern = k_fused_reduce<Phys, Phys::kBatchStaged, Phys::kMinBlocksStaged, TS>;
  static bool attr_set[64] = {false};  // per instantiation and device (benign if set twice)
  if (plan->device >= 0 && plan->device < 64 && !attr_set[plan->device]) {
    ATL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[plan->device] = true;
  }
  kern<<<grid, CTA_THREADS, smem, st>>>(phys, gd, pd, acc, (int)nt, tb);
  return ATL_OK;
}

// The (unit, bus) target of a fused reduce over `nu` units (time steps, or days).  `kernel(pd, acc)`
// launches the fused kernel, which accumulates into `acc` through the plan view `pd`: `out`
// itself, or in deterministic mode a private (unit, slot) buffer with one writer per address
// that k_gather_slots then sums into `out` in a fixed order.  An empty plan leaves zeros.
template <class Kernel>
int reduce_into(const AtlPlan* plan, float* out, int64_t nu, cudaStream_t st, Kernel kernel) {
  if (plan->n_active == 0) {
    ATL_CUDA(cudaMemsetAsync(out, 0, (size_t)nu * plan->n_bus * sizeof(float), st));
    return ATL_OK;
  }
  const bool det = deterministic() && plan->n_slots > 0;
  float* acc = out;
  PlanDev pd = plan->dev();
  if (det) {
    ATL_CUDA(cudaMallocAsync((void**)&acc, (size_t)nu * plan->n_slots * sizeof(float), st));
    pd = plan->dev_partial();
  }
  cudaError_t e = cudaMemsetAsync(acc, 0, (size_t)nu * pd.n_bus * sizeof(float), st);
  int rc = e == cudaSuccess ? kernel(pd, acc) : cuda_fail(e, "cudaMemsetAsync(acc)");
  if (det) {
    if (rc == ATL_OK) rc = launch_gather_slots(plan, acc, nu, out, st);
    cudaFreeAsync(acc, st);
  }
  return rc;
}

// Two-pass fallback for matrices that do not tile (e.g. one bus per cell): `cells(scratch, u0, n)`
// writes the per-cell rows of units [u0, u0 + n) into an unpadded scratch block of at most
// 256 MiB, which a CSR gather then reduces into rows [u0, u0 + n) of `out`.
template <class Cells>
int two_pass(const AtlPlan* plan, float* out, int64_t nu, cudaStream_t st, Cells cells) {
  const int64_t S = plan->grid.S_out;
  int64_t blk = (256LL << 20) / (S * 4);
  if (blk < 1) blk = 1;
  if (blk > nu) blk = nu;
  float* scratch = nullptr;
  ATL_CUDA(cudaMallocAsync((void**)&scratch, (size_t)blk * S * sizeof(float), st));
  for (int64_t u = 0; u < nu; u += blk) {
    const int64_t n = (nu - u < blk) ? nu - u : blk;
    int rc = cells(scratch, u, n);
    if (rc == ATL_OK) rc = launch_csr_spmm(plan, scratch, n, out + (size_t)u * plan->n_bus, st);
    if (rc != ATL_OK) {
      cudaFreeAsync(scratch, st);
      return rc;
    }
  }
  ATL_CUDA(cudaFreeAsync(scratch, st));
  return ATL_OK;
}

// Fused path of one slab.  `Phys` must use the plan's lane layout.
template <class Phys>
int launch_fused(const Phys& phys, const AtlPlan* plan, float* out, int64_t nt, cudaStream_t st) {
  return reduce_into(plan, out, nt, st, [&](const PlanDev& pd, float* acc) {
    const int gx = (plan->n_active + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    int tb = tuning().tb > 0 ? tuning().tb : pick_tb(gx, nt);
    const GridDev gd = plan->grid;
    const int variant = tuning().variant;
    // ATL_VARIANT: 0 = the functor's own choice (Phys::kStaged), 1 = shuffle reduce against dense
    // weight vectors, 2 = staged reduce (chunk Phys::kStage), 3 = staged reduce, the other chunk length
    const bool staged = variant == 0 ? Phys::kStaged : variant != 1;
    if (!staged) {
      dim3 grid(gx, (unsigned)((nt + tb - 1) / tb));
      k_fused_reduce_v1<Phys, Phys::kBatch, Phys::kMinBlocks, 1>
          <<<grid, CTA_THREADS, Phys::kSmemFloats * sizeof(float), st>>>(phys, gd, pd, acc, (int)nt, tb);
    } else if (variant == 3) {
      int rc = launch_staged<Phys, (Phys::kStage == 16 ? 8 : 16)>(phys, plan, gd, pd, acc, nt, tb, gx, st);
      if (rc) return rc;
    } else {
      int rc = launch_staged<Phys, Phys::kStage>(phys, plan, gd, pd, acc, nt, tb, gx, st);
      if (rc) return rc;
    }
    ++g_launches;
    ATL_CUDA(cudaGetLastError());
    return ATL_OK;
  });
}

// Two-pass path of one slab: per-cell blocks of the physics, then the CSR gather.
template <class Phys>
int launch_two_pass(const Phys& phys, const AtlPlan* plan, float* out, int64_t nt,
                    cudaStream_t st) {
  return two_pass(plan, out, nt, st, [&](float* scratch, int64_t t, int64_t n) {
    return launch_cells(phys, plan->grid, scratch, t, t + n, false, st);
  });
}

// Dispatch on the lane layout.  `make(vec_tag)` builds the functor for a layout:
// make(std::true_type{}) -> Phys<VEC>, make(std::false_type{}) -> Phys<SCALAR>.
// `ptrs_aligned`: every field pointer is 16-byte aligned (needed for VEC).
template <class Make>
int dispatch_reduce(Make make, const AtlPlan* plan, bool ptrs_aligned, float* out, int64_t nt,
                    cudaStream_t st) {
  if (nt <= 0) return ATL_OK;
  ATL_REQUIRE(nt < (1LL << 31), "slab too long");
  if (plan->fused) {
    if (plan->vec) {
      ATL_REQUIRE(ptrs_aligned,
                  "field pointers must be 16-byte aligned (pitch % 4 == 0 uses 128-bit loads)");
      return launch_fused(make(std::true_type{}), plan, out, nt, st);
    }
    return launch_fused(make(std::false_type{}), plan, out, nt, st);
  }
  if (plan->vec && ptrs_aligned) return launch_two_pass(make(std::true_type{}), plan, out, nt, st);
  return launch_two_pass(make(std::false_type{}), plan, out, nt, st);
}

template <class Make>
int dispatch_cells(Make make, const GridDev& gd, bool ptrs_aligned, float* out, int64_t nt,
                   bool timesum, cudaStream_t st, float* cnt_out = nullptr) {
  if (gd.pitch % 4 == 0 && ptrs_aligned)
    return launch_cells(make(std::true_type{}), gd, out, 0, nt, timesum, st, cnt_out);
  return launch_cells(make(std::false_type{}), gd, out, 0, nt, timesum, st, cnt_out);
}

// ---------------------------------------------------------------- entry points
// atl_<op>_reduce / _cells / _timesum of an operator.
enum class Entry { kReduce, kCells, kTimesum };

inline int check_plan_grid(const AtlOpBase* op, const AtlPlan* plan) {
  ATL_REQUIRE(plan->grid.nx == op->grid.nx && plan->grid.ny == op->grid.ny &&
                  plan->grid.pitch == op->grid.pitch,
              "plan / operator grid (or pitch) mismatch");
  return ATL_OK;
}

// Every entry point of a physics-functor operator runs this one sequence: all argument checks,
// then cudaSetDevice, then the dispatch by kind, so a malformed call is refused before the
// library touches the device.  The operator's binding `B` supplies
//   using Op, Fields;                        the handle (derived from AtlOpBase), the field pointers
//   static int check(const Op*, const Fields*, int64_t t0, int64_t nt);   the operator's own checks
//   static void each_field(const Op*, F& fields, Visit visit);
//                                            visit(pointer member, bytes per element) for every field
//                                            pointer, in one fixed order: the VEC layout needs them all
//                                            16-byte aligned, host streaming copies and rebinds them
//   static int with_phys(const Op*, const Fields*, int64_t t0, Run run);
//                                            run(make) with the functor maker of the operator's
//                                            compile-time mode, make(vec_tag) -> Phys (dispatch_reduce)
// Operators without a time axis ignore t0.
template <class B>
int run_entry(Entry kind, const typename B::Op* op, const AtlPlan* plan, const typename B::Fields* f,
              int64_t t0, int64_t nt, float* out, float* cnt_out, void* stream) {
  if (int rc = B::check(op, f, t0, nt)) return rc;
  ATL_REQUIRE(out && (plan || kind != Entry::kReduce), "NULL argument");
  if (kind == Entry::kReduce)
    if (int rc = check_plan_grid(op, plan)) return rc;
  ATL_CUDA(cudaSetDevice(op->device));
  bool al = true;
  B::each_field(op, *f, [&](const void* p, size_t) { al = al && aligned16(p); });
  const cudaStream_t st = (cudaStream_t)stream;
  return B::with_phys(op, f, t0, [&](auto make) {
    if (kind == Entry::kReduce) return dispatch_reduce(make, plan, al, out, nt, st);
    return dispatch_cells(make, op->grid, al, out, nt, kind == Entry::kTimesum, st, cnt_out);
  });
}

// ---------------------------------------------------------------- host streaming (host_stream.cu)
// atl_<op>_reduce_host: the fields live in host memory and are streamed in time slabs through a
// device ring.  The ring holds ny * nx elements per step, so the operator must be unpadded.
struct SlabField {
  const char* host;  // nullptr = unused
  size_t elem;       // bytes per element
};
// Reduces units [u0, u0 + n) of the call (steps, or days) whose fields the ring holds at `dev`
// (one pointer per SlabField, nullptr for unused ones) into `out_dev`.
using SlabLaunch = std::function<int(const std::vector<void*>& dev, int64_t u0, int64_t n, float* out_dev,
                                     cudaStream_t st)>;

// The checks every host entry point makes before any CUDA call.
inline int check_host(const AtlOpBase* op, const AtlPlan* plan, const float* out_host) {
  ATL_REQUIRE(out_host, "NULL output");
  if (int rc = check_plan_grid(op, plan)) return rc;
  ATL_REQUIRE(op->grid.pitch == op->grid.nx,
              "host entry points take unpadded fields (operator pitch must be nx)");
  return ATL_OK;
}

// Streams `n_units` units, unit u starting at step unit_start[u] (n_units + 1 entries; NULL:
// one step per unit), `chunk_units` per slab (<= 0: about 192 MiB of input), and copies the
// (unit, bus) result to `out_host`.  The caller has run check_host.
int stream_slabs(const AtlOpBase* op, const AtlPlan* plan, const std::vector<SlabField>& fields,
                 int64_t n_units, const int64_t* unit_start, int64_t chunk_units, float* out_host,
                 const SlabLaunch& launch);

template <class B>
int run_reduce_host(const typename B::Op* op, const AtlPlan* plan, const typename B::Fields* f, int64_t t0,
                    int64_t nt, float* out_host, int64_t chunk_steps) {
  ATL_REQUIRE(op && plan && f, "NULL argument");
  if (int rc = check_host(op, plan, out_host)) return rc;
  if (int rc = B::check(op, f, t0, nt)) return rc;
  std::vector<SlabField> fields;
  B::each_field(op, *f, [&](const auto& p, size_t elem) { fields.push_back({(const char*)p, elem}); });
  auto launch = [&](const std::vector<void*>& dev, int64_t u0, int64_t n, float* out_dev, cudaStream_t st) {
    typename B::Fields df = *f;
    size_t i = 0;
    B::each_field(op, df, [&](auto& p, size_t) {
      p = static_cast<std::remove_reference_t<decltype(p)>>(dev[i++]);  // nullptr stays nullptr
    });
    return run_entry<B>(Entry::kReduce, op, plan, &df, t0 + u0, n, out_dev, nullptr, st);
  };
  return stream_slabs(op, plan, fields, nt, nullptr, chunk_steps, out_host, launch);
}

}  // namespace atl

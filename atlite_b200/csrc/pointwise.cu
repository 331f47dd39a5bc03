// pointwise.cu -- conversions that are a pointwise function of ONE field, fused
// with the shape reduce: temperature / dewpoint (K -> deg C, convert.py:292-329),
// soil temperature (NaN over sea -> 0, :306-316), heat-pump coefficient of
// performance (quadratic in sink_T - source_T, :338-366) and runoff weighted by
// the static height field (:1028-1034).  4 B per cell-timestep.
#include <vector>

#include "kernels.cuh"

namespace atl {

template <bool VEC>
struct PointwisePhys {
  static constexpr bool kVec = VEC;
  using Geom = TileGeomT<VEC>;
  const float* f;
  const float* cell_scale;  // device (ny, nx) or nullptr
  int nx, ny;
  float shift, sink, c0, c1, c2;
  int nan_to_zero, poly;

  struct Cell {
    float sc[4];
  };
  struct Raw {
    float v[4];
  };
  static constexpr int kSmemFloats = 0;
  static constexpr int kBatch = 4, kMinBlocks = 6;
  static constexpr bool kHasExact = false;
  static constexpr bool kStaged = false;
  static constexpr int kStage = 8, kBatchStaged = kBatch, kMinBlocksStaged = kMinBlocks;
  __device__ void stage(float*) const {}
  __device__ void init(Cell& c, const Geom& g, const float*) const {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      c.sc[i] = 1.f;
      if (cell_scale)
        c.sc[i] = __ldg(cell_scale + min(g.cell_y(i), ny - 1) * nx + min(g.cell_x(i), nx - 1));
    }
  }
  __device__ void load(const Cell&, const Geom& g, int64_t sb, Raw& r) const { load4(f, sb, g, r.v); }
  __device__ void compute(const Cell& c, const Geom&, int, const Raw& r, float (&v)[4],
                          const float*) const {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float y = r.v[i] + shift;
      if (nan_to_zero) y = (y == y) ? y : 0.f;  // .fillna(0.0)
      if (poly) {
        const float d = sink - y;
        y = fmaf(fmaf(c2, d, c1), d, c0);  // c0 + c1 d + c2 d^2
      }
      v[i] = y * c.sc[i];
    }
  }
};

}  // namespace atl

using namespace atl;

struct AtlPointwiseOp : AtlOpBase {
  float shift, sink, c0, c1, c2;
  int nan_to_zero, poly;
  float* d_scale = nullptr;
};

template <bool VEC>
static PointwisePhys<VEC> make_phys(const AtlPointwiseOp* op, const float* field) {
  PointwisePhys<VEC> p;
  p.f = field;
  p.cell_scale = op->d_scale;
  p.nx = op->grid.nx;
  p.ny = op->grid.ny;
  p.shift = op->shift;
  p.sink = op->sink;
  p.c0 = op->c0;
  p.c1 = op->c1;
  p.c2 = op->c2;
  p.nan_to_zero = op->nan_to_zero;
  p.poly = op->poly;
  return p;
}

// The pointwise operator's part of the shared entry sequence (kernels.cuh: run_entry): its one
// field, which the C ABI passes as a bare pointer.  No time axis: t0 is ignored.
struct PointwiseFields {
  const float* field;
};
struct PointwiseBinding {
  using Op = AtlPointwiseOp;
  using Fields = PointwiseFields;
  static int check(const AtlPointwiseOp* op, const PointwiseFields* f, int64_t, int64_t) {
    ATL_REQUIRE(op && f->field, "NULL argument");
    return ATL_OK;
  }
  template <class F, class Visit>
  static void each_field(const AtlPointwiseOp*, F& f, Visit visit) {
    visit(f.field, 4);
  }
  template <class Run>
  static int with_phys(const AtlPointwiseOp* op, const PointwiseFields* f, int64_t, Run run) {
    return run([&](auto vec) { return make_phys<decltype(vec)::value>(op, f->field); });
  }
};

extern "C" {

int atl_pointwise_create(int device, const AtlPointwiseConfig* cfg, AtlPointwiseOp** op_out) {
  ATL_REQUIRE(cfg && op_out, "NULL argument");
  *op_out = nullptr;
  ATL_REQUIRE(cfg->ny > 0 && cfg->nx > 0, "bad grid");
  AtlPointwiseOp* op = new AtlPointwiseOp();
  op->device = device;
  ATL_REQUIRE(cfg->pitch == 0 || cfg->pitch >= cfg->nx, "pitch must be >= nx");
  op->grid = make_grid(cfg->ny, cfg->nx, cfg->pitch);
  op->shift = (float)cfg->shift;
  op->sink = (float)cfg->sink;
  op->c0 = (float)cfg->c0;
  op->c1 = (float)cfg->c1;
  op->c2 = (float)cfg->c2;
  op->nan_to_zero = cfg->nan_to_zero;
  op->poly = cfg->poly;
  if (cfg->cell_scale) {
    const size_t bytes = (size_t)op->grid.S_out * sizeof(float);
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc((void**)&op->d_scale, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(op->d_scale, cfg->cell_scale, bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      atl_pointwise_destroy(op);
      return cuda_fail(e, "atl_pointwise_create");
    }
  }
  *op_out = op;
  return ATL_OK;
}

void atl_pointwise_destroy(AtlPointwiseOp* op) {
  if (!op) return;
  if (op->d_scale) {
    cudaSetDevice(op->device);
    cudaFree(op->d_scale);
  }
  delete op;
}

int atl_pointwise_op_info(const AtlPointwiseOp* op, int32_t* device, int32_t* ny, int32_t* nx) {
  return op_info(op, device, ny, nx);
}

int atl_pointwise_reduce(const AtlPointwiseOp* op, const AtlPlan* plan, const float* field_dev,
                         int64_t nt, float* out_dev, void* stream) {
  const PointwiseFields f{field_dev};
  return run_entry<PointwiseBinding>(Entry::kReduce, op, plan, &f, 0, nt, out_dev, nullptr, stream);
}

int atl_pointwise_cells(const AtlPointwiseOp* op, const float* field_dev, int64_t nt,
                        float* out_dev, void* stream) {
  const PointwiseFields f{field_dev};
  return run_entry<PointwiseBinding>(Entry::kCells, op, nullptr, &f, 0, nt, out_dev, nullptr, stream);
}

int atl_pointwise_timesum(const AtlPointwiseOp* op, const float* field_dev, int64_t nt,
                          float* out_dev, float* count_dev, void* stream) {
  const PointwiseFields f{field_dev};
  return run_entry<PointwiseBinding>(Entry::kTimesum, op, nullptr, &f, 0, nt, out_dev, count_dev, stream);
}

int atl_pointwise_reduce_host(const AtlPointwiseOp* op, const AtlPlan* plan,
                              const float* field_host, int64_t nt, float* out_host,
                              int64_t chunk_steps) {
  const PointwiseFields f{field_host};
  return run_reduce_host<PointwiseBinding>(op, plan, &f, 0, nt, out_host, chunk_steps);
}

}  // extern "C"

/*
 * atlite_b200.h -- C ABI of libatlite_b200.so
 *
 * B200-native (sm_100a) replacement for the conversion-and-aggregation hot
 * path of PyPSA/atlite.  Plain C: pointers, sizes, opaque handles; no torch
 * or C++ types cross this boundary.  The reference is pure Python, so the
 * "FFI a maintainer would bind" is a ctypes stub (see INTEGRATION.md); the
 * entry points below are cut exactly where the reference hands work to
 * NumPy/dask/scipy:
 *
 *   reference (paths relative to /root/reference/atlite/)      entry point
 *   ---------------------------------------------------------  ------------------------
 *   aggregate.py:16-35  aggregate_matrix (dense x CSR^T)        atl_plan_create + *_reduce, atl_spmm
 *   convert.py:840-854  convert_pv  (+ pv/*.py)                 atl_pv_create, atl_pv_reduce/cells/timesum
 *   convert.py:634-662  convert_wind (+ wind.py:24-128)         atl_wind_create, atl_wind_*
 *   convert.py:405-418  convert_heat_demand                     atl_heat_create, atl_heat_*
 *   convert.py:475-491  convert_cooling_demand                  atl_heat_* with AtlHeatConfig.cooling = 1
 *   convert.py:748-767  convert_irradiation                     atl_pv_* with AtlPvConfig.output = ATL_OUT_TOTAL..GROUND
 *   convert.py:550-573  convert_solar_thermal                   atl_pv_* with AtlPvConfig.output = ATL_OUT_SOLAR_THERMAL
 *   convert.py:292-366  temperature / soil / dewpoint / COP     atl_pointwise_*
 *   convert.py:1028-1034 convert_runoff                         atl_pointwise_* with cell_scale = height
 *   convert.py:940-972  convert_csp (+ csp.py:18-58)            atl_csp_*
 *   convert.py:200-211  no-matrix branch (_aggregate_time)      *_cells, *_timesum
 *   convert.py:257-271  reduce + time aggregation               *_reduce (+ host finalisation in Python)
 *
 * Conventions
 *   - All weather fields are C-contiguous (time, y, x) float32 slabs, x fastest
 *     (the cutout's NetCDF layout; SURVEY.md section 8).  A "slab" covers time
 *     steps [t0, t0+nt) of the operator's time axis and its pointers address
 *     the slab's first step.
 *   - `pitch` (0 = nx): elements per stored row of the DEVICE input fields.  A
 *     device-resident cutout whose width is not a multiple of 4 may be stored
 *     row-padded (pitch = round_up(nx, 4), padding contents arbitrary) so that
 *     the 128-bit kernels apply; operator and plan must be created with the same
 *     pitch.  Host entry points (*_reduce_host) always take unpadded arrays
 *     (pitch = nx operators; a padded one is refused with ATL_ERR_INVALID);
 *     per-cell OUTPUTS are never padded.
 *   - Pointers named *_dev are device pointers on the operator's device, those
 *     named *_host are host pointers.  Small tables (coordinates, time axis,
 *     power curve) are always host pointers and are copied at create time.
 *   - The aggregated output is (nt, n_bus) float32, time-major -- the dim
 *     order of the reference's dask branch (aggregate.py:24-32) -- and is
 *     OVERWRITTEN (zero-filled, then accumulated) by each *_reduce call.
 *   - Every function returns ATL_OK (0) or a negative error code;
 *     atl_last_error() returns a thread-local message.  Nothing here falls
 *     back to a CPU implementation: without a CUDA device every compute entry
 *     point fails with ATL_ERR_CUDA.
 *   - stream: a cudaStream_t passed as void* (NULL = default stream).  Calls
 *     are asynchronous w.r.t. the host unless stated otherwise.
 */
#ifndef ATLITE_B200_H
#define ATLITE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ATL_OK 0
#define ATL_ERR_INVALID (-1) /* bad argument / unsupported combination */
#define ATL_ERR_CUDA (-2)    /* CUDA runtime error (see atl_last_error) */
#define ATL_ERR_NOMEM (-3)

#define ATL_ABI_VERSION 4

int atl_abi_version(void);
const char* atl_last_error(void);
int atl_device_count(int* count_out);
/* Host-only: 128-bit content hash of a byte range (MurmurHash3-style mixing, ~5 GB/s).  The
 * Python layer keys its plan cache on it: the reference rebuilds nothing per call, here a
 * matrix that is already planned must be recognised faster than it could be re-planned
 * (convert.py:213-249 hands over a fresh scipy matrix every call). */
int atl_hash128(const void* data, int64_t nbytes, uint64_t seed, uint64_t out[2]);
/* Deterministic reduce mode (default off, or env ATL_DETERMINISTIC=1): the fused
 * kernels accumulate every (tile, bus) partial in a private slot and a second
 * kernel sums each bus's slots in a fixed order -> bitwise-repeatable results at
 * ~2 % extra traffic.  Returns the previous setting. */
int atl_set_deterministic(int on);
/* Which fused kernel serves the *_reduce entry points (default 0, or env ATL_VARIANT / ATL_TB):
 * 0 = each operator's measured best, 1 = shuffle reduce against dense per-slot weight vectors,
 * 2 = staged reduce over the per-slot entry lists (8-step chunks), 3 = the same with 16-step
 * chunks; tb = time steps per thread block (0 = automatic).  Results are the same up to
 * float32 summation order. */
int atl_set_tuning(int variant, int tb);
/* CPUs the kernel lists as local to the GPU's PCI device (its NUMA node): host-streaming
 * calls bind their staging threads there for the duration of the call (ATL_NUMA_BIND=0
 * disables).  Fills up to `capacity` CPU ids, *n_out = how many there are (0 = unknown). */
int atl_device_local_cpus(int device, int32_t* cpus_out, int32_t capacity, int32_t* n_out);

/* ------------------------------------------------------------------ */
/* Aggregation plan: the (n_bus x S) CSR indicator/layout matrix       */
/* (convert.py:213-254) pre-tiled for the fused reduce kernels.        */
/* ------------------------------------------------------------------ */
typedef struct AtlPlan AtlPlan;

typedef struct {
  int32_t ny, nx, n_bus;
  int64_t nnz;            /* stored entries after merging duplicates   */
  int32_t n_tiles;        /* 32x4-cell warp tiles covering the grid     */
  int32_t n_active_tiles; /* tiles touched by at least one entry        */
  int64_t n_slots;        /* distinct (tile, bus) pairs                 */
  double slots_per_active_tile;
  int32_t fused;          /* 1: fused tile path, 0: two-pass CSR fallback */
  int32_t pitch;          /* row pitch of the input fields (elements), >= nx */
  int32_t vec;            /* 1: 128-bit lane layout (pitch % 4 == 0), 0: scalar */
  int64_t n_pairs;        /* stored (slot, cell) entries the staged reduce walks     */
} AtlPlanInfo;

/* indptr/indices/data: host CSR arrays (scipy layout), column index
 * s = iy*nx + ix (cutout.grid order, cutout.py:355-376). */
int atl_plan_create(int device, int32_t ny, int32_t nx, int32_t n_bus,
                    const int64_t* indptr_host, const int32_t* indices_host,
                    const double* data_host, AtlPlan** plan_out);
int atl_plan_create_pitched(int device, int32_t ny, int32_t nx, int32_t pitch, int32_t n_bus,
                            const int64_t* indptr_host, const int32_t* indices_host,
                            const double* data_host, AtlPlan** plan_out);
int atl_plan_info(const AtlPlan* plan, AtlPlanInfo* info_out);
/* Host-only view of the tiling (no CUDA needed; used by the CPU tests and for
 * inspection): fills *info_out; when the three output arrays are given
 * (slot_capacity >= n_slots) also tile_slot_ptr[n_tiles+1], slot_row[n_slots] and
 * slot_w[n_slots*128] (weights in lane order; VEC layout iff nx % 4 == 0:
 * cell (iy, ix) of a tile sits at ((iy%4)*8 + (ix%32)/4)*4 + ix%4, else at
 * (ix%32)*4 + iy%4). */
int atl_plan_tiling_host(int32_t ny, int32_t nx, int32_t n_bus, const int64_t* indptr_host,
                         const int32_t* indices_host, const double* data_host,
                         AtlPlanInfo* info_out, int32_t* tile_slot_ptr_out,
                         int32_t* slot_row_out, float* slot_w_out, int64_t slot_capacity);
/* Host-only view of the entry lists the staged reduce kernel walks (CPU tests): for slot s
 * (same numbering as atl_plan_tiling_host) the entries slot_pair_ptr[s] .. slot_pair_ptr[s+1],
 * each {pair_cell = position 32*i + lane of the cell in the warp's staging row, pair_w}.
 * Duplicates of one (bus, cell) are summed, explicit zeros kept (scipy CSR semantics:
 * aggregate.py:25 multiplies exactly the stored entries).  Always fills *n_pairs_out; the
 * arrays only when all three are given. */
int atl_plan_pairs_host(int32_t ny, int32_t nx, int32_t n_bus, const int64_t* indptr_host,
                        const int32_t* indices_host, const double* data_host,
                        int64_t* n_pairs_out, int32_t* slot_pair_ptr_out, int32_t* pair_cell_out,
                        float* pair_w_out, int64_t slot_capacity, int64_t pair_capacity);
void atl_plan_destroy(AtlPlan* plan);

/* Generic (time, S) dense  x  CSR^T  ->  (time, n_bus)  (aggregate.py:24-32):
 * the path for unknown convert_func results. */
int atl_spmm(const AtlPlan* plan, const float* dense_dev, int64_t nt,
             float* out_dev, void* stream);

/* ------------------------------------------------------------------ */
/* Cutout ingest: parallel decode of compressed (time, y, x) chunks      */
/* (the storage format of data.py:139,245-248: zlib + byte shuffle; the  */
/* read path of cutout.py:142-154)                                       */
/* ------------------------------------------------------------------ */
typedef struct {
  int32_t ny, nx;       /* grid of the variable                                   */
  int32_t elem_bytes;   /* 2, 4 or 8                                              */
  int32_t shuffle;      /* 1: HDF5 byte-shuffle filter was applied before deflate */
  int32_t deflate;      /* 1: chunks are zlib streams; 0: stored raw              */
  int64_t chunk[3];     /* chunk shape (time, y, x); edge chunks are stored whole */
} AtlChunkSpec;
/* Decode the listed chunks of one variable into dst_host, a C-contiguous (nt, ny, nx) slab
 * holding steps [t0, t0 + nt): every chunk is pread from `path` at file_offset[c]
 * (stored_bytes[c] bytes), inflated, un-shuffled and its part inside the slab copied to its
 * place; chunk_origin[3c..3c+2] = (t, y, x) of the chunk's first element.  Chunks run in
 * parallel on n_threads host threads (0 = all cores, at most 64).  Bytes are copied as
 * stored (the caller converts endianness / packing).  No GPU involved. */
int atl_decode_chunks(const char* path, const AtlChunkSpec* spec, int64_t n_chunks,
                      const int64_t* file_offset, const int64_t* stored_bytes,
                      const int64_t* chunk_origin, int64_t t0, int64_t nt, void* dst_host,
                      int32_t n_threads);

/* ------------------------------------------------------------------ */
/* PV: SolarPosition -> SurfaceOrientation -> TiltedIrradiation ->     */
/* SolarPanelModel (convert.py:840-854)                                */
/* ------------------------------------------------------------------ */
enum { ATL_TRACK_NONE = 0, ATL_TRACK_HORIZONTAL = 1, ATL_TRACK_TILTED_HORIZONTAL = 2,
       ATL_TRACK_VERTICAL = 3, ATL_TRACK_DUAL = 4 };       /* pv/orientation.py:114-176 */
enum { ATL_TRIGON_SIMPLE = 0, ATL_TRIGON_HAY_DAVIES = 1 };  /* pv/irradiation.py:214-236 */
enum { ATL_CLEARSKY_SIMPLE = 0, ATL_CLEARSKY_ENHANCED = 1 };/* pv/irradiation.py:33-65  */
enum { ATL_IRR_DIRECT_DIFFUSE = 0, ATL_IRR_INFLUX = 1 };    /* pv/irradiation.py:202-208 */
enum { ATL_ALBEDO_VAR = 0, ATL_ALBEDO_OUTFLUX = 1 };        /* pv/irradiation.py:128-139 */
enum { ATL_SOLAR_COMPUTED = 0, ATL_SOLAR_STORED_F32 = 1, ATL_SOLAR_STORED_F64 = 2 }; /* pv/solar_position.py:54-60 vs 69-116 */
enum { ATL_PANEL_HULD = 0, ATL_PANEL_BOFINGER = 1 };        /* pv/solar_panel_model.py:12-74 */
/* what the PV operator emits: panel power (convert_pv), one tilted-irradiation
 * component (convert_irradiation, pv/irradiation.py:238-245), or solar-thermal
 * collector output (convert_solar_thermal, convert.py:565-573) */
enum { ATL_OUT_PANEL = 0, ATL_OUT_TOTAL = 1, ATL_OUT_DIRECT = 2, ATL_OUT_DIFFUSE = 3,
       ATL_OUT_GROUND = 4, ATL_OUT_SOLAR_THERMAL = 5 };

typedef struct {
  int32_t ny, nx;
  int64_t nt;                 /* length of the time axis                        */
  const int64_t* time_ns;     /* host, nt: datetime64[ns] UTC                   */
  int64_t time_shift_ns;      /* SolarPosition(time_shift=...), default 0       */
  const double* lon_deg;      /* host, nx   (ds["lon"])                          */
  const double* lat_deg;      /* host, ny   (ds["lat"])                          */
  const double* slope_rad;    /* host, ny (ny*nx if orientation_2d)  orientation(lon,lat,sp)["slope"]   */
  const double* azimuth_rad;  /* host, ny (ny*nx if orientation_2d)  orientation(...)["azimuth"]        */
  int32_t tracking, trigon_model, clearsky_model, irr_branch, albedo_src,
      solar_src, panel_model;
  double altitude_threshold_deg; /* pv/irradiation.py:155, default 1.0         */
  /* Huld: c_temp_amb, c_temp_irrad, r_tmod, r_irradiance, k_1..k_6, inverter_efficiency
   * Bofinger: A, B, C, D, NOCT, Tamb, Intc, Tstd, ta, threshold, inverter_efficiency */
  double panel[16];
  int32_t output;             /* ATL_OUT_*; panel[] is ignored unless ATL_OUT_PANEL */
  double thermal[3];          /* ATL_OUT_SOLAR_THERMAL: c0, c1, t_store in deg C  */
  int32_t pitch;              /* row pitch of the device fields, 0 = nx            */
  int32_t orientation_2d;     /* 1: slope_rad / azimuth_rad vary per cell, (ny, nx) row-major:
                                 an orientation callback (pv/orientation.py:107) that returns
                                 (y, x) arrays */
} AtlPvConfig;

typedef struct { /* device pointers to (nt_slab, ny, nx) slabs; unused = NULL */
  const float* influx_toa;
  const float* influx_direct;
  const float* influx_diffuse;
  const float* influx;
  const float* albedo;
  const float* outflux;
  const float* temperature;
  const float* humidity;
  const void* solar_altitude; /* float or double per solar_src */
  const void* solar_azimuth;
} AtlPvFields;

typedef struct AtlPvOp AtlPvOp;
int atl_pv_create(int device, const AtlPvConfig* cfg, AtlPvOp** op_out);
void atl_pv_destroy(AtlPvOp* op);
/* fused convert + aggregate of slab [t0, t0+nt): out_dev (nt, n_bus) */
int atl_pv_reduce(const AtlPvOp* op, const AtlPlan* plan, const AtlPvFields* f,
                  int64_t t0, int64_t nt, float* out_dev, void* stream);
/* per-cell result (aggregate_time=None, no matrix): out_dev (nt, ny, nx) */
int atl_pv_cells(const AtlPvOp* op, const AtlPvFields* f, int64_t t0, int64_t nt,
                 float* out_dev, void* stream);
/* per-cell NaN-skipping time sum, ACCUMULATED into out_dev (ny, nx) (caller zero-fills);
 * count_dev (ny, nx, may be NULL) accumulates the number of non-NaN steps per cell: the
 * reference's `da.mean("time")` divides by it (convert.py:51-56).  Same for every *_timesum. */
int atl_pv_timesum(const AtlPvOp* op, const AtlPvFields* f, int64_t t0, int64_t nt,
                   float* out_dev, float* count_dev, void* stream);

/* ------------------------------------------------------------------ */
/* Wind: extrapolate_wind_speed + np.interp power curve                */
/* (wind.py:24-128, convert.py:634-662)                                */
/* ------------------------------------------------------------------ */
enum { ATL_WIND_NONE = 0 /* wnd{hub}m present, wind.py:75-78 */,
       ATL_WIND_LOG = 1 /* wind.py:91-102 */, ATL_WIND_POWER = 2 /* wind.py:103-112 */ };

typedef struct {
  int32_t ny, nx;
  int32_t method;
  double from_height, to_height;
  int32_t n_knots;         /* <= 255 */
  const double* V;         /* host, n_knots, non-decreasing (resource.py:346-355) */
  const double* POW_norm;  /* host, n_knots: POW / P  (convert.py:649)            */
  int32_t pitch;           /* row pitch of the device fields, 0 = nx              */
} AtlWindConfig;

typedef struct {
  const float* wnd; /* wnd{from}m, (nt, ny, nx)                           */
  const float* aux; /* roughness (LOG) or wnd_shear_exp (POWER) or NULL   */
} AtlWindFields;

typedef struct AtlWindOp AtlWindOp;
int atl_wind_create(int device, const AtlWindConfig* cfg, AtlWindOp** op_out);
void atl_wind_destroy(AtlWindOp* op);
int atl_wind_reduce(const AtlWindOp* op, const AtlPlan* plan, const AtlWindFields* f,
                    int64_t nt, float* out_dev, void* stream);
int atl_wind_cells(const AtlWindOp* op, const AtlWindFields* f, int64_t nt,
                   float* out_dev, void* stream);
int atl_wind_timesum(const AtlWindOp* op, const AtlWindFields* f, int64_t nt,
                     float* out_dev, float* count_dev, void* stream);

/* ------------------------------------------------------------------ */
/* Heat demand: daily mean temperature -> degree days                  */
/* (convert.py:405-418)                                                */
/* ------------------------------------------------------------------ */
typedef struct {
  int32_t ny, nx;
  double threshold_c, a, constant; /* convert.py:413-418 (threshold in deg C) */
  int32_t cooling;                 /* 1: a * (Tmean - threshold), convert.py:475-491 */
  int32_t pitch;                   /* row pitch of the device field, 0 = nx            */
} AtlHeatConfig;

typedef struct AtlHeatOp AtlHeatOp;
int atl_heat_create(int device, const AtlHeatConfig* cfg, AtlHeatOp** op_out);
void atl_heat_destroy(AtlHeatOp* op);
/* day_start_host: n_days+1 offsets into the slab's time steps (calendar-day
 * bins of time+hour_shift, convert.py:408-412); out_dev (n_days, n_bus). */
int atl_heat_reduce(const AtlHeatOp* op, const AtlPlan* plan, const float* temperature_dev,
                    const int64_t* day_start_host, int64_t n_days, float* out_dev,
                    void* stream);
int atl_heat_cells(const AtlHeatOp* op, const float* temperature_dev,
                   const int64_t* day_start_host, int64_t n_days, float* out_dev,
                   void* stream);
int atl_heat_timesum(const AtlHeatOp* op, const float* temperature_dev,
                     const int64_t* day_start_host, int64_t n_days, float* out_dev,
                     float* count_dev, void* stream);

/* ------------------------------------------------------------------ */
/* Pointwise conversions of ONE (time, y, x) field:                    */
/*   y = x + shift;  nan_to_zero: y = 0 where NaN;                     */
/*   poly: d = sink - y, out = c0 + c1 d + c2 d^2  else out = y;       */
/*   out *= cell_scale[y, x] (optional static (ny, nx) field)          */
/* temperature / dewpoint (shift = -273.15), soil temperature          */
/* (+ nan_to_zero), coefficient_of_performance (poly), runoff          */
/* (cell_scale = height): convert.py:292-366, 1028-1034.               */
/* ------------------------------------------------------------------ */
typedef struct {
  int32_t ny, nx;
  double shift;
  int32_t nan_to_zero;
  int32_t poly;
  double sink, c0, c1, c2;
  const float* cell_scale; /* host, ny*nx (unpadded), or NULL */
  int32_t pitch;           /* row pitch of the device field, 0 = nx */
} AtlPointwiseConfig;

typedef struct AtlPointwiseOp AtlPointwiseOp;
int atl_pointwise_create(int device, const AtlPointwiseConfig* cfg, AtlPointwiseOp** op_out);
void atl_pointwise_destroy(AtlPointwiseOp* op);
int atl_pointwise_reduce(const AtlPointwiseOp* op, const AtlPlan* plan, const float* field_dev,
                         int64_t nt, float* out_dev, void* stream);
int atl_pointwise_cells(const AtlPointwiseOp* op, const float* field_dev, int64_t nt,
                        float* out_dev, void* stream);
int atl_pointwise_timesum(const AtlPointwiseOp* op, const float* field_dev, int64_t nt,
                          float* out_dev, float* count_dev, void* stream);
int atl_pointwise_reduce_host(const AtlPointwiseOp* op, const AtlPlan* plan,
                              const float* field_host, int64_t nt, float* out_host,
                              int64_t chunk_steps);

/* ------------------------------------------------------------------ */
/* CSP: solar position -> direct irradiation (horizontal | DNI) x        */
/* efficiency(altitude, azimuth) table (convert.py:940-972, csp.py)     */
/* ------------------------------------------------------------------ */
enum { ATL_CSP_PARABOLIC_TROUGH = 0, ATL_CSP_SOLAR_TOWER = 1 };
typedef struct {
  int32_t ny, nx;
  int64_t nt;
  const int64_t* time_ns;      /* host, nt (needed unless the solar position is stored) */
  int64_t time_shift_ns;
  const double* lon_deg;       /* host, nx */
  const double* lat_deg;       /* host, ny */
  int32_t solar_src;           /* ATL_SOLAR_* */
  int32_t technology;          /* ATL_CSP_* */
  double r_irradiance;         /* W/m^2 */
  double dni_altitude_threshold_deg; /* csp.py:18, default 3.75 */
  int32_t n_alt, n_az;         /* efficiency table, each 2..128, product <= 8192 */
  const double* altitude_rad;  /* host, n_alt, increasing */
  const double* azimuth_rad;   /* host, n_az, increasing */
  const double* efficiency;    /* host, n_alt * n_az row-major, p.u. */
  int32_t pitch;               /* row pitch of the device fields, 0 = nx */
} AtlCspConfig;

typedef struct {
  const float* influx_direct;
  const void* solar_altitude; /* float or double per solar_src, or NULL */
  const void* solar_azimuth;
} AtlCspFields;

typedef struct AtlCspOp AtlCspOp;
int atl_csp_create(int device, const AtlCspConfig* cfg, AtlCspOp** op_out);
void atl_csp_destroy(AtlCspOp* op);
int atl_csp_reduce(const AtlCspOp* op, const AtlPlan* plan, const AtlCspFields* f, int64_t t0,
                   int64_t nt, float* out_dev, void* stream);
int atl_csp_cells(const AtlCspOp* op, const AtlCspFields* f, int64_t t0, int64_t nt,
                  float* out_dev, void* stream);
int atl_csp_timesum(const AtlCspOp* op, const AtlCspFields* f, int64_t t0, int64_t nt,
                    float* out_dev, float* count_dev, void* stream);
int atl_csp_reduce_host(const AtlCspOp* op, const AtlPlan* plan, const AtlCspFields* f_host,
                        int64_t t0, int64_t nt, float* out_host, int64_t chunk_steps);

/* ------------------------------------------------------------------ */
/* Host-buffer entry points: the call the reference-facing Python API  */
/* makes when the cutout lives in host memory (NumPy / NetCDF).  The   */
/* library streams time slabs through a pinned ring (H2D overlapped    */
/* with the kernels) and returns the (nt, n_bus) result in host memory.*/
/* Synchronous.  chunk_steps <= 0 picks a default.                     */
/* ------------------------------------------------------------------ */
int atl_pv_reduce_host(const AtlPvOp* op, const AtlPlan* plan, const AtlPvFields* f_host,
                       int64_t t0, int64_t nt, float* out_host, int64_t chunk_steps);
int atl_wind_reduce_host(const AtlWindOp* op, const AtlPlan* plan,
                         const AtlWindFields* f_host, int64_t nt, float* out_host,
                         int64_t chunk_steps);
int atl_heat_reduce_host(const AtlHeatOp* op, const AtlPlan* plan,
                         const float* temperature_host, const int64_t* day_start_host,
                         int64_t n_days, float* out_host, int64_t chunk_days);

/* Introspection of operator handles (device, grid). */
int atl_pv_op_info(const AtlPvOp* op, int32_t* device, int32_t* ny, int32_t* nx,
                   int32_t* solar_src);
/* Host-only: evaluates the power-curve interpolation exactly as the kernels do
 * (same tables, same fp32 formula), no CUDA needed; the CPU tests compare it with
 * np.interp.  force_mode: -1 = the table atl_wind_create would pick, 0 = binary
 * search, 1 = general bucket LUT, 2 = lattice LUT (knots on a uniform lattice) with the
 * steps added back by compares, 3 = saturating lattice LUT (256 rows, steps folded into
 * the table, no clamps; what -1 picks when the curve qualifies);
 * *mode_out (optional) = the table actually built (a forced LUT mode the curve does
 * not qualify for falls back to 0). */
int atl_wind_curve_eval_host(const double* V, const double* POW_norm, int32_t n_knots,
                             int32_t force_mode, const float* x, int64_t n, float* y_out,
                             int32_t* mode_out);
/* Host-only: which table a power curve gets.  info[0] = table (0 binary search, 1 general
 * LUT, 2 lattice LUT, 3 saturating lattice LUT), info[1] = steps the kernel adds back by compares (0 when the curve has
 * none or they are folded into the lattice table), info[2] = steps in the curve (duplicate
 * knots with different powers), info[3] = bytes staged to shared memory. */
int atl_wind_curve_info_host(const double* V, const double* POW_norm, int32_t n_knots,
                             int32_t force_mode, int32_t info[4]);
int atl_wind_op_info(const AtlWindOp* op, int32_t* device, int32_t* ny, int32_t* nx);
int atl_heat_op_info(const AtlHeatOp* op, int32_t* device, int32_t* ny, int32_t* nx);
int atl_pointwise_op_info(const AtlPointwiseOp* op, int32_t* device, int32_t* ny, int32_t* nx);
int atl_csp_op_info(const AtlCspOp* op, int32_t* device, int32_t* ny, int32_t* nx,
                    int32_t* solar_src);

/* Number of kernel launches issued by this library since load (bench.py's
 * "gpu_launches" evidence). */
int64_t atl_launch_count(void);
/* The atl_*_reduce_host calls keep their pinned staging buffers (used for pageable
 * inputs) for the next call; this frees them. */
void atl_release_host_staging(void);

/* ------------------------------------------------------------------ */
/* Indicator matrix: shapes -> CSR (n_shapes, ny*nx) of covered cell   */
/* fractions (cutout.py:492-515 -> gis.py:104-145 on the regular grid  */
/* of cutout.py:355-376).  SURVEY section 8 f1.                        */
/* ------------------------------------------------------------------ */
typedef struct AtlIndicator AtlIndicator;
/* Grid: cell (iy, ix) is the box of half-width (dx/2, dy/2) about (x0 + ix*dx,
 * y0 + iy*dy); dx, dy > 0.  Shapes: shape s owns rings
 * shape_ring_ptr[s] .. shape_ring_ptr[s+1]-1; ring r owns the vertices
 * ring_ptr[r] .. ring_ptr[r+1]-1 of xy (x, y interleaved, float64, same CRS as the
 * grid; the closing vertex may be repeated or not); ring_is_hole[r] != 0 marks an
 * interior ring.  Ring orientation is free.  All pointers are HOST pointers; the
 * areas are computed on `device`.  Entries are kept when the covered fraction
 * exceeds 1e-10; columns are sorted (iy*nx + ix). */
int atl_indicator_compute(int device, int32_t ny, int32_t nx, double x0, double dx, double y0,
                          double dy, int32_t n_shapes, const int64_t* shape_ring_ptr,
                          const int64_t* ring_ptr, const int8_t* ring_is_hole, const double* xy,
                          AtlIndicator** out);
int atl_indicator_nnz(const AtlIndicator* ind, int64_t* nnz_out);
/* indptr_out[n_shapes+1], indices_out[nnz], data_out[nnz] (host, caller-owned) */
int atl_indicator_export(const AtlIndicator* ind, int64_t* indptr_out, int32_t* indices_out,
                         double* data_out);
void atl_indicator_destroy(AtlIndicator* ind);

/* ------------------------------------------------------------------ */
/* ERA5 prepare-time derivations (datasets/era5.py:120-201), SURVEY    */
/* section 8 f4.  All field pointers are DEVICE pointers to n float32  */
/* values (any shape); outputs may not alias inputs.                   */
/* ------------------------------------------------------------------ */
/* get_data_wind (era5.py:120-135) [+ sanitize_wind :141-146 if sanitize != 0]:
 * wnd100m = |(u100, v100)|, wnd_shear_exp = ln(|(u10, v10)| / wnd100m) / ln(10/100),
 * wnd_azimuth = atan2(u100, v100) mapped to [0, 2 pi), roughness = fsr (< 0 -> 2e-4). */
int atl_era5_wind(int device, int64_t n, const float* u100, const float* v100, const float* u10,
                  const float* v10, const float* fsr, int32_t sanitize, float* wnd100m,
                  float* wnd_shear_exp, float* wnd_azimuth, float* roughness, void* stream);
/* get_data_influx (era5.py:163-175) [+ sanitize_influx :195-201]: albedo =
 * ((ssrd - ssr) / ssrd, 0 where ssrd == 0 or NaN), influx_diffuse = ssrd - fdir, and
 * influx_{toa, direct, diffuse} converted J m-2 -> W m-2 (/ 3600) [clipped at 0]. */
int atl_era5_influx(int device, int64_t n, const float* ssrd, const float* ssr, const float* tisr,
                    const float* fdir, int32_t sanitize, float* influx_toa, float* influx_direct,
                    float* influx_diffuse, float* albedo, void* stream);
/* SolarPosition (pv/solar_position.py:69-116) materialised as the cutout variables
 * solar_altitude / solar_azimuth (era5.py:182-188 uses time_shift = -30 min):
 * (nt, ny, nx) float64 each, device; time / lon / lat are host arrays. */
int atl_solar_position(int device, const int64_t* time_ns_host, int64_t nt, int64_t time_shift_ns,
                       const double* lon_deg_host, int32_t nx, const double* lat_deg_host, int32_t ny,
                       double* altitude_dev, double* azimuth_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ATLITE_B200_H */

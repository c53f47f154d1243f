/*
 * geokernels.h -- C ABI of libgeokernels.so: the sm_100a implementation of
 * dask-geomodeling's per-tile raster compute path.
 *
 * The reference (nens/dask-geomodeling) is pure Python and has no FFI of its
 * own; every entry point below therefore cites the reference *Python function*
 * it replaces (paths relative to the reference checkout, file:line).  The
 * Python blocks in dask_geomodeling_b200/ bind these symbols with ctypes (see
 * INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure;
 *     gm_last_error() returns a thread-local message for the last failure.
 *   - rasters are C-contiguous (bands, height, width), row 0 = north.
 *   - `space` says where `data` lives: host memory (the library stages it
 *     through device buffers, copies included in the call) or device memory
 *     (no copies; the call only enqueues kernels on `stream`).
 *   - `stream` is a cudaStream_t passed as void*; NULL = the library stream.
 *   - no torch / Python types anywhere in the signatures.
 */
#ifndef GEOKERNELS_H
#define GEOKERNELS_H

#include <stdint.h>
#include "gm_bytecode.h"

#ifdef __cplusplus
extern "C" {
#endif

#define GM_ABI_VERSION 1

/* ---- dtypes (storage) ---------------------------------------------------- */
enum GmDType {
  GM_BOOL = 0, GM_U8 = 1, GM_I8 = 2, GM_U16 = 3, GM_I16 = 4,
  GM_U32 = 5, GM_I32 = 6, GM_I64 = 7, GM_F32 = 8, GM_F64 = 9
};

enum GmSpace { GM_HOST = 0, GM_DEVICE = 1 };

typedef struct GmArray {
  void*   data;      /* host or device pointer, 16-byte aligned            */
  int32_t dtype;     /* GmDType                                            */
  int32_t space;     /* GmSpace                                            */
  int64_t shape[3];  /* (bands, height, width)                             */
} GmArray;

/* ---- fused element-wise evaluator ----------------------------------------
 * The instruction set (GmClass, GmOp, GmReduce, GmSrcKind, GmFlags, GmTableKind)
 * is in gm_bytecode.h.
 */
#define GM_NREG       4
#define GM_MAX_INSTR  40
#define GM_MAX_INPUTS 8
#define GM_MAX_OUTPUTS 4
#define GM_MAX_TABLES 2

typedef struct GmInstr {
  uint8_t  op;        /* GmOp                                               */
  uint8_t  cls;       /* class the operation computes / compares in         */
  uint8_t  cls_a;     /* class of acc on entry                              */
  uint8_t  cls_b;     /* class of b as materialised                         */
  uint8_t  cls_out;   /* class of acc on exit                               */
  uint8_t  src_kind;  /* GmSrcKind                                          */
  uint8_t  src;       /* register / input index                             */
  uint8_t  flags;     /* GmFlags                                            */
  uint32_t aux;       /* register (ST), output (OUT) or table index         */
  uint32_t reserved;
  uint64_t k[6];      /* constants, raw bits; meaning depends on op:
                         k0 immediate b / threshold / location / mask value
                         k1 sentinel of acc   k2 sentinel of b
                         k3 fill of the result  k4 isclose tolerance / right
                         k5 spare                                           */
} GmInstr;

typedef struct GmTable {
  const void* keys;   /* host ptr: n sorted keys (int64 or float64 bits)    */
  const void* vals;   /* host ptr: n 8-byte values (Reclassify) or NULL     */
  const uint8_t* hit; /* host ptr: dense tables, 1 where the key is mapped,
                         2 where it is mapped onto the fill value           */
  int64_t base;       /* dense tables: key of entry 0                       */
  int32_t n;
  int32_t kind;       /* GmTableKind                                        */
} GmTable;

typedef struct GmProgram {
  int32_t n_instr;
  int32_t n_inputs;
  int32_t n_outputs;
  int32_t word;       /* 4: every class is 32-bit; 8: 64-bit slots          */
  int32_t n_tables;
  int32_t reserved;
  GmInstr instr[GM_MAX_INSTR];
  GmTable tables[GM_MAX_TABLES];
} GmProgram;

/* runtime ------------------------------------------------------------------ */
int  gm_abi_version(void);
int  gm_init(int device);                 /* idempotent; selects the device  */
int  gm_shutdown(void);
const char* gm_last_error(void);
int  gm_device_info(int* sm_count, int64_t* total_mem, int* cc_major, int* cc_minor);
int64_t gm_launch_count(void);            /* kernels launched by this lib    */
void* gm_default_stream(void);
int  gm_stream_sync(void* stream);

int  gm_malloc(void** ptr, int64_t bytes, void* stream);   /* stream-ordered pool */
int  gm_free(void* ptr, void* stream);
int  gm_host_alloc(void** ptr, int64_t bytes);             /* pinned           */
int  gm_host_free(void* ptr);
int  gm_host_register(void* ptr, int64_t bytes);           /* pin user memory  */
int  gm_host_unregister(void* ptr);
int  gm_memcpy_h2d(void* dst, const void* src, int64_t bytes, void* stream);
int  gm_memcpy_d2h(void* dst, const void* src, int64_t bytes, void* stream);  /* syncs */
int  gm_memcpy_d2h_async(void* dst, const void* src, int64_t bytes, void* stream);  /* no sync */
int  gm_memcpy_d2d(void* dst, const void* src, int64_t bytes, void* stream);
/* extra streams for chunk pipelines (upload / evaluate / download of row chunks overlap) */
int  gm_stream_create(void** stream);
int  gm_stream_destroy(void* stream);
/* rectangle copy host->device: rows x row_bytes, pitches in bytes           */
int  gm_memcpy2d_h2d(void* dst, int64_t dpitch, const void* src, int64_t spitch,
                     int64_t row_bytes, int64_t rows, void* stream);
int  gm_fill(void* dst, int32_t dtype, const void* value, int64_t count, void* stream);

/* fused element-wise programs (replaces the `process` staticmethods of
 * raster/elemwise.py and raster/misc.py cited above)                        */
int  gm_eval_program(const GmProgram* prog, const GmArray* inputs,
                     GmArray* outputs, int64_t n_pixels, void* stream);

/* Evaluator back ends.  Both execute the same GmProgram with the same results:
 *   GM_EVAL_INTERPRET   one resident kernel interprets the bytecode (no compile);
 *   GM_EVAL_SPECIALISE  the bytecode is translated to a straight-line kernel,
 *                       compiled once for sm_100a with NVRTC and cached;
 *   GM_EVAL_AUTO        (default; env GM_EVAL=auto|interp|jit) specialise from
 *                       2^18 pixels on, interpret below.                      */
enum GmEvalMode { GM_EVAL_AUTO = 0, GM_EVAL_INTERPRET = 1, GM_EVAL_SPECIALISE = 2 };
int  gm_set_eval_mode(int mode);
int  gm_get_eval_mode(void);
/* inspection: generated CUDA source of a program / NVRTC compile check (neither
 * needs a GPU); number of kernels compiled so far                            */
int  gm_jit_source(const GmProgram* prog, const int32_t* in_dtype, const int32_t* out_dtype,
                   char* buffer, int64_t capacity, int64_t* length);
/* the same with the program's constants as literals: the kernel a program gets
 * when its constants repeat on large rasters (tools/jit_sass.py)              */
int  gm_jit_baked_source(const GmProgram* prog, const int32_t* in_dtype, const int32_t* out_dtype,
                         char* buffer, int64_t capacity, int64_t* length);
int  gm_jit_check(const GmProgram* prog, const int32_t* in_dtype, const int32_t* out_dtype,
                  int64_t* cubin_bytes);
int64_t gm_jit_compile_count(void);

/* reduce_rasters over stacks of any length (raster/reduction.py:38-119) and Place at any number of
 * coordinates (raster/spatial.py:657-731).  Each raster of a stack is reduced exactly as by a
 * GM_OP_OVERLAY step of kind `kind` (GmReduce) into an accumulator of class `acc_cls` that starts at
 * `init`; its has-data test is that of GM_OP_OVERLAY (utils.get_index: np.isclose for floats, ==
 * otherwise) on the stored value converted to class `cls`.  The result is stored in the output
 * dtype: for max / min / sum / product a NaN accumulator (no raster had data) becomes `fill`
 * (raw bits of the output's class), other values are converted; last / count store acc as it is.
 * 'first' is 'last' over the reversed stack.                                                      */
typedef struct GmStackInput {
  const void* data;    /* device pointer, n_pixels cells; any alignment                          */
  int32_t dtype;       /* GmDType of the storage                                                  */
  uint8_t cls;         /* GmClass the value is tested and reduced in                              */
  uint8_t flags;       /* GM_F_ND_T | GM_F_CLOSE | GM_F_ND_FINITE                                 */
  uint16_t reserved;
  uint64_t k2, k4;     /* sentinel, isclose tolerance: raw bits of class `cls`                    */
} GmStackInput;
/* one kernel launch whatever n_inputs is; `inputs` is a host array, `out` a device array        */
int  gm_reduce_stack(const GmStackInput* inputs, int64_t n_inputs, int kind, int acc_cls,
                     uint64_t init, uint64_t fill, GmArray* out, void* stream);
/* out[b, j, i] = reduction over copies c (in order) of src[b, j - dj_c, i - di_c]; a cell outside
 * the source or holding a non-finite float is `nodata` (src dtype), as gm_resample_nn makes it.
 * `offsets` = host (di_0, dj_0, di_1, dj_1, ...); `test` = has-data test of the source (its
 * data is ignored).  Work is proportional to the output tiles each copy meets.                  */
int  gm_place(const GmArray* src, GmArray* dst, const void* nodata, const int32_t* offsets,
              int64_t n_copies, const GmStackInput* test, int kind, int acc_cls, uint64_t init,
              uint64_t fill, void* stream);

/* The statistics of reduce_rasters that keep more than one value per pixel, over the same stacks:
 * the rasters are stacked in the working float dtype W (`work_bytes` = 2, 4 or 8: float16 / 32 /
 * 64), a slot holding the value converted to W where the has-data test holds and NaN elsewhere,
 * then reduced as NumPy's nan-functions reduce axis 0:
 *   mean:   sum in W in stack order, divided by the count in float64, rounded to W   (np.nanmean)
 *   var:    sum of W((x - mean)^2) in stack order, divided likewise; ddof 0          (np.nanvar)
 *   std:    sqrt(var) in W                                                            (np.nanstd)
 *   argmin / argmax: first index reaching the extreme, a NaN slot counting as +inf / -inf
 *                    (np.nanargmin / np.nanargmax), converted to the output dtype.
 * A pixel where every slot is NaN holds `fill` (raw bits of the output's class); other results,
 * NaN and inf included, are stored as they are.  mean / var / std need W == the output dtype. */
enum GmStackStat { GM_STACK_MEAN = 0, GM_STACK_VAR = 1, GM_STACK_STD = 2, GM_STACK_ARGMIN = 3,
                  GM_STACK_ARGMAX = 4 };
/* one kernel launch whatever n_inputs is (var and std read the stack twice within it)           */
int  gm_reduce_stack_stat(const GmStackInput* inputs, int64_t n_inputs, int stat, int work_bytes,
                          uint64_t fill, GmArray* out, void* stream);
/* gm_place with a GmStackStat.  A cell outside a copy's footprint is a NaN slot.  The stack holds
 * the copies that put at least one data cell (any band) inside `dst`, in order, so the index of
 * argmin / argmax is a copy's rank among those.                                                  */
int  gm_place_stat(const GmArray* src, GmArray* dst, const void* nodata, const int32_t* offsets,
                   int64_t n_copies, const GmStackInput* test, int stat, int work_bytes, uint64_t fill,
                   void* stream);

/* input adaptor: nearest-neighbour resample of a source window into the
 * request grid; equals the aligned crop/pad for aligned requests
 * (raster/sources.py:119-149, MemorySource).  src_i = floor(i0 + (i+0.5)*si)  */
int  gm_resample_nn(const GmArray* src, GmArray* dst, const void* nodata,
                    double col0, double col_step, double row0, double row_step,
                    void* stream);

/* input adaptor across projections: nearest-neighbour warp of a source window into a request
 * grid in another CRS (raster/sources.py:119-149, the reference's gdal.ReprojectImage).  Target
 * cell (i, j) takes the value of source cell (floor(row), floor(col)) where (col, row) =
 * ((x - src_geo[0]) / src_geo[1] + 1e-10, (y - src_geo[3]) / src_geo[5] + 1e-10) and (x, y) is
 * the centre (dst_geo[0] + (j + 0.5) dst_geo[1], dst_geo[3] + (i + 0.5) dst_geo[5]) transformed
 * exactly in float64 into the source CRS; no data outside the source, for non-finite source values
 * and for coordinates the source CRS cannot represent.  CRSs are WGS 84 only: EPSG:4326
 * (x = lon, y = lat in degrees), EPSG:3857, and UTM (zone +z north / -z south, transverse
 * Mercator by Krueger's series to sixth order).  `src` holds rows/cols [win_row0, +shape[1]) x
 * [win_col0, +shape[2]) of the whole (src_height x src_width) source described by src_geo.
 * Reads of source cells outside that window give no data and are counted: with misses != NULL
 * (host pointer) the call synchronises `stream` and stores the count, and the caller repeats the
 * call with a larger window when it is not 0.                                                   */
enum GmCrsKind { GM_CRS_GEOGRAPHIC = 0, GM_CRS_MERCATOR = 1, GM_CRS_UTM = 2 };
typedef struct GmWarp {
  int32_t dst_kind, dst_zone;     /* GmCrsKind; UTM zone (+north / -south), else 0 */
  int32_t src_kind, src_zone;
  double  dst_geo[6];             /* geotransform of the request grid              */
  double  src_geo[6];             /* geotransform of the whole source              */
  int64_t src_height, src_width;  /* whole source                                  */
  int64_t win_row0, win_col0;     /* source cell of src[:, 0, 0]                   */
} GmWarp;
int  gm_warp_nn(const GmArray* src, GmArray* dst, const void* nodata, const GmWarp* warp,
                int64_t* misses, void* stream);

/* stencils (raster/spatial.py): src carries the halo the reference requests.  gm_hillshade and
 * gm_moving_max accept rows with extra columns on the right (src.shape[2] >= dst.shape[2] + halo):
 * on a 16-byte row pitch HillShade reads four columns per load and MovingMax stages tiles by TMA */
int  gm_hillshade(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
                  double fill, double xres, double yres, double altitude_deg,
                  double azimuth_deg, void* stream);            /* :353-417 */
int  gm_moving_max(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
                   int size, void* stream);                     /* :192-213 */
int  gm_dilate(const GmArray* src, GmArray* dst, const void* values, int n_values,
               void* stream);                                   /* :146-155 */
/* Gaussian: weights are scipy's _gaussian_kernel1d (host, float64), radius
 * ly/lx taps; margins my/mx are cropped ("exact" mode).  zoom=1 applies the
 * nearest-neighbour zoom-back instead (:296-305).                           */
/* Arithmetic of the Gaussian's tap sums when both radii are <= 8 taps (every "exact"-mode request):
 *   GM_SMOOTH_EXACT    float64, multiply and add rounded separately -- scipy.ndimage.gaussian_filter
 *                      bit for bit;
 *   GM_SMOOTH_FMA      (default; env GM_SMOOTH=exact|fma|float32) float64 with fused multiply-add:
 *                      equal to SciPy except where a double sum lies within one rounding of a
 *                      boundary of the array dtype (then the last bit of the result may differ);
 *   GM_SMOOTH_FLOAT32  float32 rasters: float32 accumulation, relative error <= 1e-6.
 * Other radii and the zoom mode always use the exact arithmetic.                               */
enum GmSmoothMode { GM_SMOOTH_EXACT = 0, GM_SMOOTH_FMA = 1, GM_SMOOTH_FLOAT32 = 2 };
int  gm_set_smooth_mode(int mode);
int  gm_get_smooth_mode(void);
int  gm_smooth(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
               double fill, const double* wy, int ly, const double* wx, int lx,
               int my, int mx, int zoom, double zy, double zx, double oy, double ox,
               void* stream);                                   /* :273-307 */

/* temporal (raster/temporal.py:722-768 TemporalAggregate, :959-1005 Cumulative)
 * frames of bin g are frame_index[bin_offsets[g] .. bin_offsets[g+1])        */
enum GmStat { GM_STAT_SUM = 0, GM_STAT_COUNT, GM_STAT_MIN, GM_STAT_MAX, GM_STAT_MEAN,
              GM_STAT_MEDIAN, GM_STAT_STD, GM_STAT_VAR, GM_STAT_PERCENTILE };
int  gm_temporal_aggregate(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
                           int stat, double q, const int32_t* bin_offsets,
                           const int32_t* frame_index, int n_bins, void* stream);
int  gm_temporal_cumulative(const GmArray* src, GmArray* dst, const void* nodata, int has_nodata,
                            int stat, const int32_t* bin_offsets, const int32_t* frame_index,
                            const int32_t* out_frame, int n_bins, void* stream);

/* polygons: CSR layout.  ring r of polygon p: rings poly_offsets[p]..[p+1),
 * vertices ring_offsets[r]..[r+1) (closed rings, xy interleaved float64).
 * geo: GDAL geotransform of the target grid (6 doubles).                    */
typedef struct GmPolygons {
  const double*  xy;            /* host, 2*n_vertices                        */
  const int64_t* ring_offsets;  /* host, n_rings+1                           */
  const int64_t* poly_offsets;  /* host, n_polygons+1                        */
  int64_t n_polygons;
  int64_t n_rings;
  int64_t n_vertices;
  const void* resident;         /* NULL, or a handle from gm_polygons_upload: the
                                   CSR arrays already live in HBM (no per-call copy) */
} GmPolygons;

/* keep a polygon soup in HBM between calls (AggregateRaster over many frames /
 * requests, multi-GPU stripes); the host arrays must still be valid in the
 * descriptor, the handle only replaces their upload                          */
int  gm_polygons_upload(const GmPolygons* polys, void** handle);
int  gm_polygons_free(void* handle);

/* utils.rasterize_geoseries (utils.py:638-756): burn value[p] (dst dtype) for
 * every pixel whose centre is inside polygon p, later polygons on top.      */
int  gm_rasterize_polygons(const GmPolygons* polys, const double geo[6],
                           const void* burn_values, const void* nodata,
                           GmArray* dst, void* stream);

/* geometry/aggregate.py:113-203 aggregate_polygons + measurements.py:18-137:
 * out[t*n_polygons + p] (float32); covered[p] = pixel centres inside p
 * (0 => caller applies the centroid fallback, aggregate.py:561-571).
 * row_begin/row_end restrict the rows this call reads (multi-GPU stripes);
 * partial != NULL receives (count,sum,min,max) partials instead of `out`.   */
typedef struct GmZonalPartial { int64_t count; double sum; double vmin; double vmax; } GmZonalPartial;
int  gm_zonal_stats(const GmArray* raster, const void* nodata, int has_nodata,
                    const GmPolygons* polys, const double geo[6],
                    int stat, double q, const float* thresholds,
                    int64_t row_begin, int64_t row_end,
                    float* out, int64_t* covered, GmZonalPartial* partial,
                    void* stream);

/* Multi-GPU order statistics (SURVEY.md section 8e, measurements.py:18-137): a rank
 * extracts the ACTIVE cell values under every polygon of its row stripe
 * (counts[p] = partial[p].count of a previous gm_zonal_stats call; values are
 * packed polygon by polygon, `values` has sum(counts) elements of the raster
 * dtype), the segments are routed to the polygons' owner ranks, and the owner
 * selects median / percentile per segment with the reference's interpolation. */
int  gm_zonal_values(const GmArray* raster, const void* nodata, int has_nodata,
                     const GmPolygons* polys, const double geo[6], const float* thresholds,
                     const int64_t* counts, void* values, void* stream);
int  gm_segment_order_stat(const void* values, int32_t dtype, const int64_t* offsets,
                           int64_t n_segments, int stat, double q, float* out, void* stream);

/* Multi-GPU count / sum / mean / min / max (SURVEY.md section 8e): a rank reduces the polygons
 * over its row stripe into partials that STAY IN HBM, laid out for two all-reduces --
 * sums[3N] = (count, covered cells, sum) as float64 for a SUM, extremes[2N] = (min, -max) for a
 * MIN -- and after the collectives the statistic of scipy.ndimage sum/mean/minimum/maximum
 * (geometry/aggregate.py:311-316) is formed from them.  `sums` / `extremes` are DEVICE
 * pointers (e.g. torch tensors); `out` / `covered` are host buffers.  `stat` (GmStat, or -1 for
 * everything) lets the stripe pass compute only what the statistic needs: the sums for
 * sum / mean / count, one extreme for min / max.  With a resident soup (gm_polygons_upload) the
 * stripe pass keeps what it derives from the soup for this grid (pixel-space vertices, row
 * ranges, the ids of the polygons with rows in the stripe) from the second call on the same grid
 * on (a sweep of ever new windows stays on the stream-ordered per-call path) and does not
 * synchronise: its crossing-overflow flag is read back by gm_zonal_finalize_device, which takes
 * the same `polys` (NULL: nothing deferred).                                                  */
int  gm_zonal_partials_device(const GmArray* raster, const void* nodata, int has_nodata,
                              const GmPolygons* polys, const double geo[6],
                              const float* thresholds, int64_t row_begin, int64_t row_end,
                              double* sums, double* extremes, int stat, void* stream);
int  gm_zonal_finalize_device(const double* sums, const double* extremes, int64_t n_polygons,
                              int stat, float* out, int64_t* covered, const GmPolygons* polys,
                              void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GEOKERNELS_H */

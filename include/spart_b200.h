/*
 * spart_b200.h -- C ABI of libspart_b200.so, the B200 (sm_100a) implementation of the
 * SPART forward model (BSM soil -> PROSPECT-5D/PRO leaf -> SAILH canopy -> SMAC atmosphere
 * -> sensor bands) evaluated over large batches of parameter sets.
 *
 * The reference (wirrell/SPART-python) has no FFI layer: its boundary is the Python call
 * surface `SPART(soilpar, leafbio, canopy, atm, angles, sensor, DOY).run()`
 * (reference src/SPART/SPART.py:83-95, 162-269).  Each entry point below names the part of
 * that surface it replaces.  INTEGRATION.md shows the ctypes binding a maintainer of the
 * reference would add.
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success, a negative SPART_E* code
 *     for an argument error, or a positive cudaError_t value for a CUDA failure;
 *     spart_last_error() returns a thread-local description of the last failure;
 *   - no exception ever crosses this boundary;
 *   - `*_dev` pointers are device pointers owned by the caller (e.g. PyTorch's caching
 *     allocator); the library never allocates per call on the device paths and all work is
 *     enqueued asynchronously on the caller's stream (a cudaStream_t passed as void*);
 *   - a context is immutable after spart_create and may be used concurrently from several
 *     host threads until spart_destroy, which no other thread may overlap; create one context
 *     per GPU;
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 *
 * Batch parameter layout ("params"): struct-of-arrays, double, [SPART_NPAR][ld] with
 * ld >= n, row order
 *   0..8   leaf    Cab Cdm Cw Cs Cca Cant N PROT CBC   (LeafBiology, prospect_5d.py:73-81)
 *   9..14  soil    B lat lon SMp SMC film              (SoilParameters, bsm.py:269-287)
 *   15..18 canopy  LAI LIDFa LIDFb q                   (CanopyStructure, sailh.py:340-348)
 *   19..21 angles  sol_angle obs_angle rel_angle, deg  (Angles, sailh.py:298-301)
 *   22..25 atm     aot550 uo3 uh2o Pa                  (AtmosphericProperties, smac.py:307-317)
 *   26     DOY                                         (SPART.__init__, SPART.py:83)
 *
 * Broadcast rows: `broadcast_rows` is a bit mask over these 27 rows.  A set bit r says that row r
 * is constant over the batch (a look-up table with fixed geometry, fixed SMC / film, PROSPECT-5D
 * without PROT / CBC ...): only params[r * ld + 0] is ever read, the host path copies one element
 * of that row instead of n, and when bits 19, 20 and 21 are all set -- one sun / observer geometry
 * for the whole batch BY CONSTRUCTION -- the library evaluates the sample-independent volume
 * scattering terms (_volscatt, sailh.py:401-446) and the geometry-only sub-expressions of SMAC
 * (smac.py:125-201) once per thread block instead of once per sample.  Results agree with the
 * general path to a few ulp (sums are re-associated).  When bits 16 and 17 (LIDFa, LIDFb) are both
 * set the leaf inclination distribution (calculate_leafangles, sailh.py:351-398) is iterated once for
 * the whole batch (bit-identical results).  There is no unchecked "the caller promises" flag: a row
 * is either read per sample or read once.
 */
#ifndef SPART_B200_H
#define SPART_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPART_ABI_VERSION 5

#define SPART_NPAR 27       /* rows of a parameter batch                                   */
#define SPART_NWL 2001      /* 400..2400 nm, 1 nm (SpectralBands.wlP, SPART.py:303)        */
#define SPART_NWL_S 2162    /* + 161 thermal wavelengths (SpectralBands.wlS, SPART.py:310) */
#define SPART_NLC 17        /* per-wavelength constants, see SpartTables                   */
#define SPART_NSMAC 60      /* per-band host-folded SMAC constants, see SpartSensor        */
#define SPART_NOUT 3        /* R_TOC, R_TOA, L_TOA                                         */
#define SPART_NSPEC 9       /* planes of spart_forward_spectrum                            */
#define SPART_NKERNELS 3    /* kernels of spart_forward_bands: leaf angles, geometry, bands */

enum {
  SPART_OK = 0,
  SPART_EINVAL = -1,   /* bad argument (null pointer, negative size, unknown sensor index) */
  SPART_ENODEV = -2,   /* no usable CUDA device                                            */
  SPART_ENOMEM = -3    /* host allocation failed                                           */
};

enum { SPART_FP64 = 64, SPART_FP32 = 32 };

/* flags of spart_forward_bands (bit 0 was ABI 4's unchecked uniform-geometry promise; it is now
 * derived from broadcast_rows and the value 1 is rejected) */
enum {
  /* the context was created with a user-supplied dry-soil spectrum in row 11 of SpartTables.lc
   * (rows 12, 13 zero): B / lat / lon are ignored and rdry = that spectrum, as with the reference's
   * SoilParametersFromFile (bsm.py:42-43, 155-226) */
  SPART_FLAG_SOIL_SPECTRUM = 2,
  /* band values of the four canopy reflectances are SRF-weighted means over the band
   * (calculate_spectral_convolution, SPART.py:358-396, applied to canopyopt) instead of the
   * reference's np.interp sample at the band centre (SPART.py:216-223); SPART_FP64 only */
  SPART_FLAG_SRF_BANDS = 4,
  /* the workspace still holds the per-sample record of a previous spart_forward_bands call for
   * the same params / n / precision / soil flag (any sensor): skip the per-sample kernels and run
   * only the band kernel.  This is how one batch is evaluated for several sensors (e.g.
   * Sentinel-2A and -2B) while paying for the sensor-independent work once. */
  SPART_FLAG_REUSE_RECORD = 8,
  /* SPART_FP32 only: params are float [SPART_NPAR][ld] and the results are written as float, which
   * halves the bytes on every copy and on the final gather of a sharded run.  The model is
   * evaluated at the float-rounded inputs. */
  SPART_FLAG_F32_IO = 16,
  /* compact result: out = [n][n_bands][2] (R_TOC, R_TOA) followed by etscale[n], the per-sample
   * extraterrestrial scale cf(DOY) cos(sza) / pi (SPART.py:345-353).  L_TOA is then rebuilt by the
   * consumer bit for bit as (conv_ea[b] * etscale[s]) * R_TOA[s][b] -- the product the kernels
   * themselves form (SPART.py:252); conv_ea is the SpartSensor member.  Two thirds of the bytes. */
  SPART_FLAG_COMPACT_OUT = 32,
  /* SPART_FP64, device path: the workspace already holds a caller-supplied leaf inclination
   * distribution (spart_set_lidf on the same workspace and stream): LIDFa / LIDFb are ignored, the
   * leaf-angle kernel is skipped and the 13 values enter k, K, bf, sob, sof as they are -- what the
   * reference does with an assigned CanopyStructure.lidf (sailh.py:81-97 read canopy.lidf). */
  SPART_FLAG_USER_LIDF = 64,
  /* the context was created with a soil library (spart_create_with_soils): params row 9 (B) holds each
   * sample's 0-based library index as a whole number in the row's element type, rows 10 and 11 (lat, lon)
   * are ignored and rdry = library[index] -- a LUT whose entries each take one measured dry-soil spectrum,
   * as the reference does with one SoilParametersFromFile per SPART object (bsm.py:42-43, 155-226).
   * Row 9 may be a broadcast row.  An index that is not a whole number in [0, n_soils) (NaN included)
   * gives NaN in every output that depends on the soil; nothing outside the library is read.  Excludes
   * SPART_FLAG_SOIL_SPECTRUM; combines with every other flag.  Each sample's result equals bit for bit a
   * run of that sample with SPART_FLAG_SOIL_SPECTRUM and the spectrum library[index]. */
  SPART_FLAG_SOIL_LIBRARY = 128
};

/* elements of the result buffer of spart_forward_bands for n samples, nb bands and these flags */
#define SPART_OUT_ELEMS(n, nb, flags) \
  (((flags) & SPART_FLAG_COMPACT_OUT) ? (size_t)(n) * (size_t)(nb) * 2 + (size_t)(n) : (size_t)(n) * (size_t)(nb) * 3)

typedef struct SpartCtx SpartCtx;

/* Sample-independent per-wavelength constants, host pointer, double [SPART_NLC][SPART_NWL]:
 *   0 Kab 1 Kca 2 Kdm 3 Kw 4 Ks 5 Kant 6 cbc 7 prot          optical_params.pkl (SPART.py:399-406)
 *   8 tav(40,nr)  9 tav(90,nr)  10 tav(90,nr)/nr^2            prospect_5d.py:200-205
 *   11..13 GSV[:,0..2]                                         bsm.py:45-52
 *   14 tav(90,2/nw)/tav(90,2)  15 1-tav(90,nw)/nw^2  16 1-tav(40,nw)   bsm.py:110-119
 * calculate_tav (prospect_5d.py:249-311) only ever receives table arguments, so these are
 * folded once on the host. */
typedef struct {
  int32_t n_wl;            /* must be SPART_NWL */
  const double* lc;        /* [SPART_NLC][n_wl] */
} SpartTables;

/* One sensor = the content of sensor_information/<name>.pkl the hot path uses
 * (SPART.py:216-232, 358-396), with sample-independent sub-expressions folded on the host. */
typedef struct {
  int32_t n_bands;
  const int32_t* wl_lo;    /* [n_bands] index into 400..2400 nm of the knot at/below wl_smac      */
  const int32_t* wl_hi;    /* [n_bands] upper knot (== wl_lo when wl_smac hits a knot exactly)     */
  const double* wl_frac;   /* [n_bands] wl_smac - knot(wl_lo): np.interp weight (SPART.py:220-223) */
  const double* smac;      /* [SPART_NSMAC][n_bands] folded SMAC coefficients (smac.py:44-92)      */
  const double* conv_ea;   /* [n_bands] SRF-convolved Ea (SPART.py:358-396 applied to ETpar['Ea']) */
  /* optional (all three NULL = not available): spectral response per band for
   * SPART_FLAG_SRF_BANDS, already reduced to the 1-nm grid with the nearest-index rule of
   * get_closest_index (SPART.py:381-387) and normalised by sum(p_srf): band b has srf_len[b]
   * non-zero weights; its (wavelength index, weight) pairs follow those of band b-1 in
   * srf_idx / srf_w */
  const int32_t* srf_len;  /* [n_bands] */
  const int32_t* srf_idx;  /* [sum(srf_len)] index into 400..2400 nm */
  const double* srf_w;     /* [sum(srf_len)] */
} SpartSensor;

/* ABI version of the loaded library (== SPART_ABI_VERSION of the header it was built from). */
int spart_abi_version(void);

/* Thread-local text of the last error returned on this thread ("" if none). */
const char* spart_last_error(void);

/* Number of CUDA devices visible (0 when there is no driver/GPU). Never fails. */
int spart_device_count(void);

/* Replaces SPART.__init__'s table loads (SPART.py:92-95): uploads the immutable tables and
 * all sensors to `device` once.  *out must be released with spart_destroy. */
int spart_create(const SpartTables* tables, const SpartSensor* sensors, int32_t n_sensors,
                 int32_t device, SpartCtx** out);
/* spart_create plus a soil library for SPART_FLAG_SOIL_LIBRARY: soils is host memory, double
 * [n_soils][SPART_NWL] (dry-soil reflectance on 400..2400 nm), uploaded once; 1 <= n_soils <= 2^24 (a float
 * holds every whole number up to 2^24, so the index stays exact under SPART_FLAG_F32_IO).  The context
 * serves runs without the flag exactly like one from spart_create. */
int spart_create_with_soils(const SpartTables* tables, const SpartSensor* sensors, int32_t n_sensors,
                            const double* soils, int32_t n_soils, int32_t device, SpartCtx** out);
/* Frees the context.  It first waits for all work on the context's device (cudaDeviceSynchronize), so
 * device-path calls still queued on any stream finish before their tables are freed.  The caller must not
 * destroy a context while another thread is inside a call on it, or call it afterwards. */
int spart_destroy(SpartCtx* ctx);

/* Device scratch the caller must provide to the *_dev entry points for a batch of n samples. */
size_t spart_workspace_bytes(const SpartCtx* ctx, int64_t n);

/* Replaces the per-sample loop over SPART(...).run() (SPART.py:162-269): for every sample
 * s < n and band b of sensor `sensor`, out_dev[(s * n_bands + b) * 3 + {0,1,2}] =
 * {R_TOC, R_TOA, L_TOA} (or the compact layout of SPART_FLAG_COMPACT_OUT).  params_dev:
 * [SPART_NPAR][ld] (see top) of double, or of float with SPART_FLAG_F32_IO; out_dev has the same
 * element type.  broadcast_rows: see top.  precision: SPART_FP64 or SPART_FP32 (arithmetic type of
 * the spectral / atmosphere stage).  Asynchronous on `stream`; makes the context's device current
 * for the duration of the call and restores the caller's. */
int spart_forward_bands(const SpartCtx* ctx, int32_t sensor, const void* params_dev,
                        int64_t n, int64_t ld, uint32_t broadcast_rows, int32_t precision,
                        int32_t flags, void* workspace_dev, void* out_dev, void* stream);

/* spart_forward_bands with the broadcast rows read from a separate base: element 0 of broadcast row r
 * is params_bc_dev[r * ld] (same element type and ld as params_dev), every other row is read from
 * params_dev.  A caller that splits a batch of more than 65535 * 128 samples into calls passes
 * params_dev = batch + first sample of the call and params_bc_dev = batch, so that every call reads the
 * batch's own element 0 of each broadcast row; spart_forward_bands(..., p, ...) is
 * spart_forward_bands_bc(..., p, p, ...).  params_bc_dev must not be NULL. */
int spart_forward_bands_bc(const SpartCtx* ctx, int32_t sensor, const void* params_dev,
                           const void* params_bc_dev, int64_t n, int64_t ld, uint32_t broadcast_rows,
                           int32_t precision, int32_t flags, void* workspace_dev, void* out_dev, void* stream);

/* Same computation with HOST buffers: params_host [SPART_NPAR][ld] and out_host (layout and
 * element type as above, SPART_OUT_ELEMS elements) are ordinary host memory.  The parameters travel
 * in spans of up to 128 Ki samples (one 2-D copy per run of per-sample rows) into three device
 * buffers; each span is evaluated in place in chunks of up to 64 Ki samples whose results flow back
 * as they complete.  One stream per copy direction, one per output slot, tied by events, so both
 * copy engines and the SMs run side by side.  Pinned or registered buffers (cudaHostAlloc /
 * cudaHostRegister / torch pin_memory) are
 * DMA'd directly; pageable buffers (plain NumPy arrays) are staged through internal pinned
 * buffers by a small pool of copy threads (SPART_HOST_THREADS, default 12), because an asynchronous
 * copy on pageable memory degenerates to a synchronous single-threaded driver copy.  Broadcast
 * rows move one element.  Returns when out_host is complete; on failure no copy is left in
 * flight.  This is the drop-in for a caller that holds NumPy arrays. */
int spart_forward_bands_host(SpartCtx* ctx, int32_t sensor, const void* params_host,
                             int64_t n, int64_t ld, uint32_t broadcast_rows, int32_t precision,
                             int32_t flags, void* out_host);

/* Stores a caller-supplied leaf inclination distribution, lidf_dev [n][13] of double (the 13 classes
 * of sailh.py:49, each row summing to 1), in the workspace of a batch of n samples; the following
 * spart_forward_bands call on that workspace passes SPART_FLAG_USER_LIDF.  Asynchronous on stream. */
int spart_set_lidf(const double* lidf_dev, int64_t n, void* workspace_dev, void* stream);

/* Replaces the leafopt / soilopt / canopyopt attributes of a SPART object after run()
 * (SPART.py:192-214, 427-470): full 2162-wavelength spectra.
 * out_dev: double [n][SPART_NSPEC][SPART_NWL_S], planes
 *   0 leaf refl  1 leaf tran  2 kChlrel (0 beyond 2400 nm)  3 soil refl (wet)  4 soil refl dry
 *   (value at 2400 nm beyond)  5 rso  6 rdo  7 rsd  8 rdd.
 * rho_thermal / tau_thermal: leaf reflectance / transmittance beyond 2400 nm
 * (LeafBiology.rho_thermal / tau_thermal, prospect_5d.py:82-83, SPART.py:461-466; the reference's
 * default is 0.01 each).  flags: 0, SPART_FLAG_SOIL_SPECTRUM or SPART_FLAG_SOIL_LIBRARY (plane 4 is then the
 * sample's library spectrum), and / or SPART_FLAG_USER_LIDF. */
int spart_forward_spectrum(const SpartCtx* ctx, const double* params_dev, int64_t n, int64_t ld,
                           int32_t flags, double rho_thermal, double tau_thermal,
                           void* workspace_dev, double* out_dev, void* stream);

/* Replaces SMAC(angles, atm, coefs) (smac.py:14-213) for sensor `sensor`.  params_dev:
 * [SPART_NPAR][ld]; only the angle and atmosphere rows 19..25 matter, the others must merely be
 * finite.  out_dev: double [n][9][n_bands] in the field order of the reference's
 * AtmosphericOptics: Ta_s, Ta_o, Tg, Ra_dd, Ra_so, Ta_ss, Ta_sd, Ta_oo, Ta_do. */
int spart_smac(const SpartCtx* ctx, int32_t sensor, const double* params_dev, int64_t n, int64_t ld,
               void* workspace_dev, double* out_dev, void* stream);

/* Replaces SAILH(soil, leafopt, canopy, angles) on caller-supplied spectra (sailh.py:14-237).
 * params_dev: [SPART_NPAR][ld]; only the canopy and angle rows 15..21 matter, the others must
 * merely be finite.  soil_refl / leaf_refl / leaf_tran: double spectra of SPART_NWL_S (2162)
 * wavelengths, sample s at offset s * spectra_stride (spectra_stride = 0: one spectrum shared by
 * all samples).  out_dev: double [n][4][2162] = rso, rdo, rsd, rdd. */
int spart_sailh(const SpartCtx* ctx, const double* params_dev, int64_t n, int64_t ld,
                const double* soil_refl_dev, const double* leaf_refl_dev, const double* leaf_tran_dev,
                int64_t spectra_stride, void* workspace_dev, double* out_dev, void* stream);

/* Replaces CanopyStructure.__init__'s calculate_leafangles (sailh.py:340-398): the 13-class
 * leaf inclination distribution for n (LIDFa, LIDFb) pairs.  ab_dev: double [2][ld];
 * out_dev: double [n][13].  Needs no context. */
int spart_leafangles(const double* ab_dev, int64_t n, int64_t ld, double* out_dev, void* stream);

/* Consumer of a LUT (new; the reference has no retrieval step): for each of m observed band
 * vectors obs_dev [m][n_bands] (float) the index of the LUT entry lut_dev [n][n_bands] (float, e.g.
 * one output column of spart_forward_bands cast to float) with the smallest weighted squared
 * distance sum_b (sqrt_w[b] (obs_b - lut_b))^2, ties to the lowest index.  weights_dev: sqrt of the
 * band weights [n_bands] or NULL (all 1).  workspace_dev: spart_lut_workspace_bytes(m) bytes.
 * Outputs best_index_dev int64 [m] (= index_offset + local index), best_cost_dev float [m].  An entry whose
 * cost is NaN (NaN in the entry or the observation) or not below 3e38 is never chosen; an observation without
 * any other entry gets the "no entry" result: index 2^32 - 1 and cost NaN (packed word all ones).
 * Sharded tables: every GPU searches its own slice with index_offset = first global entry of the
 * slice and packed_dev != NULL; the call then leaves one word (cost bits << 32 | global index)
 * per observation in packed_dev [m] instead of unpacking it, the caller min-reduces the words
 * over the GPUs (ncclMin on 64-bit integers: costs are >= 0, so integer order = (cost, index)
 * order, ties to the lowest global index) and calls spart_lut_unpack.  The all-ones "no entry" word is -1 as a
 * signed integer: replace it by 2^63 - 1 (which unpacks to index 2^32 - 1, cost NaN) before a signed
 * reduction.  The full table never has
 * to be gathered on one GPU.  index_offset + n < 2^32. */
size_t spart_lut_workspace_bytes(int64_t m);
int spart_lut_nearest(const float* lut_dev, int64_t n, int32_t n_bands, const float* obs_dev, int64_t m,
                      const float* weights_dev, int64_t index_offset, void* workspace_dev,
                      int64_t* best_index_dev, float* best_cost_dev, unsigned long long* packed_dev,
                      void* stream);
/* The same search on the tensor cores (3xTF32 mma.sync over the band axis, n_bands <= 30): the entry is
 * chosen by an approximate comparison (error ~1e-6 |obs||entry|, so near-ties may resolve differently),
 * its reported cost is recomputed exactly in FP32.  Same arguments as spart_lut_nearest. */
int spart_lut_nearest_tc(const float* lut_dev, int64_t n, int32_t n_bands, const float* obs_dev, int64_t m,
                         const float* weights_dev, int64_t index_offset, void* workspace_dev,
                         int64_t* best_index_dev, float* best_cost_dev, unsigned long long* packed_dev,
                         void* stream);
int spart_lut_unpack(const unsigned long long* packed_dev, int64_t m, int64_t* best_index_dev,
                     float* best_cost_dev, void* stream);

/* The k nearest LUT entries of each observation (1 <= k <= 128, n_bands <= 32), with the cost of
 * spart_lut_nearest bit for bit (so k = 1 returns its index and cost).  Per observation the k smallest words
 * (cost bits << 32 | index_offset + local index) in unsigned order, i.e. ascending cost, ties to the lowest index
 * (also at the k-th place), whatever the launch plan.  Entries whose cost is NaN or not below 3e38 are never chosen;
 * slots beyond the qualifying entries hold the "no entry" word (all ones: index 2^32 - 1, cost NaN), which sorts
 * last.  Outputs best_index_dev int64 [m][k] and best_cost_dev float [m][k]; with packed_dev != NULL the call
 * instead leaves the sorted words in packed_dev [m][k], for spart_lut_topk_merge with the lists of other GPUs.
 * workspace_dev: spart_lut_topk_workspace_bytes(n, m, k) bytes (depends on its arguments only).  Other arguments
 * and limits as in spart_lut_nearest. */
size_t spart_lut_topk_workspace_bytes(int64_t n, int64_t m, int32_t k);
int spart_lut_topk(const float* lut_dev, int64_t n, int32_t n_bands, const float* obs_dev, int64_t m, int32_t k,
                   const float* weights_dev, int64_t index_offset, void* workspace_dev, int64_t* best_index_dev,
                   float* best_cost_dev, unsigned long long* packed_dev, void* stream);
/* n_lists ascending lists of k words per observation, lists_dev [n_lists][m][k] (e.g. the packed_dev results of
 * several GPUs, gathered), reduced to the k smallest words, ascending: best_index_dev [m][k] + best_cost_dev [m][k],
 * or (packed_dev != NULL) the words in packed_dev [m][k].  1 <= n_lists <= 4096. */
int spart_lut_topk_merge(const unsigned long long* lists_dev, int64_t n_lists, int64_t m, int32_t k,
                         int64_t* best_index_dev, float* best_cost_dev, unsigned long long* packed_dev,
                         void* stream);

/* Moments of the parameters of the chosen entries, over a parameter table that may be sharded: a call sees the
 * entries [index_offset, index_offset + n_local) (index_offset + n_local < 2^32).  Parameter p of local entry e is
 * params_dev[p * stride_param + e * stride_entry] (elements; double, or float with SPART_FLAG_F32_IO), so both the
 * [n_params][n] batch layout and an [n][n_params] table are read without a copy.  For each observation o and each
 * of its k neighbours index_dev [m][k] (int64, e.g. spart_lut_topk's best_index_dev) that falls in the local range,
 * in neighbour order, in FP64, added to acc_dev [m][n_params + 1] (zero it first):
 *   centre_dev == NULL: acc[o][p] += x, and acc[o][n_params] += 1 (the count);
 *   centre_dev [m][n_params]: acc[o][p] += (x - centre[o][p])^2, and the count as above.
 * Pieces of a table accumulate into one acc_dev (on several GPUs: one sum all-reduce of acc_dev per pass).
 * spart_lut_moments_finish: mean [m][n_params] = sum / count, count_dev int64 [m]; with sq_dev (the acc_dev of a
 * second pass centred on that mean) also std_dev [m][n_params] = sqrt(sq / count), the population standard
 * deviation.  count 0 gives NaN mean and std. */
int spart_lut_moments_accumulate(const void* params_dev, int32_t n_params, int64_t stride_param,
                                 int64_t stride_entry, int32_t flags, int64_t index_offset, int64_t n_local,
                                 const int64_t* index_dev, int64_t m, int32_t k, const double* centre_dev,
                                 double* acc_dev, void* stream);
int spart_lut_moments_finish(const double* sum_dev, const double* sq_dev, int64_t m, int32_t n_params,
                             double* mean_dev, double* std_dev, int64_t* count_dev, void* stream);

/* Variance-based sensitivity analysis (new; the reference has none): a scrambled Sobol' design in the batch layout
 * and the Saltelli (2010) estimators of the first-order and total Sobol' indices.  No context is needed; the
 * calls run on the current device.
 *
 * spart_sobol_design writes rows rows[0..n_vary-1] (distinct, 0..26) of params_dev [SPART_NPAR][ld]; the other
 * rows are the caller's.  rows, lo and hi are HOST arrays of n_vary entries; 1 <= n_vary <= 27.
 *   Point i (0 <= first <= i < first + count <= 2^32) of dimension d is k_d(i) = XOR of v'[d][j] over the set
 *   bits j of i ^ (i >> 1), XOR s_d, and u = k_d(i) 2^-32; v are the Joe-Kuo direction numbers that SciPy ships
 *   (sobol_dirs.h).  Varied parameter p gets x = lo[p] + (hi[p] - lo[p]) u, rounded once per operation (no fused
 *   multiply-add), and moved to the double below hi[p] if it rounds up to it, so x is in [lo[p], hi[p]).
 *   scramble = 0: v' = v, s = 0, which is scipy.stats.qmc.Sobol(D, scramble=False, bits=32) bit for bit.
 *   scramble = 1: v'[d][j] = L_d v[d][j] over GF(2) and a random digital shift s_d.  L_d is unit lower-triangular
 *   (rows counted from the most significant bit); with the SplitMix64 stream of `seed`, dimension d draws the
 *   words 32 d .. 32 d + 31: the strictly-lower part of row r = 1..31 is the low r bits of word 32 d + r - 1
 *   (its bit r - 1 - c is column c), and s_d is the low 32 bits of word 32 d + 31.  Dimension d thus gets the
 *   same scramble whatever the number of dimensions, and the net property of the points is kept.
 *   saltelli = 0: `count` samples 0..count-1 of dimensions 0..n_vary-1 (ld >= count), e.g. a quasi-random LUT.
 *   saltelli = 1: (n_vary + 2) count samples in blocks A, B, AB_1 .. AB_n_vary (sample block * count + j,
 *   ld >= (n_vary + 2) count): A uses dimensions 0..n_vary-1, B dimensions n_vary..2 n_vary-1, and AB_i is A
 *   with varied parameter i taken from B.  The A block equals the saltelli = 0 output.
 *
 * spart_sobol_accumulate adds the sums of one chunk of n base points to acc_dev (spart_sobol_acc_elems(n_out,
 * n_vary) doubles; zero it before the first chunk).  f_dev [(n_vary + 2) n][n_out]: the outputs of the chunk's
 * design blocks, f[(block n + j) n_out + o] -- spart_forward_bands' [samples][nb][3] over the blocks A, B, AB_i
 * of the chunk, with n_out = 3 nb.  ref_dev [(n_vary + 2)][n_out]: the outputs of base point 0 of the whole
 * design (A, B, AB_1 .. AB_n_vary), by which every summed quantity is shifted, so an output whose mean is far
 * above its spread keeps its variance.  acc_dev [128][n_vary + 1][n_out][8]: per slice of the chunk's base
 * points, for varied parameter i < n_vary, with D = f_ABi - f_A, p = (f_B - f_A0) D and u = D^2 (f_A0 = ref's
 * f_A), the sums of (p - p_0), (p - p_0)^2, (D - D_0), (D - D_0)^2, (p - p_0)(D - D_0), (u - u_0), (u - u_0)^2
 * and a zero (x_0: x at base point 0); slot n_vary: the sums of (f - f_A0) and (f - f_A0)^2 over f_A and f_B,
 * then zeros.  All sums are FP64 in a fixed order, so a run is bit-reproducible; the accumulators of design
 * pieces on several GPUs (each with the same ref) merge with one sum all-reduce.
 *
 * spart_sobol_finish, over n_total base points, with the estimators of scipy.stats.sobol_indices (method
 * "saltelli_2010", outputs centred on their mean): mean_dev, var_dev [n_out]: mean and population variance V of
 * f_A and f_B together; first_dev, total_dev [n_out][n_vary]: S_i = mean(t) / V with t = (f_B - mean) D, and
 * ST_i = mean(u) / (2 V); first_se_dev, total_se_dev: std(t) / (sqrt(N) V) and std(u) / (2 sqrt(N) V),
 * population standard deviations, which ignore the uncertainty of V (and of the mean).  V = 0 gives NaN
 * indices. */
int spart_sobol_design(const int32_t* rows, const double* lo, const double* hi, int32_t n_vary, uint64_t seed,
                       int32_t scramble, int64_t first, int64_t count, int32_t saltelli, double* params_dev,
                       int64_t ld, void* stream);
size_t spart_sobol_acc_elems(int32_t n_out, int32_t n_vary);
int spart_sobol_accumulate(const double* f_dev, int64_t n, int32_t n_out, int32_t n_vary, const double* ref_dev,
                           double* acc_dev, void* stream);
int spart_sobol_finish(const double* acc_dev, const double* ref_dev, int64_t n_total, int32_t n_out,
                       int32_t n_vary, double* mean_dev, double* var_dev, double* first_dev, double* total_dev,
                       double* first_se_dev, double* total_se_dev, void* stream);

/* Retrieval by bounded Levenberg-Marquardt (new; the reference has none): fit n_vary = P (1..16) varied rows of
 * each observation's parameters to its band vector, from n_starts starts per observation.  A track is one start of
 * one observation: track t (0 <= t < n_tracks) belongs to observation t / n_starts.  It is iterated in normalised
 * coordinates u in [0, 1]^P, x_p = lo[p] + (hi[p] - lo[p]) u_p (each operation rounded once, no fused
 * multiply-add).  lo and hi are HOST arrays of P finite values with lo < hi.  One iteration is
 * spart_invert_design -> spart_forward_bands -> spart_invert_step over the active tracks, whose indices the caller
 * lists in active_dev (int32 [n_active], distinct); a track is active while its status is SPART_INV_ACTIVE.  No
 * context is needed; the calls run on the current device and on the caller's stream.
 *
 * State: double state_dev [spart_invert_state_rows(P)][n_tracks] (column t = track t); rows u [P], trial [P],
 * J^T W J [P (P + 1) / 2] (lower triangle, (i, j <= i) at row i (i + 1) / 2 + j), J^T W r [P], C, lambda, status,
 * forward calls.  The caller initialises it: trial = the start clipped to [0, 1] in u, C = NaN, lambda = 1e-3,
 * status SPART_INV_ACTIVE (SPART_INV_INVALID for a start that is not finite), forward calls 0; u, J^T W J and
 * J^T W r are written by the first step.  spart_invert_state_rows returns 0 for P outside 1..16.
 *
 * spart_invert_design writes the P + 1 samples of each active track, columns slot (P + 1) .. slot (P + 1) + P of
 * params_dev [SPART_NPAR][ld] (ld >= n_active (P + 1)) for active_dev[slot]: sample 0 at the trial point and
 * sample p + 1 with u_p moved by h = 2^-17, upwards when u_p + h <= 1, otherwise downwards.  Varied rows
 * rows[0..P-1] get x; the n_obs_rows rows obs_rows[] (distinct, not varied) get the track's observation's value
 * obs_values_dev[k ld_values + o]; every other row is a broadcast row: base[row] (HOST [27]) is written at element
 * 0 only, so run the batch with those rows in broadcast_rows (fixed angles then select the folded geometry).
 *
 * spart_invert_step reads the forward outputs f_dev [n_active (P + 1)][n_bands][3] of that batch, column `column`
 * (0 R_TOC, 1 R_TOA, 2 L_TOA), the observations obs_dev [n_tracks / n_starts][n_bands] and the weights
 * weights_dev [n_bands] (NULL: all 1), and advances each active track by one step:
 *   - C(trial) = sum_b w_b (f_b - y_b)^2 in band order.  On the first call the trial (the start) is accepted; a
 *     non-finite observation value or C gives SPART_INV_INVALID.  Later, the trial is accepted if
 *     C(trial) < C, strictly: then u = trial, C = C(trial), J^T W J and J^T W r are those of the trial (column p of
 *     J = (f(sample p + 1) - f(sample 0)) / du_p, du_p the difference of the two x written over hi - lo), lambda =
 *     max(lambda / 10, 1e-15), and SPART_INV_CONVERGED_COST if C_old - C <= ftol C_old.  On rejection lambda =
 *     10 lambda.
 *   - SPART_INV_STALLED if lambda > 1e16, else SPART_INV_MAX_ITER if the track has made max_iter forward calls.
 *   - Otherwise (J^T W J + lambda D) delta = -J^T W r with D = diag(max(J^T W J_pp, 1e-30)) is solved by
 *     Cholesky, with lambda = 10 lambda and a new factorisation while one fails (SPART_INV_STALLED past 1e16);
 *     the next trial is clip(u + delta, 0, 1), and SPART_INV_CONVERGED_STEP if max_p |trial_p - u_p| <= xtol.
 *   ftol, xtol >= 0 and finite; max_iter >= 1.  Each track's result depends on its own data only.
 *
 * spart_invert_finish, per observation o of n_obs (n_tracks = n_obs n_starts): the track with the lowest finite C
 * (ties to the lowest start) gives x_dev [n_obs][P] (x of its u), cost_dev, status_dev, start_dev (the start's
 * index, 0..n_starts-1) and iterations_dev (its forward calls); n_forward_dev is the forward runs of all the
 * observation's tracks, sum of forward calls x (P + 1).  std_dev [n_obs][P] = (hi - lo) sqrt(s (A^-1)_pp) with
 * A = J^T W J of that track, s = C / (n_bands - P) (absolute_sigma = 0, as scipy.optimize.curve_fit) or 1
 * (absolute_sigma = 1: the weights are 1 / sigma_b^2); NaN when A is not positive definite, or when n_bands <= P
 * with absolute_sigma = 0.  An observation without a finite-cost track gets NaN x, cost and std,
 * SPART_INV_INVALID, start -1 and 0 iterations. */
#define SPART_INV_ACTIVE 0
#define SPART_INV_CONVERGED_COST 1
#define SPART_INV_CONVERGED_STEP 2
#define SPART_INV_MAX_ITER 3
#define SPART_INV_STALLED 4
#define SPART_INV_INVALID 5
size_t spart_invert_state_rows(int32_t n_vary);
int spart_invert_design(const int32_t* rows, const double* lo, const double* hi, int32_t n_vary,
                        const int32_t* obs_rows, int32_t n_obs_rows, const double* obs_values_dev,
                        int64_t ld_values, const double* base, int32_t n_starts, const double* state_dev,
                        int64_t n_tracks, const int32_t* active_dev, int64_t n_active, double* params_dev,
                        int64_t ld, void* stream);
int spart_invert_step(const double* lo, const double* hi, int32_t n_vary, int32_t n_starts, const double* f_dev,
                      int32_t n_bands, int32_t column, const double* obs_dev, const double* weights_dev, double ftol,
                      double xtol, int32_t max_iter, double* state_dev, int64_t n_tracks, const int32_t* active_dev,
                      int64_t n_active, void* stream);
int spart_invert_finish(const double* lo, const double* hi, int32_t n_vary, int32_t n_starts, int32_t n_bands,
                        int32_t absolute_sigma, const double* state_dev, int64_t n_obs, double* x_dev,
                        double* cost_dev, double* std_dev, int32_t* status_dev, int32_t* start_dev,
                        int32_t* iterations_dev, int64_t* n_forward_dev, void* stream);

/* Per-kernel timing of spart_forward_bands with CUDA events recorded on the caller's stream
 * (used by bench.py for the roofline).  After spart_profile_enable(ctx, 1) every
 * spart_forward_bands call records events around its SPART_NKERNELS kernels; spart_profile_read
 * waits for them and returns in kernel_ms[0..2] the summed durations [ms] of the leaf-angle
 * kernel, the per-sample geometry kernel and the per-(sample, band) kernel over `*calls` calls,
 * then clears the list. */
int spart_profile_enable(SpartCtx* ctx, int32_t on);
int spart_profile_read(SpartCtx* ctx, double* kernel_ms, int64_t* calls);

/* Micro-benchmarks used as roofline denominators by bench.py: dependent-free DFMA / FFMA
 * chains on all SMs.  Results in TFLOP/s (FMA = 2 flop). */
int spart_measure_peaks(int32_t device, double* fp64_tflops, double* fp32_tflops);

/* The FP64 rate of DEPENDENT DFMA chains on register operands, one chain per warp, eight warps per
 * scheduler (a degree-6 Horner step): on the B200 FP64 instructions of different warps issue every
 * 3 cycles, not 2, so this is ~2/3 of spart_measure_peaks' FP64 figure -- the issue ceiling of the
 * leaf-angle / geometry / band kernels, reported by bench.py beside the DFMA-chain peak. */
int spart_measure_fp64_chain(int32_t device, double* tflops);

/* Number of kernel launches this library has enqueued on this thread since load. */
int64_t spart_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SPART_B200_H */

/*
 * lidar_snow_sim.h -- C ABI of the B200-native LiDAR snowfall / wet-ground augmentation engine.
 *
 * The reference (SysCV/LiDAR_snow_sim) has no FFI: its boundary is plain Python functions on NumPy arrays
 * (SURVEY.md 8b).  This header is what a binding for that boundary would bind; lidar_snow_sim_b200/_lib.py is the
 * ctypes binding and lidar_snow_sim_b200/snowfall/simulation.py mirrors the reference signatures on top of it.
 * Each entry point cites the reference interface it replaces (paths relative to the reference root).
 *
 * Conventions
 *   - every function returns an lss_status (0 = LSS_OK); lss_last_error() gives a human-readable message;
 *   - "d_" pointers are DEVICE pointers on the engine's device, "h_" pointers are HOST pointers;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all device work of a call is
 *     enqueued on it and the call returns without synchronising unless stated otherwise;
 *   - clouds are float32 rows (x, y, z, intensity, channel), the STF / reference layout (tools/snowfall/precompute.py:78);
 *   - no torch / C++ types cross this boundary.
 */
#ifndef LIDAR_SNOW_SIM_H
#define LIDAR_SNOW_SIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LSS_API __attribute__((visibility("default")))
#else
#define LSS_API
#endif

typedef struct lss_engine lss_engine;

typedef enum {
    LSS_OK = 0,
    LSS_ERR_INVALID_ARG = 1,
    LSS_ERR_CUDA = 2,
    LSS_ERR_NO_TABLE = 3,         /* FileNotFoundError analogue: particle table set not uploaded (simulation.py:329) */
    LSS_ERR_RANGE_INDEX = 4,      /* IndexError analogue: a waveform sample index >= 1230, i.e. a return beyond
                                     ~120 m on a beam that has occluders (simulation.py:149) */
    LSS_ERR_NEGATIVE_INTENSITY = 5,  /* AssertionError analogue (simulation.py:184) */
    LSS_ERR_OCCLUDER_OVERFLOW = 6,   /* more than 128 occluders on one beam (or > 65536 beams with more than 24) */
    LSS_ERR_WORKSPACE = 7,        /* caller-supplied workspace too small */
    LSS_ERR_NO_SENSOR = 8,        /* AssertionError analogue: sensor constants missing (simulation.py:35,474-480) */
    LSS_ERR_TOO_FEW_GROUND = 9    /* TypeError analogue: fewer than 3 ground points, estimate_laser_parameters returns
                                     None (tools/wet_ground/augmentation.py:213-214) and simulation.py:462 fails */
} lss_status;

/* flags for lss_snowfall_batch */
#define LSS_FLAG_THRESHOLD_FILTER 0x1u   /* apply keep = (label==2) | (round(I) > threshold(d))  (simulation.py:516-523) */
#define LSS_FLAG_CAMERA_FOV 0x2u         /* apply the camera field-of-view filter (simulation.py:532-540) */
#define LSS_FLAG_DEVICE_PREPASS 0x4u     /* compute ground plane + noise-threshold polynomial on the device
                                            (simulation.py:449-467) instead of taking h_thresh_poly */
#define LSS_FLAG_ASSUME_SORTED 0x8u      /* accepted for compatibility, no effect: the channel sort (simulation.py:447) is
                                            fused into the final scatter pass and costs nothing extra */

#define LSS_N_CHANNELS 64
#define LSS_POINT_STRIDE 5

/* ---- lifetime -------------------------------------------------------------------------------------------------- */
LSS_API lss_status lss_create(int device, lss_engine **out);
LSS_API void lss_destroy(lss_engine *e);
LSS_API const char *lss_status_string(lss_status s);
LSS_API const char *lss_last_error(const lss_engine *e);
LSS_API int lss_version(void);

/* ---- sensor constants ------------------------------------------------------------------------------------------
 * Replaces the YAML read of calib/20171102_64E_S3.yaml (simulation.py:474-480) and the per-channel lookups at
 * simulation.py:72-76 (min_intensity default 0, focal_distance [m as in the YAML], focal_slope) and :123-126
 * (max_intensity 255, or 230 for channels 53/55/56/58).  All arrays: n_channels doubles, host.                    */
LSS_API lss_status lss_set_sensor(lss_engine *e, int n_channels, const double *h_focal_distance, const double *h_focal_slope,
                          const double *h_min_intensity, const double *h_max_intensity);

/* Camera calibration for the FOV filter: replaces get_calib() (simulation.py:32-36) +
 * lib/OpenPCDet/pcdet/utils/calibration_kitti.py:5-20.  Row-major float32: P2[3*4], R0[3*3], V2C[3*4].            */
LSS_API lss_status lss_set_camera(lss_engine *e, const float *h_P2, const float *h_R0, const float *h_V2C, int img_h,
                          int img_w);

/* ---- particle tables ---------------------------------------------------------------------------------------------
 * Replaces np.load('<prefix>_<k>.npy') per channel (simulation.py:78,324-329).  One "table set" = the n_planes
 * (x, y, r) float64 tables of one particle_file_prefix; plane k (file index k+1) is rows
 * h_plane_offsets[k] .. h_plane_offsets[k+1] of h_xyr.  The set is preprocessed on the device into an
 * azimuth-bucketed, range-sorted candidate index and stays resident (L2-sized) until freed.
 * max_beam_divergence_rad bounds the beam_divergence later calls may use with this set.
 * Synchronises the stream before returning (the host arrays may be released afterwards).                           */
LSS_API lss_status lss_upload_particles(lss_engine *e, int n_planes, const double *h_xyr, const int64_t *h_plane_offsets,
                                double max_beam_divergence_rad, int n_azimuth_buckets, void *stream,
                                int *table_id_out);
/* same, from device-resident tables (e.g. written by lss_sample_particles) */
LSS_API lss_status lss_upload_particles_device(lss_engine *e, int n_planes, const double *d_xyr,
                                       const int64_t *h_plane_offsets, double max_beam_divergence_rad,
                                       int n_azimuth_buckets, void *stream, int *table_id_out);
LSS_API lss_status lss_free_particles(lss_engine *e, int table_id);
/* bytes of device memory held by a table set, and its number of candidate-index entries */
LSS_API lss_status lss_table_info(lss_engine *e, int table_id, int64_t *n_particles, int64_t *n_entries, int64_t *bytes);

/* ---- snowfall augmentation ---------------------------------------------------------------------------------------
 * Batched augment() (simulation.py:427-544) on device-resident clouds.
 *
 *   d_points         float32[n_total*5]   clouds concatenated; cloud b = rows h_cloud_offsets[b] .. [b+1]
 *   h_cloud_offsets  int64[n_clouds+1]    host
 *   h_order          int32[n_clouds*64]   channel -> plane index per cloud: the `order` list of simulation.py:483-486
 *                                         (the caller owns the random.shuffle so results are reproducible)
 *   beam_divergence_deg                   as in the reference (degrees; callers pass degrees(3e-3))
 *   d_theta          float32[n_total] or NULL.  Optional beam azimuths atan2(y,x) in ORIGINAL row order.  The
 *                                         reference's float32 np.arctan2 is host/SIMD dependent (SURVEY.md App. D);
 *                                         parity harnesses pass the oracle host's bits here.  NULL: computed on
 *                                         device as the correctly rounded float32 of the float64 atan2.
 *   h_thresh_poly    float64[n_clouds*3] or NULL: np.polyfit coefficients p of simulation.py:467-469 per cloud
 *                                         (required with LSS_FLAG_THRESHOLD_FILTER unless LSS_FLAG_DEVICE_PREPASS)
 *   h_plane_in       float64[n_clouds*4] or NULL, h_ymins_in int32[n_clouds*50] or NULL: with LSS_FLAG_DEVICE_PREPASS,
 *                                         the two library-defined choices of the reference's pre-pass replayed from a
 *                                         reference run (see lss_noise_threshold_poly); NULL = the device's own choice
 *   noise_floor                           simulation.py:428 (used by the device pre-pass only)
 *   flags                                 LSS_FLAG_*
 *   d_out_points     float32[n_total*5]   augmented rows (x, y, z, intensity, label), sorted by channel (stable), cloud b
 *                                         compacted to the front of its own slot: rows h_cloud_offsets[b] ..
 *                                         h_cloud_offsets[b] + count[b]; rows behind that are unspecified
 *   d_out_counts     int32[n_clouds]      rows kept per cloud
 *   d_out_stats      float64[n_clouds*4]  num_attenuated, num_removed, avg_intensity_diff, intensity_diff_sum
 *                                         (simulation.py:525-542)
 *   d_out_full       float32[n_total*5] or NULL: optional un-filtered channel-sorted rows (label column filled)
 *   d_out_perm       int32[n_total] or NULL: optional original row index (within its cloud) of each sorted row
 *   d_out_nocc       int32[n_total] or NULL: optional number of claiming occluders per (sorted) beam
 *   d_workspace / workspace_bytes         scratch; query the size with lss_snowfall_workspace_bytes
 *
 * Errors raised by the device (LSS_ERR_RANGE_INDEX, ...) are latched in the engine and reported by
 * lss_check_async() after the stream has been synchronised by the caller.                                          */
LSS_API lss_status lss_snowfall_batch(lss_engine *e, int table_id, const float *d_points, const int64_t *h_cloud_offsets,
                              int n_clouds, const int32_t *h_order, double beam_divergence_deg, const float *d_theta,
                              const double *h_thresh_poly, const double *h_plane_in, const int32_t *h_ymins_in,
                              double noise_floor, uint32_t flags, float *d_out_points,
                              int32_t *d_out_counts, double *d_out_stats, float *d_out_full, int32_t *d_out_perm,
                              int32_t *d_out_nocc, void *d_workspace, int64_t workspace_bytes, void *stream);
LSS_API int64_t lss_snowfall_workspace_bytes(int64_t n_total, int n_clouds);
/* Host-to-host batched augment(): the reference's call shape (numpy cloud in -> numpy cloud out,
 * simulation.py:427-544) for a batch.  h_points / h_out_* are HOST buffers (page-locked memory gives full PCIe speed;
 * pageable works).  The batch is cut into `n_chunks` groups of whole clouds (<= 0: default 4) that flow through
 * engine-owned streams and device buffers: H2D copy -> pre-pass -> beam stage -> D2H copy, the transfers and the
 * pre-pass of one chunk overlapping the beam kernels of another.  Arguments and the slot-compacted output layout are
 * those of lss_snowfall_batch (no d_theta / debug views); results are bit-identical to it for any n_chunks.
 *
 *   lss_snowfall_batch_host          synchronous; returns the batch's device status (LSS_ERR_RANGE_INDEX, ...) directly
 *   lss_snowfall_batch_host_submit   enqueues the batch and returns a ticket; up to 3 batches may be in flight (the
 *                                    4th submit without a wait fails with LSS_ERR_INVALID_ARG).  The host buffers must
 *                                    stay valid and untouched until the ticket has been waited for.  With 2-3 batches
 *                                    in flight -- a prefetching data loader -- batch k+1's copy-in, batch k's kernels
 *                                    and batch k-1's copy-out run concurrently.
 *   lss_snowfall_batch_host_wait     blocks until that batch's results are in its host buffers; returns its status   */
LSS_API lss_status lss_snowfall_batch_host(lss_engine *e, int table_id, const float *h_points,
                                           const int64_t *h_cloud_offsets, int n_clouds, const int32_t *h_order,
                                           double beam_divergence_deg, const double *h_thresh_poly, double noise_floor,
                                           uint32_t flags, int n_chunks, float *h_out_points, int32_t *h_out_counts,
                                           double *h_out_stats);
LSS_API lss_status lss_snowfall_batch_host_submit(lss_engine *e, int table_id, const float *h_points,
                                                  const int64_t *h_cloud_offsets, int n_clouds, const int32_t *h_order,
                                                  double beam_divergence_deg, const double *h_thresh_poly,
                                                  double noise_floor, uint32_t flags, int n_chunks, float *h_out_points,
                                                  int32_t *h_out_counts, double *h_out_stats, int *ticket_out);
LSS_API lss_status lss_snowfall_batch_host_wait(lss_engine *e, int ticket);
/* Diagnostic: device timeline of the most recently waited batch.  out[4*c + k] = milliseconds from the batch's first
 * enqueued operation until chunk c's rows are on the device (k=0), its threshold polynomial is ready (1), its beam stage
 * is done (2), its results are on the host (3).  Returns the number of chunks written (<= cap_chunks).               */
LSS_API int lss_host_pipe_trace(lss_engine *e, float *out, int cap_chunks);
/* Synchronises `stream`, then returns and clears the latched asynchronous device status.                          */
LSS_API lss_status lss_check_async(lss_engine *e, void *stream);
/* number of kernel launches the engine has enqueued since creation (bench.py's gpu_launches) */
LSS_API int64_t lss_launch_count(const lss_engine *e);
/* ---- per-cloud pre-pass ----------------------------------------------------------------------------------------------
 * Ground plane (calculate_plane, tools/wet_ground/planes.py:12-50), ground mask + incident angle
 * (simulation.py:450-455), estimate_laser_parameters (tools/wet_ground/augmentation.py:195-266, 'linear') and the
 * degree-2 noise-threshold polynomial (simulation.py:462-467) for every cloud of a batch.  lss_snowfall_batch runs
 * the same code with LSS_FLAG_DEVICE_PREPASS; this entry point exposes the results.
 *   h_plane_in   float64[n_clouds*4] (w0, w1, w2, h) or NULL.  NULL: estimated on the device (deterministic RANSAC).
 *                The reference's plane comes from sklearn's RANSAC on NumPy's global RNG (planes.py:35).
 *   h_ymins_in   int32[n_clouds*50] or NULL: per cloud and range bin, the intensity-bin index the reference host picked
 *                with np.argpartition(hist, 2, axis=1)[:, 0] (augmentation.py:236) -- an implementation-defined one of the
 *                least populated bins (AVX-512 / AVX2 / scalar NumPy builds pick differently).  NULL: the device takes the
 *                FIRST least populated bin (NumPy's portable introselect).  With both inputs replayed from a reference
 *                run everything downstream is comparable with that run's outputs (tests/golden/).
 *   d_poly_out   float64[n_clouds*3]  np.polyfit order (highest power first), device
 *   d_plane_out  float64[n_clouds*4] or NULL, device
 *   d_fit_out    float64[n_clouds*8] or NULL, device: linregress slope, intercept of I/cos over range
 *                (augmentation.py:216-219); slope, intercept of the per-bin minima fit (:249); ymax (:233); n_ground;
 *                points in the mounting window (planes.py:21-27); 1 if the flat-earth fallback was taken (:29-32)
 *   d_ymins_out  int32[n_clouds*50] or NULL, device: the picks used (-1: fewer than 3 ground points)                    */
LSS_API lss_status lss_noise_threshold_poly(lss_engine *e, const float *d_points, const int64_t *h_cloud_offsets,
                                    int n_clouds, double noise_floor, const double *h_plane_in,
                                    const int32_t *h_ymins_in, double *d_poly_out, double *d_plane_out,
                                    double *d_fit_out, int32_t *d_ymins_out, void *d_workspace,
                                    int64_t workspace_bytes, void *stream);
LSS_API int64_t lss_prepass_workspace_bytes(int64_t n_total, int n_clouds);

/* ---- wet-ground augmentation ------------------------------------------------------------------------------------------
 * Batched ground_water_augmentation() (tools/wet_ground/augmentation.py:25-161, estimation_method='linear') with the
 * Fresnel chain of tools/wet_ground/phy_equations.py:35-108, on device-resident clouds.
 *   d_points          float32[n_total*5]; cloud b starts at row h_cloud_offsets[b]
 *   d_cloud_counts    int32[n_clouds] device or NULL: valid rows per cloud when the input is the slot-compacted output of
 *                     lss_snowfall_batch (fused snow -> wet path); NULL: h_cloud_offsets[b+1] - h_cloud_offsets[b]
 *   water_height, pavement_depth, noise_floor, power_factor, flat_earth, delta, replace: as in the reference signature
 *   h_plane_in        float64[n_clouds*4] (w0, w1, w2, h) or NULL (device RANSAC, planes.py:12-50)
 *   h_ymins_in        int32[n_clouds*50] or NULL: replayed np.argpartition picks, see lss_noise_threshold_poly
 *   d_out_points      float32[n_total*5]: per cloud, non-ground rows first, then the kept ground rows (:150-159),
 *                     compacted to the front of the cloud's slot
 *   d_out_intensity64 float64[n_total] or NULL: column 3 of the output rows in the reference's float64
 *   d_out_counts      int32[n_clouds]
 *   d_out_passthrough int32[n_clouds] or NULL: 1 where the cloud had < 1000 ground points and is returned unchanged (:51-52)
 *   d_out_plane       float64[n_clouds*4] or NULL                                                                       */
LSS_API lss_status lss_wet_ground_batch(lss_engine *e, const float *d_points, const int64_t *h_cloud_offsets,
                                const int32_t *d_cloud_counts, int n_clouds, double water_height, double pavement_depth,
                                double noise_floor, double power_factor, int flat_earth, double delta, int replace,
                                const double *h_plane_in, const int32_t *h_ymins_in, float *d_out_points,
                                double *d_out_intensity64, int32_t *d_out_counts, int32_t *d_out_passthrough,
                                double *d_out_plane, void *d_workspace, int64_t workspace_bytes, void *stream);
LSS_API int64_t lss_wet_ground_workspace_bytes(int64_t n_total, int n_clouds);

/* ---- fog simulation ("next" row, SURVEY.md 8f-3) -----------------------------------------------------------------------
 * Batched simulate_fog() (lib/LiDAR_fog_sim/fog_simulation.py:299-316: P_R_fog_hard :183-189, P_R_fog_soft :192-296) on
 * device-resident clouds of n_features (>= 4: x, y, z, intensity, ...) float32 columns.
 *   alpha, beta, beta_0   the ParameterSet fields the reference reads (:66, :73, :168)
 *   d_lut     float64[2001*2]  the integral look-up table the reference unpickles (get_integral_dict, :174-180) as
 *                              (fog_distance, fog_response) per 0.1 m of range 0 .. 200 m; device memory
 *   flags     LSS_FOG_HARD | LSS_FOG_SOFT | LSS_FOG_GAIN   (hard=, soft=, gain= of simulate_fog)
 *   noise, noise_variant       `noise` (0: none) and 1..4 for 'v1'..'v4' (:237-266)
 *   h_rng_state  uint64[n_clouds*4] or NULL: per cloud the PCG64 state {state_hi, state_lo, inc_hi, inc_lo} of the
 *                caller's numpy Generator AFTER the one `integers` draw of :207.  Fog point number k of a cloud (in point
 *                order) uses the generator's k-th next double, exactly like the reference's sequential draws; the
 *                caller advances its generator by the returned count afterwards.  Used for variants 1-3.
 *   d_ext_noise  float64[n_total] or NULL: externally drawn values by (cloud offset + rank) instead: uniforms in [0,1)
 *                for variants 1-3, Generator.beta(2, 20) draws for variant 4 (rejection sampling cannot jump ahead:
 *                call once without it to get ranks and counts, draw, call again).  Variant 4 without it: no noise.
 *   d_out        float64[n_total*n_features]  augmented rows in input order (float32 valued when only LSS_FOG_HARD)
 *   d_out_fog_mask uint8[n_total]             1 = the fog response replaced the return (simulated_fog_pc = rows with 1)
 *   d_out_rank   int32[n_total] or NULL       rank of each fog point among its cloud's fog points, -1 elsewhere
 *   d_out_info   float64[n_clouds*3]          min_fog_response (inf if none), max_fog_response, num_fog_responses
 * Parity: masks, ranks, counts and the random stream are exact; intensities / coordinates agree to float64 rounding
 * except where the reference itself is host-defined (float32 np.exp, scalar float32 power, pow): DESIGN.md 8.          */
#define LSS_FOG_HARD 0x1u
#define LSS_FOG_SOFT 0x2u
#define LSS_FOG_GAIN 0x4u
LSS_API lss_status lss_fog_batch(lss_engine *e, const float *d_points, int n_features, const int64_t *h_cloud_offsets,
                                 int n_clouds, double alpha, double beta, double beta_0, const double *d_lut,
                                 uint32_t flags, int noise, int noise_variant, const uint64_t *h_rng_state,
                                 const double *d_ext_noise, double *d_out, uint8_t *d_out_fog_mask, int32_t *d_out_rank,
                                 double *d_out_info, void *d_workspace, int64_t workspace_bytes, void *stream);
LSS_API int64_t lss_fog_workspace_bytes(int64_t n_total, int n_clouds);

/* ---- LISA Monte-Carlo rain / snow augmenter ("next" row, SURVEY.md 8f-3) ----------------------------------------------
 * LISA.monte_carlo_augment (lib/LISA/python/lisa.py:293-341) with the per-return experiment monte_carlo_lisa (:34-190) on
 * device-resident returns; caller: DenseDataset.__getitem__ (lib/OpenPCDet/pcdet/datasets/dense/dense_dataset.py:713-746).
 *   d_points      float64[n_points * n_features] (x, y, z, intensity in [0, 1], ...), n_features >= 4 -- the reference
 *                 feeds float64 (dense_dataset.py:732-734)
 *   rain_rate     Rr [mm/h];  mode 0 'rain' (Marshall-Palmer), 1 'gunn' (Marshall-Gunn), 2 'sekhon' (Sekhon-Srivastava)
 *   alpha         extinction coefficient [1/m] = LISA.alpha(LISA.Nd(D, Rr)) (:468-482), integrated by the caller from the
 *                 Mie efficiency table (the reference's data file mie_<n>_lambda_<wl>.npz)
 *   r_min, r_max, beam_divergence, min_diameter, range_accuracy   the LISA constructor arguments (:193-195)
 *   signal_last   0 = 'strongest' return, 1 = 'last'
 *   d_draw_table  float64[table_len] device or NULL.  Not NULL = the reference's fixed_seed mode (:54-55: every return
 *                 re-seeds NumPy's MT19937 with 666): the doubles np.random.RandomState(666).random_sample(table_len)
 *                 produces, which every return consumes from the start (one for the particle count, then ranges, then
 *                 diameters, then pairs for the polar Gaussian).  LSS_ERR_WORKSPACE (asynchronous, lss_check_async) if a
 *                 return needs more than table_len draws.  NULL: counter-based generator keyed by (seed, return index).
 *   d_out         float64[n_points * (n_features + 2)]: x, y, z, intensity, label (0 lost, 1 not scattered, 2 scattered),
 *                 intensity_diff, zeros
 * Parity (fixed-seed): labels, particle choices and the stream position exact; values to libm rounding (pow, log, exp).  */
LSS_API lss_status lss_lisa_batch(lss_engine *e, const double *d_points, int n_features, int64_t n_points, double rain_rate,
                                  int mode, double alpha, double r_min, double r_max, double beam_divergence,
                                  double min_diameter, double range_accuracy, int signal_last,
                                  const double *d_draw_table, int table_len, uint64_t seed, double *d_out, void *stream);

/* ---- point-range mask + voxelisation ("next" row, SURVEY.md 8f-4) ---------------------------------------------------------
 * The detector-input stage of the reference's data path on device-resident clouds, e.g. the slot-compacted output of
 * lss_snowfall_batch / lss_wet_ground_batch, so that the augmented batch reaches the detector without a host round trip:
 *   DataProcessor.mask_points_and_boxes_outside_range (points part)   lib/OpenPCDet/pcdet/datasets/processor/data_processor.py:78-91
 *       = mask_points_by_range, lib/OpenPCDet/pcdet/utils/common_utils.py:60-63: x and y inside the range, ends inclusive
 *   DataProcessor.transform_points_to_voxels                             data_processor.py:115-143 -> VoxelGeneratorWrapper
 *       (:15-58) -> spconv's point-to-voxel rule (third party; restated in oracle/voxel.py): float32
 *       c = floor((p - range_min) / voxel_size), points outside the grid skipped, voxels numbered by first appearance in
 *       point order, at most max_voxels voxels, the first max_points_per_voxel points of a voxel kept in point order
 *   batch index column of DatasetTemplate.collate_batch                  lib/OpenPCDet/pcdet/datasets/dataset.py:199-204
 *
 *   d_points            float32[n_total * n_features], n_features >= 3 (x, y, z, ...); cloud b starts at row h_cloud_offsets[b]
 *   d_cloud_counts      int32[n_clouds] device or NULL: valid rows per cloud slot (slot-compacted input)
 *   h_point_cloud_range float32[6] (x0, y0, z0, x1, y1, z1); h_voxel_size float32[3]     (dense_dataset.yaml:4,71)
 *   mask_xy_range       != 0: apply the x / y range mask first (it differs from the grid test at the upper edge)
 *   d_out_voxels        float32[n_clouds * max_voxels * max_points_per_voxel * n_features], zero padded
 *   d_out_coords        int32[n_clouds * max_voxels * 4]   (cloud index, z, y, x)
 *   d_out_num_points    int32[n_clouds * max_voxels]
 *   d_out_n_voxels      int32[n_clouds]; cloud b's voxels are rows [0, n_voxels[b]) of its slot of max_voxels rows
 * Results are bit-identical to the sequential rule (integer reductions only).                                           */
LSS_API lss_status lss_voxelize_batch(lss_engine *e, const float *d_points, int n_features, const int64_t *h_cloud_offsets,
                                      const int32_t *d_cloud_counts, int n_clouds, const float *h_point_cloud_range,
                                      const float *h_voxel_size, int max_points_per_voxel, int max_voxels,
                                      int mask_xy_range, float *d_out_voxels, int32_t *d_out_coords,
                                      int32_t *d_out_num_points, int32_t *d_out_n_voxels, void *d_workspace,
                                      int64_t workspace_bytes, void *stream);
LSS_API int64_t lss_voxelize_workspace_bytes(int64_t n_total, int n_clouds, int max_points_per_voxel, int max_voxels);

/* ---- dynamic radius outlier removal (DROR) ----------------------------------------------------------------------------
 * dynamic_radius_outlier_filter (lib/cadc_devkit/other/dror.py:288-334), the de-snowing filter whose snow indices the DENSE
 * data path reads from per-frame pickles (lib/OpenPCDet/pcdet/datasets/dense/dense_dataset.py:588-616), computed on
 * device-resident clouds, e.g. the slot-compacted output of lss_snowfall_batch.  Rule (DESIGN.md 7.4): with
 *     sr_i = max(alpha_deg * beta * pi / 180 * sqrt(x_i^2 + y_i^2), sr_min)     float64 (dror.py:316-321)
 *     d2_ij = ((0 + dx^2) + dy^2) + dz^2                                        float32, FLANN's L2_Simple order
 * point i is kept iff at least k_min + 1 points j of its cloud, i included, have sqrt((double)d2_ij) < sr_i -- what the
 * reference's k = k_min + 1 nearest-neighbour count decides (dror.py:311-334).  Integer result: exact, deterministic.
 *   d_points        float32[n_total * n_features], n_features >= 3; xyz are read, every column is copied
 *   d_cloud_counts  int32[n_clouds] device or NULL: valid rows per cloud slot (slot-compacted input)
 *   h_crop_xy       float32[4] (x0, x1, y0, y1) or NULL.  Not NULL = the `crop` variant of process_dense (dror.py:238-256):
 *                   only rows with x0 <= x <= x1 and y0 <= y <= y1 (get_cube_mask, :73-84, whose z test has no effect)
 *                   take part; the others get code 2
 *   d_codes         uint8[n_total]: 0 snow, 1 kept, 2 outside the crop (rows behind a cloud's count are not written)
 *   d_out_points    float32[n_total * n_features] or NULL (codes and counts only): per cloud the kept rows in input
 *                   order, compacted to the front of the cloud's slot, as lss_snowfall_batch lays out its output
 *   d_out_counts    int32[n_clouds] kept rows;  d_out_n_snow  int32[n_clouds] rows with code 0
 *   d_workspace     lss_dror_workspace_bytes(n_total, n_clouds) bytes (-1 there: no usable CUDA device)            */
LSS_API lss_status lss_dror_batch(lss_engine *e, const float *d_points, int n_features, const int64_t *h_cloud_offsets,
                                  const int32_t *d_cloud_counts, int n_clouds, double alpha_deg, double beta, int k_min,
                                  double sr_min, const float *h_crop_xy, uint8_t *d_codes, float *d_out_points,
                                  int32_t *d_out_counts, int32_t *d_out_n_snow, void *d_workspace,
                                  int64_t workspace_bytes, void *stream);
LSS_API int64_t lss_dror_workspace_bytes(int64_t n_total, int n_clouds);

/* ---- exchange step of the sharded batch (SURVEY.md 8e, BASELINE.json configs[3]) ------------------------------------------
 * The reference has no multi-GPU augmentation; its collectives are OpenPCDet's result merging
 * (lib/OpenPCDet/pcdet/utils/commu_utils.py:77,90: all_gather of pickled, variable-size objects).  The sharded engine
 * reassembles the augmented batch on every rank instead: gathered row buffer float32[world * n_rows * 5] (rank r's
 * slot-compacted batch at rows [r * n_rows, (r + 1) * n_rows)) and gathered counts int32[world * n_clouds].
 * lss_gather_push writes the KEPT rows of this rank's batch (cloud b: rows [off[b], off[b] + count[b])) and its counts into
 * every rank's gathered buffers with peer-to-peer stores over NVLink -- one small kernel (CTAs of 128 threads x 32 registers,
 * which fit next to the persistent solve kernel of the following step), no library collective, no whole-slot copy.
 *   d_points / d_counts / d_cloud_offsets   this rank's output of lss_snowfall_batch (counts may be NULL: all rows), offsets on
 *                       the DEVICE (int64[n_clouds + 1])
 *   h_peer_points[world], h_peer_counts[world]   host arrays of DEVICE pointers: every rank's gathered buffers as mapped into
 *                       this process (peer mappings of a symmetric allocation; entry `rank` is the local buffer)
 *   d_mc_points / d_mc_counts   multicast (NVLS) mappings of the same allocations, or both NULL: then one store per peer
 *   n_blocks            CTAs to launch (<= 0: a quarter of the SMs with multicast, 64 with per-peer stores: the measured optima)
 * Stream-ordered on `stream`; a consumer on ANOTHER rank needs a barrier across ranks after this rank's kernel has finished. */
LSS_API lss_status lss_gather_push(lss_engine *e, const float *d_points, const int32_t *d_counts,
                                   const int64_t *d_cloud_offsets, int n_clouds, int64_t n_rows, int world, int rank,
                                   float *const *h_peer_points, int32_t *const *h_peer_counts, float *d_mc_points,
                                   int32_t *d_mc_counts, int n_blocks, void *stream);

/* ---- snowflake table sampler ---------------------------------------------------------------------------------------
 * dart_throwing(occupancy_ratio, precipitation_rate, R_0, rng, distribution) of tools/snowfall/sampling.py:90-194:
 * sequential rejection sampling of non-overlapping disks in a disk of radius R_0 until the occupied area reaches
 * occupancy_ratio * pi * R_0^2.  Host-native (uniform grid instead of the reference's O(N^2) scan); consumes NumPy's
 * PCG64 stream exactly like the reference, so the same Generator state yields the same table.
 *   distribution   0 = 'gunn', 1 = 'sekhon'                       (sampling.py:108-113)
 *   pcg_state      uint64[4] in/out: {state_hi, state_lo, inc_hi, inc_lo} of numpy's PCG64
 *   h_xyr          float64[capacity*3] out: (x, y, r) rows         n_out: rows written
 * Needs no GPU.  LSS_ERR_WORKSPACE if `capacity` rows do not suffice.                                               */
LSS_API lss_status lss_dart_throwing(double occupancy_ratio, double precipitation_rate, double R_0, int distribution,
                             uint64_t *pcg_state, double *h_xyr, int64_t capacity, int64_t *n_out);
/* n_planes independent planes (sampling.py:410-413), one host thread per plane up to n_threads (<= 0: all cores).
 * pcg_states uint64[n_planes*4]; plane k -> h_xyr + 3*k*capacity_per_plane, h_counts[k] rows.                        */
LSS_API lss_status lss_dart_throwing_planes(int n_planes, double occupancy_ratio, double precipitation_rate, double R_0,
                                    int distribution, uint64_t *pcg_states, double *h_xyr,
                                    int64_t capacity_per_plane, int64_t *h_counts, int n_threads);

/* Device-resident sampler: the same greedy dart throwing for n_planes planes at once, entirely on the GPU, written to
 * device memory (feed lss_upload_particles_device).  The acceptance rule and the stop criterion are the reference's;
 * the random stream is a counter-based generator keyed by (seed, plane, dart) instead of NumPy's PCG64, so parity with
 * the reference's tables is statistical (use lss_dart_throwing for stream-exact tables).
 *   n_candidates       darts thrown per plane (must be enough to reach the occupancy: LSS_ERR_WORKSPACE otherwise)
 *   d_xyr_out          float64[n_planes * capacity_per_plane * 3]: plane p at offset p * capacity_per_plane rows
 *   d_counts           int32[n_planes] accepted rows per plane
 *   d_candidates_out   float64[n_planes * n_candidates * 3] or NULL: every dart in throw order (test hook)
 * Synchronises the stream.                                                                                              */
LSS_API lss_status lss_sample_particles(lss_engine *e, int n_planes, double occupancy_ratio, double precipitation_rate,
                                double R_0, int distribution, uint64_t seed, int64_t n_candidates, double *d_xyr_out,
                                int64_t capacity_per_plane, int32_t *d_counts, double *d_candidates_out,
                                void *d_workspace, int64_t workspace_bytes, void *stream);
LSS_API int64_t lss_sample_particles_workspace_bytes(int n_planes, int64_t n_candidates);

/* Optional per-kernel timing for bench.py's roofline: when enabled every kernel launch is bracketed by CUDA events
 * on the launching stream.  lss_kernel_times() (call after synchronising) accumulates and returns, per kernel id
 * 0..n-1 (names via lss_kernel_name), total milliseconds and number of launches; reset != 0 clears the totals.     */
LSS_API lss_status lss_set_profiling(lss_engine *e, int enable);
LSS_API lss_status lss_kernel_times(lss_engine *e, int reset, double *h_ms, int64_t *h_calls, int n);
LSS_API const char *lss_kernel_name(int kernel);
/* test hook: the beam azimuth the kernels compute when no d_theta is supplied, (float)atan2((double)y, (double)x)
 * (simulation.py:91), element-wise on device arrays of n float32 values                                              */
LSS_API lss_status lss_debug_azimuth(lss_engine *e, const float *d_y, const float *d_x, int64_t n, float *d_out, void *stream);
/* test hook: the engine's range grid R = np.round(np.linspace(0, 120 + c*tau_h, 1230), 2) (simulation.py:111-116),
 * 1230 doubles written to h_out.  Host only, needs no GPU.                                                          */
LSS_API lss_status lss_debug_range_grid(double *h_out);

#ifdef __cplusplus
}
#endif
#endif /* LIDAR_SNOW_SIM_H */

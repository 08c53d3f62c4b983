/*
 * drs.h -- C-ABI of libdrs.so, the B200-native (sm_100a) hot path of
 * keillernogueira/dynamic-rs-segmentation.
 *
 * The reference has no FFI: its compute seam is `tf.Session.run(fetches, feed_dict)`
 * called from the three Python scripts, plus the NumPy host loops either side of it
 * (SURVEY.md section 8b).  Each entry point below names the reference interface it
 * replaces (file:line under /root/reference).  Conventions:
 *   - one handle per process / GPU, not thread-safe;
 *   - every function returns 0 on success, non-zero on error; the message is
 *     available from drs_last_error();
 *   - pointers ending in _host are host memory owned by the caller (the NumPy buffers
 *     of feed_dict / the fetched arrays); pointers ending in _dev are device memory
 *     owned by the caller; the library owns weights, optimizer slots and workspace;
 *   - work is enqueued on the handle's stream (drs_set_stream); *_host entry points
 *     synchronise that stream before returning, *_dev entry points do not;
 *   - tensors are NHWC, weights HWIO [kh,kw,Ci,Co], labels/pred are class ids.
 * There is no CPU fallback: every compute entry point fails if no sm_100 device is present.
 */
#ifndef DRS_H_
#define DRS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct drs_handle_s* drs_handle_t;

/* net_type keys of the scripts' CLI (isprs:1660-1680, contest:996-1013, coffee:1197-1220) */
enum drs_net_type {
  DRS_NET_DILATED6 = 0,          /* dilated_icpr_original      isprs:761-788  */
  DRS_NET_DILATED6_POOLING = 1,  /* dilated_grsl               isprs:962-993  */
  DRS_NET_DENSE_DILATED6 = 2,    /* dilated_icpr_rate6_densely isprs:914-959  */
  DRS_NET_DILATED8_POOLING = 3,  /* dilated_grsl_rate8 / dilated8_grsl isprs:996-1033 */
  /* plain six-layer stacks of the same primitives (SURVEY section 8f, N4) */
  DRS_NET_RATE6 = 4,             /* dilated_icpr_rate6            isprs:886-911  rates 1..6, ReLU, no pooling */
  DRS_NET_RATE6_SMALL = 5,       /* dilated_icpr_rate6_small      isprs:791-816  64,64,64,128,128,128 */
  DRS_NET_RATE6_NODILATION = 6,  /* dilated_icpr_rate6_nodilation isprs:852-883  tf.nn.conv2d (rate 1) */
  DRS_NET_RATE1 = 7,             /* dilated_icpr_rate1            coffee:788-813 every rate 1 */
  DRS_NET_VARY_RATE = 8,         /* dilated_icpr_vary_rate        coffee:816-841 rates 1,2,4,1,2,4 */
  DRS_NET_ICPR_OLD = 9,          /* dilated_icpr_old              contest:574-603 three layers, scopes conv1/conv3/conv5 */
  /* structural variants (csrc/variants.cuh): same conv stack as dilated_icpr_rate6 plus a new layer type */
  DRS_NET_RATE6_AVGPOOL = 10,    /* dilated_icpr_rate6_avgpool    isprs:819-849  SAME average pooling 5x5 / 7x7 behind conv1..5 */
  DRS_NET_RATE6_SE = 11,         /* dilated_icpr_rate6_SE         isprs:1036-1061 squeeze-and-excitation gate behind conv2/4/6 */
  DRS_NET_RATE6_SQUEEZE = 12     /* dilated_icpr_rate6_squeeze    isprs:1064-1086 conv2..6 as squeeze modules (1x1 -> 1x1 || kxk) */
  /* contest's dilated_grsl_old (contest:606-636) is dilated_grsl with 3 input channels: DRS_NET_DILATED6_POOLING */
};

/* arithmetic of the convolution stack */
enum drs_precision {
  DRS_PREC_FP32 = 0,  /* CUDA-core fp32, fixed reduction order (exact-order mode)          */
  DRS_PREC_F16 = 1,   /* tcgen05 kind::f16, fp16 operands, fp32 accumulate in TMEM           */
  DRS_PREC_BF16 = 2   /* tcgen05 kind::f16, bf16 operands, fp32 accumulate (training default) */
};

enum drs_scene_dtype { DRS_SCENE_F64 = 0, DRS_SCENE_F32 = 1 };

/* sliding-window variants (SURVEY.md Appendix C): which script's create_patches_per_map */
enum drs_grid_variant { DRS_GRID_ISPRS = 0, DRS_GRID_CONTEST = 1, DRS_GRID_COFFEE = 2 };

typedef struct drs_config {
  int32_t net_type;        /* enum drs_net_type */
  int32_t channels;        /* input channels C (Vaihingen 4, Potsdam 5, contest/coffee 3) */
  int32_t num_classes;     /* K (6 / 7 / 2) */
  int32_t precision;       /* enum drs_precision */
  float weight_decay;      /* isprs:640-652: wd * l2_loss(W) for every `weights` variable */
  float lr_initial;        /* isprs:1686 exponential_decay(lr_initial, step, decay_steps, decay_rate, staircase) */
  int32_t decay_steps;     /* 50000 */
  float decay_rate;        /* 0.5 isprs / 0.1 contest, coffee */
  float momentum;          /* 0.9, isprs:1687 MomentumOptimizer */
  float bn_decay;          /* 0.999, tf.contrib.layers.batch_norm default (isprs:658) */
  float bn_eps;            /* 0.001 */
  int32_t bn_unbiased_ema; /* 1: moving_variance EMA fed with the Bessel-corrected batch variance (fused TF path) */
  int32_t device;          /* CUDA device ordinal */
  int32_t isprs_scopes;    /* 1: Dilated6 variables are named main_conv1..6 (isprs:766-777) instead of conv1..6 */
} drs_config;

/* ---- life cycle ------------------------------------------------------------------- */
int drs_create(drs_handle_t* out, const drs_config* cfg);
int drs_destroy(drs_handle_t h);
const char* drs_last_error(void);
int drs_version(void);
/* cudaStream_t to enqueue on: any stream handle incl. 0 (the legacy default stream, what torch uses unless told otherwise);
 * (void*)-1 = back to the handle's own non-blocking stream, which is the initial state. */
int drs_set_stream(drs_handle_t h, void* cuda_stream);
int drs_synchronize(drs_handle_t h);

/* ---- variables: tf.train.Saver / sess.run(init) (isprs:1693-1717) ------------------- */
/* Variables are addressed by TF scope name: "<scope>/weights", "<scope>/biases",
 * "<scope>/moving_mean", "<scope>/moving_variance", "<scope>/weights/Momentum",
 * "<scope>/biases/Momentum", and the scalar "global_step". */
int drs_num_variables(drs_handle_t h);
int drs_variable_name(drs_handle_t h, int index, char* name_out, int name_cap, int64_t* count_out);
int drs_set_variable(drs_handle_t h, const char* name, const float* data_host, int64_t count);
int drs_get_variable(drs_handle_t h, const char* name, float* data_host, int64_t count);
/* gradient of the last train step w.r.t. a trainable variable (parity tests) */
int drs_get_gradient(drs_handle_t h, const char* name, float* data_host, int64_t count);

/* ---- checkpoints: saver.save(sess, output_path + 'model', global_step=step) (isprs:1797-1802) and
 * saver.restore(sess, model_path) (isprs:1693-1717; contest:1035-1056; coffee:1233-1262) ------------------------------- */
/* One uncompressed .npz (what numpy.savez writes, numpy.load reads): a float32 array per variable of drs_variable_name(),
 * named by the TF variable with '/' written as "__" ("conv1__weights", "conv1__weights__Momentum", "conv1__moving_mean",
 * "global_step"), filters in TF's HWIO shape, so that a TF checkpoint can be converted with tf.train.load_variable +
 * numpy.savez alone.  drs_save writes "<path>.tmp.<pid>" and renames it over <path> (a reader never sees half a file);
 * drs_load validates every member against the model (names, element counts, CRC-32) before it changes anything, accepts
 * float32 / float64 / int32 / int64 payloads, any subset of the variables, and refuses compressed archives.
 * Restoring and continuing is bit-identical to not having stopped (tests/test_gpu_parity.py). */
int drs_save(drs_handle_t h, const char* path);
int drs_load(drs_handle_t h, const char* path);
/* The container without a handle or a device (inspection / conversion tools, CPU tests).
 *   drs_npz_write: n arrays; names[i] is the member name without ".npy"; dims is n x 4 (the first ndim[i] entries used).
 *   drs_npz_entry: *total_out = number of arrays; index < 0 asks for the count only; otherwise name / shape / element count
 *                  of the index-th array in archive order.
 *   drs_npz_read:  the named array converted to float32 into out[count]. */
int drs_npz_write(const char* path, int32_t n, const char* const* names, const float* const* data, const int32_t* ndim,
                  const int64_t* dims);
int drs_npz_entry(const char* path, int32_t index, char* name_out, int32_t name_cap, int32_t* ndim_out, int64_t* dims_out,
                  int64_t* count_out, int32_t* total_out);
int drs_npz_read(const char* path, const char* name, float* out, int64_t count);

/* ---- compute seam: sess.run ---------------------------------------------------------- */
/* infer:  sess.run([pred_up, logits], is_training=False)   isprs:1274-1275, contest:929-931, coffee:1058-1059
 *   x       [B, crop*crop*C] fp32 (row-major NHWC, isprs:763)
 *   logits  [B, crop, crop, K] fp32 (may be NULL)
 *   pred    [B, crop, crop] int64 on the host path (tf.argmax, isprs:1690), uint8 on the device path (may be NULL) */
int drs_forward_host(drs_handle_t h, const float* x_host, int32_t B, int32_t crop,
                     float* logits_host, int64_t* pred_host);
int drs_forward_dev(drs_handle_t h, const float* x_dev, int32_t B, int32_t crop,
                    float* logits_dev, uint8_t* pred_dev);

/* train:  sess.run([optimizer, loss, pred_up], is_training=True)  isprs:1750-1752, contest:1083-1086, coffee:1295-1297
 *   y     [B, crop*crop] class ids fed as float32 (isprs:1654, cast isprs:1091)
 *   mask  [B, crop*crop] 0/1 bytes or NULL (contest boolean_mask, contest:886-888)
 *   loss  CE mean (+mask) + sum wd*l2_loss(W), with pre-update weights (isprs:1089-1099)
 *   pred  argmax of the same train-mode forward
 *   cm    K*K uint32 confusion counts + [K*K] = #correct, of (y, pred)
 *         (calc_accuracy_by_crop, isprs:510-531) -- fused so that the host loop disappears; may be NULL.
 *         Counted over acc_mask when given (isprs b_mask: False in the corners of rotated patches,
 *         isprs:285-296, 1754), else over mask, else over every pixel. */
int drs_train_step_host(drs_handle_t h, const float* x_host, const float* y_host, const uint8_t* mask_host,
                        const uint8_t* acc_mask_host, int32_t B, int32_t crop, float* loss_out, int64_t* pred_host,
                        uint32_t* cm_host);
int drs_train_step_dev(drs_handle_t h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                       const uint8_t* acc_mask_dev, int32_t B, int32_t crop, float* loss_out_host, uint8_t* pred_dev,
                       uint32_t* cm_dev);

/* The train step of the pipelined loop: identical work, but nothing is waited for.  The loss and the confusion counts of
 * the step are copied into a pinned result slot behind an event; drs_train_result(ticket) waits for that event only and
 * returns them.  At most 8 steps may be outstanding (the result ring); tickets count up from 0.  The reference's loop
 * needs loss / counts only for the score update and the log lines (isprs:1754-1778), which do not feed the next draws. */
int drs_train_step_async(drs_handle_t h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                         const uint8_t* acc_mask_dev, int32_t B, int32_t crop, uint8_t* pred_dev, int64_t* ticket_out);
int drs_train_result(drs_handle_t h, int64_t ticket, float* loss_out, uint32_t* cm_out);

/* Size the workspace (and the host-path staging buffers) once for the largest batch / patch size of the run, so that no
 * re-allocation happens when a larger patch size is drawn later (the patch-size interval is known up front: probValues). */
int drs_reserve_workspace(drs_handle_t h, int32_t B, int32_t crop_max, int32_t training);

/* Optional warm-up for the dynamic patch sizes: captures the CUDA graph of drs_train_step_dev for this (B, crop, buffers)
 * without executing it, so that the first real step of every patch size replays instead of capturing (the analogue of
 * TF building its graph before the loop, isprs:1652-1693).  Nothing is computed and no variable changes. */
int drs_train_prepare(drs_handle_t h, const float* x_dev, const float* y_dev, const uint8_t* mask_dev,
                      const uint8_t* acc_mask_dev, int32_t B, int32_t crop, uint8_t* pred_dev, uint32_t* cm_dev);

/* contest: pixels whose label equals `label` (7 = unlabelled, contest:236-239) are excluded from the loss mean, the
 * gradient and the fused confusion counts when no explicit mask is passed -- the boolean_mask of contest:886-897 derived
 * on the device from the labels the gather kernel produced.  label < 0 (default) disables it. */
int drs_set_ignore_label(drs_handle_t h, int32_t label);

/* Data-parallel exchange hook: called on the handle's stream order with a device buffer that must be
 * summed over ranks in place (flat gradients ++ loss numerator ++ confusion counts; and, when
 * sync_bn != 0, the per-layer BN statistics).  NULL = single process.  The reference has no
 * multi-device code; this is the one exchange step of the sharded path (SURVEY.md section 8e). */
typedef int (*drs_allreduce_fn)(void* user, float* buf_dev, int64_t count, void* cuda_stream);
int drs_set_allreduce(drs_handle_t h, drs_allreduce_fn fn, void* user, int32_t world_size, int32_t sync_bn);

/* In-library exchange (csrc/drs_comm.cuh): NCCL over NVLink / NVSwitch, dlopen'ed at run time (libnccl.so.2; a process that
 * already holds torch's bundled copy gets the same instance).  Rank 0 obtains a 128-byte id, the host distributes it (any
 * transport: torch.distributed, MPI, a file), every rank calls drs_comm_init.  From then on the step's exchanges are
 * ncclAllReduce calls on the handle's streams -- no host callback, so the data-parallel step is captured as a CUDA graph
 * like the single-GPU one -- and drs_set_allreduce is ignored.  sync_bn != 0: the per-layer BN sums are reduced over the
 * global batch forward and backward (single-process parity mode, SURVEY.md section 8e). */
int drs_comm_unique_id(uint8_t* id128_out);
int drs_comm_init(drs_handle_t h, const uint8_t* id128, int32_t rank, int32_t world, int32_t sync_bn);
int drs_comm_destroy(drs_handle_t h);
/* Stripe-sharded scene pass: after drs_scene_infer over this rank's rows [row_cuts[rank], row_cuts[rank+1]) (labels_out_host
 * may be NULL there), every rank sends its uint8 label stripe to rank 0 device-to-device; rank 0 receives [H, W] and copies it
 * to labels_out_host once (NULL on the other ranks; with all_ranks != 0 the assembled map is broadcast and every rank
 * receives it).  row_cuts has world+1 entries. */
int drs_scene_gather_labels(drs_handle_t h, int32_t H, int32_t W, const int32_t* row_cuts, int32_t all_ranks,
                            uint8_t* labels_out_host);

/* ---- scene path: NumPy loops around sess.run ----------------------------------------- */
/* Keep a scene resident in HBM (replaces the per-batch NumPy slicing of isprs:259, 364).
 * scene [H,W,C] float64 (isprs img_as_float) or float32 (contest/coffee); labels [H,W] uint8 or NULL. */
int drs_scene_upload(drs_handle_t h, int32_t scene_id, const void* scene_host, int32_t H, int32_t W, int32_t C,
                     int32_t dtype, const uint8_t* labels_host);
/* Stripe-sharded inference: keep only rows [row0, row0+rows) of the H-row scene resident (the rank's output stripe plus the
 * patch rows that straddle its borders).  rows_host points at the first resident row. */
int drs_scene_upload_rows(drs_handle_t h, int32_t scene_id, const void* rows_host, int32_t H, int32_t W, int32_t C,
                          int32_t dtype, const uint8_t* labels_rows_host, int32_t row0, int32_t rows);
int drs_scene_free(drs_handle_t h, int32_t scene_id);
/* normalize_images (isprs:74-81): (x - mean)/std on channels 0..2 only, in the scene's dtype. */
int drs_set_normalization(drs_handle_t h, const double* mean3, const double* std3);

/* coffee only: training patches are cast to float16 BEFORE normalisation (coffee:293; test patches stay float32, coffee:346);
 * when on, the gather of float32 scenes reproduces NumPy's float16 arithmetic (half operands, float32 operation, half result). */
int drs_set_gather_fp16(drs_handle_t h, int32_t on);

/* dynamically_create_patches + normalize_images (isprs:245-334, 74-81; contest:192-254; coffee:241-293)
 *   inst   [B,3] int32 (scene_id, row, col) AFTER the caller's shift-back (host keeps RNG + border rule)
 *   flips  [B] uint8: 0 none, 1 flipud, 2 fliplr (isprs:304-318)
 *   noise  [B,crop,crop,C] float64 added before normalisation where noise_on[b]!=0 (isprs:298-301), or NULL
 *   x_out  [B,crop,crop,C] fp32 device; y_out [B,crop,crop] fp32 device (labels as fed), may be NULL
 *   over_x [B,crop,crop,C] float64 / over_y [B,crop,crop] uint8: patches that replace the scene crop where
 *          over_on[b]!=0 (the host-rotated patches of isprs:292-296; GPU rotation is a "next" row), or NULL */
int drs_gather_dev(drs_handle_t h, const int32_t* inst_host, const uint8_t* flips_host, int32_t B, int32_t crop,
                   const double* noise_host, const uint8_t* noise_on_host, const double* over_x_host,
                   const uint8_t* over_y_host, const uint8_t* over_on_host, float* x_out_dev, float* y_out_dev);

/* The same gather with the nearest-neighbour rotation of isprs:287-296 done on the device (SURVEY section 8f, N1):
 *   rot    [B,6] float64 per patch: m00 m01 m10 m11 off0 off1 of scipy.ndimage.rotate(angle, order=0, reshape=False)'s
 *          affine map (built on the host exactly as scipy builds it: cosdg/sindg of the integer angle, centre offsets);
 *          the kernel evaluates cc = (off + i*m_0) + j*m_1 in float64 in scipy's order, takes floor(cc + 0.5), and
 *          writes the constant 0 (patch, label) where cc < 0 or cc > crop-1 -- bit-identical to scipy for all 360 angles.
 *   rot_on [B] uint8, rotation applied where != 0 (before noise, normalisation and flip, as in the reference)
 *   amask_out [B,crop,crop] uint8 device or NULL: rotate(np.ones) then flip = the mask calc_accuracy_by_crop receives. */
int drs_gather_rot_dev(drs_handle_t h, const int32_t* inst_host, const uint8_t* flips_host, int32_t B, int32_t crop,
                       const double* noise_host, const uint8_t* noise_on_host, const double* rot_host,
                       const uint8_t* rot_on_host, float* x_out_dev, float* y_out_dev, uint8_t* amask_out_dev);

/* ---- host-side step planner (no device needed) ------------------------------------------------------------------
 * dynamically_create_patches (isprs:245-334) draws, per patch, randint(0,2) rotate? / randint(0,2) noise? /
 * normal(0, 0.01, patch.shape) / randint(0,3) flip from the legacy global NumPy generator, which the patch-size draw of
 * the next step shares.  These entry points restate NumPy's MT19937, randint and legacy_gauss bit for bit
 * (csrc/host_plan.cpp) on a generator state the caller takes from np.random.get_state() and writes back with
 * np.random.set_state(), so a seeded run consumes the stream exactly like the reference at a fraction of the cost. */
typedef struct drs_mt_state {
  uint32_t key[624];  /* np.random.get_state()[1] */
  int32_t pos;        /* [2] */
  int32_t has_gauss;  /* [3] */
  double gauss;       /* [4] cached_gaussian */
} drs_mt_state;
typedef struct drs_planner_s* drs_planner_t;   /* scratch + worker pool of the deferred Gaussian transform */
int drs_planner_create(drs_planner_t* out);
int drs_planner_destroy(drs_planner_t p);
/* np.random.normal(loc, scale, n) / np.random.randint(0, n, count) on the caller's state (unit tests, building blocks) */
int drs_mt_normal(drs_planner_t p, drs_mt_state* st, double loc, double scale, double* out, int64_t n, int32_t threads);
int drs_mt_randint(drs_mt_state* st, uint32_t n, int32_t* out, int64_t count);
/* One batch of dynamically_create_patches' decisions (isprs:255-318):
 *   batch_inst [B,4] int64 (map, x, y, rotation angle) = selected_training_instances[batch]
 *   scene_hw   [n_scenes,2] int32 scene heights / widths (border rule isprs:259-269)
 *   rot_table  [360,6] float64: scipy.ndimage.rotate's affine map per integer angle for THIS crop (host.rotation_table)
 *   inst_out [B,3] int32 (scene, row, col after the shift-back); flips_out [B] (0 none, 1 flipud, 2 fliplr);
 *   rot_on_out [B], rot_out [B,6]; noise_on_out [B]; noise_slot_out [B] int32 = index of the patch's noise block
 *   in noise_out or -1; noise_out: compact float64 noise, block k = values [k*crop*crop*C, (k+1)*crop*crop*C)
 *   (noise_cap >= n_noise*crop*crop*C + 2 doubles); *n_noise_out = number of noisy patches.
 *   is_train == 0: only inst_out is produced and the generator is not touched (validation batches, isprs:1586).
 *   threads: workers of the deferred transform.  [own_b0, own_b1): patches whose noise values the caller needs (data
 *   parallel ranks scan the whole batch but transform only their slice); pass 0, B for all.
 * Returns 0, or 2 bad scene index, 3 window outside the scene (the reference prints an error, isprs:273-280),
 * 4 rotation angle outside [0,360), 5 noise_out too small, 1 bad argument. */
int drs_plan_isprs_batch(drs_planner_t p, drs_mt_state* st, const int64_t* batch_inst, int32_t B, const int32_t* scene_hw,
                         int32_t n_scenes, int32_t crop, int32_t C, int32_t is_train, const double* rot_table,
                         int32_t* inst_out, uint8_t* flips_out, uint8_t* rot_on_out, double* rot_out, uint8_t* noise_on_out,
                         int32_t* noise_slot_out, double* noise_out, int64_t noise_cap, int32_t* n_noise_out, int32_t threads,
                         int32_t own_b0, int32_t own_b1);

/* Gather of a planned batch (drs_plan_isprs_batch) with no host synchronisation: the plan arrays must be page-locked host
 * memory that stays untouched until the step's result has been fetched; they are uploaded on a separate stream into a
 * two-slot device staging ring and the gather kernel is ordered behind the copy.  noise_host is the compact noise
 * (noise_count doubles, block noise_slot[b] belongs to patch b); rotation and the accuracy mask as drs_gather_rot_dev. */
int drs_gather_plan_dev(drs_handle_t h, const int32_t* inst_host, const uint8_t* flips_host, int32_t B, int32_t crop,
                        const uint8_t* rot_on_host, const double* rot_host, const uint8_t* noise_on_host,
                        const int32_t* noise_slot_host, const double* noise_host, int64_t noise_count, float* x_out_dev,
                        float* y_out_dev, uint8_t* amask_out_dev);

/* create_patches_per_map index arithmetic (isprs:344-375, contest:267-301 incl. the offset_h bug, coffee:302-322):
 * (row, col) of every patch in visiting order, batch after batch.  Pure host code (no device needed).
 *   pos_out [cap_pairs,2] int32 or NULL (query the count through n_out). */
int drs_grid_positions(int32_t H, int32_t W, int32_t crop, int32_t batch, int32_t variant, int32_t* pos_out,
                       int64_t cap_pairs, int64_t* n_out);

/* accumulate + argmax (isprs:1261-1284, contest:916-941, coffee:1045-1068), standalone:
 *   logits [P,crop,crop,K] fp32 device, pos [P,2] int32 host (row, col) in visiting order.
 *   labels_out [H,W] uint8 host; mean_out [H,W,K] float64 host or NULL (prob_im / occur_im).
 * Adds per pixel in visiting order (bit-identical to NumPy's sequential fp32 `+=`), no atomics. */
int drs_accumulate_argmax(drs_handle_t h, const float* logits_dev, const int32_t* pos_host, int32_t P, int32_t crop,
                          int32_t K, int32_t H, int32_t W, uint8_t* labels_out_host, double* mean_out_host);

/* Whole validate_test / test / generate_final_maps inner loop (isprs:1249-1284) for rows [row_begin,row_end)
 * of an uploaded scene: grid -> gather+normalise -> forward -> ordered accumulate -> argmax.
 *   batch     the script's batch_size (fixes the contest/coffee visiting order; results do not depend on
 *             the internal chunking because eval-mode BN is batch-independent)
 *   labels_out [row_end-row_begin, W] uint8 host.
 * A rank that owns an output stripe evaluates every patch intersecting it, so stripes need no exchange. */
int drs_scene_infer(drs_handle_t h, int32_t scene_id, int32_t crop, int32_t batch, int32_t variant,
                    int32_t row_begin, int32_t row_end, uint8_t* labels_out_host, double* mean_out_host);

/* The same pass over a scene that is still in host memory (a fresh tile): scene rows are copied on a separate stream,
 * in pieces, just ahead of the chunk that first reads them, so the upload (1.44 GB for a
 * 6000x6000x5 float64 tile) overlaps the convolutions instead of preceding them.  Equivalent to drs_scene_upload (without
 * labels) followed by drs_scene_infer over all rows; the scene stays resident as scene_id afterwards. */
int drs_scene_infer_host(drs_handle_t h, int32_t scene_id, const void* scene_host, int32_t H, int32_t W, int32_t C,
                         int32_t dtype, int32_t crop, int32_t batch, int32_t variant, uint8_t* labels_out_host,
                         double* mean_out_host);

/* validate_test_multiscale (isprs:1347-1474): one drs_scene_infer pass per crop, in the order given, over rows
 * [row_begin,row_end); after each pass every pixel adds softmax(float32(prob_im/occur_im)) with NumPy's float32 arithmetic
 * to a float32 sum; the label map is its first argmax.  labels_out_host NULL = stay on the device for
 * drs_scene_confusion / drs_scene_gather_labels; prob_sum_out_host [rows,W,K] float32 (np.sum(mean_prob, axis=0)) or NULL. */
int drs_scene_infer_multiscale(drs_handle_t h, int32_t scene_id, int32_t n_scales, const int32_t* crops_host, int32_t batch,
                               int32_t variant, int32_t row_begin, int32_t row_end, uint8_t* labels_out_host,
                               float* prob_sum_out_host);
/* host-only (no device): the kernel's per-pixel softmax, compiled for the host, for CPU tests. in/out [n_pixels, K] float32 */
int drs_debug_np_softmax(const float* in_host, int64_t n_pixels, int32_t K, float* out_host);
/* host-only: the exp of that softmax (NumPy's float32 exp restated) on n float32 values */
int drs_debug_np_expf(const float* in_host, int64_t n, float* out_host);
/* unit-test entry: one launch of the multi-scale kernel on given sums and counts (K = the net's classes):
 * acc += softmax(float32(prob/occur)) (acc ignored on input when first != 0), labels_out_host (or NULL) = first argmax(acc).
 * prob [npix,K] float32, occur [npix] uint32, acc_inout [npix,K] float32, labels [npix] uint8, all host memory. */
int drs_debug_multiscale_softmax_add(drs_handle_t h, const float* prob_host, const uint32_t* occur_host, int64_t npix,
                                     int32_t first, float* acc_inout_host, uint8_t* labels_out_host);

/* calc_accuracy_by_crop (isprs:510-531) / per-pixel scene confusion (isprs:1289-1296, contest:944-948):
 *   truth, pred [n] uint8 device; mask [n] or NULL; ignore_label <0 = none.
 *   cm_out [K*K+1] uint32 host: counts[true][pred] then #correct. */
int drs_confusion_dev(drs_handle_t h, const uint8_t* truth_dev, const uint8_t* pred_dev, const uint8_t* mask_dev,
                      int64_t n, int32_t K, int32_t ignore_label, uint32_t* cm_out_host);

/* Scene-level confusion matrix on the device (isprs:1289-1296, contest:944-951, SURVEY section 8f N2): the label map of
 * the last drs_scene_infer pass over scene_id against the ground truth uploaded with that scene.  Pixels whose truth is
 * ignore_label (isprs: eroded class 6, contest: unlabelled class 7; -1 = none) or >= K are skipped.
 * cm_out_host: K*K counts [truth][pred] followed by the number of correct pixels. */
int drs_scene_confusion(drs_handle_t h, int32_t scene_id, int32_t K, int32_t ignore_label, uint32_t* cm_out_host);

/* ---- introspection for bench / tests ---------------------------------------------------- */
/* number of kernels this library has launched since creation (bench.py "gpu_launches") */
int64_t drs_launch_count(drs_handle_t h);
/* Per-launch timing of the tensor-core convolution kernels with CUDA events on the handle's stream:
 * drs_set_profiling(h,1) starts a record; drs_profile_read returns the summed device time (ms), the number of
 * launches and their algorithmic FLOPs since then, and resets the record. */
int drs_set_profiling(drs_handle_t h, int32_t on);
int drs_profile_read(drs_handle_t h, float* conv_ms, int64_t* conv_launches, double* conv_flops);
int drs_last_conv_ms(drs_handle_t h, float* ms_out);
/* debug: copy the activation of conv scope `name` from the last forward (post act/pool) as fp32 NHWC.  After a training step
 * under DRS_DEBUG_KEEP=1 also "z:<scope>" (raw conv output), "pre:<scope>" (activation in front of an average pool or SE
 * gate), "logits", "dlogits", "dout:<scope>" (gradient of the layer output), "da:<scope>" (gradient in front of the BN
 * backward; not for the fused bf16 pool + BN backward, which never stores it) and "dz:<scope>". */
int drs_debug_activation(drs_handle_t h, const char* name, float* out_host, int64_t count);
/* unit-test entry: one dilated SAME convolution through the tcgen05 path (or SIMT when precision=FP32).  In F16 / BF16
 * the conv1 shape (5x5, rate 1, Ci <= 8, Co 32 or 64) runs on conv1's tensor-core kernel, as the first layer of both
 * forwards does; every other shape on the generic tcgen05 kernel.
 *   x [B,crop,crop,Ci] fp32 host, w HWIO fp32 host, scale/shift [Co] (y = act(conv*scale+shift)), act 0/1/2 */
int drs_debug_conv(drs_handle_t h, const float* x_host, const float* w_host, const float* scale_host,
                   const float* shift_host, int32_t B, int32_t crop, int32_t k, int32_t rate, int32_t Ci, int32_t Co,
                   int32_t act, int32_t precision, float* y_host);

/* kernel micro-benchmark: average milliseconds of `reps` launches of one tcgen05 convolution (the kernel behind
 * _conv_layer, isprs:700-723) on pseudo-random resident operands; exp_mode >= 0 selects a DRS_EXP_MODE timing
 * experiment (outputs are then meaningless), -1 the production kernel.  exp_mode bit 16 runs the instrumented twin of
 * the kernel; instr_out (10 words, may be NULL) then receives CTA 0's cycle counters: producer {total, waiting for a
 * free slot, stages, expect_tx issue, TMA issue}, MMA issuer {total, waiting for operands, MMA issue, commit issue,
 * waiting for an accumulator}. */
int drs_bench_conv(drs_handle_t h, int32_t B, int32_t crop, int32_t k, int32_t rate, int32_t Ci, int32_t Co,
                   int32_t precision, int32_t exp_mode, int32_t reps, float* ms_out, uint32_t* instr_out);

/* unit-test entry: filter gradient of one dilated SAME convolution (the wgrad inside isprs:1687 minimize):
 *   x [B,crop,crop,Ci], dy [B,crop,crop,Co] fp32 host -> dw [k,k,Ci,Co] fp32 host.
 *   precision BF16: tcgen05 MN-major path (operands rounded to bf16); FP32: CUDA-core fixed-order path. */
int drs_debug_wgrad(drs_handle_t h, const float* x_host, const float* dy_host, int32_t B, int32_t crop, int32_t k,
                    int32_t rate, int32_t Ci, int32_t Co, int32_t precision, float* dw_host);
/* host-only: the schedule of conv_tc_kernel (csrc/conv_tc.cuh, ConvSched): the 128-pixel units CTA `block` of a `grid`-CTA
 * launch over `num_units` units works on, in order; pair_out[i] = 1 when unit i is the first of a pair of consecutive
 * units that share one filter slice (mt = 2, Co <= 128).  *n_out = number of entries (may exceed cap). */
int drs_debug_conv_schedule(int32_t num_units, int32_t mt, int32_t grid, int32_t block, int32_t* units_out, uint8_t* pair_out,
                            int32_t cap, int32_t* n_out);

/* unit-test entry: data gradient of one dilated SAME convolution exactly as the step computes it (a convolution of dy
 * with tap-flipped, Ci/Co-transposed weights and the before/after padding swapped):
 *   dy [B,crop,crop,Co], w HWIO [k,k,Ci,Co] fp32 host -> dx [B,crop,crop,Ci] fp32 host.  precision BF16 (tcgen05) or FP32. */
int drs_debug_dgrad(drs_handle_t h, const float* dy_host, const float* w_host, int32_t B, int32_t crop, int32_t k, int32_t rate,
                    int32_t Ci, int32_t Co, int32_t precision, float* dx_host);

/* unit-test entry: one layer's train-mode batch-norm (no gamma/beta, isprs:655-663) + activation (+ 3x3 max-pool, isprs:745-750)
 * forward and backward with the step's own kernels: z [B,crop,crop,C] raw conv output, dout = gradient w.r.t. the layer
 * output -> out (layer output), dz (gradient w.r.t. z), batch mean / inverse std.  act: 0 none, 1 ReLU, 2 LeakyReLU(0.1). */
int drs_debug_layer(drs_handle_t h, const float* z_host, const float* dout_host, int32_t B, int32_t crop, int32_t C, int32_t pool,
                    int32_t act, int32_t precision, float* out_host, float* dz_host, float* mean_host, float* inv_std_host);

#ifdef __cplusplus
}
#endif
#endif /* DRS_H_ */

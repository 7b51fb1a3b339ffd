/*
 * dcscn_b200.h - C-ABI of the B200-native DCSCN forward / backward hot path.
 *
 * The reference (jiny2001/dcscn-super-resolution) has no FFI: its seam is the Python class
 * DCSCN.SuperResolution and the four `sess.run` call sites.  Each entry point below names the
 * reference interface it stands in for (paths relative to the reference checkout).
 *
 * All tensors are contiguous fp32 NHWC with C == 1 at the boundary (TF placeholders
 * x / x2 / y, DCSCN.py:224-226).  Functions return 0 on success, non-zero on error;
 * dcscn_last_error() returns the message of the last failure on the calling thread.
 * A handle is not re-entrant; use one handle per GPU / host thread.
 */
#ifndef DCSCN_B200_H_
#define DCSCN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dcscn_handle dcscn_handle;

/* Arithmetic of the tensor-core layers. */
enum {
  DCSCN_PRECISION_F16X3 = 0, /* fp32-equivalent: fp16 hi/lo split operands, 3 UMMA passes, fp32 accumulate */
  DCSCN_PRECISION_F16X1 = 1  /* single-pass fp16 operands (PSNR-neutral, not 1e-3-pixel exact) */
};

/*
 * Graph hyper-parameters: the subset of helper/args.py:16-98 flags that shape the graph built by
 * DCSCN.SuperResolution.__init__ (DCSCN.py:29-106) and build_graph (DCSCN.py:222-332).
 */
typedef struct dcscn_config {
  int32_t struct_size;            /* sizeof(dcscn_config), for ABI checking */
  int32_t scale;                  /* --scale (2, 3 or 4) */
  int32_t layers;                 /* --layers */
  int32_t filters;                /* --filters */
  int32_t min_filters;            /* --min_filters */
  float filters_decay_gamma;      /* --filters_decay_gamma */
  int32_t use_nin;                /* --use_nin (only 1 is supported) */
  int32_t nin_filters;            /* --nin_filters  (A1) */
  int32_t nin_filters2;           /* --nin_filters2 (B1, B2) */
  int32_t cnn_size;               /* --cnn_size (3) */
  int32_t reconstruct_layers;     /* --reconstruct_layers (max(flag,1) == 1 supported) */
  int32_t reconstruct_filters;    /* --reconstruct_filters */
  int32_t pixel_shuffler_filters; /* --pixel_shuffler_filters (0 = same as input) */
  int32_t depthwise_separable;    /* --depthwise_separable */
  int32_t channels;               /* --channels (1) */
  float dropout_keep;             /* --dropout_rate (keep probability, training only) */
  float l2_decay;                 /* --l2_decay */
  float clipping_norm;            /* --clipping_norm */
  float beta1, beta2, epsilon;    /* --beta1 --beta2 --epsilon (Adam) */
  int32_t device_id;              /* --gpu_device_id */
  int32_t precision;              /* DCSCN_PRECISION_* */
} dcscn_config;

/* SuperResolution(flags) + build_graph() + init_session (DCSCN.py:29, :222; tf_graph.py:65).  Fails on a device that is
 * not sm_100a or has an odd SM count (the tensor-core kernels run on CTA pairs). */
int dcscn_create(const dcscn_config* cfg, dcscn_handle** out);
/* sess.close() */
int dcscn_destroy(dcscn_handle* h);
const char* dcscn_last_error(void);

/*
 * Variables of the graph, named exactly like the TF variables in the reference's checkpoints
 * (tf.train.Saver, tf_graph.py:263-296): "CNN1/conv_W" [k,k,cin,cout] HWIO, "CNN1/conv_B",
 * "CNN1/prelu/CNN1_prelu", "A1/...", "B1/...", "B2/...", "Up-PS/Up-PS_CNN/conv_W", "R-CNN1/conv_W" ...
 */
int dcscn_num_params(dcscn_handle* h);
int dcscn_param_info(dcscn_handle* h, int index, char* name_buf, int name_buf_len, int64_t* dims4, int* ndim);
/* saver.restore (tf_graph.py:276): host fp32 -> engine.  numel must match the variable. */
int dcscn_set_param(dcscn_handle* h, const char* name, const float* host_data, int64_t numel);
/* saver.save (tf_graph.py:291): engine -> host fp32. */
int dcscn_get_param(dcscn_handle* h, const char* name, float* host_data, int64_t numel);

/*
 * sess.run(self.y_, {x, x2, dropout: 1.0, is_training: 0})  (DCSCN.py:565, :575).
 * x [n,h,w,1], x2 and y [n,scale*h,scale*w,1]: DEVICE pointers; asynchronous on `stream` (cudaStream_t).
 */
int dcscn_forward(dcscn_handle* h, const float* x_dev, const float* x2_dev, float* y_dev, int n, int height,
                  int width, void* stream);
/* Same call with HOST buffers (pinned or pageable): H2D, forward, D2H, synchronises before returning.  x2 may be NULL:
 * the bicubic up-scale of x is then formed on the device, bit for bit what `util.resize_image_by_pil(x, scale)` returns
 * (dcscn_bicubic_resize), and only x crosses PCIe (the default of `SuperResolution.do`, DCSCN.py:551-553). */
int dcscn_forward_host(dcscn_handle* h, const float* x, const float* x2, float* y, int n, int height, int width);
/* `util.resize_image_by_pil` (helper/utilty.py:211-239) for single-channel float images on the device: Pillow's bicubic
 * `Image.resize` of mode 'F' images restated bit-exactly (two passes, double accumulation, float32 intermediate; up- or
 * down-scaling).  src [n, height, width] -> dst [n, out_height, out_width], fp32 device tensors. */
int dcscn_bicubic_resize(dcscn_handle* h, const float* src_dev, float* dst_dev, int n, int height, int width, int out_height,
                         int out_width, void* stream);

/* The self-ensemble of `SuperResolution.do` (DCSCN.py:547-586) for ONE image, entirely on the device: the first `flips`
 * (1..8) transforms of helper/utilty.py:595-617 are applied to x [height,width] and x2 [scale*height, scale*width],
 * transforms 0..3 and 4..7 each run as one batched forward, and y [scale*height, scale*width] receives the float64 mean
 * of the inverse-transformed outputs, summed in the order 0, 1, ... like the reference's float64 accumulator. */
int dcscn_forward_ensemble(dcscn_handle* h, const float* x_dev, const float* x2_dev, double* y_dev, int height, int width,
                           int flips, void* stream);
int dcscn_forward_ensemble_host(dcscn_handle* h, const float* x, const float* x2, double* y, int height, int width, int flips);
/* (x2 may be NULL in dcscn_forward_ensemble_host as well: formed on the device from x.) */
/* One rank's share of the same ensemble when the 8 transforms are spread over several GPUs (SURVEY.md section 8e): bit t of
 * `transform_mask` selects transform t; y receives the float64 SUM of the selected inverse-transformed outputs (no
 * division), ready for one ncclAllReduce(sum) over the ranks followed by the division by the ensemble size. */
int dcscn_forward_ensemble_partial(dcscn_handle* h, const float* x_dev, const float* x2_dev, double* y_dev, int height,
                                   int width, int transform_mask, void* stream);

/*
 * sess.run([self.training_optimizer, self.image_loss, self.mse], {x, x2, y, lr, dropout: keep, is_training: 1})
 * (DCSCN.py:415-425; graph: build_optimizer / add_optimizer_op, DCSCN.py:334-413): forward with inverted dropout
 * (keep = cfg.dropout_keep, masks from a counter hash of `seed`), mse loss + l2_decay * sum(l2_loss(conv_W)),
 * gradients of every variable, tf.clip_by_global_norm(cfg.clipping_norm), TF-Adam with learning rate `lr`.
 * `apply_update` = 0 computes loss and gradients only (dcscn_get_grad), leaving the weights untouched.
 * x / x2 / y are DEVICE pointers (dcscn_train_step) or HOST pointers (dcscn_train_step_host); both synchronise.
 */
int dcscn_train_step(dcscn_handle* h, const float* x_dev, const float* x2_dev, const float* y_dev, int n, int height, int width,
                     float lr, uint32_t seed, int apply_update, float* out_loss, float* out_mse, void* stream);
int dcscn_train_step_host(dcscn_handle* h, const float* x, const float* x2, const float* y, int n, int height, int width, float lr,
                          uint32_t seed, int apply_update, float* out_loss, float* out_mse);
/*
 * Training data path on the device (reference: helper/loader.py:70-275 BatchDataSets + DCSCN.py:186-190 build_input_batch,
 * which assemble every mini-batch patch by patch in Python).  dcscn_patch_store_set copies the data set's uint8 patch
 * arrays - LR input [count, ph, pw], its bicubic up-scale and the ground truth [count, scale*ph, scale*pw] - into HBM
 * once.  dcscn_train_step_indexed is dcscn_train_step on the mini-batch {patch indices[i]}: one gather launch per tensor
 * converts uint8 -> fp32 * (max_value / 255) (loader.py:251-255); bit 31 of an index mirrors that patch left-right
 * (the augmentation of loader.py:318-319).  dcscn_patch_gather returns the same gathered fp32 tensors to the host
 * (parity checks against the host loader).
 */
int dcscn_patch_store_set(dcscn_handle* h, const uint8_t* lr, const uint8_t* bicubic, const uint8_t* truth, int64_t count,
                          int patch_height, int patch_width);
int dcscn_train_step_indexed(dcscn_handle* h, const int32_t* indices, int n, float max_value, float lr, uint32_t seed,
                             int apply_update, float* out_loss, float* out_mse);
int dcscn_patch_gather(dcscn_handle* h, const int32_t* indices, int n, float max_value, float* x, float* x2, float* y);
/* d loss / d variable of the LAST train step (after the L2 term, before clipping): tf.gradients(loss, trainables). */
int dcscn_get_grad(dcscn_handle* h, const char* name, float* host_data, int64_t numel);
/* Adam slots of a variable ("<var>/Adam" = slot 0, "<var>/Adam_1" = slot 1 in the reference's checkpoints). */
int dcscn_get_adam_slot(dcscn_handle* h, const char* name, int slot, float* host_data, int64_t numel);
/* Restoring optimizer state from a checkpoint (what tf.train.Saver.restore does for the graph sr.py / train.py build,
 * helper/tf_graph.py:263-280): the slots, and the number of applied updates t (the reference stores it as
 * beta1_power = beta1^(t+1), beta2_power = beta2^(t+1)). */
int dcscn_set_adam_slot(dcscn_handle* h, const char* name, int slot, const float* host_data, int64_t numel);
int dcscn_get_adam_step(dcscn_handle* h, int64_t* step);
int dcscn_set_adam_step(dcscn_handle* h, int64_t step);
/* tf.global_variables_initializer() on the optimizer's variables (helper/tf_graph.py:73-75 re-runs it for every trial of
 * train.py:100-103): both Adam slots of every variable back to zero and the update count t to 0. */
int dcscn_reset_optimizer(dcscn_handle* h);
/* Data-parallel training: after dcscn_train_step(..., apply_update = 0) on every rank, all-reduce the flat buffer
 * returned here (device pointer, `count` floats: the gradient of every trainable in dcscn_param_info order followed by
 * this rank's {image_loss, mse}) - ONE ncclAllReduce(sum) over NVLink - then call dcscn_apply_gradients_avg on every
 * rank with grad_scale = 1 / ranks: it scales the summed gradients to their mean, applies the global-norm clip of the
 * averaged gradient + Adam identically everywhere (SURVEY.md section 8e) and returns the job-wide mean loss / mse.
 * Every rank must hold the same number of patches (each normalises by its own pixel count).
 * dcscn_apply_gradients is the same with grad_scale = 1 (gradients already averaged by the caller). */
int dcscn_grad_buffer(dcscn_handle* h, float** dev_ptr, int64_t* count);
int dcscn_apply_gradients(dcscn_handle* h, float lr, void* stream);
int dcscn_apply_gradients_avg(dcscn_handle* h, float lr, float grad_scale, float* out_loss, float* out_mse, void* stream);
/* Global gradient norm of the last train step (what clip_by_global_norm computed). */
float dcscn_last_grad_norm(dcscn_handle* h);
/* The keep mask (1 = kept) the train step with `seed` applies to `tensor` ("CNNi", "A1", "B1", "B2"), [n,h,w,C] uint8:
 * lets a CPU oracle replay the exact same dropout. */
int dcscn_dropout_mask(dcscn_handle* h, const char* tensor, uint32_t seed, int n, int height, int width, uint8_t* mask, int64_t numel);

/*
 * Parity / debug: output of one layer of the LAST forward as fp32 NHWC [n, H_l, W_l, cout_l]
 * (`tensor` is the reference's self.H entry: "CNN1".."CNNL", "A1", "B1", "B2", "Up-PS", "Up-PS2").
 */
int dcscn_get_activation(dcscn_handle* h, const char* tensor, float* host_data, int64_t numel);

/* Options: "conv_impl" 0 = tcgen05 (default), 1 = CUDA-core fp32 validation kernels;
 *          "seg_chunks" = pipeline stages per fp32-promotion segment (default 0 = automatic: 2, or 3 for thin layers);
 *          "fuse_last" 1 | 0 = compute the per-pixel half of R-CNN1 inside the last Up-PS epilogue (default 1);
 *          "timing" 0 | 1 = record per-launch CUDA events (see dcscn_get_timings);
 *          "store_mode" 2 | 0 | 1 = fp16 plane stores of the tensor-core epilogues: 32-byte stores with neighbouring lanes
 *          exchanging halves so that each instruction writes 64 contiguous bytes of a pixel (default; streaming 3x3 kernel,
 *          elsewhere like 0), one 32-byte store per lane and plane, or two 16-byte stores (the round-1/2 form, cross-check);
 *          "wide_tiles" 1 | 0 = column tiles of the streaming 3x3 kernel capped at 256 (default: layers wider than 160
 *          columns use two TMEM buffers and read each input box once per pixel tile) or at 160 (three buffers);
 *          "ds_impl" 0 | 1 = depthwise-separable layers on the tile kernels (default) or the first-generation kernels (cross-check);
 *          "act_grad_impl" 0 | 1 = activation gradients with 16-byte (default) or channel-pair accesses (cross-check);
 *          "ds_cache" 1 | 0 = depthwise-separable pixel-shuffler layers keep their depthwise values across column groups;
 *          "gather_impl" 0 | 1 = R-CNN1 gather with four pixels per thread (default where W % 4 == 0) or the generic kernel;
 *          "graph" 1 | 0 = replay the launches of a forward (all but the last kernel) as one CUDA graph per (n, h, w) once
 *          the same input pointer has been seen twice in a row (default 1; off while "timing" = 1 or "conv_impl" = 1);
 *          "l1_loss" 0 | 1 = image_loss of the train step is mean |y_ - y| instead of the MSE (--use_l1_loss,
 *          DCSCN.py:342-344; the returned mse stays the MSE);
 *          "wgrad_impl" 0 | 1 = filter gradients on tcgen05 (default) or on CUDA cores (cross-check);
 *          "wgrad_taps" 0..3 = filter taps per wgrad CTA (0 = automatic);
 *          "host_repack" 0 | 1 = after an optimizer step rebuild the packed tensor-core weight images on the host
 *          (validation of the default device-side refresh). */
int dcscn_set_option(dcscn_handle* h, const char* key, int64_t value);
/* With option "timing" = 1 every launch of a forward is bracketed by CUDA events on its stream; this returns the
 * device time in ms of each launch of the LAST forward (in launch order) and their comma-separated names. */
int dcscn_get_timings(dcscn_handle* h, float* ms, int capacity, int* count, char* names, int names_len);
/* Number of kernels this handle has launched so far (bench.py "gpu_launches"). */
int64_t dcscn_launch_count(dcscn_handle* h);
/* Forwards served by a CUDA-graph replay so far (option "graph"). */
int64_t dcscn_graph_replays(dcscn_handle* h);
/* Bytes of device memory currently held by the handle. */
int64_t dcscn_device_bytes(dcscn_handle* h);
/* Measurement only (no reference counterpart; bench.py's roofline denominator): kind::f16 tcgen05.mma throughput with
 * both operands resident in shared memory, every SM busy.  group = 1 | 2 (cta_group), n = accumulator width of one
 * product (multiple of 16), mode 0 = the three hi/lo products of the conv kernels per K = 16 slice, 1 = the stacked
 * form (one UMMA of width 2n + one of width n; group 1, n <= 128), 2 = a single product; iters x 4 slices are issued by
 * each cluster.  Returns the launch duration (ms, CUDA events) and the longest issuing-thread span (SM cycles). */
int dcscn_umma_probe(int device_id, int group, int n, int mode, int iters, float* out_ms, double* out_cycles);

#ifdef __cplusplus
}
#endif
#endif /* DCSCN_B200_H_ */

/*
 * include/pcnn.h -- C ABI of the B200-native LeNet/MNIST training engine (libpcnn.so).
 *
 * This is the drop-in boundary for the hot path of Tamerkobba/Parallel-CNN: the 18 layer functions of
 * Sequential/layer.h and the driver entry points of Sequential/Main.cpp.  The reference has no FFI layer
 * (its boundary is `#include "layer.h"`), so include/layer.h in this repo re-declares the reference's own
 * class and functions and forwards each of them to the entry points below; INTEGRATION.md shows the binding.
 * Every entry point cites the reference interface it replaces as  [ref: <file>:<lines>]  relative to
 * /root/reference/.
 *
 * Conventions
 *   - plain C: pointers, sizes, ints.  No torch / C++ types.  All functions return 0 on success or a negative
 *     pcnn_status; pcnn_last_error_string() describes the most recent failure on the calling thread.
 *   - "dev" pointers are CUDA device pointers on the context's device; "host" pointers are ordinary memory.
 *   - every call enqueues on the context's stream; only *_sync / *_d2h / get_* / *_host calls block.
 *   - one context per GPU, not thread-safe per context (the reference is single-threaded global state).
 *   - there is NO CPU fallback: on a machine without a usable sm_100 GPU pcnn_create fails with
 *     PCNN_ERR_NOGPU and nothing else computes.
 *
 * Packed parameter vector (PCNN_NPARAM = 2,343 floats), also the layout of the packed gradient:
 *     [0,150) c1.weight[6][5][5] | [150,156) c1.bias | [156,172) s1.weight[1][4][4] | [172] s1.bias |
 *     [173,2333) f.weight[10][6][6][6] | [2333,2343) f.bias             [ref: Sequential/Main.cpp:17-20]
 * The packed gradient holds what the reference multiplies by dt (the NEGATIVE gradient, layer.h:93): d_weight
 * for the weight blocks and the raw bias accumulators (sum d_preact) for the bias blocks; the /576 and /216
 * of layer.h:412 and layer.h:316 are applied by the update.  Element PCNN_NPARAM of the device-side vector
 * carries the sum of per-sample error norms (Main.cpp:168-169).
 */
#ifndef PCNN_H_
#define PCNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCNN_NPARAM 2343
#define PCNN_OFF_C1W 0
#define PCNN_OFF_C1B 150
#define PCNN_OFF_S1W 156
#define PCNN_OFF_S1B 172
#define PCNN_OFF_FW 173
#define PCNN_OFF_FB 2333
#define PCNN_IMG 784   /* 28 x 28 */
#define PCNN_C1 3456   /* 6 x 24 x 24 */
#define PCNN_S1 216    /* 6 x 6 x 6 */
#define PCNN_F 10

typedef enum {
    PCNN_OK = 0,
    PCNN_ERR_ARG = -1,    /* null pointer, negative size, bad enum */
    PCNN_ERR_CUDA = -2,   /* a CUDA runtime call or kernel failed */
    PCNN_ERR_NCCL = -3,   /* NCCL missing or a collective failed */
    PCNN_ERR_STATE = -4,  /* call not valid in the current state (no dataset bound, comm not initialised...) */
    PCNN_ERR_IO = -5,     /* file problems other than the mnist_load codes */
    PCNN_ERR_NOGPU = -6   /* no CUDA device / not compute capability 10.x */
} pcnn_status;

#define PCNN_MAX_PEERS 8   /* GPUs of one NVSwitch domain the in-kernel gradient exchange addresses */
typedef enum { PCNN_MODE_AUTO = 0, PCNN_MODE_GRAPH = 1, PCNN_MODE_PERSISTENT = 2 } pcnn_step_mode;
typedef enum { PCNN_U8 = 0, PCNN_F32 = 1 } pcnn_pixel_type;   /* IDX bytes, or the reference's float[28][28] */
typedef enum { PCNN_TRAIN_SET = 0, PCNN_TEST_SET = 1 } pcnn_split;

typedef struct pcnn_ctx pcnn_ctx;

/* ------------------------------------------------------------------ library / context */
int pcnn_version(void);
const char *pcnn_last_error_string(void);
/* device < 0: current device.  stream: a cudaStream_t to enqueue on (e.g. the caller's torch stream) or NULL
 * for a private non-blocking stream. */
int pcnn_create(pcnn_ctx **out, int device, void *stream);
int pcnn_destroy(pcnn_ctx *ctx);
int pcnn_sync(pcnn_ctx *ctx);
int pcnn_device_info(pcnn_ctx *ctx, int *sm_count, int *cc_major, int *cc_minor, size_t *hbm_bytes);

/* ------------------------------------------------------------------ device buffers owned by `Layer`
 * [ref: Sequential/layer.h:39-79  Layer::Layer / ~Layer / setOutput / clear / bp_clear] */
int pcnn_malloc(pcnn_ctx *ctx, void **dev, size_t bytes);             /* zero-initialised, like new float[n]() */
int pcnn_free(pcnn_ctx *ctx, void *dev);
int pcnn_memset0(pcnn_ctx *ctx, void *dev, size_t bytes);            /* Layer::clear, Layer::bp_clear */
int pcnn_h2d(pcnn_ctx *ctx, void *dev, const void *host, size_t bytes);   /* Layer::setOutput (blocking) */
int pcnn_d2h(pcnn_ctx *ctx, void *host, const void *dev, size_t bytes);   /* host reads of l_f.output etc. */
int pcnn_d2d(pcnn_ctx *ctx, void *dst, const void *src, size_t bytes);

/* ------------------------------------------------------------------ parameters
 * pcnn_init_params_reference replays the constructor draws of the three static Layer objects: glibc rand()
 * with the default seed, per neuron bias then weights, c1 -> s1 -> f  [ref: layer.h:48-54, Main.cpp:17-20].
 * It is a host-side utility (private re-implementation of the glibc TYPE_3 generator; global rand() state
 * is not touched) and needs no GPU. */
int pcnn_init_params_reference(float *host_params);
int pcnn_set_params(pcnn_ctx *ctx, const float *host_params);
int pcnn_get_params(pcnn_ctx *ctx, float *host_params);
int pcnn_get_grads(pcnn_ctx *ctx, float *host_grads);                /* packed gradient of the last step */
int pcnn_params_dev(pcnn_ctx *ctx, float **dev_params);              /* the context's own packed vector */
int pcnn_set_learning_rate(pcnn_ctx *ctx, float dt);                 /* default 0.1f  [ref: layer.h:12] */
/* 9,372-byte packed checkpoint with a 16-byte header (the reference has none; SURVEY.md 8f.3) */
int pcnn_save_params(pcnn_ctx *ctx, const char *path);
int pcnn_load_params(pcnn_ctx *ctx, const char *path);

/* ------------------------------------------------------------------ per-operator API (drop-in for layer.h)
 * Device pointers; row-major arrays shaped as in the reference with a leading batch dimension B (B = 1 is the
 * reference call).  Arithmetic follows the reference's evaluation order in fp32 without FMA contraction and
 * evaluates the sigmoid in double, so B = 1 results are bit-identical to Sequential/layer.h up to the last-ulp
 * difference between CUDA's and glibc's double exp().  For B > 1 the weight-gradient ops sum over the batch
 * and the in-place bias updates use dt / B (DESIGN.md "mini-batch semantics"). */
int pcnn_apply_step_function(pcnn_ctx *ctx, const float *in, float *out, long n);        /* [ref: layer.h:85-89] */
int pcnn_make_error(pcnn_ctx *ctx, float *err, const float *out, unsigned Y, int n);     /* [ref: layer.h:91-95] */
int pcnn_make_error_batch(pcnn_ctx *ctx, float *err, const float *out, const uint8_t *labels, int B);
int pcnn_apply_grad(pcnn_ctx *ctx, float *w, const float *g, long n);                    /* [ref: layer.h:97-101] */
int pcnn_apply_grad_scaled(pcnn_ctx *ctx, float *w, const float *g, long n, float step);
int pcnn_vector_norm(pcnn_ctx *ctx, const float *v, int n, int B, float *norms_dev);     /* [ref: Main.cpp:28-34] */
int pcnn_fp_c1(pcnn_ctx *ctx, const float *in, float *pre, const float *w, const float *b, int B);   /* [ref: layer.h:105-140] */
int pcnn_fp_s1(pcnn_ctx *ctx, const float *in, float *pre, const float *w, const float *b, int B);   /* [ref: layer.h:143-181] */
int pcnn_fp_preact_f(pcnn_ctx *ctx, const float *in, float *pre, const float *w, int B);             /* [ref: layer.h:184-203] */
int pcnn_fp_bias_f(pcnn_ctx *ctx, float *pre, const float *b, int B);                                /* [ref: layer.h:206-211] */
int pcnn_bp_weight_f(pcnn_ctx *ctx, float *dw, const float *dpre, const float *pout, int B);         /* [ref: layer.h:214-227] */
int pcnn_bp_bias_f(pcnn_ctx *ctx, float *bias, const float *dpre, int B);                            /* [ref: layer.h:229-234] */
int pcnn_bp_output_s1(pcnn_ctx *ctx, float *dout, const float *nw, const float *ndpre, int B);       /* [ref: layer.h:237-257] */
int pcnn_bp_preact_s1(pcnn_ctx *ctx, float *dpre, const float *dout, const float *pre, int B);       /* [ref: layer.h:260-270] */
int pcnn_bp_weight_s1(pcnn_ctx *ctx, float *dw, const float *dpre, const float *pout, int B);        /* [ref: layer.h:272-300] */
int pcnn_bp_bias_s1(pcnn_ctx *ctx, float *bias, const float *dpre, int B);                           /* [ref: layer.h:302-317] */
int pcnn_bp_output_c1(pcnn_ctx *ctx, float *dout, const float *nw, const float *ndpre, int B);       /* [ref: layer.h:319-346] */
int pcnn_bp_preact_c1(pcnn_ctx *ctx, float *dpre, const float *dout, const float *pre, int B);       /* [ref: layer.h:348-369] */
int pcnn_bp_weight_c1(pcnn_ctx *ctx, float *dw, const float *dpre, const float *pout, int B);        /* [ref: layer.h:371-395] */
int pcnn_bp_bias_c1(pcnn_ctx *ctx, float *bias, const float *dpre, int B);                           /* [ref: layer.h:398-414] */

/* ------------------------------------------------------------------ data  [ref: Sequential/mnist.h:79-160, Main.cpp:36-42]
 * pcnn_mnist_load_u8 keeps mnist_load's return codes (0 ok, -1 no such files, -2 bad image file, -3 bad label
 * file, -4 count mismatch) but returns the raw u8 pixels instead of the double[28][28] staging. */
int pcnn_mnist_load_u8(const char *image_file, const char *label_file, uint8_t **images, uint8_t **labels,
                       unsigned *count);
void pcnn_mnist_free(void *p);
/* copy a host dataset to the device and bind it as the train / test split (u8 IDX payload or float[784]) */
int pcnn_dataset_upload(pcnn_ctx *ctx, int split, const void *host_images, int pixel_type,
                        const uint8_t *host_labels, long n);
/* bind caller-owned device buffers instead (no copy; caller keeps them alive) */
int pcnn_dataset_bind(pcnn_ctx *ctx, int split, const void *dev_images, int pixel_type,
                      const uint8_t *dev_labels, long n);

/* ------------------------------------------------------------------ fused training / evaluation path
 * One step = forward_pass + makeError + vectorNorm + back_pass for every sample of the batch with frozen
 * parameters, batch-sum of the packed gradient, (optional all-reduce), update  w += (dt / B_global) * g.
 * At B = 1 this is the body of learn()'s loop  [ref: Main.cpp:157-171, 59-144]. */
int pcnn_train_step(pcnn_ctx *ctx, long first, int B);                 /* samples [first, first+B) of the bound train split */
/* consecutive batches starting at `first` (or continuing at the device-side cursor when first == -1), wrapping at the
 * end of the split; replayed from cached CUDA graphs.  _prepare instantiates the graphs such a call needs (untimed). */
int pcnn_train_steps(pcnn_ctx *ctx, long first, int B, int nsteps);
int pcnn_train_steps_prepare(pcnn_ctx *ctx, int B, int nsteps);
int pcnn_train_step_dev(pcnn_ctx *ctx, const void *dev_images, int pixel_type, const uint8_t *dev_labels, int B);
/* host buffers in, H2D inside the call, error-norm sum of the step back out (blocking) */
int pcnn_train_step_host(pcnn_ctx *ctx, const void *host_images, int pixel_type, const uint8_t *host_labels,
                         int B, float *err_sum_out);
/* frozen-parameter gradient only (no update): fills the packed gradient (+ error sum); used by parity tests */
int pcnn_compute_grads(pcnn_ctx *ctx, const void *dev_images, int pixel_type, const uint8_t *dev_labels, int B);
/* learn(): `epochs` passes over the bound train split in dataset order with batch B (tail batch kept);
 * mean_err_out = sum of error norms / n of the LAST epoch, as learn() prints  [ref: Main.cpp:146-184] */
int pcnn_learn(pcnn_ctx *ctx, int B, int epochs, float *mean_err_out);
/* same, with the dataset in HOST memory.  Page-locked images (cudaHostAlloc / cudaHostRegister, 16-byte aligned): the training
 * kernel reads them across PCIe itself, one image per CTA and step, a step ahead -- no staging copy, one label copy + one launch
 * per epoch.  Pageable images: staged through a chunked H2D copy stream that the kernel follows chunk by chunk.  Same samples,
 * same order, bit-identical results either way; returns when the last step's results are in host memory. */
int pcnn_learn_host(pcnn_ctx *ctx, const void *host_images, int pixel_type, const uint8_t *host_labels,
                    long n, int B, int epochs, float *mean_err_out);
int pcnn_err_sum(pcnn_ctx *ctx, double *sum_out, int reset);           /* running sum of per-sample error norms */
/* forward_pass for B samples; f_out_dev [B][10] may be NULL, pred_dev [B] (first-max argmax) may be NULL
 * [ref: Main.cpp:59-105, 186-200] */
int pcnn_forward_batch(pcnn_ctx *ctx, const void *dev_images, int pixel_type, int B, float *f_out_dev,
                       uint8_t *pred_dev);
/* test(): misclassification count over the bound test split  [ref: Main.cpp:202-214] */
int pcnn_test(pcnn_ctx *ctx, long *wrong_out);
/* number of kernels this context has launched since creation (bench.py's gpu_launches) */
int pcnn_launch_count(pcnn_ctx *ctx, long *count_out);
/* per-step error sums recorded by the most recent pcnn_learn_host epoch (device -> pinned host, one float per step) */
int pcnn_step_errs(pcnn_ctx *ctx, float *host_out, long cap, long *count_out);
/* measurement helpers for bench.py (CUDA events on the context's stream, after `iters / 10 + 3` warm-up launches):
 * average duration of the fused gradient kernel alone over `iters` launches walking the bound train split, and the
 * sustained fp32 FMA rate of this GPU under its current clocks (dependent-chain-free FFMA micro-benchmark). */
int pcnn_time_fused_kernel(pcnn_ctx *ctx, int B, int iters, float *avg_ms_out);
int pcnn_measure_fp32_peak(pcnn_ctx *ctx, float *tflops_out);
/* streaming-read rate (GB/s) of a TMA load pipeline with no consumer work over a bf16 tensor [N][P][Q][64] in HBM:
 * mode 0 = 1-D bulk copies of 16 KB, 1 = 2-D boxes of 128 pixels, 2 = the input-gradient kernel's pattern (boxes of
 * 1 pixel x 32 rows), 3 = the weight-gradient kernel's pattern (one row of pixels per box).  The ceiling the convolution
 * backward kernels are measured against next to the HBM copy peak. */
int pcnn_measure_tma_read(pcnn_ctx *ctx, const void *dev_bf16, int N, int P, int Q, int mode, int iters, float *gbps_out);
/* store rate (GB/s) of the forward convolution's epilogue with everything but the stores removed: y viewed as [N][P][row_elems]
 * bf16, tiles of 128 rows x 256 columns walked like the forward kernel (image height H on the input side, H % 32 == 0).  mode 0 =
 * the kernel's own pattern (boxes {64 columns, 32 rows}, 128-byte swizzle), 1 / 2 = boxes of 128 / 256 columns without swizzle,
 * 3 = per-row 1-D bulk stores of 128 bytes, 4 = four boxes per commit group, 5 = 32-byte st.global.v8 from registers (no TMA),
 * 6 = half TMA boxes, half direct stores; hot = 1 aims every tile at the first row block (an
 * L2-resident target).  The ceiling the forward kernel's store phase is measured against.  The tensor is OVERWRITTEN with
 * unspecified values (the staging buffers are never filled). */
int pcnn_measure_tma_write(pcnn_ctx *ctx, void *dev_bf16, int N, int P, int H, int row_elems, int mode, int hot, int iters, float *gbps_out);
/* SM clocks per tcgen05.mma (kind::f16 bf16, K = 16, shape M x N, operands K- or MN-major in shared memory) when one thread
 * issues `reps` of them back to back over `nacc` rotating accumulators: the issue-rate table the convolution kernels are
 * designed against (small-N instructions are far from the tensor-pipe peak). */
int pcnn_measure_mma_rate(pcnn_ctx *ctx, int M, int N, int a_mn_major, int b_mn_major, int nacc, int reps, float *clk_per_mma);

/* ------------------------------------------------------------------ data parallelism (not in the reference; SURVEY.md 8e)
 * Sample-sharded replicas, one process per GPU.  After pcnn_comm_init_rank every train step all-reduces the
 * packed gradient (2,344 floats) once and divides the step by B * world. */
int pcnn_comm_unique_id(void *id_out, size_t *id_bytes);               /* rank 0; 128 bytes */
int pcnn_comm_init_rank(pcnn_ctx *ctx, const void *id, int rank, int world);
int pcnn_comm_destroy(pcnn_ctx *ctx);
int pcnn_allreduce_grads(pcnn_ctx *ctx);
/* In-kernel exchange over NVLink / NVSwitch peer memory (no NCCL launch per step): every rank exports one IPC handle
 * (64 bytes) for its inbox, the handles of all ranks are gathered by any rendezvous and attached.  Afterwards the
 * persistent training kernel pushes its chunk of the reduced gradient straight into every peer's inbox and adds the
 * ranks' chunks in rank order, inside the step. */
int pcnn_p2p_export(pcnn_ctx *ctx, void *handle_out, size_t *handle_bytes);
int pcnn_p2p_attach(pcnn_ctx *ctx, const void *handles, int rank, int world);
int pcnn_p2p_detach(pcnn_ctx *ctx);
/* How cursor-driven steps (pcnn_train_steps, pcnn_learn, pcnn_learn_host) execute: PCNN_MODE_PERSISTENT = one
 * cooperative kernel running all steps (thread-block clusters + tagged words through L2 instead of grid barriers,
 * in-kernel reduction/update/exchange); PCNN_MODE_GRAPH = CUDA graphs of per-step kernels (+ NCCL all-reduce when
 * distributed); PCNN_MODE_AUTO (default) = persistent whenever it can serve the configuration (single GPU, or peers
 * attached), else graph. */
int pcnn_set_step_mode(pcnn_ctx *ctx, int mode);
/* Geometry of the most recent persistent launch and what the device can hold: out6 = { grid, cluster size, co-resident CTAs,
 * co-resident CTAs when launched as clusters, the cluster size the kernel is built for, 1 if the launches are cooperative }.
 * pcnn_persist_tune(ctx, mask): bit 0 forces the variant without clusters; bit 1 keeps the clusters but launches without the
 * cooperative attribute (profilers that re-issue cooperative launches drop the cluster dimension); bit 2 makes
 * pcnn_learn_host enqueue its host copies BEFORE the kernel launch (needed wherever launches block the calling thread:
 * kernel-replay profilers; CUDA_LAUNCH_BLOCKING=1 is detected by itself); bit 3 keeps the two-stage gradient exchange on 2
 * GPUs (default there: cluster shares stored straight into the peer's memory); bit 4 sends pinned host images of
 * pcnn_learn_host through the staged copy stream instead of letting the kernel pull them.  Measurement knobs for the runs
 * under profiles/.
 * out6[5] of pcnn_persist_info: bit 0 = cooperative launch, bit 1 = direct exchange used. */
int pcnn_persist_info(pcnn_ctx *ctx, int *out6);
int pcnn_persist_tune(pcnn_ctx *ctx, int max_cluster);
/* Phase timestamps of the persistent kernel (ns; 6 per step: step start, parameters resident, images done, cluster slot
 * written, owned chunk gathered, parameters published; first 256 steps of a launch, CTA 0).  host_out == NULL arms tracing for the
 * following launches, host_out != NULL reads the stamps back. */
int pcnn_persist_trace(pcnn_ctx *ctx, long long *host_out, int cap_steps);
/* the same six stamps of EVERY CTA at step 128 of the traced launch, rows of 8 (six stamps, SM id, spare): their spread is
 * the skew between CTAs that the gradient owners have to wait for */
int pcnn_persist_trace_ctas(pcnn_ctx *ctx, long long *host_out, int cap_ctas);

/* ------------------------------------------------------------------ north_star extension ops (parity unpinned by the reference)
 * max-pool k x k stride k over [C][H][W] planes with argmax cache (flat index i*k+j, first maximum wins) */
int pcnn_maxpool_fwd(pcnn_ctx *ctx, const float *in, float *out, int32_t *argmax, int planes, int H, int W, int k);
int pcnn_maxpool_bwd(pcnn_ctx *ctx, const float *dout, const int32_t *argmax, float *din, int planes, int H, int W, int k);
/* softmax cross-entropy over n logits per row; d = onehot - p (the reference's sign convention for d_preact) */
int pcnn_softmax_ce(pcnn_ctx *ctx, const float *logits, const uint8_t *labels, int B, int n, float *prob,
                    float *d, float *loss);

/* ------------------------------------------------------------------ LeNet-5-style variant with a second convolution layer
 * (SURVEY.md 8f row 4; PARITY UNPINNED: the reference has exactly one conv layer, layer.h:105-140 / Main.cpp:17-20).
 *     28x28 -> c1 6@5x5 -> s2 shared 2x2/2 weighted sum -> c3 16@5x5 over 6 channels -> s4 shared 2x2/2 -> f 256 -> 10,
 * sigmoid everywhere, the reference's loss (d_preact_f = onehot - output) and its gradient / update rules generalised by
 * rule; oracle/lenet5_oracle.c is the definition.  Packed parameters, PCNN_L5_NPARAM = 5,152 floats:
 *     c1w 150 | c1b 6 | s2w 4 | s2b 1 | c3w [16][6][5][5] 2400 | c3b 16 | s4w 4 | s4b 1 | fw [10][256] 2560 | fb 10.
 * All pointers are device pointers; grads_dev holds PCNN_L5_NPARAM + 1 floats (packed gradient, then the batch sum of
 * error norms) and may be NULL for pcnn_l5_train_step.  One fused kernel per batch (activations and parameters in shared
 * memory) + a fixed-order slot reduction: deterministic.  Update: w += (dt / B) * g with the bias divisors of the rules. */
#define PCNN_L5_NPARAM 5152
int pcnn_l5_compute_grads(pcnn_ctx *ctx, const float *params_dev, const void *images_dev, int pixel_type,
                          const uint8_t *labels_dev, int B, float *grads_dev);
int pcnn_l5_train_step(pcnn_ctx *ctx, float *params_dev, const void *images_dev, int pixel_type, const uint8_t *labels_dev,
                       int B, float *grads_dev);
int pcnn_l5_forward(pcnn_ctx *ctx, const float *params_dev, const void *images_dev, int pixel_type, int B, float *f_out_dev);

/* ------------------------------------------------------------------ bf16 tensor-core convolution (SURVEY.md x3; BASELINE configs 3, 5)
 * The reference's conv semantics (valid, stride 1, cross-correlation, layer.h:118-130) generalised to C input channels,
 * K filters of R x S taps, on tcgen05 tensor cores with TMEM accumulators and TMA-fed operands (csrc/conv_tc.cu).
 * Activations are NHWC bf16 with a row pitch of `row_pitch` elements (>= W*C, multiple of 8); filters fp32 KRSC on the
 * host (rounded to bf16 once, at plan creation); output NHWC bf16 [N][H-R+1][W-S+1][K], bias and optional sigmoid fused.
 * Constraint of this round: some pixel block Qt with (Qt+S-1)*C <= 32, Qt*K <= 256 and Qt*K % 16 == 0 must exist
 * (LeNet c1: Qt = 24; 224x224x3 -> 64 x 3x3: Qt = 4).  PARITY UNPINNED by the reference (it has no bf16 path): the
 * checker is orc_conv_fwd_nhwc in oracle/lenet_oracle.c on the bf16-rounded operands. */
typedef struct pcnn_conv_plan pcnn_conv_plan;
int pcnn_conv_tc_plan_create(pcnn_ctx *ctx, int N, int H, int W, int C, int K, int R, int S, int row_pitch,
                             int image_rows /* rows between consecutive images in memory, >= H; 0 = H.  A multiple of
                                               32 lets the epilogue use asynchronous TMA stores */,
                             int act, const float *filt_host, const float *bias_host, pcnn_conv_plan **plan_out);
/* the same with a window step of `stride` (1..4) in both directions (SURVEY.md 8f row 4): y [N][(H-R)/stride+1][(W-S)/stride+1][K];
 * rows per image (image_rows, or H) must be a multiple of the stride; the pixel block then needs ((Qt-1)*stride+S)*C <= 32.
 * Its backward passes are pcnn_conv_wgrad_strided / pcnn_conv_dgrad_strided below. */
int pcnn_conv_tc_plan_create_strided(pcnn_ctx *ctx, int N, int H, int W, int C, int K, int R, int S, int stride, int row_pitch,
                                     int image_rows, int act, const float *filt_host, const float *bias_host,
                                     pcnn_conv_plan **plan_out);
int pcnn_conv_tc_plan_destroy(pcnn_ctx *ctx, pcnn_conv_plan *plan);
int pcnn_conv_tc_fwd(pcnn_ctx *ctx, pcnn_conv_plan *plan, const void *x_bf16_dev, void *y_bf16_dev);
/* Backward passes of the same convolution (bf16 operands, fp32 accumulation, deterministic; tcgen05 kernels, see
 * pcnn_conv_bwd_select): weight gradient fp32 KRSC [ref: layer.h:371-395 bp_weight_c1, without its /576] and input gradient
 * bf16 NHWC in x's layout.  row_pitch / image_rows as for the forward plan (0 = dense). */
int pcnn_conv_wgrad(pcnn_ctx *ctx, const void *x_bf16_dev, const void *dy_bf16_dev, float *dw_f32_dev, int N, int H, int W, int C,
                    int K, int R, int S, int row_pitch, int image_rows);
int pcnn_conv_dgrad(pcnn_ctx *ctx, const void *dy_bf16_dev, const float *filt_f32_dev, void *dx_bf16_dev, int N, int H, int W,
                    int C, int K, int R, int S, int row_pitch, int image_rows);
/* The same with a window step of `stride` (1..4, else PCNN_ERR_ARG) in both directions: dy [N][(H-R)/stride+1][(W-S)/stride+1][K],
 *     dw[k][r][s][c] = sum dy[n][p][q][k] * x[n][p*stride+r][q*stride+s][c]
 *     dx[n][h][w][c] = sum over (h-r) % stride == 0, (w-s) % stride == 0 of dy[n][(h-r)/stride][(w-s)/stride][k] * f[k][r][s][c].
 * Rows per image need not be a multiple of the stride.  Every dx element is written, rows and columns no tap reaches as 0.
 * stride = 1 is pcnn_conv_wgrad / pcnn_conv_dgrad.  The tensor-core weight gradient needs ((RB-1)*stride + R)*S*C <= 64 for some
 * RB >= 1 and a row pitch that is a multiple of 8 elements; the tensor-core input gradient is built for 3x3 taps with C in
 * {1,2,3,4,8}, 5x5 with C in {1,3} and 7x7 with C = 1 at strides 1 and 2, 3x3 with C in {1,2,3} at stride 3, 3x3x3 and 5x5x1 at
 * stride 4.  Other shapes are refused as for stride 1 (see pcnn_conv_bwd_select). */
int pcnn_conv_wgrad_strided(pcnn_ctx *ctx, const void *x_bf16_dev, const void *dy_bf16_dev, float *dw_f32_dev, int N, int H, int W,
                            int C, int K, int R, int S, int stride, int row_pitch, int image_rows);
int pcnn_conv_dgrad_strided(pcnn_ctx *ctx, const void *dy_bf16_dev, const float *filt_f32_dev, void *dx_bf16_dev, int N, int H, int W,
                            int C, int K, int R, int S, int stride, int row_pitch, int image_rows);
/* Which kernels pcnn_conv_wgrad / pcnn_conv_dgrad may use.  PCNN_CONV_BWD_TENSOR (default): the tcgen05 kernels only (any filter
 * count up to 256: counts that are not a multiple of 64 are zero-padded to one in an extra pass over dy) -- a shape they
 * cannot take is an ERROR (PCNN_ERR_ARG naming the restriction), never a silent detour.  PCNN_CONV_BWD_REFERENCE: the
 * deterministic FMA-pipe kernels of csrc/conv_bwd.cu for every shape (any C, K, taps): a second implementation the tests
 * compare the tensor-core kernels against, ~1 % of the HBM roofline at BASELINE config 5 -- an explicit opt-in. */
typedef enum { PCNN_CONV_BWD_TENSOR = 0, PCNN_CONV_BWD_REFERENCE = 1 } pcnn_conv_bwd_path;
int pcnn_conv_bwd_select(pcnn_ctx *ctx, int path);
/* Host-only query (works without a GPU): which kernels pcnn_conv_wgrad / pcnn_conv_dgrad pick for a shape and how they tile it.
 * out9 = { wgrad on tensor cores, dy rows per tile, pixels per tile, stages,
 *          dgrad on tensor cores, column strips, output pixels per lane quarter, TMEM slot groups in flight, stages } */
int pcnn_conv_bwd_plan_info(int N, int H, int W, int C, int K, int R, int S, int *out9);
/* the same for a window step of `stride` (1..4, else PCNN_ERR_ARG); out9[6] counts dx columns per lane quarter */
int pcnn_conv_bwd_plan_info_strided(int N, int H, int W, int C, int K, int R, int S, int stride, int *out9);
/* Zero padding for the valid-padding kernels above (SURVEY.md 8f row 4): pcnn_pad_nhwc_bf16 embeds dense [N][H][W][C] images into
 * a zeroed canvas [N][dst_image_rows][dst_row_pitch] at row offset pad_h, pixel offset pad_w (0 = the tight canvas
 * [H + 2 pad_h][(W + 2 pad_w) * C]); a "same" convolution is pad -> pcnn_conv_tc_fwd, its input gradient is
 * pcnn_conv_dgrad into a padded canvas -> pcnn_crop_nhwc_bf16, its weight gradient is pcnn_conv_wgrad on the padded x. */
int pcnn_pad_nhwc_bf16(pcnn_ctx *ctx, const void *src_bf16_dev, void *dst_bf16_dev, int N, int H, int W, int C, int pad_h, int pad_w,
                       int dst_row_pitch, int dst_image_rows);
int pcnn_crop_nhwc_bf16(pcnn_ctx *ctx, const void *src_bf16_dev, void *dst_bf16_dev, int N, int H, int W, int C, int pad_h, int pad_w,
                        int src_row_pitch, int src_image_rows);
/* fp32 [rows][w] -> bf16 [rows][pitch] with zero padding (builds the padded activation rows the TMA descriptor needs) */
int pcnn_f32_to_bf16_rows(pcnn_ctx *ctx, const float *src_dev, void *dst_bf16_dev, long rows, int w, int pitch);

#ifdef __cplusplus
}
#endif
#endif /* PCNN_H_ */

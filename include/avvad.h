/*
 * libavvad -- B200-native (sm_100a) hot path of sp-uhh/audio-visual-vad, C ABI.
 *
 * Every entry point takes plain device pointers, sizes and a CUDA stream (as void*); nothing
 * allocates across the ABI except the opaque per-model handles, and all scratch memory is passed
 * in by the caller after a *_workspace_bytes() query.  All functions return 0 on success or a
 * negative avvad_status; avvad_last_error() returns a thread-local description.  There is no CPU
 * fallback: a call without a CUDA device fails with AVVAD_ERR_CUDA.
 *
 * The reference (pure Python) has no FFI of its own; each entry point below names the reference
 * code it replaces (paths relative to the reference repo root).  INTEGRATION.md shows the
 * ctypes stubs a maintainer would add to packages/ to bind them.
 */
#ifndef AVVAD_H_
#define AVVAD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  AVVAD_OK = 0,
  AVVAD_ERR_ARG = -1,     /* bad shape / null pointer / unsupported parameter        */
  AVVAD_ERR_CUDA = -2,    /* CUDA runtime error (see avvad_last_error)               */
  AVVAD_ERR_STATE = -3,   /* handle not fully loaded                                 */
  AVVAD_ERR_WORKSPACE = -4 /* workspace too small                                    */
} avvad_status;

const char* avvad_last_error(void);
int avvad_version(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
uint64_t avvad_launch_count(void);

/* Per-launch device timing of the tensor-core kernels (CUDA events on the launching stream), used by
 * bench.py for the roofline figure.  cat: 0 = implicit-GEMM convolution, 1 = plain GEMM, 2 = LSTM step, 3 = stem,
 * 4 = audio front end, 5 = MCB fusion (for 4 and 5 the "flops" field carries the stage's algorithmic BYTES).
 * avvad_profile_read sums the launches of one category recorded since the last avvad_profile_clear
 * (it synchronises the device); flops = 2*M*N*K per launch. */
int avvad_profile_enable(int on);
int avvad_profile_read(int cat, double* ms, double* flops, uint64_t* launches);
int avvad_profile_clear(void);
/* Per-launch records (launch order) of one category; returns how many were written (<= max_n). */
int64_t avvad_profile_dump(int cat, double* ms, double* flops, int64_t max_n);
/* Debug aid (tools/micro/lstm_ab.py): while `buf` is non-null, the CTA-pair LSTM recurrence runs its tracing
 * instantiation and writes u64 [CTA][T][8] %globaltimer stamps (first K block ready, last TMA issued, first MMA, last
 * commit, accumulator observed, h stored, CTA barrier passed, flag published) into this device buffer. */
void avvad_debug_lstm_trace(void* buf);

/* ------------------------------------------------------------------------------------------
 * Audio front end (SURVEY §8a A1-A4)
 * replaces: packages/processing/stft.py:102-152 (stft_pytorch: pad-at-end rule, periodic Hann,
 *           1024-pt rFFT, hop 256, center=False), packages/data_handling.py:441 (x / max|x|),
 *           :454-457 (re^2+im^2, log(.+eps)), scripts/evaluate_AV_net.py:225-230 ((x-mu)/(sigma+eps)),
 *           and the zero-pad-to-max-T of packages/utils.py:157-166 (collate).
 * ---------------------------------------------------------------------------------------- */

/* Frame count of stft_pytorch(center=False) for an n_samples-long signal, including the
 * pad-at-end rule evaluated in the reference's double arithmetic (stft.py:134-139). */
int64_t avvad_stft_num_frames(int64_t n_samples, double fs, double wlen_sec, double hop_percent,
                              int pad_at_end);

/* wave      : f32 [B][wave_stride] device, utterance b uses the first n_samples[b] samples
 * n_samples : i32 [B] device
 * n_frames  : i32 [B] device -- frames to emit per utterance (<= avvad_stft_num_frames; the
 *             reference trims to the label/video length, data_handling.py:483-486)
 * mean,std  : f32 [513] device or NULL (no standardisation)
 * out       : f32 [B][t_max][513] device.  Rows t >= n_frames[b] get the collate value
 *             (0-mean)/(std+eps) (or 0 when mean==NULL).
 * normalise : 0 = none, 1 = divide by max|x| over the utterance's samples (AV_Net.py:117's peak normalisation),
 *             2 = divide by the peaks the caller put in peak_scratch (a stream cannot see the whole utterance)
 * peak_scratch : f32 [B] device scratch (per-utterance max|x|) with normalise == 1, the given peaks with 2
 * nfft must be 1024 and hop 256 (the reference's 64 ms / 25 % at 16 kHz). */
int avvad_frontend_logpower(const float* wave, int64_t wave_stride, const int32_t* n_samples,
                            const int32_t* n_frames, int32_t B, int32_t t_max, int normalise,
                            const float* mean, const float* std, float eps, float* out,
                            float* peak_scratch, void* stream);

/* avvad_frontend_logpower written straight into a bf16 LSTM layer-0 operand (the audio-only model has nothing between
 * the front end and the recurrence):
 * out_bf16 : bf16 [B][t_max][ld] device.  Row (b, t) gets __float2bfloat16_rn of the value avvad_frontend_logpower
 *            writes to out[b][t][k] at column col_off + k (k < 513), and zeros in columns [col_off + 513, ld); columns
 *            below col_off are not touched.  == avvad_frontend_logpower + avvad_pack_rows_bf16(zero_tail = 1), bit
 *            for bit.
 * ld       : multiple of 8, >= col_off + 513.  Every other argument as avvad_frontend_logpower.  Always runs the
 *            register-FFT kernel (AVVAD_FE_REG only selects the kernel of the f32 output). */
int avvad_frontend_logpower_bf16(const float* wave, int64_t wave_stride, const int32_t* n_samples,
                                 const int32_t* n_frames, int32_t B, int32_t t_max, int normalise,
                                 const float* mean, const float* std, float eps, void* out_bf16, int64_t ld,
                                 int64_t col_off, float* peak_scratch, void* stream);

/* Raw STFT, (B, 513, t_max, 2) real view like the legacy torch.stft the reference calls
 * (stft.py:145-151).  No normalisation / log. */
int avvad_stft(const float* wave, int64_t wave_stride, const int32_t* n_samples,
               const int32_t* n_frames, int32_t B, int32_t t_max, float* out_ft2, void* stream);

/* ------------------------------------------------------------------------------------------
 * Video frame-rate conversion (SURVEY §8a U + A4)
 * replaces: scripts/create_video_train_files_upsampled.py:116-173 (ffmpeg fps=62.5 + x264 + decode)
 *           and scripts/evaluate_AV_net.py:176-182 ((H,W,T)->(T,H,W), standardise).
 * src(k) = (den*(2k+1)-1) / (2*num) with num/den = fps_out/fps_in (25/12 for 30 -> 62.5).
 * ---------------------------------------------------------------------------------------- */
int64_t avvad_upsampled_length(int64_t n_src, int32_t num, int32_t den);

/* src      : u8 or f32 [B][f_max][hw] device (src_is_f32 selects)
 * n_src    : i32 [B] source frames per utterance; n_out: i32 [B] frames to emit
 * out      : f32 [B][t_max][hw]; rows k >= n_out[b] get (0-mean)/(std+eps). */
int avvad_upsample_gather(const void* src, int src_is_f32, const int32_t* n_src, const int32_t* n_out,
                          int32_t B, int32_t f_max, int32_t t_max, int32_t hw, int32_t num, int32_t den,
                          float mean, float std, float eps, int standardise, float* out, void* stream);

/* Just the index map (i32 [n_out]) -- exposed so callers/tests can check it bit-exactly. */
/* Feature-level form of the same gather (optional "dedup" path of the pipeline): the eval-mode trunk is a pure
 * per-frame function and the 62.5 fps sequence is a duplication of the 30 fps one, so the trunk may run on the source
 * frames and its 512-d features be gathered instead:
 *   out[b][k][:] = feat_src[b][avvad_upsample_index(k, n_src[b])][:]  for k < n_out[b],  feat_pad[:] otherwise
 * (feat_pad = trunk feature of the collate zero frame).  Writes f32 [B][t_max][C] and/or bf16 rows at column col_off. */
int avvad_feature_gather(const float* feat_src, const float* feat_pad, const int32_t* n_src, const int32_t* n_out,
                         int32_t B, int32_t f_max, int32_t t_max, int32_t C, int32_t num, int32_t den,
                         float* out_f32, void* out_bf16, int64_t ld_bf16, int64_t col_off, void* stream);

int avvad_upsample_index(int32_t n_src, int32_t n_out, int32_t num, int32_t den, int32_t* out_idx,
                         void* stream);

/* ------------------------------------------------------------------------------------------
 * ResNet-18 trunk on single-channel 67x67 ROIs (SURVEY §8a V1-V3, eval-mode BN folded)
 * replaces: packages/models/AV_Net.py:78-94 / Video_Net.py:60-75 (repeat to 3 channels +
 *           torchvision resnet18 children[:-1]).
 * ---------------------------------------------------------------------------------------- */
typedef struct avvad_resnet18 avvad_resnet18;

int avvad_resnet18_create(avvad_resnet18** out);
void avvad_resnet18_destroy(avvad_resnet18* h);

/* Conv layer order (index): 0 conv1(7x7/2,3->64); 1..4 layer1.{0,1}.conv{1,2};
 * 5 l2.0.conv1, 6 l2.0.conv2, 7 l2.0.downsample, 8 l2.1.conv1, 9 l2.1.conv2; 10..14 layer3 likewise;
 * 15..19 layer4 likewise.  w is the f32 OIHW torch weight; gamma/beta/mean/var the following
 * BatchNorm2d's weight/bias/running_mean/running_var (eps 1e-5).  The layer is folded
 * (w*gamma/sqrt(var+eps), beta-mean*gamma/sqrt(var+eps)) and repacked to bf16 [O][R][S][I]
 * (conv1: 3 input channels summed to 1, K padded 49->64) on the device. */
int avvad_resnet18_set_conv(avvad_resnet18* h, int layer, const float* w, const float* gamma,
                            const float* beta, const float* mean, const float* var, float bn_eps,
                            void* stream);

/* Workspace of one forward call: four rotating NHWC bf16 activation buffers of min(n_frames, chunk_frames) frames
 * (36,992 bytes per frame each).  chunk_frames <= 0 selects 2048; large passes are faster (one launch per layer and
 * pass), the Python engine uses 24,576. */
size_t avvad_resnet18_workspace_bytes(int64_t n_frames, int64_t chunk_frames);

/* frames : f32 [n_frames][67][67] device (already standardised, as the reference's forward gets)
 * feat   : f32 [n_frames][512] device (may be NULL)
 * feat_bf16 : optional bf16 [n_frames][ld_bf16] destination written at column col_off (the LSTM
 *          operand buffer of the concat fusion), may be NULL */
int avvad_resnet18_forward(avvad_resnet18* h, const float* frames, int64_t n_frames,
                           int64_t chunk_frames, void* workspace, size_t workspace_bytes,
                           float* feat, void* feat_bf16, int64_t ld_bf16, int64_t col_off,
                           void* stream);

/* The same trunk fed straight from the 30 fps u8 source frames (rows U + A4 + V1/V2 of SURVEY 8a in one pass):
 * output frame (b, k), k < t_max, is source frame avvad_upsample_index(k, n_src[b]) standardised as
 * (v - mean) / (std + eps) when k < n_out[b] and the collate zero frame otherwise -- bit-identical to
 * avvad_upsample_gather followed by avvad_resnet18_forward, without the fp32 (B, t_max, 67, 67) tensor.
 * src : u8 [B][f_max][67][67] device.  Outputs as avvad_resnet18_forward with n_frames = B * t_max
 * (workspace: avvad_resnet18_workspace_bytes(B * t_max, chunk_frames)). */
int avvad_resnet18_forward_u8(avvad_resnet18* h, const uint8_t* src, const int32_t* n_src,
                              const int32_t* n_out, int32_t B, int32_t f_max, int32_t t_max, int32_t num,
                              int32_t den, float mean, float std, float eps, int standardise,
                              int64_t chunk_frames, void* workspace, size_t workspace_bytes, float* feat,
                              void* feat_bf16, int64_t ld_bf16, int64_t col_off, void* stream);

/* Test hook: run the trunk up to and including conv layer `upto` (see order above; 0 = conv1 +
 * maxpool) and copy that activation (bf16 NHWC) to out_act. */
int avvad_resnet18_forward_upto(avvad_resnet18* h, const float* frames, int64_t n_frames, int upto,
                                void* workspace, size_t workspace_bytes, void* out_act, void* stream);

/* Training-mode forward (SURVEY §8a V3): BatchNorm uses the batch statistics of this call (all n_frames frames) and
 * updates running_mean / running_var (arrays of 20 device pointers in the conv layer order above; NULL = leave
 * untouched) with `momentum`, as nn.BatchNorm2d does while scripts/train_AV_net.py:253 keeps the frozen trunk in
 * train() mode.  avvad_resnet18_set_conv_train loads the un-folded conv weight and the BN affine parameters. */
int avvad_resnet18_set_conv_train(avvad_resnet18* h, int layer, const float* w, const float* gamma, const float* beta,
                                  void* stream);
size_t avvad_resnet18_train_workspace_bytes(int64_t n_frames);
int avvad_resnet18_forward_train(avvad_resnet18* h, const float* frames, int64_t n_frames, void* workspace,
                                 size_t workspace_bytes, float bn_eps, float momentum, float* const* running_mean,
                                 float* const* running_var, float* feat, void* feat_bf16, int64_t ld_bf16,
                                 int64_t col_off, void* stream);

/* Trainable trunk (scripts/train_video_net.py:145-173 hands ALL parameters to Adam, the ResNet included).
 * replaces: autograd of packages/models/Video_Net.py:60-99 (torchvision resnet18 children[:-1] in train() mode).
 * avvad_resnet18_forward_tape = avvad_resnet18_forward_train that also keeps, in the caller-owned `tape`
 * (avvad_resnet18_tape_bytes), every tensor the backward needs (raw conv outputs, post-activation tensors, batch mean /
 * inverse std per BatchNorm layer).  avvad_resnet18_backward turns dfeat (f32 [n][512], the gradient w.r.t. the trunk's
 * features) into the gradients of the 20 convolution weights (PyTorch layout [O][I][k][k] fp32; layer 0: [64][3][7][7])
 * and of the 20 BatchNorm affine parameter pairs (dgamma, dbeta fp32 [C]); dW / dgamma / dbeta are arrays of 20 device
 * pointers in the conv layer order above.  `frames` must be the tensor the matching forward saw. */
size_t avvad_resnet18_tape_bytes(int64_t n_frames);
size_t avvad_resnet18_tape_workspace_bytes(int64_t n_frames);
/* Byte offsets of the tape's tensors (inspection hook used by the parity tests): offsets[0..37] = raw conv1 output
 * (n,34,34,64), its BN+ReLU (n,34,34,64), the pooled map (n,17,17,64), the raw outputs of conv layers 1..19, then
 * (first activation, block output) of the 8 BasicBlocks -- NHWC bf16 --, offsets[38] = float [20][1024] (mean | invstd). */
int avvad_resnet18_tape_layout(int64_t n_frames, int64_t* offsets, int count);
int avvad_resnet18_forward_tape(avvad_resnet18* h, const float* frames, int64_t n_frames, void* workspace,
                                size_t workspace_bytes, void* tape, size_t tape_bytes, float bn_eps, float momentum,
                                float* const* running_mean, float* const* running_var, float* feat, void* feat_bf16,
                                int64_t ld_bf16, int64_t col_off, void* stream);
size_t avvad_resnet18_backward_workspace_bytes(int64_t n_frames);
int avvad_resnet18_backward(avvad_resnet18* h, const float* frames, int64_t n_frames, void* tape, const float* dfeat,
                            void* workspace, size_t workspace_bytes, float bn_eps, float* const* dW,
                            float* const* dgamma, float* const* dbeta, void* stream);

/* ------------------------------------------------------------------------------------------
 * Data preparation on the device (SURVEY 8f rows 1 and 3)
 *
 * avvad_dct_roi_decode: NTCD-TIMIT `.mat` rows (67x67 2-D DCT coefficients per 30 fps frame) -> mouth-ROI frames.
 *   replaces: scripts/create_video_train_files_upsampled.py:137-162, packages/processing/video.py:5-24
 *   (scipy idct(idct(x).T).T in float64, normalisation, np.rot90(., 3)).
 *   dct [n_frames][67*67] f32.  mode 0: per-frame min-max -> u8 [n_frames][67][67] in out_u8 (the variant that produced
 *   the reference's shipped *_upsampled.h5 files), optional raw decode (un-rotated, f32) in out_f32.
 *   mode 1: the script as shipped: (A - A.min()) / max_row_range * 255 over ALL frames of the call, rotated, f32 in
 *   out_f32; needs avvad_dct_roi_workspace_bytes(n_frames).
 * avvad_vad_labels: packages/processing/target.py:5-48 (clean_speech_VAD, center=False): fp32 frame energies summed
 *   in the reference's order, label = energy > 10^vad_threshold * min(energy) (fp64 compare).  labels [B][t_max] f32.
 * avvad_ibm_labels: target.py:50-70 (clean_speech_IBM) on an STFT [B][bins][t_max][2] (avvad_stft layout):
 *   20*log10(|X|+eps) > max - ibm_threshold per utterance.  mask [B][bins][t_max] f32; scratch db same size, max [B].
 * avvad_stats_accumulate / _finalize: scripts/create_audio_train_files.py:273-280,365-368: per-bin running sum and sum
 *   of squares (fp64, caller-zeroed accumulators) over the valid frames of x [B][t_max][bins]; mean = S/n,
 *   std = sqrt((Q - n*mean^2)/(n-1)).
 * ---------------------------------------------------------------------------------------- */
size_t avvad_dct_roi_workspace_bytes(int64_t n_frames);
int avvad_dct_roi_decode(const float* dct, int64_t n_frames, int mode, uint8_t* out_u8, float* out_f32,
                         void* workspace, size_t workspace_bytes, void* stream);
int avvad_vad_labels(const float* wave, int64_t wave_stride, const int32_t* n_samples, const int32_t* n_frames,
                     int32_t B, int32_t t_max, int32_t nfft, int32_t hop, double vad_threshold,
                     float* energy_scratch, float* labels, void* stream);
int avvad_ibm_labels(const float* stft_ft2, const int32_t* n_frames, int32_t B, int32_t t_max, int32_t bins,
                     float eps, float ibm_threshold, float* db_scratch, float* max_scratch, float* mask,
                     void* stream);
int avvad_stats_accumulate(const float* x, const int32_t* n_frames, int32_t B, int32_t t_max, int32_t bins,
                           double* sum, double* sumsq, void* stream);
int avvad_stats_finalize(const double* sum, const double* sumsq, double n, int32_t bins, float* mean, float* std,
                         void* stream);

/* ------------------------------------------------------------------------------------------
 * bf16 tensor-core GEMM  C[M][N] = A[M][K] * W[N][K]^T (+bias)   (tcgen05 / TMEM)
 * Exposed for tests and for the LSTM / head projections.  A, W bf16 row-major with K % 64 == 0
 * and 16-byte aligned rows; C f32 or bf16.
 * ---------------------------------------------------------------------------------------- */
int avvad_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                    void* C, int64_t ldc, int c_is_bf16, int relu, int64_t M, int64_t N, int64_t K,
                    void* stream);

/* Generic NHWC bf16 convolution through the same engine (tests; ResNet uses it internally).
 * in [n][H][W][Cin], w [Cout][R][S][Cin], out [n][OH][OW][Cout], residual optional (same as out). */
int avvad_conv2d_nhwc_bf16(const void* in, const void* w, const float* bias, const void* residual,
                           void* out, int64_t n, int H, int W, int Cin, int Cout, int R, int S,
                           int stride, int pad, int relu, void* stream);

/* Same convolution with a second operand appended along K (ResNet downsample blocks, torchvision BasicBlock with
 * `downsample`: out = relu(bn2(conv2(y)) + bn_ds(conv1x1_s2(x))), AV_Net.py:25-30 via torchvision resnet18):
 *   out = act( conv_{RxS,stride,pad}(in; w[:, :R*S*Cin]) + conv_{1x1,stride2,0}(in2; w[:, R*S*Cin:]) + bias )
 * in2 [n][H2][W2][Cin2]; w [Cout][R*S*Cin + Cin2]; both convolutions must produce the same OH x OW grid. */
int avvad_conv2d_nhwc_bf16_dual(const void* in, const void* in2, const void* w, const float* bias, void* out,
                                int64_t n, int H, int W, int Cin, int H2, int W2, int Cin2, int stride2, int Cout,
                                int R, int S, int stride, int pad, int relu, void* stream);

/* f32 -> bf16 row repack: dst[m][col_off + j] = bf16(src[m][j]) for j < cols; optional zero fill of
 * [col_off+cols, ld_dst) when zero_tail != 0. */
int avvad_pack_rows_bf16(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int64_t col_off,
                         int64_t rows, int64_t cols, int zero_tail, void* stream);

/* ------------------------------------------------------------------------------------------
 * MCB fusion (SURVEY §8a F2-F3)
 * replaces: packages/models/compact_bilinear_pooling.py:140-173 and AV_Net.py:111-121
 *           (count sketches -> circular convolution -> signed sqrt -> whole-tensor L2 -> BN1d eval).
 * ---------------------------------------------------------------------------------------- */
typedef struct avvad_mcb avvad_mcb;
int avvad_mcb_create(avvad_mcb** out);
void avvad_mcb_destroy(avvad_mcb* h);
/* h1,h2: i64 [513]/[512] device; s1,s2 f32; BN1d(1024) eval parameters. */
int avvad_mcb_load(avvad_mcb* h, const int64_t* h1, const float* s1, const int64_t* h2, const float* s2,
                   const float* bn_gamma, const float* bn_beta, const float* bn_mean,
                   const float* bn_var, float eps, void* stream);
size_t avvad_mcb_workspace_bytes(int64_t rows);
/* audio f32 [rows][513], video f32 [rows][512] -> out_bf16 [rows][ld_out] (first 1024 columns),
 * optional out_f32 [rows][1024] (post-BN, for tests). */
int avvad_mcb_forward(avvad_mcb* h, const float* audio, const float* video, int64_t rows,
                      void* workspace, size_t workspace_bytes, void* out_bf16, int64_t ld_out,
                      float* out_f32, void* stream);

/* Grouped forward: rows = n_groups utterances x t_max rows ([b][t] layout), lengths i32 [n_groups] (device) valid rows
 * each.  Every utterance is divided by its OWN L2 norm over its valid rows, i.e. a batched call reproduces n_groups
 * stand-alone forward calls of the reference module -- what scripts/evaluate_AV_net.py:186-236 does (x[None], v[None],
 * lengths = [T]: one utterance per call, so AV_Net.py:117's whole-tensor norm is a per-utterance norm there).  Rows
 * behind an utterance's length are skipped and written as zeros. */
size_t avvad_mcb_grouped_workspace_bytes(int64_t n_groups, int64_t t_max);
int avvad_mcb_forward_grouped(avvad_mcb* h, const float* audio, const float* video, int64_t n_groups, int64_t t_max,
                              const int32_t* lengths, void* workspace, size_t workspace_bytes, void* out_bf16,
                              int64_t ld_out, float* out_f32, void* stream);
/* As avvad_mcb_forward_grouped; norms_in (f32 [n_groups] device or NULL): divide by these norms instead of computing
 * them (streaming: every block of an utterance uses one norm); norms_out (or NULL): receives the norms used. */
int avvad_mcb_forward_grouped_norms(avvad_mcb* h, const float* audio, const float* video, int64_t n_groups,
                                    int64_t t_max, const int32_t* lengths, const float* norms_in, float* norms_out,
                                    void* workspace, size_t workspace_bytes, void* out_bf16, int64_t ld_out,
                                    float* out_f32, void* stream);

/* Training mode (module in train()): BatchNorm1d uses this call's batch statistics and the CURRENT gamma/beta, updates
 * running_mean/var in place (NULL = leave); the workspace then carries what avvad_mcb_backward_bn needs to turn the
 * gradient w.r.t. the BN output (dx, f32 [rows][ld_dx]) into dgamma / dbeta [1024]. */
int avvad_mcb_forward_train(avvad_mcb* h, const float* audio, const float* video, int64_t rows, void* workspace,
                            size_t workspace_bytes, const float* gamma, const float* beta, float momentum,
                            float* running_mean, float* running_var, void* out_bf16, int64_t ld_out, float* out_f32,
                            void* stream);
int avvad_mcb_backward_bn(avvad_mcb* h, void* workspace, const float* dx, int64_t ld_dx, int64_t rows, float* dgamma,
                          float* dbeta, void* stream);

/* ------------------------------------------------------------------------------------------
 * Host-side codec of the reference's on-disk format (SURVEY §8f row 3): LZF, the chunk filter (HDF5 filter id 32000)
 * the reference writes every *.h5 with (scripts/create_video_train_files_upsampled.py:99,261; create_audio_train_files.py:86).
 * replaces: the h5py/liblzf dependency of packages/data_handling.py:6 for reading and of the create_*_train_files
 *           scripts for writing; the HDF5 container itself is handled by avvad/h5min.py.  Host pointers, no CUDA.
 * compress: returns the compressed size, 0 if it does not fit in `cap`; hlog = log2 of the hash-table size (h5py: 17);
 *           table = NULL or a caller-owned uint32[2^hlog] carried from chunk to chunk (reproduces h5py byte for byte).
 * decompress: returns the number of bytes produced, -1 on a malformed stream.
 * ---------------------------------------------------------------------------------------- */
int64_t avvad_lzf_compress(const uint8_t* in, int64_t in_len, uint8_t* out, int64_t cap, int hlog, uint32_t* table);
int64_t avvad_lzf_decompress(const uint8_t* in, int64_t in_len, uint8_t* out, int64_t cap);

/* Stand-alone CountSketch / CompactBilinearPooling modules
 * replaces: packages/models/compact_bilinear_pooling.py:7-57 (CountSketchFn forward/backward) and :140-220
 *           (CompactBilinearPoolingFn forward and hand-written backward).
 * off/idx: CSR of the inverse map j -> {i : h_i = j} (ascending i; off has out_size+1 entries), h: int32 copy of the
 * sketch indices, s: +-1.  The raw MCB entry points are fixed to the model's sizes (513, 512 -> 1024). */
int avvad_count_sketch_forward(const float* x, int64_t rows, int in_size, int out_size, const int32_t* off,
                               const int32_t* idx, const float* s, float* out, void* stream);
int avvad_count_sketch_backward(const float* grad_out, int64_t rows, int in_size, int out_size, const int32_t* h,
                                const float* s, float* grad_x, void* stream);
int avvad_mcb_raw_forward(const int32_t* off1, const int32_t* idx1, const float* s1, const int32_t* off2,
                          const int32_t* idx2, const float* s2, const float* x, const float* y, int64_t rows,
                          float* out, void* stream);
/* grad_x [rows][513] and/or grad_y [rows][512] (NULL = skip) from grad_out [rows][1024]. */
int avvad_mcb_raw_backward(const int32_t* off1, const int32_t* idx1, const float* s1, const int32_t* h1,
                           const int32_t* off2, const int32_t* idx2, const float* s2, const int32_t* h2,
                           const float* x, const float* y, const float* grad_out, int64_t rows, float* grad_x,
                           float* grad_y, void* stream);

/* ------------------------------------------------------------------------------------------
 * 2-layer (generic L) unidirectional LSTM over padded batches + Linear head (SURVEY R1,R2,H1,H2)
 * replaces: AV_Net.py:127-140, Audio_Net.py:50-59, Video_Net.py:101-116
 *           (pack_padded_sequence -> nn.LSTM -> pad_packed_sequence -> nn.Linear) and the
 *           sigmoid / >0.5 of scripts/evaluate_AV_net.py:239-240.
 * ---------------------------------------------------------------------------------------- */
typedef struct avvad_lstm avvad_lstm;
int avvad_lstm_create(avvad_lstm** out, int layers, int input_size, int hidden, int y_dim);
void avvad_lstm_destroy(avvad_lstm* h);
/* PyTorch layout: w_ih [4H][I_l], w_hh [4H][H], b_ih/b_hh [4H]; gate order i,f,g,o. */
int avvad_lstm_set_layer(avvad_lstm* h, int layer, const float* w_ih, const float* w_hh,
                         const float* b_ih, const float* b_hh, void* stream);
int avvad_lstm_set_head(avvad_lstm* h, const float* w, const float* b, void* stream);
/* Padded input width (bf16 elements) the caller must lay the layer-0 operand out with. */
int64_t avvad_lstm_input_ld(const avvad_lstm* h);
size_t avvad_lstm_workspace_bytes(const avvad_lstm* h, int64_t B, int64_t T);
/* x_bf16  : bf16 [B][T][ld_x] device, ld_x == avvad_lstm_input_ld(h), columns >= input_size zero
 * lengths : i32 [B] device
 * logits  : f32 [B][T][y_dim]; rows t >= len_b receive the head bias (zeros through the Linear)
 * post, dec : optional f32 / i32 [B][T][y_dim]: sigmoid(logit) and (sigmoid > 0.5)
 * last_logits: optional f32 [B][y_dim]: head applied to the last valid step (return_last=True)
 * Streams: with two layers the call forks onto a handle-owned side stream (layer 1 follows layer 0 one chunk of time
 * steps behind) and joins `stream` again before it returns; every output is ordered on `stream` as usual.  One call at a
 * time per handle (the handle owns the side stream, its events and the flag area inside `workspace`). */
int avvad_lstm_forward(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                       void* workspace, size_t workspace_bytes, float* logits, float* post,
                       int32_t* dec, float* last_logits, void* stream);
/* Streaming: as avvad_lstm_forward, continuing from a recurrent state and returning the state after the call.
 * h_in / h_out : bf16 [layers][B][H] (the h the recurrence feeds its MMA), c_in / c_out : f32 [layers][B][H].
 * Row b carries lengths[b] new steps (0 <= lengths[b] <= T; 0 passes the state through).  h_in / c_in NULL = zero
 * state; h_out / c_out may be NULL or alias h_in / c_in (the call reads its input state before it writes the output).
 * h_out[l][b] / c_out[l][b] are layer l's h and c at step lengths[b] - 1.  Running a sequence in blocks with the state
 * carried gives the logits of one call on the whole sequence, bit for bit, on every recurrence path.
 * workspace: avvad_lstm_state_workspace_bytes(h, B, T).  The logit outputs may all be NULL when h_out or c_out is set. */
size_t avvad_lstm_state_workspace_bytes(const avvad_lstm* h, int64_t B, int64_t T);
int avvad_lstm_forward_state(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                             const void* h_in, const float* c_in, void* h_out, float* c_out,
                             void* workspace, size_t workspace_bytes, float* logits, float* post,
                             int32_t* dec, float* last_logits, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training step of the LSTM + head (SURVEY §8a O1): forward that keeps activations, BPTT, fused Adam
 * replaces: autograd of packages/models/AV_Net.py:127-140 and torch.optim.Adam (scripts/train_AV_net.py:238,305-307).
 * ---------------------------------------------------------------------------------------- */
size_t avvad_lstm_tape_bytes(int layers, int hidden, int64_t B, int64_t T);
/* Byte offsets of the tape's tensors (inspection hook used by the state tests, host only): offsets[3l + 0, 1, 2] =
 * layer l's
 *   gates : bf16 [B][T][4H] post-activation gates, gate-interleaved (element 4u+g, g = i, f, g, o);
 *   c     : f32  [B][T][H] cell state c_t;
 *   hseq  : bf16 [B][T][H] output h_t in PyTorch unit order, exactly 0 for t >= len_b.
 * count must be 3 * layers. */
int avvad_lstm_tape_layout(int layers, int hidden, int64_t B, int64_t T, int64_t* offsets, int count);
int avvad_lstm_forward_train(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                             void* workspace, size_t workspace_bytes, void* tape, size_t tape_bytes, float* logits,
                             void* stream);
size_t avvad_lstm_backward_workspace_bytes(const avvad_lstm* h, int64_t B, int64_t T);
/* dlogits f32 [B][T][1]; gradients fp32 in PyTorch layout: dW_ih[l] [4H][I_l], dW_hh[l] [4H][H], db[l] [4H] (bias_ih
 * and bias_hh share it), dW_head [1][H], db_head [1]; dx optional f32 [B][T][input_size]. */
int avvad_lstm_backward(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T, void* tape,
                        const float* dlogits, void* workspace, size_t workspace_bytes, float* const* dW_ih,
                        float* const* dW_hh, float* const* db, float* dW_head, float* db_head, float* dx, void* stream);
/* Training with a carried state (nn.LSTM's hx, truncated BPTT over blocks of a long sequence).  State shapes and the
 * NULL / aliasing rules are those of avvad_lstm_forward_state: h bf16 and c f32, both [layers][B][H].
 * The stateful tape holds T + 1 positions per row (tape_bytes >= avvad_lstm_tape_bytes(layers, H, B, T + 1); inspect it
 * with avvad_lstm_tape_layout(layers, H, B, T + 1, ...)): position 0 holds the initial state -- h_in in hseq, c_in in
 * c, zero gates -- and positions 1..lengths[b] the call's steps.
 * workspace: avvad_lstm_train_state_workspace_bytes(h, B, T). */
size_t avvad_lstm_train_state_workspace_bytes(const avvad_lstm* h, int64_t B, int64_t T);
int avvad_lstm_forward_train_state(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                                   const void* h_in, const float* c_in, void* h_out, float* c_out,
                                   void* workspace, size_t workspace_bytes, void* tape, size_t tape_bytes,
                                   float* logits, void* stream);
/* BPTT over a stateful tape; x_bf16, lengths, B and T as given to avvad_lstm_forward_train_state, dlogits f32
 * [B][T][y_dim], the gradients as in avvad_lstm_backward.  dh_out / dc_out f32 [layers][B][H] (NULL = zero): the
 * gradient w.r.t. h_out / c_out, entering each row at its last step lengths[b] - 1.  dh_in / dc_in f32 [layers][B][H]
 * (NULL = not wanted; the recurrent GEMM that produces them is then skipped): the gradient w.r.t. h_in / c_in.  A row
 * of length 0 passes dh_out / dc_out through.  The outputs may alias dh_out / dc_out.
 * workspace: avvad_lstm_backward_state_workspace_bytes(h, B, T). */
size_t avvad_lstm_backward_state_workspace_bytes(const avvad_lstm* h, int64_t B, int64_t T);
int avvad_lstm_backward_state(avvad_lstm* h, const void* x_bf16, const int32_t* lengths, int64_t B, int64_t T,
                              void* tape, const float* dlogits, const float* dh_out, const float* dc_out,
                              float* dh_in, float* dc_in, void* workspace, size_t workspace_bytes,
                              float* const* dW_ih, float* const* dW_hh, float* const* db,
                              float* dW_head, float* db_head, float* dx, void* stream);
/* torch.optim.Adam update (no weight decay, no amsgrad): step >= 1 is the 1-based update count. */
int avvad_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                    float beta1, float beta2, float eps, int64_t step, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training-loop loss and metrics over padded batches (SURVEY §8a L1, L2)
 * replaces: the per-utterance Python loops of scripts/train_AV_net.py:298-301 (sum over utterances of
 *           packages/models/utils.py:113 binary_cross_entropy) and :311-329 (packages/models/utils.py:164-203 f1_loss).
 * ---------------------------------------------------------------------------------------- */
/* logits,target: f32 [B][T][y_dim]; lengths i32 [B]; loss f32[1]; per_utt f32[B] (per-utterance mean BCE);
 * dlogits: optional f32 [B][T][y_dim] = d loss / d logits (zero on padded steps). */
int avvad_bce_loss(const float* logits, const float* target, const int32_t* lengths, int32_t B, int32_t T,
                   int32_t y_dim, float eps, float* loss, float* per_utt, float* dlogits, void* stream);
/* y_dim == 1.  metrics f32 [B][4] = (accuracy, precision, recall, f1) per utterance; dec optional i32 [B][T]. */
int avvad_f1_metrics(const float* logits, const float* target, const int32_t* lengths, int32_t B, int32_t T,
                     float epsilon, float* metrics, int32_t* dec, void* stream);

/* ------------------------------------------------------------------------------------------
 * WaveNet-style encoder (SURVEY §8a W1; unused by the reference's scripts but on the path by north_star decree)
 * replaces: packages/models/wavenet_autoencoder.py:74-93 (_encode).
 * ---------------------------------------------------------------------------------------- */
typedef struct avvad_wavenet avvad_wavenet;
int avvad_wavenet_create(avvad_wavenet** out, int filter_width, int quantization_channel, const int32_t* dilations,
                         int n_dilations, int residual_channel, int dilation_channel, int bottleneck_width,
                         int pool_size);
void avvad_wavenet_destroy(avvad_wavenet* h);
/* kind: 0 en_causal_layer, 1 en_dilation_layer_stack[index], 2 en_dense_layer_stack[index], 3 bottleneck_layer.
 * w: torch Conv1d weight f32 [O][I][k]; bias f32 [O] or NULL. */
int avvad_wavenet_set_layer(avvad_wavenet* h, int kind, int index, const float* w, const float* bias, void* stream);
int64_t avvad_wavenet_encoded_length(const avvad_wavenet* h, int64_t n_samples);
size_t avvad_wavenet_workspace_bytes(const avvad_wavenet* h, int64_t B, int64_t N);
/* x f32 (B, quantization_channel, N) -> out f32 (B, bottleneck_width, pool_size) */
int avvad_wavenet_encode(avvad_wavenet* h, const float* x, int64_t B, int64_t N, void* workspace,
                         size_t workspace_bytes, float* out, void* stream);
/* Training.  The forward with a tape computes exactly what avvad_wavenet_encode computes and also keeps, in the caller's
 * tape buffer (avvad_wavenet_tape_bytes), every layer input S_i (bf16), every dense-layer operand relu(dilated_i + bias)
 * (bf16) and the bottleneck output (f32).  Same workspace as avvad_wavenet_encode. */
size_t avvad_wavenet_tape_bytes(const avvad_wavenet* h, int64_t B, int64_t N);
int avvad_wavenet_encode_train(avvad_wavenet* h, const float* x, int64_t B, int64_t N, void* workspace,
                               size_t workspace_bytes, void* tape, size_t tape_bytes, float* out, void* stream);
size_t avvad_wavenet_backward_workspace_bytes(const avvad_wavenet* h, int64_t B, int64_t N);
/* Gradients of a loss given dout = d loss / d out, f32 (B, bottleneck_width, pool_size) contiguous, from the tape of
 * avvad_wavenet_encode_train on the same x, B, N and weights.  dw[i] (f32 [O][I][k], torch Conv1d layout) and db[i]
 * (f32 [O]) for i = 0 en_causal_layer, 1 + 2j en_dilation_layer_stack[j], 2 + 2j en_dense_layer_stack[j],
 * 1 + 2n bottleneck_layer; every dw[i] is required, db may be NULL or hold NULL entries (use_bias=False: nothing is
 * written).  dx: f32 (B, quantization_channel, N) or NULL.  Deterministic: identical calls give identical bits. */
int avvad_wavenet_backward(avvad_wavenet* h, const float* x, int64_t B, int64_t N, const void* tape, size_t tape_bytes,
                           const float* dout, float* dx, float* const* dw, float* const* db, void* workspace,
                           size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AVVAD_H_ */

/*
 * aniportrait_b200 — C ABI of the B200-native (sm_100a) AniPortrait denoising hot path.
 *
 * The reference (Zejun-Yang/AniPortrait) is pure Python/PyTorch and has no FFI: its "operator interface" for this
 * path is the set of torch/diffusers library calls issued by src/models/*.py. Each entry point below replaces one such
 * family of calls (cited per function as reference file:line); the Python host mirror in aniportrait_b200/models and
 * aniportrait_b200/pipelines binds them with ctypes (see INTEGRATION.md for the binding a reference maintainer adds).
 *
 * Conventions
 *   - plain C types only; all tensors are raw CUDA device pointers owned by the caller (torch in practice)
 *   - activations are fp16, channels-last: images [frames, H, W, C] == token matrices [frames*H*W, C]
 *   - `stream` is a cudaStream_t passed as void*; functions only enqueue work: no allocation, no synchronisation
 *   - return 0 on success, a negative AP_ERR_* otherwise; ap_last_error() gives a thread-local message
 *   - there is NO CPU fallback: every function fails if the CUDA device is not a compute-capability 10.x GPU
 */
#ifndef ANIPORTRAIT_B200_H_
#define ANIPORTRAIT_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define AP_VERSION 200

#define AP_OK 0
#define AP_ERR_INVALID (-1)  /* bad argument / unsupported shape */
#define AP_ERR_CUDA (-2)     /* CUDA runtime / driver error      */
#define AP_ERR_DEVICE (-3)   /* not an sm_100 device             */

/* flags for ap_gemm_f16 */
#define AP_GEMM_GEGLU 1 /* weight rows interleaved [16 value | 16 gate]; out = value * gelu_erf(gate), N/2 columns */
#define AP_GEMM_OUT_F32 2 /* `out` is fp32 [M, ldo] (used for the small per-step bias tables) */
/* out = gelu_erf(acc + bias) (bias optional; no residual, no epilogue statistics): the wav2vec2 feature-extractor convolutions
 * 1-6 (Conv1d without bias + GELUActivation, transformers Wav2Vec2NoLayerNormConvLayer) and each encoder layer's
 * feed_forward.intermediate_dense + intermediate_act_fn (reference src/audio_models/wav2vec2.py:30,47 -> transformers) */
#define AP_GEMM_GELU 4

/*
 * Optional epilogue extensions of ap_gemm_f16 / ap_conv3x3_nhwc_f16 (pass NULL for none). They need the TMA epilogue
 * (16-byte aligned fp16 output with ldo % 8 == 0); the functions fail otherwise.
 *
 * Statistics for the NEXT normalisation, fused into this op's epilogue (reference: the standalone nn.LayerNorm /
 * nn.GroupNorm passes of src/models/attention.py:331-362, motion_module.py:228-241, resnet.py:221-238): computed from the
 * fp16-rounded outputs, written as per-warp partials in a fixed layout (no atomics; consumers add them in a fixed order).
 *   row_stat_out  fp32 pairs {sum, sumsq} [parts][row_stat_ld]: output row m over the columns one epilogue warp handled;
 *                 parts = 2 * ap_gemm_row_stat_parts(...) ; row_stat_ld >= M rounded up to 128
 *   col_stat_out  fp32 pairs per output column over 32 consecutive rows: [ceil(M / 128) * 4][col_stat_ld]
 *                 (conv: 32-row sub-boxes of the output tile; needs Ho * Wo % 32 == 0 so that no sub-box spans two frames)
 * LayerNorm folded into this GEMM: A = [x | a2] with a2 = the [M, 8] fp16 matrix written by ap_layernorm_finalize_f16
 * (columns -mean_hi, -mean_lo, -mean_hi, 0...), weights [W diag(gamma) | colsum_hi, colsum_hi, colsum_lo, 0...] (K1 + 8
 * columns), `bias` = beta.W^T + b; the accumulator then holds x.W'^T - mean colsum(W') and the epilogue applies
 *   out = ln_rstd[m] * acc + bias.
 *   bias_ld       row stride of the bias table in floats (0 = N): lets several ops share one [groups, sum of N] table
 */
typedef struct ap_epilogue_ext {
  void* row_stat_out;
  long long row_stat_ld;
  void* col_stat_out;
  long long col_stat_ld;
  const float* ln_rstd;
  long long bias_ld;
} ap_epilogue_ext;

int ap_version(void);
const char* ap_last_error(void);
/* Binds the library to `device` (cudaSetDevice), verifies sm_100, resolves the driver entry points it needs. */
int ap_init(int device);

/*
 * out[M, N] = A[M, K1 (+K2)] . W[N, K1+K2]^T (+ bias) (+ residual)            -- fp16 in, fp32 accumulate, fp16 out
 * Replaces nn.Linear / 1x1 Conv2d / diffusers Attention.to_{q,k,v,out} / FeedForward projections:
 *   reference src/models/transformer_3d.py:64-66,93-95,124-160; src/models/attention.py:323-361;
 *   src/models/motion_module.py:122,144,163-170,233; src/models/resnet.py:207-209 (1x1 conv_shortcut, two-source
 *   K = torch.cat([hidden, skip]) of src/models/unet_3d_blocks.py:697,826 without materialising the concat).
 * a/a2: row-major fp16, leading dims lda/lda2 (elements); a2 may be NULL. w: [N, K1+K2] row-major contiguous.
 * bias: fp32 [groups, N] or NULL; output row m uses bias row m / bias_group_rows (<=0: one shared row).
 * residual: fp16 [M, ldr] or NULL. n_valid: columns >= n_valid are not written (<=0: all).
 * block_n: 0 = auto (N must be a multiple of 32).
 */
int ap_gemm_f16(const void* a, long long lda, int K1, const void* a2, long long lda2, int K2, const void* w,
                long long M, int N, const float* bias, long long bias_group_rows, const void* residual,
                long long ldr, void* out, long long ldo, int n_valid, int flags, int block_n, void* stream,
                const ap_epilogue_ext* ext);
/* Number of n-groups (work items along N) ap_gemm_f16 will use for this shape: row_stat_out needs 2x this many parts. */
int ap_gemm_row_stat_parts(long long M, int N, int K, int flags, int block_n);

/*
 * 3x3 convolution, zero padding 1, stride 1|2, channels-last fp16, as an implicit GEMM (no im2col buffer).
 * Replaces InflatedConv3d / Downsample3D / Upsample3D.conv (reference src/models/resnet.py:10-18,52,107,166,195)
 * and conv_in/conv_out (src/models/unet_3d.py:90,250).
 * x: [Nf, H, W, C1]; x2: optional [Nf, H, W, C2] concatenated after x along channels; C1, C2 multiples of 64.
 * w: [Cout, 3, 3, C1+C2] (tap-major, channel-minor) fp16. out/residual: [Nf, H/stride, W/stride, ldo].
 */
int ap_conv3x3_nhwc_f16(const void* x, int C1, const void* x2, int C2, int Nf, int H, int W, int stride,
                        const void* w, int Cout, const float* bias, long long bias_group_rows,
                        const void* residual, void* out, long long ldo, int n_valid, int block_n, void* stream,
                        const ap_epilogue_ext* ext);

/*
 * GroupNorm over channels-last activations, optional fused SiLU, optional second source concatenated along channels
 * (the normalised concat of [hidden, skip] is written once, replacing torch.cat + GroupNorm + SiLU).
 * Replaces InflatedGroupNorm / nn.GroupNorm (reference src/models/resnet.py:21-29,221-222,232-238;
 * src/models/transformer_3d.py:124; src/models/motion_module.py:156; src/models/unet_3d.py:573-574).
 * x: [Nf, HW, C1], x2: [Nf, HW, C2] or NULL, out: [Nf, HW, C1+C2]; statistics per (frame, group) in fp32.
 * stats: caller-provided fp32 workspace of 2*groups*(Nf + 2*AP_GN_MAX_BLOCKS) floats ({mean, rstd} per (frame, group)
 * followed by per-block partial sums: the reduction is atomic-free, results are bit-reproducible run to run).
 */
#define AP_GN_MAX_BLOCKS 2368
int ap_groupnorm_nhwc_f16(const void* x, int C1, const void* x2, int C2, int Nf, int HW, int groups, float eps,
                          const float* gamma, const float* beta, int silu, float* stats, void* out, void* stream);

/*
 * The same GroupNorm with the statistics pass removed: {sum, sumsq} per channel and 32-row block were written by the
 * epilogue of the op that produced x (ap_epilogue_ext.col_stat_out of ap_gemm_f16 / ap_conv3x3_nhwc_f16); this call only
 * reduces them per (frame, group) and applies the normalisation. colstat*: fp32 pairs [Nf * HW / 32][ld*]; HW % 32 == 0,
 * at most 32 groups. stats: fp32 workspace of 2 * groups * Nf floats.
 */
int ap_groupnorm_apply_nhwc_f16(const void* x, int C1, const void* colstat1, long long ld1, const void* x2, int C2,
                                const void* colstat2, long long ld2, int Nf, int HW, int groups, float eps,
                                const float* gamma, const float* beta, int silu, float* stats, void* out, void* stream);

/*
 * Row statistics -> the two small operands of a LayerNorm-folded GEMM. row_stat: fp32 pairs [parts][ld] as written by
 * ap_epilogue_ext.row_stat_out of the op that produced x [M, K]; a2_out: fp16 [M, 8] = (-mean_hi, -mean_lo, -mean_hi, 0 x 5)
 * (mean split into two halves so that the fp16 operand carries it to ~2^-22); rstd_out: fp32 [M] = 1 / sqrt(var + eps).
 * Partials are added in a fixed order (bit-reproducible).
 */
int ap_layernorm_finalize_f16(const void* row_stat, int parts, long long ld, long long M, int K, float eps, void* a2_out,
                              float* rstd_out, void* stream);

/*
 * LayerNorm over the last dim (+ optional additive table pe[(row / rows_per_pe) % pe_period][C], the motion module's
 * sinusoidal frame encoding which the reference adds to the LayerNorm output, src/models/motion_module.py:365-366).
 * Replaces nn.LayerNorm (reference src/models/attention.py:331-362; src/models/motion_module.py:228-241).
 */
int ap_layernorm_f16(const void* x, long long rows, int C, float eps, const float* gamma, const float* beta,
                     const float* pe, int rows_per_pe, int pe_period, void* out, void* stream);

/*
 * BatchNorm2d with BATCH statistics (train mode: biased variance over all `rows` = frames*H*W of the call) + optional ReLU,
 * channels-last. Replaces nn.BatchNorm2d + nn.ReLU of the PoseGuider, which the reference never switches to eval mode
 * (reference src/models/pose_guider.py:19-89; scripts/pose2vid.py:102-110). x/out: [rows, C] fp16, C % 8 == 0.
 * workspace: fp32, at least 2*C*(AP_BN_MAX_BLOCKS+1) floats (per-block partial sums, then the per-channel affine pair);
 * two-stage order-fixed reduction, double-precision finalize.
 */
#define AP_BN_MAX_BLOCKS 2048
int ap_batchnorm_train_nhwc_f16(const void* x, long long rows, int C, const float* gamma, const float* beta, float eps,
                                int relu, float* workspace, long long workspace_floats, void* out, void* stream);

/*
 * Direct convolution for the PoseGuider stem's small channel counts (reference src/models/pose_guider.py:19-40):
 * x [Nf, H, W, Cin] fp16 with Cin in {8 (3 padded), 16, 32}; w [Cout, K, K, Cin] fp16; (K, stride) in {(3,1), (4,2)};
 * out [Nf, Ho, Wo, Cout], Cout % 16 == 0 (% 8 for Cin = 8, K = 3); bias fp32 [Cout] or NULL. Wider 3x3 convolutions go
 * through ap_conv3x3_nhwc_f16.
 */
int ap_conv2d_direct_nhwc_f16(const void* x, int Cin, int Nf, int H, int W, const void* w, int Cout, int K, int stride,
                              int pad, const float* bias, void* out, void* stream);

/* Row softmax, fp16 in/out (may be in place), fp32 math: the VAE mid-block attention (single head, d = 512) is evaluated as
 * GEMM -> softmax -> GEMM (diffusers AutoencoderKL [dep], reference pipeline_pose2vid_long.py:118-121). */
int ap_softmax_rows_f16(const void* x, void* out, long long rows, int cols, long long ld, void* stream);

/*
 * Fused spatial self / reference attention (flash-style, tcgen05). q/k/v: [n_frames*tokens, ld_qkv] fp16 with head h
 * at columns [h*dpad, h*dpad + head_dim) (zero padded to dpad in {64,128,192}); frames >= first_bank_frame also attend
 * to bank (frame - first_bank_frame) / frames_per_bank of bank_k/bank_v: [n_banks*bank_tokens, ld_bank] (NULL = none).
 * out: [n_frames*tokens, ldo], head h at columns [h*head_dim, (h+1)*head_dim).
 * Replaces F.scaled_dot_product_attention under ReferenceAttentionControl's read-mode forward, including the CFG
 * redo for the unconditional half (reference src/models/mutual_self_attention.py:147-186; src/models/attention.py:323-330).
 */
int ap_attention_f16(const void* q, const void* k, const void* v, long long ld_qkv, const void* bank_k,
                     const void* bank_v, long long ld_bank, int bank_tokens, int n_banks, int n_frames, int tokens,
                     int heads, int head_dim, int dpad, int first_bank_frame, int frames_per_bank, float scale,
                     void* out, long long ldo, void* stream);

/*
 * Temporal attention core of the motion module: softmax over the F frames of each (batch, position, head).
 * qkv: [B*F*N, ld] = [q | k | v] (C columns each, token row (b*F+f)*N+p); out: [B*F*N, ldo].
 * Replaces VersatileAttention's rearrange + SDPA + rearrange (reference src/models/motion_module.py:351-388).
 */
int ap_temporal_attention_f16(const void* qkv, long long ld, void* out, long long ldo, int B, int F, int N, int C,
                              int heads, float scale, void* stream);

/* Elementwise / layout helpers (fp16, n % 8 == 0 where vectorised). */
int ap_add_f16(const void* a, const void* b, void* out, long long n, void* stream);          /* unet_3d.py:485-486,508-510 */
int ap_silu_f16(const void* x, void* out, long long n, void* stream);                        /* resnet.py:226-230 */
/* out[i] = a[i] + b[i % nb] (b broadcast over the leading CFG-branch dim) */
int ap_add_bcast_f16(const void* a, const void* b, void* out, long long n, long long nb, void* stream);
/* diffusers Timesteps(dim, flip_sin_to_cos=True, freq_shift=0): out[b] = [cos(t_b w_i) | sin(t_b w_i)], unet_3d.py:463 */
int ap_timestep_embedding_f16(const float* t, int B, int dim, void* out, void* stream);
int ap_upsample2x_nhwc_f16(const void* x, void* out, int Nf, int H, int W, int C, void* stream); /* resnet.py:71-78 */
int ap_ncfhw_to_nhwc_f16(const void* x, void* out, int B, int C, int F, int HW, int Cpad, void* stream);
int ap_nhwc_to_ncfhw_f16(const void* x, void* out, int B, int C, int F, int HW, int ld, void* stream);

/*
 * Denoising-loop elementwise ops (reference src/pipelines/pipeline_pose2vid_long.py:521-559 and diffusers
 * DDIMScheduler.step [dep], eta = 0). latents: fp16 [L, HW, 4] channels-last; acc: fp32 [B, L, HW, 4].
 * ap_cfg_ddim_step_f16: overlap average + classifier-free guidance + one DDIM update, in place on `latents`; `acc` is
 * zeroed. prediction_type: AP_PRED_* (configs/inference/inference_v2.yaml:30 uses v_prediction, inference_v1.yaml
 * epsilon); clip_range > 0 clamps the predicted x0 to [-clip_range, clip_range] (DDIMScheduler clip_sample), <= 0: off.
 */
#define AP_PRED_V 0
#define AP_PRED_EPSILON 1
#define AP_PRED_SAMPLE 2
int ap_gather_window_f16(const void* latents, const int* frame_idx, void* out, int dup, int F, int HW, int Cpad,
                         void* stream);
int ap_scatter_accumulate_f16(const void* pred, int ld, const int* frame_idx, float* acc, int B, int F, int L, int HW,
                              void* stream);
int ap_cfg_ddim_step_f16(float* acc, const float* inv_count, int cfg, float guidance, float alpha_t, float alpha_prev,
                         int prediction_type, float clip_range, void* latents, int L, int HW, void* stream);

/*
 * Decoded video -> packed 8-bit RGB frames on the device (reference src/utils/util.py:87-104 save_videos_grid does
 * `(x * 255).numpy().astype(np.uint8)`, after `(x + 1) / 2` if rescale, on the fp32 host copy that
 * pipeline_pose2vid_long.py:123-125 makes: 4 bytes per sample over PCIe instead of 1). video: fp16 [B, 3, F, H, W] addressed
 * through `strides` = element strides of (b, c, f, h, w) (host array of 5); out: [B, F, H, W, 3] bytes. Bit-identical to
 * the host arithmetic for values in range; out-of-range values saturate, NaN -> 0.
 */
int ap_pack_frames_u8(const void* video, const long long* strides, int B, int F, int H, int W, int rescale, void* out,
                      void* stream);

/*
 * Audio front-end of audio2vid (reference scripts/audio2vid.py:162,189-195 -> src/audio_models/model.py:58-69,
 * pose_model.py:97-105 -> wav2vec2.py:13-64): the wav2vec2-base encoder (transformers Wav2Vec2Model with
 * feat_extract_norm="group") on sm_100a. The transformer layers use ap_gemm_f16 / ap_attention_f16 / ap_layernorm_f16;
 * the three entry points below are the parts no existing kernel covers. Feature-extractor layers 1-6 (k = 3 / 2,
 * stride 2, 512 channels, no bias) are ap_gemm_f16 calls with AP_GEMM_GELU over strided views of the channels-last input
 * (row stride 1024 = two input frames; k = 2: A = x as [T_out, 1024]; k = 3: A = [x as [T_out, 1024] | x from frame 2 on
 * as [T_out, 512]]) with tap-major weights [512, k * 512]: no im2col buffer, and no TMA box reads past frame T_in - 1.
 */

/*
 * Feature-extractor layer 0: Conv1d(1, 512, k = 10, stride 5, no bias) on the raw waveform + GroupNorm(512, 512) (one
 * channel per group: statistics over time, biased variance) + exact-erf GELU (transformers Wav2Vec2GroupNormConvLayer).
 * wav: fp32 [S], S >= 10; w: fp32 [512, 10]; gamma/beta: fp32 [512]; out: fp16 [T0, 512] channels-last,
 * T0 = (S - 10) / 5 + 1. workspace: fp32, at least ap_wav_conv0_workspace_floats(S) floats (per-block partial sums and
 * the per-channel affine pair): the reduction is atomic-free in a fixed order, double-precision finalize (bit-reproducible).
 */
int ap_wav_conv0_workspace_floats(long long S); /* AP_ERR_INVALID if S needs more than 2^31 - 1 floats */
int ap_wav_conv0_gn_gelu_f16(const float* wav, long long S, const float* w, const float* gamma, const float* beta,
                             float eps, float* workspace, long long workspace_floats, void* out, void* stream);

/*
 * F.interpolate(mode="linear", align_corners=True) along time of a channels-last fp16 matrix (reference
 * src/audio_models/torch_utils.py:17-20, applied at wav2vec2.py:32): x [T_in, C] -> out [T_out, C], C % 8 == 0,
 * fp32 weights computed as torch does (scale = (T_in - 1) / (T_out - 1), 0 for T_out = 1).
 */
int ap_interp_linear_time_f16(const void* x, int T_in, int C, void* out, int T_out, void* stream);

/*
 * wav2vec2 positional convolution (transformers Wav2Vec2PositionalConvEmbedding + the residual add of Wav2Vec2Encoder):
 *   out[t] = x[t] + gelu_erf(b + sum_k W_k x[t + k - 64])   on [T, 768], 16 groups of 48 channels, k = 128, padding 64,
 * the last of the T + 1 conv outputs dropped (Wav2Vec2SamePadLayer). w: the weight-norm-resolved weight packed
 * [16 groups][128 taps][48 in][48 out] fp16; bias: fp32 [768]. Tensor cores (mma.sync through WMMA), fp32 accumulation,
 * taps summed in a fixed order. out must not alias x.
 */
int ap_pos_conv_gelu_f16(const void* x, int T, const void* w, const float* bias, void* out, void* stream);

/*
 * out[i] = (sum over s = 0 .. n_src-1 of x[s * n + i]) / n_src, summed in fp32 in order s = 0, 1, ... (the reference's
 * `sum(hidden_states) / len(hidden_states)`, src/audio_models/model.py:63-66; n_src = 1 is an fp16 -> fp32 copy).
 * x: fp16 [n_src, n]; out_f32 (fp32 [n]) and/or out_f16 (fp16 [n]) may be NULL.
 */
int ap_mean_f16(const void* x, int n_src, long long n, float* out_f32, void* out_f16, void* stream);

/*
 * Face-mesh pose maps (audio2vid / vid2vid conditioning; reference src/utils/pose_util.py, src/utils/draw_util.py).
 *
 * ap_pose_smooth: smooth_pose_seq(x, window) (pose_util.py:81-88) on x [L, 6], fp32 (f64 = 0) or fp64 (f64 = 1), out the
 * same dtype: out[i] = mean of rows max(0, i - window/2) .. min(L, i + window/2 + 1) - 1, summed row after row in the
 * input dtype and divided by the count, without FMA contraction: bit-identical to numpy. out must not alias x.
 */
int ap_pose_smooth(const void* x, int L, int window, int f64, void* out, void* stream);

/*
 * ap_project_points: project_points / project_points_with_trans (pose_util.py:30-59) in fp64. points [L, N, 3] (fp32 or
 * fp64 per points_f64); `pose` [L, 6] (xyz Euler degrees, extrinsic, then a translation) with one 4 x 4 `trans`, or
 * pose = NULL with per-frame `trans` [L, 4, 4]; out fp64 [L, N, 2] pixel coordinates of a W x H image, through
 * create_perspective_matrix(W / H) (63 degree vertical FOV, near 1, far 10000, y flipped, fp32 entries).
 */
int ap_project_points(const void* points, int points_f64, int L, int N, const void* trans, int trans_f64, const void* pose,
                      int pose_f64, int W, int H, double* out, void* stream);

/*
 * ap_facemesh_raster: FaceMeshVisualizer.draw_landmarks (draw_util.py:124-148) for L frames. keypoints [L, N, 2] (fp32 or
 * fp64 per kp_f64): pixel coordinates of a W x H image (normed = 0) or normalised ones (normed = 1). Each landmark is
 * normalised, rounded to fp32, valid iff both coordinates lie in [0, 1], and placed at pixel min(floor(v * 512), 511) of
 * a 512 x 512 canvas. Every edge e of `edges` (int32 [E, 3]: landmark a, landmark b, colour group g; a, b < N) whose two
 * landmarks are valid is drawn as cv2.line(thickness=2, LINE_8); a pixel takes the colour of the highest group that
 * covers it, colours[g] (uint8 [G, 3], written as given: BGR in the reference). The canvas is then resized to W x H as
 * cv2.resize(INTER_LINEAR) does (W, H multiples of 8). canvas: uint8 workspace [L, 512, 512], 16-byte aligned; out: uint8
 * [L, H, W, 3]. Deterministic: two calls give the same bytes.
 */
int ap_facemesh_raster(const void* keypoints, int kp_f64, int L, int N, int normed, int W, int H, const int* edges, int E,
                       const unsigned char* colours, int G, void* canvas, void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ANIPORTRAIT_B200_H_ */

/* zeggs_b200 -- C ABI of the B200-native ZeroEGGS audio->gesture hot path (libzeggs_b200.so).
 *
 * The reference (ubisoft/ubisoft-laforge-ZeroEGGS) is pure Python/PyTorch and has no FFI today; its
 * "plugin API" for this path is the Python call surface of ZEGGS/modules.py, ZEGGS/audio/spectrograms.py,
 * ZEGGS/data_pipeline.py:33 and the train step body of ZEGGS/train.py.  Each entry point below names the
 * reference function it replaces (file:line relative to /root/reference).  INTEGRATION.md shows the
 * ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - every function returns int: 0 = ok, <0 = error (ZEGGS_ERR_*); text via zeggs_last_error().
 *   - the CALLER owns every buffer; the library allocates nothing persistent.  Workspace sizes come
 *     from the *_workspace_bytes() functions.  All pointers are DEVICE pointers unless named h_*.
 *   - every call is asynchronous on the given cudaStream_t (passed as void*), re-entrant per stream.
 *   - tensors are dense row-major float32 unless stated; quaternions are w-first (anim/tquat.py:8-15);
 *     pose vector order is [root_vel 3 | root_vrt 3 | lpos 225 | ltxy 450 | lvel 225 | lvrt 225 | gaze 3]
 *     (modules.py:699-710) and the output order of modules.py:731-736.
 */
#ifndef ZEGGS_B200_H
#define ZEGGS_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZEGGS_OK 0
#define ZEGGS_ERR_ARG (-1)
#define ZEGGS_ERR_CUDA (-2)
#define ZEGGS_ERR_UNSUPPORTED (-3)
#define ZEGGS_ERR_TIMEOUT (-4)

#define ZEGGS_NJ 75
#define ZEGGS_P_OUT 1131 /* modules.py:731-736 */
#define ZEGGS_P_IN 1134  /* modules.py:699-710 */

const char* zeggs_last_error(void);
int zeggs_version(void);
/* sizeof of an args struct of this header by its C name, e.g. "zeggs_decoder_bwd_args" (0 = unknown name): bindings check their mirror. */
size_t zeggs_struct_size(const char* name);
/* number of kernels this library has launched since load (bench.py's gpu_launches claim) */
long long zeggs_launch_count(void);
/* Live device timing of the main kernel groups ("decoder_fwd", "decoder_bwd", "decoder_wgrad", "mel", "loss",
 * "encoders_fwd", "encoders_bwd"): CUDA events recorded on the launching stream around each group; read after a sync. */
void zeggs_timing_enable(int on);
void zeggs_timing_reset(void);
int zeggs_timing_read(const char* name, double* total_ms, int* count);

/* ------------------------------------------------------------------------------------------------
 * Per-call context of the batched-GEMM front end (caller-owned, plain data; no library globals are needed when it is passed):
 * every args struct below ends in `const zeggs_ctx* ctx`.  NULL selects the process-wide defaults of the legacy setters
 * (zeggs_set_scratch / zeggs_set_gemm_mode / zeggs_set_fast_wgrad), kept for callers of the plain-argument entry points.
 * Two host threads driving two streams with two contexts never share mutable library state.
 */
typedef struct {
  void* scratch;          /* device scratch for the bf16 operand copies of the tcgen05 GEMMs (and split-K partials) */
  size_t scratch_bytes;
  int gemm_mode;          /* 0: fp32 SIMT everywhere, 1: tcgen05 split-bf16 (x3, ~fp32 accuracy), 2: tcgen05 plain bf16 */
  int fast_wgrad;         /* 1: weight-gradient products run as ONE bf16 pass (set together with the tensor-core recurrence) */
} zeggs_ctx;

/* ------------------------------------------------------------------------------------------------
 * Mel front end.  Replaces audio/spectrograms.py:8-54 (extract_mel_spectrogram_for_tts, pre-emphasis
 * off), :216-269 (extract_spectrogram), :161-183 + :386-503 (Slaney filterbank), :57-131 (clip/dB/[0,1])
 * and, for `feat`, data_pipeline.py:62-82 (ln(10^(s/20)), 80->60 fps linear resample, energy channel).
 *   wav      [n_clips, n_samples] f32
 *   mel_out  [n_clips, n_mels, L] f32 or NULL   (the reference's (n_mels, L) layout, values in [0,1])
 *   feat_out [n_clips, anim_length, n_mels+1] f32 or NULL
 * L = zeggs_mel_num_frames(n_samples, n_fft, hop) (spectrograms.py:242-245, centered).
 * fb_* describe the sparse filterbank built on the host by zeggs_b200.audio (same closed form as the
 * reference): band i covers FFT bins [fb_start[i], fb_start[i]+fb_len[i]) with weights fb_w[fb_off[i]..].
 */
typedef struct {
  int n_clips, n_samples, n_fft, hop, n_mels;
  int anim_length;        /* rows of feat_out per clip (60 fps frames) */
  float min_amp;          /* min_clipping / n_fft, spectrograms.py:86-88 */
  double frames_per_anim; /* (fs/hop)/anim_fs, data_pipeline.py:68 (kept in double: floor() must match the f64 reference) */
  const float* wav;
  const float* window;   /* [n_fft] symmetric Hann, spectrograms.py:230 */
  const float* twiddle;  /* (cos,-sin) pairs: [n_fft/2] of exp(-2*pi*i*k/(n_fft/2)) then [n_fft/2+1] of exp(-2*pi*i*k/n_fft) */
  const int* fb_start;
  const int* fb_len;
  const int* fb_off;
  const float* fb_w;
  float* mel_out;
  float* feat_out;
  int fb_total;          /* number of weights in fb_w (<= 4096: staged in shared memory; 0: read from global memory) */
  const float* gain;     /* optional [n_clips] per-clip gain applied to every sample at load (loudness normalisation, data_pipeline.py:34-39) */
  const short* wav_i16;  /* optional int16 PCM input instead of `wav` (x / 32768, audio_files.py:211-236) */
} zeggs_mel_args;
int zeggs_mel_num_frames(int n_samples, int n_fft, int hop);
int zeggs_mel_forward(const zeggs_mel_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Loudness normalisation ahead of the mel front end: replaces data_pipeline.py:34-39
 * (pyloudnorm 0.1.0 Meter(rate).integrated_loudness + normalize.loudness(x, L, -20)).  Per clip:
 * K-weighting (two biquads, coef = {b0,b1,b2,a1,a2} of the high shelf then of the high pass, a0-normalised, built on the
 * host by zeggs_b200.audio in float64), gating-block energies, absolute/relative gates, integrated LUFS and
 * gain_out[clip] = 10^((target - LUFS)/20).  The host also builds the block geometry with the package's own float64
 * expressions: seg_bounds[n_seg+1] = sorted boundaries of all blocks, block j = segments [blk_seg_lo[j], blk_seg_hi[j]).
 * The gain is consumed by zeggs_mel_forward (args.gain); the waveform is not rewritten.
 */
typedef struct {
  int n_clips, n_samples, n_seg, n_blocks, warm;
  double coef[10];
  double inv_block_len;   /* 1 / (0.4 * rate) */
  double target_lufs;
  const float* wav;       /* [n_clips, n_samples] f32, or NULL with wav_i16 set */
  const short* wav_i16;
  const int* seg_bounds;  /* [n_seg + 1] */
  const int* blk_seg_lo;  /* [n_blocks] */
  const int* blk_seg_hi;  /* [n_blocks] */
  float* gain_out;        /* [n_clips] */
  float* lufs_out;        /* [n_clips] or NULL */
  void* workspace;
  size_t workspace_bytes;
} zeggs_loudness_args;
size_t zeggs_loudness_workspace_bytes(int n_clips, int n_seg);
int zeggs_loudness_gain(const zeggs_loudness_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Decoder (modules.py:11-243, 677-742): CellStateEncoder + T-1 autoregressive steps of
 * vectorize_input -> Linear+ELU -> 2-layer GRU -> Linear -> devectorize_output, one persistent kernel.
 */
typedef struct {
  int B, T, H, S, Z; /* batch, frames, hidden (modules.py:18), speech / style encoding sizes */
  float dt;
  /* reference state-dict tensors (SURVEY.md 8b), fp32 row-major */
  const float *W0, *b0;                 /* recurrent_decoder.layer0  [H, 1134+S+Z] */
  const float *W_ih0, *b_ih0;           /* layer1.weight_ih_l0 [3H, H+1134+S+Z] */
  const float *W_hh0, *b_hh0;           /* layer1.weight_hh_l0 [3H, H] */
  const float *W_ih1, *b_ih1, *W_hh1, *b_hh1;
  const float *W2, *b2;                 /* layer2 [1131, H] */
  const float *Wc0, *bc0, *Wc1, *bc1, *Wc2, *bc2; /* cell_state_encoder.layer{0,1,2} */
  const float* packed;                  /* zeggs_decoder_pack_weights output */
  const float *in_mean, *in_std, *out_mean, *out_std; /* [1134],[1134],[1131],[1131] */
  /* inputs */
  const float* root_pos0; /* [B,3] */
  const float* root_rot0; /* [B,4] */
  const float* pose0;     /* [B,1131] first frame: vel|vrt|lpos|ltxy|lvel|lvrt (un-normalised) */
  const float* gaze_pos;  /* [B,T,3] */
  const float* speech;    /* [B,T,S] */
  const float* style;     /* [B,T,Z] */
  /* outputs (frame 0 = the given pose, modules.py:72-79) */
  float* Y;        /* [B,T,1131] de-normalised pose vector per frame */
  float* root_pos; /* [B,T,3] */
  float* root_rot; /* [B,T,4] */
  void* workspace;
  size_t workspace_bytes;
  int save_for_backward; /* 1: keep every step's activations in the workspace for zeggs_decoder_window_bwd */
  int engine;            /* 0: fp32 SIMT recurrence (parity grade); 1: tcgen05 recurrence, bf16 operands / fp32 state (B <= 32) */
  const void* packed_tc; /* engine 1: zeggs_decoder_pack_weights_tc output */
  void* workspace_tc;    /* engine 1: zeggs_decoder_tc_workspace_bytes bytes (bf16 activation images) */
  const zeggs_ctx* ctx;  /* GEMM context of this call (NULL: process defaults) */
} zeggs_decoder_fwd_args;

size_t zeggs_decoder_packed_bytes(int H, int S, int Z);
/* one-off re-layout of the decoder weights into per-CTA k-major slices (re-run after each optimizer step) */
int zeggs_decoder_pack_weights(const zeggs_decoder_fwd_args* a, float* packed, void* stream);
size_t zeggs_decoder_workspace_bytes(int B, int T, int H, int S, int Z, int save_for_backward);
/* tensor-core engine: bf16 shared-memory images of the per-CTA weight slices + activation image buffers */
size_t zeggs_decoder_packed_tc_bytes(int H, int S, int Z);
size_t zeggs_decoder_tc_workspace_bytes(int H, int S, int Z);
int zeggs_decoder_pack_weights_tc(const zeggs_decoder_fwd_args* a, void* packed, void* stream);
/* development aid: device buffer [64][32] of int64 receiving CTA 0's per-step phase timestamps (NULL = off) */
void zeggs_debug_set_tc_trace(void* device_buffer);
void zeggs_debug_set_tc_nacc(int n); /* development aid: forward recurrence kernel variant (0 = shipped) */
int zeggs_debug_set_tc_gemm_variant(int v);  /* tcgen05 GEMM tile variant: -1 automatic (128x256 tiles for one-pass products with N >= 256, fused three-pass), 0 = 128x128 tiles with streamed passes */
void zeggs_debug_set_loss_impl(int v); /* development aid: 1 = warp-per-frame loss kernels (default), 0 = round-1 thread-per-frame version */
void zeggs_debug_set_tc_cluster(int n); /* development aid: cap the thread-block cluster size of the tc recurrences (1 = no clusters) */
int zeggs_debug_get_tc_cluster(void);   /* cluster size the last tc forward launch used */
int zeggs_decoder_window_fwd(const zeggs_decoder_fwd_args* a, void* stream);

/* Resumable window (streaming inference): zeggs_decoder_window_fwd with the GRU state of frame 0 taken from the caller and the
 * state of frame T-1 handed back.  Frame 0 is still the given pose (pose0, root_pos0, root_rot0); only the state that frame 1
 * starts from changes.  A continuation is a literal sub-window of the one-shot window: pass the pose, root and state of the last
 * emitted frame and the speech / style / gaze rows from that frame onward.  s == NULL is zeggs_decoder_window_fwd.
 * Inference only: save_for_backward must be 0.  With T == 1, h_final is the initial state. */
typedef struct {
  const float* h_init;          /* [2,B,H] GRU state (layer, sample, unit) = nn.GRU's h layout, as zeggs_decoder_step_args.h_in; NULL = CellStateEncoder */
  const int* init_from_state;   /* [B] int32 device: 1 = sample b starts from h_init[:,b], 0 = from the CellStateEncoder; NULL with h_init set = all 1 */
  float* h_final;               /* [2,B,H] state at frame T-1, or NULL */
} zeggs_decoder_state_args;
int zeggs_decoder_window_fwd_state(const zeggs_decoder_fwd_args* a, const zeggs_decoder_state_args* s, void* stream);

/* Backward of zeggs_decoder_window_fwd (the autograd of modules.py:47-162: full BPTT through the GRU stack,
 * the pose feedback, the gaze transform and the root integration).  Needs the forward's workspace
 * (save_for_backward = 1) and outputs (Y, root_pos, root_rot) untouched.  Gradient buffers have the shapes
 * of the corresponding weights and are overwritten. */
typedef struct {
  const float* dY;       /* [B,T,1131] upstream gradient of the pose vectors (NULL = 0) */
  const float* dRootPos; /* [B,T,3] (NULL = 0) */
  const float* dRootRot; /* [B,T,4] (NULL = 0) */
  const float* packed_bwd; /* zeggs_decoder_pack_weights_bwd output */
  float *dW0, *db0, *dW_ih0, *db_ih0, *dW_hh0, *db_hh0, *dW_ih1, *db_ih1, *dW_hh1, *db_hh1, *dW2, *db2;
  float *dWc0, *dbc0, *dWc1, *dbc1, *dWc2, *dbc2;
  float* dSpeech; /* [B,T,S] or NULL */
  float* dStyle;  /* [B,T,Z] or NULL */
  void* workspace;
  size_t workspace_bytes;
  const void* packed_bwd_tc; /* tensor-core engine (fwd args' engine == 1): zeggs_decoder_pack_weights_bwd_tc output, or NULL */
  void* workspace_tc;        /* zeggs_decoder_bwd_tc_workspace_bytes bytes (bf16 gradient images) */
  int phase;                 /* 0: everything.  Tensor-core engine only: 1 = BPTT recurrence + CellStateEncoder gradients + dSpeech / dStyle
                                (what the encoders' backward passes wait for), 2 = all remaining parameter gradients (same args, same
                                stream or one ordered after phase 1; the ctx scratch must not be used by other calls in between).
                                Other engines do all the work in phase 1 and return at once from phase 2. */
} zeggs_decoder_bwd_args;
size_t zeggs_decoder_packed_bwd_bytes(int H, int S, int Z);
int zeggs_decoder_pack_weights_bwd(const zeggs_decoder_fwd_args* a, float* packed, void* stream);
size_t zeggs_decoder_bwd_workspace_bytes(int B, int T, int H, int S, int Z);
int zeggs_decoder_window_bwd(const zeggs_decoder_fwd_args* f, const zeggs_decoder_bwd_args* b, void* stream);
size_t zeggs_decoder_packed_bwd_tc_bytes(int H, int S, int Z);
size_t zeggs_decoder_bwd_tc_workspace_bytes(int H, int S, int Z);
int zeggs_decoder_pack_weights_bwd_tc(const zeggs_decoder_fwd_args* a, void* packed, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SpeechEncoder (modules.py:249-272): conv k1 + ELU + drop -> conv k31 (replicate 'same') + ELU + drop -> Linear + ELU.
 * x is the already normalised feature tensor (train.py:232-234).  mask0/mask1 are dropout multipliers
 * (0 or 1/(1-p), p = 0.2) in [B,T,C] layout, NULL in eval mode.  The workspace keeps the activations for _bwd.
 */
typedef struct {
  int B, T, C_in, H, O;
  const float *W0, *b0; /* layer0.weight [H, C_in, 1] */
  const float *W1, *b1; /* layer1.weight [O, H, 31]  */
  const float *W2, *b2; /* layer2.weight [O, O]      */
  const float* x;       /* [B,T,C_in] */
  const float* mask0;   /* [B,T,H] or NULL */
  const float* mask1;   /* [B,T,O] or NULL */
  float* y;             /* [B,T,O] */
  void* workspace;
  size_t workspace_bytes;
  const zeggs_ctx* ctx;
} zeggs_speech_enc_args;
typedef struct {
  const float* dy; /* [B,T,O] */
  float *dW0, *db0, *dW1, *db1, *dW2, *db2;
} zeggs_speech_enc_grads;
size_t zeggs_speech_enc_workspace_bytes(int B, int T, int C_in, int H, int O);
int zeggs_speech_enc_fwd(const zeggs_speech_enc_args* a, void* stream);
int zeggs_speech_enc_bwd(const zeggs_speech_enc_args* a, const zeggs_speech_enc_grads* g, void* stream);

/* StyleEncoder, type "attn", use_vae (modules.py:278-304, 346-420, 484-651): two conv k3 + ReLU + LayerNorm + drop,
 * + sinusoidal positions, one FFT block (4-head self-attention + residual LN, 2x conv k3 feed-forward + residual LN),
 * mean over time, mu/logvar split, z = mu + eps * exp(logvar/2) / temperature.
 * x is the normalised style example [B,T,C_in]; eps [B,E/2] is the N(0,1) sample (NULL = 0); pe [T,E] the
 * positional table; masks are dropout multipliers (NULL = eval): c1 [B,T,H], c2/ao/ff [B,T,E], attn [B,nheads,T,T].
 */
typedef struct {
  int B, T, C_in, H, E, nheads;
  float temperature;
  const float *Wc1, *bc1, *ln1_g, *ln1_b; /* encoder.convs.0.conv, encoder.convs.2 */
  const float *Wc2, *bc2, *ln2_g, *ln2_b; /* encoder.convs.4.conv, encoder.convs.6 */
  const float *Win, *bin, *Wout, *bout, *ln3_g, *ln3_b; /* blocks.0.attention.* */
  const float *Wf1, *bf1, *Wf2, *bf2, *ln4_g, *ln4_b;   /* blocks.0.feed_forward.* */
  const float *x, *eps, *pe;
  const float *mask_c1, *mask_c2, *mask_attn, *mask_ao, *mask_ff;
  float *z, *mu, *logvar; /* [B, E/2] each */
  void* workspace;
  size_t workspace_bytes;
  const zeggs_ctx* ctx;
} zeggs_style_enc_args;
typedef struct {
  const float *dz, *dmu, *dlogvar; /* [B,E/2], any may be NULL */
  float *dWc1, *dbc1, *dln1_g, *dln1_b, *dWc2, *dbc2, *dln2_g, *dln2_b;
  float *dWin, *dbin, *dWout, *dbout, *dln3_g, *dln3_b;
  float *dWf1, *dbf1, *dWf2, *dbf2, *dln4_g, *dln4_b;
} zeggs_style_enc_grads;
size_t zeggs_style_enc_workspace_bytes(int B, int T, int C_in, int H, int E, int nheads);
int zeggs_style_enc_fwd(const zeggs_style_enc_args* a, void* stream);
int zeggs_style_enc_bwd(const zeggs_style_enc_args* a, const zeggs_style_enc_grads* g, void* stream);

/* ------------------------------------------------------------------------------------------------
 * One teacher-forced decoder step (RecurrentDecoderNormal.forward, modules.py:179-185), fp32 throughout:
 *   pose [B,1134] (the normalised input vector of modules.py:699-713), speech [B,S], style [B,Z], h_in [2,B,H]
 *   -> y [B,1131] (normalised output of layer2), h_out [2,B,H].
 * The tight parity point (<= 1e-4 vs the reference per step); windows go through zeggs_decoder_window_fwd, streamed windows
 * through zeggs_decoder_window_fwd_state.
 */
typedef struct {
  int B, H, S, Z;
  const float *W0, *b0, *W_ih0, *b_ih0, *W_hh0, *b_hh0, *W_ih1, *b_ih1, *W_hh1, *b_hh1, *W2, *b2;
  const float *pose, *speech, *style, *h_in;
  float *y, *h_out;
  void* workspace;
  size_t workspace_bytes;
} zeggs_decoder_step_args;
size_t zeggs_decoder_step_workspace_bytes(int B, int H, int S, int Z);
int zeggs_decoder_step_fwd(const zeggs_decoder_step_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Training loss, forward and backward in one call (train.py:277-421): world-space transforms, 75-joint FK with
 * velocities for the output and the ground truth, 17 weighted L1 means + kl_weight * KL(mu, logvar), divided by 18.
 * (Y, root_pos, root_rot) are the decoder outputs; (WY, W_root_pos, W_root_rot) the ground-truth window in the
 * same packed layout.  losses[0] = total, losses[1..17] = loss_root_pos .. loss_gaze in train.py:397-416 order,
 * losses[18] = weighted KL term.  If dY != NULL the gradient of `total` w.r.t. Y / root_pos / root_rot (and mu /
 * logvar) is written too.  torch.cross is taken over the LAST dim (the reference's dim-less calls at
 * train.py:301,315 / txform.py:25-26 only differ when B or T == 3).
 */
typedef struct {
  int B, T, Z;
  float dt, kl_weight;
  const float *Y, *root_pos, *root_rot;
  const float *WY, *W_root_pos, *W_root_rot;
  const float* gaze_pos; /* [B,T,3] */
  const int* parents;    /* int32 [75] */
  const float *mu, *logvar; /* [B,Z] or NULL */
  float* losses;         /* [19] */
  float *dY, *dRootPos, *dRootRot, *dmu, *dlogvar;
  void* workspace;
  size_t workspace_bytes;
  const float* kl_weight_dev; /* optional DEVICE scalar overriding kl_weight (updated by the host between CUDA-graph replays) */
} zeggs_loss_args;
size_t zeggs_loss_workspace_bytes(int B, int T);
int zeggs_loss_fwd_bwd(const zeggs_loss_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Pose tensors -> the values the BVH writer prints (generate.py:389-406 + utils.py:47-87): per joint the rotation from the
 * rotated x/y axes (txform.py:23-34 -> quat.py:166-206), the root re-based on its first frame and start_pos / start_rot
 * (rebase != 0) and folded into joint 0, Euler angles in degrees in 'zyx' channel order (quat.py:111-119).
 *   root_pos [N,T,3], root_rot [N,T,4] (w first), lpos [N,T,J,3], ltxy [N,T,J,2,3]
 *   positions [N,T,J,3], euler_deg [N,T,J,3] (z, y, x angle per joint), lrot [N,T,J,4] or NULL
 */
typedef struct {
  int N, T, J, rebase;
  float start_pos[3], start_rot[4];
  const float *root_pos, *root_rot, *lpos, *ltxy;
  float *positions, *euler_deg, *lrot;
} zeggs_pose_post_args;
int zeggs_pose_to_bvh_channels(const zeggs_pose_post_args* a, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Device-resident window supplier: one launch gathers a training batch out of the processed arrays kept in HBM
 * (dataset.py:110-153 windows, :176-204 style-example windows, train.py:215-225 copies).
 *   src[k] [n_frames, width[k]] f32 (X_audio_features, Y_root_pos, ...), dst[k] [B, T, width[k]]:  dst[k][b][t] = src[k][start[b] + t]
 *   ex_out [B, L, ex_width]: the arrays ex_src[0..n_ex) side by side (root_vel, root_vrt, lpos, ltxy, lvel, lvrt), remaining columns
 *   zero; rows l >= ex_n[b] repeat the example's last L - ex_n[b] rows (dataset.py:201-203).  start / ex_start / ex_n: int32 [B] on
 *   the device (drawn on the host by the same generator as the reference's sampler).
 */
#define ZEGGS_GATHER_MAX 12
typedef struct {
  int B, T, n_arrays;
  const float* src[ZEGGS_GATHER_MAX];
  float* dst[ZEGGS_GATHER_MAX];
  int width[ZEGGS_GATHER_MAX];
  const int* start;
  float* ex_out;            /* NULL: no style example (label style) */
  int L, ex_width, n_ex;
  int ex_src[ZEGGS_GATHER_MAX];
  const int* ex_start;
  const int* ex_n;
} zeggs_gather_args;
int zeggs_window_gather(const zeggs_gather_args* a, void* stream);
/* Input normalisation of train.py:232-234 / 247-249 in one pass: out[r][c] = (x[r][c] - mean[c]) / std[c]  (x, out: [rows][C] fp32). */
int zeggs_normalize_rows(const float* x, const float* mean, const float* stdv, float* out, long long rows, int C, void* stream);

/* Fused RAdam step over a flat fp32 parameter buffer (optimizers.py:31-99; weight_decay 0,
 * degenerated_to_sgd).  `step` is the 1-based step count; gradients are multiplied by grad_scale first. */
int zeggs_radam_step(float* p, const float* g, float* m, float* v, size_t n, float lr, float beta1, float beta2,
                     float eps, int step, float grad_scale, void* stream);
/* The same step with every step-dependent scalar in DEVICE memory, so that a captured CUDA graph can be replayed:
 * hyper[0..4] = lr, beta1, beta2, eps, grad_scale (inputs; the host rewrites them between replays when they change),
 * hyper[5..7] = scratch written by the call; *step_count is the number of steps taken so far and is incremented by the call
 * (the rectification terms of optimizers.py:66-78 are evaluated on the device in double from *step_count + 1). */
int zeggs_radam_step_dev(float* p, const float* g, float* m, float* v, size_t n, float* hyper, int* step_count, void* stream);
/* Dropout mask (u >= p) / (1 - p) with a counter-based generator: one pass instead of torch's rand / compare / cast / scale
 * (the Bernoulli draw of nn.Dropout, modules.py:263-270, :383-388, :551, :606).  Reproducible for a given seed. */
int zeggs_dropout_mask(float* out, size_t n, float p, unsigned long long seed, void* stream);
/* Same, seeded from DEVICE memory: effective seed = hash(*seed_dev, salt) (CUDA-graph replays draw fresh masks when the
 * caller advances *seed_dev between replays; `salt` separates the masks of one step). */
int zeggs_dropout_mask_dev(float* out, size_t n, float p, const unsigned long long* seed_dev, unsigned long long salt, void* stream);
/* N(0,1) samples from the same device-seeded generator (the VAE noise of modules.py:299 inside a replayable graph). */
int zeggs_randn_dev(float* out, size_t n, const unsigned long long* seed_dev, unsigned long long salt, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Generic fp32 GEMM used for the batched (non-recurrent) linear layers:
 *   C[M,N] = act(A[M,K] * B[N,K]^T + bias[N])            (trans_a = 0;  nn.Linear)
 *   C[M,N] = A[K,M]^T * B[K,N] (+ C if accumulate)        (trans_a = 1;  weight gradients)
 *   C[M,N] = A[M,K] * B[K,N]                              (trans_a = 2;  input gradients)
 * act: 0 none, 1 ELU, 2 ReLU.
 */
int zeggs_sgemm(int trans_a, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                const float* bias, float* C, int ldc, int act, int accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * tcgen05 / TMEM / TMA GEMM (bf16 operands, f32 accumulate in tensor memory):
 *   C[M,N] = act(A[M,K] * B[N,K]^T + bias) (+ C)   A, B row-major bf16 (K contiguous), lda/ldb in elements (%8==0)
 * With A_lo/B_lo non-NULL the product is evaluated as A_hi*B_hi + A_lo*B_hi + A_hi*B_lo (split-bf16, ~fp32
 * product accuracy); zeggs_split_bf16 produces hi = bf16(x), lo = bf16(x - hi) with rows zero-padded to ld_out.
 */
int zeggs_tc_gemm_bf16(int M, int N, int K, const void* A_hi, const void* A_lo, int lda, const void* B_hi,
                       const void* B_lo, int ldb, const float* bias, float* C, int ldc, int act, int accumulate,
                       void* stream);
/* fp32 GEMM front end used by the encoders: mode 0 NT / 1 TN / 2 NN as zeggs_sgemm.  Large products run on tcgen05
 * with operands split to bf16 (hi, lo) in the caller-provided scratch buffer (zeggs_set_scratch); small ones on the
 * fp32 SIMT kernel.  zeggs_set_gemm_mode: 0 = fp32 SIMT only, 1 = tcgen05 split-bf16 x3 (default), 2 = tcgen05 bf16. */
int zeggs_set_scratch(void* device_ptr, size_t bytes);
int zeggs_set_gemm_mode(int mode);
/* 1: weight-gradient products of the encoders (contraction over samples/frames) use ONE bf16 pass instead of the split-bf16
 * three -- the accuracy class of the tensor-core recurrence engine's own weight gradients; set by zeggs_b200.ops.set_decoder_engine. */
int zeggs_set_fast_wgrad(int on);
int zeggs_gemm_f32(int mode, int M, int N, int K, const float* A, int lda, const float* B, int ldb, const float* bias,
                   float* C, int ldc, int act, int accumulate, void* stream);
/* same with an explicit context instead of the process defaults */
int zeggs_gemm_f32_ctx(const zeggs_ctx* ctx, int mode, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                       const float* bias, float* C, int ldc, int act, int accumulate, void* stream);
int zeggs_split_bf16(const float* x, int rows, int cols, int ld_in, void* hi, void* lo, int ld_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ZEGGS_B200_H */

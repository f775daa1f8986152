/*
 * libltb200 — C ABI of the B200-native lip-sync engine (sm_100a only, no CPU fallback).
 *
 * This is the drop-in boundary behind LiveTalking's avatar plugin surface.  Every entry point names the
 * reference interface it replaces (paths relative to the lipku/LiveTalking tree).  Conventions:
 *   - plain C types, host pointers unless a name ends in _dev; the library owns all device memory;
 *   - every function returns 0 on success, non-zero on failure; ltb_last_error() returns the message
 *     (thread-local).  Nothing aborts the process; the Python shim raises RuntimeError.
 *   - handles are opaque pointers; a session is bound to one CUDA device (every entry point restores it in the calling
 *     thread).  Threading: the reference drives ONE session from three threads (avatars/base_avatar.py:469-501: render ->
 *     asr.run_step, inference -> inference_batch, process_frames -> paste_back_frame) and several sessions concurrently
 *     (ctypes releases the GIL).  Every ltb_w2l_* entry point that takes a session is therefore serialised by a
 *     per-session mutex held from its first enqueue to its synchronise; ltb_w2l_mel_step uses its own stream, device
 *     buffers and mutex and runs concurrently with the others.  An ltb_ctx (MuseTalk op layer) is NOT internally
 *     serialised across multi-call sequences: one ctx per session and thread role, as livetalking_b200.musetalk does
 *     (its allocation list is guarded).  Models and avatars are immutable after creation and shared freely.
 */
#ifndef LTB200_H_
#define LTB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ltb_w2l_model ltb_w2l_model;
typedef struct ltb_w2l_avatar ltb_w2l_avatar;
typedef struct ltb_w2l_session ltb_w2l_session;

/* ---- library ---------------------------------------------------------------------------------------- */
int ltb_version(void);
const char* ltb_last_error(void);
/* replaces utils/device.py:4-9 (reference always picks "cuda" = device 0) */
int ltb_device_count(int* count);
int ltb_set_device(int device);

/* ---- wav2lip256 model ------------------------------------------------------------------------------- */
/* replaces load_model(path), avatars/wav2lip_avatar.py:59-70.  `blob` is the packed weight image produced by
 * livetalking_b200.w2l_pack.pack_state_dict() from the reference checkpoint's state_dict (BN folded, fp16,
 * K-major rows).  The blob is copied to the current device. */
int ltb_w2l_model_create(const void* blob, size_t nbytes, ltb_w2l_model** out);
/* same, but adopts a blob that already lives in device memory (e.g. received by ncclBroadcast at init — the one
 * collective of the multi-GPU design).  No copy is made: the caller keeps ownership and must keep it alive. */
int ltb_w2l_model_create_from_device(void* blob_dev, size_t nbytes, ltb_w2l_model** out);
int ltb_w2l_model_destroy(ltb_w2l_model* m);

/* ---- avatar assets ---------------------------------------------------------------------------------- */
/* replaces load_avatar(avatar_id), avatars/wav2lip_avatar.py:72-88: face crops (n,256,256,3) u8 BGR, full frames
 * (n,H,W,3) u8 BGR and coords (n,4) int32 = (y1,y2,x1,x2) are uploaded once and stay resident in HBM.
 * frames == NULL creates a FRAME-FREE avatar: only faces and coords go to the device (H, W still validate the coords), the
 * caller keeps the frames, and only the *_region entry points composite for it.  The full-frame forms (ltb_w2l_paste,
 * ltb_w2l_paste_pred, ltb_w2l_paste_batch, ltb_w2l_infer_paste, ltb_w2l_infer_slots, ltb_w2l_step_async,
 * ltb_w2l_step_e2e_async) fail with a message for it and leave the session usable. */
int ltb_w2l_avatar_create(const uint8_t* faces, const uint8_t* frames, const int32_t* coords, int n, int H, int W,
                          ltb_w2l_avatar** out);
int ltb_w2l_avatar_destroy(ltb_w2l_avatar* a);
/* the avatar's largest paste rectangle (max y2-y1, max x2-x1 over its frames): the per-slot pitch of region outputs */
int ltb_w2l_avatar_region_max(const ltb_w2l_avatar* a, int* rh_max, int* rw_max);
/* cudaMemGetInfo of the current device (the plugins decide an avatar's residency from it) */
int ltb_mem_get_info(size_t* free_bytes, size_t* total_bytes);

/* ---- session (one avatar stream) -------------------------------------------------------------------- */
#define LTB_SESSION_KEEP_LAYERS 1 /* keep every layer's activations (debug / per-layer parity tests) */
#define LTB_SESSION_NO_GRAPH 2    /* launch kernels eagerly instead of replaying a CUDA graph */
#define LTB_SESSION_NO_HALO 4     /* route every conv to the generic gather kernel (A/B testing of the TMA halo kernel) */
#define LTB_SESSION_NO_PDL 8      /* launch the conv kernels without programmatic dependent launch (A/B testing) */
#define LTB_SESSION_SLOTS 16      /* cross-session batch: per-slot avatar / index / mel (ltb_w2l_infer_slots) */
#define LTB_SESSION_MEL_ONLY 32   /* feature extractor only (ltb_w2l_mel_step): no activation arena / plan / graphs */
/* replaces LipReal.__init__ (avatars/wav2lip_avatar.py:101-114) + warm_up (:90-96): allocates the activation
 * arena for `batch` frames, builds the layer plan and (unless NO_GRAPH) captures it into a CUDA graph.
 * stride_left/right = opt.l / opt.r (20 ms chunks), fps = opt.fps. */
int ltb_w2l_session_create(ltb_w2l_model* m, ltb_w2l_avatar* a, int batch, int stride_left, int stride_right, int fps,
                           int flags, ltb_w2l_session** out);
int ltb_w2l_session_destroy(ltb_w2l_session* s);

/* replaces audio.melspectrogram + the window slicing of MelASR.run_step
 * (avatars/audio_features/mel.py:46-63, avatars/wav2lip/audio.py:45-51).
 * pcm: (stride_left+stride_right+2*batch)*320 float32 samples; out_mel: float32 [batch,80,16] host buffer (or NULL).
 * Runs on the session's feature-extractor stream with its own device buffers: it may be called from the render thread
 * while another thread is inside ltb_w2l_infer / ltb_w2l_paste* (avatars/base_avatar.py:483-489 vs :366) and never
 * touches the forward pass's audio input.  Synchronous. */
int ltb_w2l_mel_step(ltb_w2l_session* s, const float* pcm, int nsamples, float* out_mel);
/* upload the PCM window that the device-resident step (ltb_w2l_mel_resident / ltb_w2l_step_async) reads.  Synchronous. */
int ltb_w2l_set_pcm(ltb_w2l_session* s, const float* pcm, int nsamples);

/* replaces LipReal.inference_batch(index, audiofeat_batch), avatars/wav2lip_avatar.py:116-139.
 * mel: float32 [batch,80,16] host windows (NULL = use the windows ltb_w2l_mel_resident left on the device).
 * pred_out: float32 [batch,256,256,3] BGR in [0,255] (the reference's return value) or NULL to leave the
 * predictions on the device for ltb_w2l_paste*.  Synchronous. */
int ltb_w2l_infer(ltb_w2l_session* s, int index, const float* mel, float* pred_out);

/* replaces LipReal.paste_back_frame(pred_frame, idx), avatars/wav2lip_avatar.py:141-147, for the prediction in
 * `slot` (0..batch-1) of the last infer.  out_frame: uint8 [H,W,3] host buffer.  Synchronous. */
int ltb_w2l_paste(ltb_w2l_session* s, int slot, int idx, uint8_t* out_frame);
/* same entry point for a prediction held by the host: pred is the float32 [256,256,3] array inference_batch returned
 * (the reference's exact paste_back_frame(pred_frame, idx) signature).  Synchronous. */
int ltb_w2l_paste_pred(ltb_w2l_session* s, const float* pred, int idx, uint8_t* out_frame);
/* all `batch` frames of the last infer at once (frame i uses mirror_index(n, index+i), utils/image.py:26-32).
 * out_frames: uint8 [batch,H,W,3] host buffer (pinned recommended) or NULL to keep them on the device. */
int ltb_w2l_paste_batch(ltb_w2l_session* s, int index, uint8_t* out_frames);

/* inference_batch in the plugin's fused mode, one call: H2D of the mel windows, forward, batched paste-back, D2H of the `batch`
 * composited frames (uint8 [batch,H,W,3]; pinned memory recommended), ONE lock / synchronise instead of two.  Synchronous. */
int ltb_w2l_infer_paste(ltb_w2l_session* s, int index, const float* mel, uint8_t* out_frames);

/* Cross-session batching (SURVEY §8 f1; app.py:76-100 runs up to max_session sessions against one shared model): ONE
 * forward + paste launch whose `batch` slots carry frames of DIFFERENT sessions.  The session must have been created with
 * LTB_SESSION_SLOTS (its own avatar only fixes the frame size H x W; every slot's avatar must have the same size and live
 * on the same device).  Slot i: face / frame / rectangle of avatar->frame idx (the caller applies mirror_index,
 * utils/image.py:26-32) and the (80,16) mel window MelASR queued for that frame.  out_frames: uint8 [nslots,H,W,3] host
 * buffer.  Replaces nslots/B calls of inference_batch + nslots calls of paste_back_frame.  Synchronous. */
typedef struct ltb_w2l_slot {
  ltb_w2l_avatar* avatar;
  int idx;
  const float* mel;   /* host float32 [80,16] */
} ltb_w2l_slot;
int ltb_w2l_infer_slots(ltb_w2l_session* s, const ltb_w2l_slot* slots, int nslots, uint8_t* out_frames);

/* Region forms of the composite, for frame-free avatars (and usable with any avatar): the device writes only the paste
 * rectangle, cv2.resize(pred.astype(u8), (x2-x1, y2-y1)) of avatars/wav2lip_avatar.py:141-147, and the host writes it into its
 * own copy of frame idx at (y1, x1).  Packed outputs are uint8 [count][rh_max][rw_max][3] with (rh_max, rw_max) of the SESSION's
 * avatar (ltb_w2l_avatar_region_max); slot i's rectangle of its coords (h, w) is out[i][0:h][0:w], the rest is unspecified.
 *   infer_paste_region: ltb_w2l_infer_paste with region output (count = batch).  Synchronous.
 *   infer_slots_region: ltb_w2l_infer_slots with region output (count = nslots).  Slot avatars may have any frame size; each
 *                       rectangle must fit (rh_max, rw_max) of the session's avatar.  Synchronous.
 *   paste_pred_region:  ltb_w2l_paste_pred with region output, tightly packed uint8 [y2-y1][x2-x1][3].  Synchronous. */
int ltb_w2l_infer_paste_region(ltb_w2l_session* s, int index, const float* mel, uint8_t* out_regions);
int ltb_w2l_infer_slots_region(ltb_w2l_session* s, const ltb_w2l_slot* slots, int nslots, uint8_t* out_regions);
int ltb_w2l_paste_pred_region(ltb_w2l_session* s, const float* pred, int idx, uint8_t* out_region);

/* mel windows from the PCM buffer already resident on the device (uploaded by ltb_w2l_set_pcm):
 * the device-resident form of MelASR.run_step's feature extraction.  Asynchronous. */
int ltb_w2l_mel_resident(ltb_w2l_session* s);
/* whole step with everything resident in HBM: mel (resident PCM) + forward + batched paste-back, enqueued on the
 * session stream WITHOUT synchronising — used for device-timed throughput. */
int ltb_w2l_step_async(ltb_w2l_session* s, int index);
/* the U-Net forward only (face gather + every conv + head; mel windows as left by the last mel call), enqueued without
 * synchronising: the timed region of bench.py's roofline figure (all conv launches of one step, back to back). */
int ltb_w2l_forward_async(ltb_w2l_session* s, int index);
/* profiling pass: runs the forward eagerly with a CUDA event between every op; returns per-op milliseconds, the
 * algorithmic FLOPs of each op (2*M*N*K of the conv it implements, 0 for non-conv ops) and op kinds
 * (0 conv gather, 1 prep_faces, 2 audio_conv0, 3 head, 4 conv halo, 5 stem, 6 mel).  Call with ms == NULL to query n_ops. */
int ltb_w2l_profile_ops(ltb_w2l_session* s, int index, int max_ops, int* n_ops, float* ms, double* flops, int* kinds);
/* pipelined end-to-end step with HOST buffers: H2D of the PCM window, mel, forward, batched paste-back, and the D2H of
 * the `batch` composited frames on a copy stream (double-buffered on the device, so the copy of step i overlaps the
 * kernels of step i+1).  pcm_host / frames_host must be page-locked (ltb_host_alloc) and stay untouched until
 * ltb_w2l_sync (use two alternating buffers when steps are issued back to back). */
int ltb_w2l_step_e2e_async(ltb_w2l_session* s, int index, const float* pcm_host, int nsamples, uint8_t* frames_host);
/* blocks the host until the step issued two calls ago (which used the same alternating host buffers) has completely
 * finished, i.e. its PCM has been consumed and its frames are in host memory — call before refilling the PCM buffer */
int ltb_w2l_e2e_acquire(ltb_w2l_session* s);
int ltb_w2l_sync(ltb_w2l_session* s);
/* the session's cudaStream_t (so a caller can record CUDA events on it) */
int ltb_w2l_stream(ltb_w2l_session* s, void** cuda_stream);
/* number of kernels the engine has launched on this session so far (graph replays count their nodes) */
int ltb_w2l_launch_count(ltb_w2l_session* s, long long* n);
/* pinned host memory helpers for the e2e path */
int ltb_host_alloc(size_t nbytes, void** out);
int ltb_host_free(void* p);

/* ---- debug / test hooks ----------------------------------------------------------------------------- */
/* number of conv blocks (54) ; copy layer `layer`'s post-activation output as dense fp16 NHWC [batch,H,W,C]
 * (requires LTB_SESSION_KEEP_LAYERS).  layer = 54 returns the head input (same as 53). */
int ltb_w2l_num_layers(void);
int ltb_w2l_layer_shape(ltb_w2l_session* s, int layer, int* H, int* W, int* C);
int ltb_w2l_layer_read(ltb_w2l_session* s, int layer, void* out_f16, size_t nbytes);

/* stand-alone conv on the tensor-core kernel (unit parity tests): NHWC fp16 host tensors.
 * transposed != 0: ConvTranspose2d(k=3,s=2,p=1,op=1) via 4 sub-pixel phases; weights are passed in the PyTorch
 * layouts ([Cout,Cin,KH,KW] for conv, [Cin,Cout,3,3] for transposed) as float32 and packed internally.
 * force_path: 0 = auto, 1 = gather kernel, 2 = TMA kernel. */
typedef struct ltb_conv_desc {
  int N, IH, IW, Cin, Cout, KH, KW, sy, sx, pad, transposed, relu, has_res, force_path;
} ltb_conv_desc;
int ltb_conv2d_f16(const ltb_conv_desc* d, const void* in_f16, const float* w_f32, const float* bias_f32,
                   const void* res_f16, void* out_f16);
/* same, then `reps` more back-to-back launches of the same plan between two CUDA events: *ms_per_launch (kernel development aid) */
int ltb_conv2d_f16_timed(const ltb_conv_desc* d, const void* in_f16, const float* w_f32, const float* bias_f32,
                         const void* res_f16, void* out_f16, int reps, float* ms_per_launch);

/* ==== generic device-op layer (MuseTalk path) ==========================================================================
 * The MuseTalk networks are third-party graphs the reference only wraps: diffusers.UNet2DConditionModel
 * (avatars/musetalk/models/unet.py:29-48), diffusers.AutoencoderKL (avatars/musetalk/models/vae.py:10-38) and
 * transformers.WhisperModel (avatars/musetalk/whisper/audio2feature.py:15-23).  Host code (Python) assembles them
 * from the operators below, captures the sequence once into a CUDA graph and replays it per step.  All ops are
 * asynchronous on the context stream; pointers are device pointers obtained from ltb_dev_alloc. */
typedef struct ltb_ctx ltb_ctx;
typedef struct ltb_graph ltb_graph;
int ltb_ctx_create(ltb_ctx** out);
int ltb_ctx_destroy(ltb_ctx* c);
int ltb_ctx_stream(ltb_ctx* c, void** cuda_stream);
int ltb_ctx_sync(ltb_ctx* c);
int ltb_ctx_launch_count(ltb_ctx* c, long long* n);
int ltb_dev_alloc(ltb_ctx* c, size_t bytes, int zero, void** dptr);
int ltb_dev_free(ltb_ctx* c, void* dptr);
int ltb_h2d(ltb_ctx* c, void* dst_dev, const void* src_host, size_t bytes, int sync);
int ltb_d2h(ltb_ctx* c, void* dst_host, const void* src_dev, size_t bytes, int sync);
int ltb_set_i32(ltb_ctx* c, void* dptr, int value); /* stream-ordered scalar (per-step avatar index read by graph kernels) */
int ltb_capture_begin(ltb_ctx* c);
int ltb_capture_end(ltb_ctx* c, ltb_graph** out);
int ltb_graph_launch(ltb_ctx* c, ltb_graph* g);
int ltb_graph_destroy(ltb_graph* g);

/* conv / linear / batched GEMM on the tcgen05 kernels (nn.Conv2d, nn.Linear, attention Q.K^T and P.V):
 * out[pix, co] = act(sum_{tap,ci} in[pix*s + tap - pad, ic_off+ci] * w[co, w_koff + tap*Cin + ci] + bias[co] (+ res[pix, co]))
 * w: fp16 [Cout][Ktot] (K-major rows); w_tap: optional tap-major copy [9][Cout][Cin] enabling the TMA halo kernel for
 * 3x3 s1 p1; bias may be NULL (zero).  zbatch > 1 runs zbatch independent GEMMs (z = zo*zdiv + zi) with element
 * offsets in_z*, w_z*, out_z* added to the base pointers. */
typedef struct ltb_conv_op {
  const void* in; const void* w; const void* w_tap; const float* bias; const void* res; void* out;
  int N, IH, IW, ICtot, ic_off, Cin;
  int OH, OW, Cout, OCtot, oc_off, RCtot, rc_off;
  int KH, KW, sy, sx, pad_t, pad_l;
  int Ktot, w_koff, relu, no_halo;
  int zbatch, zdiv;
  long long in_zo, in_zi, w_zo, w_zi, out_zo, out_zi;
  /* optional: also produce the GroupNorm statistics (sum, sum of squares per (image, group); gn_hw pixels per image) of the
   * output tensor into gn_stats[N][gn_groups][2] — fused into the conv epilogue when the kernel supports it */
  void* gn_stats;
  int gn_groups, gn_hw;
  /* 1: nearest-2x upsample fused with this 3x3 p1 s1 conv (diffusers Upsample2D: F.interpolate(scale 2, nearest) + conv): the
   * input is the LOW-resolution map (N, IH, IW), OH = 2*IH, OW = 2*IW; `w` / `w_tap` hold the 16 pre-summed sub-pixel slices
   * ([Cout][16][Cin] phase-major / [16][Cout][Cin] view-major, built by livetalking_b200.ops.ConvWeight.upconv()), Ktot = 16*Cin */
  int upsample2x;
} ltb_conv_op;
int ltb_op_conv2d(ltb_ctx* c, const ltb_conv_op* d);
int ltb_op_w_tap_major(ltb_ctx* c, const void* w, void* wt, int cout, int cin);
/* torch.nn.GroupNorm (+ optional SiLU) on an NHWC channel slice; fp32 statistics */
int ltb_op_groupnorm(ltb_ctx* c, const void* x, int N, int HW, int C, int Ctot, int c_off, int groups, float eps, const float* gamma,
                     const float* beta, int silu, void* out, int OCtot, int oc_off);
/* normalisation pass only, with statistics produced by a previous ltb_op_conv2d (gn_stats) */
int ltb_op_groupnorm_apply(ltb_ctx* c, const void* x, int N, int HW, int C, int Ctot, int c_off, int groups, float eps, const void* stats,
                           const float* gamma, const float* beta, int silu, void* out, int OCtot, int oc_off);
/* torch.nn.LayerNorm over the last dim of [rows, C] */
int ltb_op_layernorm(ltb_ctx* c, const void* x, int rows, int C, float eps, const float* gamma, const float* beta, void* out);
/* softmax(scale * x[:, :valid]) per row of a [rows, ld] matrix; columns [valid, cols) are written as 0 */
int ltb_op_softmax(ltb_ctx* c, const void* x, int rows, int cols, int ld, int valid, float scale, void* out);
/* diffusers GEGLU: out[rows,H] = h[:, :H] * gelu(h[:, H:]) */
int ltb_op_geglu(ltb_ctx* c, const void* h, long long rows, int H, void* out);
/* out = act(x + y[i % period]) ; y may be NULL ; act: 0 none, 1 GELU(erf), 2 SiLU */
int ltb_op_eltwise(ltb_ctx* c, const void* x, const void* y, long long n, long long period, int act, void* out);
int ltb_op_upsample2x(ltb_ctx* c, const void* x, int N, int H, int W, int C, void* out);
int ltb_op_copy_channels(ltb_ctx* c, const void* src, long long rows, int C, int SCtot, int sc_off, void* dst, int DCtot, int dc_off);
int ltb_op_transpose_heads(ltb_ctx* c, const void* v, int B, int n_keys, int Ctot, int c_off, int heads, int d, int n_pad, void* vt);
/* Fused multi-head attention out = softmax(scale * Q K^T) V on tcgen05 (scores stay in TMEM / shared memory): the diffusers Attention
 * blocks of the UNet (avatars/musetalk/models/unet.py:29-48) and the Whisper encoder layers (whisper/audio2feature.py:106-117).
 * q [B][nq] rows of q_pitch halves, k [B][kv_rows] rows of kv_pitch halves, head h at columns [h*d, (h+1)*d); vt = the
 * ltb_op_transpose_heads output [B*heads][d][n_pad]; keys >= valid get probability 0; out [B*nq][out_pitch], head h at columns
 * h*d.  d % 16 == 0, d <= 160; pitches and n_pad multiples of 8. */
int ltb_op_attention(ltb_ctx* c, const void* q, int q_pitch, const void* k, int kv_pitch, int kv_rows, const void* vt, int n_pad, int B, int heads,
                     int nq, int valid, int d, float scale, void* out, int out_pitch);
/* ---- UltraLight + HuBERT (SURVEY 8 row f4) ----------------------------------------------------------------------------------
 * InvertedResidual's depthwise 3x3 + folded BN (+ReLU), avatars/ultralight/unet.py:18-26: x NHWC fp16 (pixel pitch ICtot, channels
 * [ic_off, ic_off+C)), w_tap fp16 [9][C], bias fp32 [C], pad 1, stride 1|2 -> out (pitch OCtot, offset oc_off). */
int ltb_op_dwconv3x3(ltb_ctx* c, const void* x, int N, int IH, int IW, int ICtot, int ic_off, int C, const void* w_tap, const float* bias, int stride,
                     int relu, void* out, int OCtot, int oc_off);
/* nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True), unet.py:76, written into a channel slice (torch.cat, unet.py:88) */
int ltb_op_upsample_bilinear2x(ltb_ctx* c, const void* x, int N, int H, int W, int ICtot, int ic_off, int C, void* out, int OCtot, int oc_off);
/* LightReal.inference_batch input glue, avatars/ultralight_avatar.py:146-160: faces u8 [nf,168,168,3], frame b = mirror_index(nf,
 * *d_index + b) -> fp16 [B,160,160,16] (ch 0-2 crop/255, ch 3-5 with the filled rectangle (5,5,150,145), ch 6-15 zero) */
int ltb_op_ul_prep(ltb_ctx* c, const void* faces_u8, int nf, const void* d_index, int B, void* out);
/* 1x1 conv 32 -> 3 + sigmoid, x 255 (OutConv + F.sigmoid, unet.py:224-225; "* 255." ultralight_avatar.py:168): x fp16 [npix][32] */
int ltb_op_head_sigmoid255(ltb_ctx* c, const void* x, const float* w3x32, const float* b3, long long npix, float* pred);
/* LightReal.paste_back_frame, ultralight_avatar.py:171-184: crop[4:164,4:164] = pred.astype(u8); cv2.resize(crop, bbox) into the
 * frame; coords int32 [nf][4] = (x1,y1,x2,y2); pred f32 [B,160,160,3]; job j < count pastes slot slot0+j into out[j] for frame
 * explicit_idx (>= 0) or mirror_index(nf, index + j).  Bit-exact with OpenCV. */
int ltb_op_ul_paste(ltb_ctx* c, const void* frames, const void* faces, const void* coords, const float* pred, void* out, int nf, int H, int W,
                    int index, int explicit_idx, int slot0, int count);
/* region twin for frame-free avatars: only the bbox rectangle cv2.resize(crop, (x2-x1, y2-y1)), no frame read.  Job j writes
 * out[j][0:y2-y1][0:x2-x1] of a packed uint8 [count][rh][rw][3] buffer (rh, rw >= every box of the jobs); the host pastes it. */
int ltb_op_ul_paste_region(ltb_ctx* c, const void* faces, const void* coords, const float* pred, void* out, int nf, int rh, int rw, int index,
                           int explicit_idx, int slot0, int count);
/* Audio2Feature.get_hubert_from_16k_speech front end, avatars/ultralight/audio2feature.py:14-20: Wav2Vec2 processor normalisation
 * (stats[2] = mean, 1/sqrt(var + 1e-7)) fused with HubertModel's conv layer 0 (w fp32 [C][10], stride 5) -> fp16 [(n-10)/5+1][C] */
int ltb_op_hubert_conv0(ltb_ctx* c, const float* pcm, int n, const float* w, const float* bias, int C, float* stats, void* out);
/* HubertPositionalConvEmbedding + residual: out = h + gelu(conv1d(h, k 128, pad 64, groups)[:T]); w fp16 [D][128][D/groups] */
int ltb_op_hubert_pos_conv(ltb_ctx* c, const void* h, int T, int D, int groups, int K, const void* w, const float* bias, void* out);
/* trim / pad to T rows (audio2feature.py:50-55) + BaseASR._feature2chunks (avatars/audio_features/base_asr.py:91-157) as
 * HubertASR.run_step calls it (hubert.py:42-45): out_f32 [B][R][D] and / or out_nhwc fp16 [B][D][R] */
int ltb_op_hubert_slice(ltb_ctx* c, const void* hidden, int Tc, int T, int D, int B, int R, float start, float mult, int win_l, float* out_f32,
                        void* out_nhwc);
/* VAE.decode_latents post-processing, avatars/musetalk/models/vae.py:104-107 -> uint8 BGR NHWC */
int ltb_op_vae_post(ltb_ctx* c, const void* x, long long npix, int Ctot, void* out_u8);
/* Encoder hand-off (SURVEY 8(f) rank 3): composited uint8 BGR frames [N,H,W,3] -> planar I420 [N, H*3/2, W] on the device,
 * replacing the CPU bgr24 -> yuv420p conversion behind VideoFrame.from_ndarray (avatars/base_avatar.py:449-453).
 * OpenCV COLOR_BGR2YUV_I420 arithmetic (BT.601 limited range); H even, W % 4 == 0. */
int ltb_op_bgr_to_i420(ltb_ctx* c, const void* bgr_u8, int N, int H, int W, void* out_i420);
/* The watermark of avatars/base_avatar.py:449 (cv2.putText(frame, "LiveTalking", (10,20), FONT_HERSHEY_SIMPLEX, 0.3, (128,128,128), 1))
 * for frames that stay on the device: writes colour (b,g,r) into the n pixels pix_yx[k] = (y, x) (int32, device) of every frame
 * [N,H,W,3]; the pixel set is what OpenCV itself rasterises for that text (livetalking_b200/watermark.py).  Bit-exact. */
int ltb_op_stamp_pixels(ltb_ctx* c, void* frames_u8, int N, int H, int W, const void* pix_yx, int n, int b, int g, int r);
/* VAE.preprocess_img, avatars/musetalk/models/vae.py:51-82 (uint8 BGR -> fp16 RGB [-1,1], 8-channel padded NHWC) */
int ltb_op_vae_pre(ltb_ctx* c, const void* img_u8, int N, int H, int W, int half_mask, void* out);
/* out[i] = table[mirror_index(n, *d_index + i)], i < B  (latent gather of MuseReal.inference_batch, musetalk_avatar.py:134-139) */
int ltb_op_gather_rows(ltb_ctx* c, const void* table, int n, const void* d_index, int B, long long row_elems, void* out);
/* transformers.WhisperFeatureExtractor as used by Audio2Feature.audio2feat (avatars/musetalk/whisper/audio2feature.py:106-111):
 * float32 PCM [n <= 480000] -> log-mel features; out_f16 = fp16 [3000][80] (conv1 input), out_f32 (optional) = float [80][3000].
 * fb_f32: the 80 x 201 Slaney mel filterbank; logspec_ws: >= 80*3000 floats; gmax_ws: one int. */
int ltb_op_whisper_logmel(ltb_ctx* c, const void* pcm_f32, int n, const void* fb_f32, void* logspec_ws, void* gmax_ws, void* out_f16,
                          void* out_f32);
/* WhisperASR._feature2chunks / BaseASR._get_sliced_feature (avatars/audio_features/whisper.py:35-56, base_asr.py:91-133):
 * frame i <- encoder steps int((i+start)*mult) + 0..9 (clamped) of the 5 hidden states -> out[i][50 rows][D]. */
int ltb_op_whisper_slice(ltb_ctx* c, const void* const* hidden5, int T, int D, int B, float start, float mult, void* out,
                         int out_rows_per_frame);
/* MuseReal.paste_back_frame + get_image_blending (avatars/musetalk_avatar.py:154-164, avatars/musetalk/myutil.py:4-25) */
typedef struct ltb_mt_paste_op {
  const void* frames; const void* coords; const void* crop; const void* masks; const void* mask_off; const void* pred; void* out;
  int nf, H, W, index, explicit_idx, slot0, count;
  int pred_hw;   /* side of the square prediction: 256 (the reference, vae.py:15) or 512 (64x64 latents); 0 = 256 */
  /* region form (frame-free avatars; zero = the full-frame form above): body = the crop box of every original frame, packed exactly
   * like the masks (same shapes, same mask_off); frames is not read and may be NULL.  Job j writes only its blended crop box,
   * out[j][0:y_e-y_s][0:x_e-x_s] of a packed uint8 [count][region_h][region_w][3] buffer (region_h/w >= every crop box of the jobs);
   * nothing outside the crop box changes, so the host pastes it into its own copy of the frame. */
  const void* body;
  int region_h, region_w;
} ltb_mt_paste_op;
int ltb_op_mt_paste(ltb_ctx* c, const ltb_mt_paste_op* d);

#ifdef __cplusplus
}
#endif
#endif /* LTB200_H_ */

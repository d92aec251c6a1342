/* dcb200 -- C ABI of the B200-native DeepConsensus model path.
 *
 * This is the drop-in boundary for the one hot path of google/deepconsensus (v1.2.0):
 *
 *   quick_inference.initialize_model()          deepconsensus/inference/quick_inference.py:485-532
 *   quick_inference.run_model_on_examples()     deepconsensus/inference/quick_inference.py:341-415
 *     -> model.predict(rows)                    deepconsensus/models/networks.py:357-365 (:221-345, :436-520)
 *     -> argmax / Phred / calibration / clip    quick_inference.py:377-389, quality_calibration/calibration_lib.py:77-99
 *     -> per-window base + quality strings      quick_inference.py:390-414, utils/utils.py:60-62
 *
 * The reference has no FFI (it is pure Python on TensorFlow); the binding a maintainer adds
 * is a ctypes stub -- see INTEGRATION.md and deepconsensus_b200/engine.py.
 *
 * Conventions: plain C, no exceptions across the boundary.  Every function returns
 * DCB_OK (0) or a negative error code; dcb_last_error() gives the message.  All buffers are
 * caller-owned and caller-sized.  One engine per device, not re-entrant (the reference
 * touches the model from its main thread only).  Results are deterministic (no atomics in
 * any reduction).
 */
#ifndef DCB200_H_
#define DCB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCB_OK 0
#define DCB_ERR_INVALID (-1)     /* bad argument / unsupported configuration */
#define DCB_ERR_CUDA (-2)        /* CUDA runtime error (message has the detail) */
#define DCB_ERR_WEIGHTS (-3)     /* missing / mis-shaped variable */
#define DCB_ERR_STATE (-4)       /* call order (e.g. forward before load_weights) */
#define DCB_ERR_INPUT_RANGE (-5) /* an embedding id was out of range (TF would raise); output still produced with clamped ids */

typedef struct dcb_engine dcb_engine;

/* Model + inference options.  Field names follow params.json / InferenceOptions
 * (models/model_configs.py:76-139,272-338; quick_inference.py:238-275). */
typedef struct dcb_config {
  int32_t struct_size;        /* sizeof(dcb_config), for ABI checking */
  int32_t device;             /* CUDA device ordinal */
  /* input geometry (data_providers.py:61-113) */
  int32_t max_passes;
  int32_t max_length;
  int32_t use_ccs_bq;
  /* transformer (transformer_basic_params.py:33-67 merged under model_configs.py) */
  int32_t hidden_size;        /* must be 280 */
  int32_t num_heads;          /* must be 2 */
  int32_t num_hidden_layers;
  int32_t filter_size;        /* multiple of 128, <= 2048 */
  int32_t attn_win_size;      /* 0 => full attention (params.attn_win_size None) */
  int32_t rezero;             /* 1: x + alpha*f(x); 0: x + f(LayerNorm(x)) (encoder_stack.py:72-93) */
  int32_t add_pos_encoding;
  int32_t condense_transformer_input; /* must be 1 (transformer_input_size == hidden_size) */
  /* embedding widths and vocabularies (networks.py:375-421) */
  int32_t per_base_hidden_size, pw_hidden_size, ip_hidden_size, strand_hidden_size,
      ccs_bq_hidden_size, sn_hidden_size;
  int32_t pw_max, ip_max, sn_max, ccs_bq_max, strand_max;
  /* post-processing (quick_inference.py:377-389) */
  int32_t max_base_quality;   /* 93 */
  int32_t calibration_enabled;
  double calibration_threshold, calibration_w, calibration_b;
  /* engine sizing */
  int32_t max_batch;          /* largest B a single dcb_forward call will see */
  int32_t chunk_tiles;        /* 128-token tiles processed per pass through the layer stack; 0 = auto */
  int32_t precision;          /* DCB_PRECISION_BF16 (default) or DCB_PRECISION_FP32: which arithmetic dcb_forward uses
                                 when the call does not say (see DCB_STRICT_FP32) */
  int32_t reserved[5];
} dcb_config;

/* Arithmetic of the forward pass.
 *   DCB_PRECISION_BF16  tensor-core path: bf16 operands, float32 accumulation / residual / LayerNorm / softmax.
 *                       Logits differ from the reference's float32 graph by the operand rounding (0.02-0.1 on
 *                       random-weight models), so the argmax can flip at near-ties.
 *   DCB_PRECISION_FP32  the reference's own arithmetic (float32 operands and accumulation, networks.py:506-507):
 *                       differs from the reference by summation order only (~1e-5 on logits); identical bases wherever
 *                       the float32 top-2 logit margin exceeds 1e-3.  CUDA-core kernels, ~25x slower. */
#define DCB_PRECISION_BF16 0
#define DCB_PRECISION_FP32 1

/* A named host tensor in the reference checkpoint's layout (SURVEY.md Appendix B), e.g.
 * "model/encoder_stack/layers/0/0/layer/query_dense_layer/kernel" float32 [280,2,140]. */
typedef struct dcb_tensor {
  const char* name;
  const float* data;   /* host pointer, C-contiguous float32 */
  int32_t ndim;
  int64_t shape[4];
} dcb_tensor;

/* flags for dcb_forward */
#define DCB_ROWS_ON_DEVICE 1u   /* `rows` is a device pointer (already resident in HBM); must be 16-byte aligned */
#define DCB_OUT_ON_DEVICE 2u    /* output pointers are device pointers */
#define DCB_STRICT_FP32 4u      /* this call runs in float32 (DCB_PRECISION_FP32) whatever dcb_config.precision says */
#define DCB_FAST_BF16 8u        /* this call runs the bf16 tensor-core path whatever dcb_config.precision says */

/* Create an engine on cfg->device.  Replaces model construction in initialize_model
 * (quick_inference.py:515-526). */
int dcb_create(const dcb_config* cfg, dcb_engine** out);

/* Load all variables (host fp32, reference shapes); the engine pads, folds (query scale,
 * ReZero alpha) and casts into its device layouts.  Replaces checkpoint.restore(...)
 * (quick_inference.py:527-529).  Unknown names are ignored (expect_partial); every variable
 * the configured model needs must be present. */
int dcb_load_weights(dcb_engine* e, const dcb_tensor* tensors, int32_t n);

/* The hot path: rows float32 [B, total_rows, max_length] (the [B,R,L,1] tensor of
 * quick_inference.py:363 with the channel axis dropped; NOT pre-clipped -- format_rows'
 * clipping happens on the device) -> per position base character (' ', 'A', 'T', 'C', 'G')
 * and Phred+33 quality character.  probs_out / logits_out ([B, L, 5] float32) may be NULL. */
int dcb_forward(dcb_engine* e, const float* rows, int32_t batch, uint32_t flags,
                uint8_t* bases_out, uint8_t* quals_out, float* probs_out, float* logits_out);

/* ---- packed input rows (SURVEY.md section 8(f)1: the feature-construction side of the path) --------------------------
 * The float32 [B, R, L] rows of quick_inference.py:363 hold small integers: bases / ccs in 0..4, pw / ip from uint8
 * BAM tags (pre_lib.py:221-226,704-744), strand in 0..2, ccs_bq in -1..93, plus four float SN values per window that
 * extract_features repeats along L (pre_lib.py:741-742).  The packed form keeps exactly that information in
 * dcb_packed_window_bytes() bytes per window (7,344 B instead of 40,800 B for 20 x 120) -- per window, in this order:
 *     u8 [P][L]   bits 0-2 = base id of subread p (row p), bits 3-4 = its strand id (row 3P + p)
 *     u8 [P][L]   pw (rows P..2P-1),   clipped to [0, 255] and truncated, as format_rows + tf.cast would
 *     u8 [P][L]   ip (rows 2P..3P-1),  same
 *     u8 [L]      ccs base id (row 4P)
 *     u8 [L]      ccs_bq + 1 (row 4P+1; only when use_ccs_bq) -- the embedding id itself (networks.py:495)
 *     padding to a multiple of 16 bytes
 *     f32 [4]     the window's SN values (rows R-4..R-1, taken at position 0; not clipped)
 * The engine turns packed bytes into table ids inside its embedding kernel (PW_MAX / IP_MAX / SN_MAX clipping included);
 * results are bit-identical to dcb_forward on the float32 rows the packed form was made from.
 *
 * dcb_pack_rows: host helper (needs no GPU and no engine -- it belongs to the producer of the rows; only max_passes,
 * max_length, use_ccs_bq and the *_max fields of `cfg` are read), float32 rows [B, R, L] -> packed.  Returns DCB_ERR_INPUT_RANGE (and still writes
 * clamped output) if a base / strand / ccs / ccs_bq value is outside its vocabulary -- the values TensorFlow's gather
 * would raise on -- or an SN row is not constant along L; DCB_ERR_INVALID if the configuration cannot be packed
 * (PW_MAX or IP_MAX above 255). */
size_t dcb_packed_window_bytes(const dcb_config* cfg);
int dcb_pack_rows(const dcb_config* cfg, const float* rows, int32_t batch, uint8_t* packed_out);
/* dcb_forward / dcb_submit on packed rows (host pointer, or device pointer with DCB_ROWS_ON_DEVICE: 16-byte aligned). */
int dcb_forward_packed(dcb_engine* e, const uint8_t* packed, int32_t batch, uint32_t flags,
                       uint8_t* bases_out, uint8_t* quals_out, float* probs_out, float* logits_out);
int dcb_submit_packed(dcb_engine* e, const uint8_t* packed, int32_t batch, uint32_t flags,
                      uint8_t* bases_out, uint8_t* quals_out, float* probs_out, float* logits_out, int64_t* ticket);

/* Pipelined form of dcb_forward for a stream of batches (the `for batch in batches: model.predict(batch)` loop of
 * quick_inference.py:352-368): dcb_submit enqueues the host->device copy of `rows` on a copy stream, the kernels and
 * the device->host copy of the results, and returns a ticket without waiting; dcb_wait(ticket) blocks until that
 * batch's outputs are in the caller's buffers and returns its status (DCB_ERR_INPUT_RANGE etc.).  At most TWO
 * submissions may be in flight, so the copy of batch i+1 overlaps the kernels of batch i; tickets must be waited for in
 * order.  `rows` and the output buffers must stay valid (and should be page-locked, dcb_alloc_host) until dcb_wait
 * returns.  dcb_forward == dcb_submit + dcb_wait. */
int dcb_submit(dcb_engine* e, const float* rows, int32_t batch, uint32_t flags,
               uint8_t* bases_out, uint8_t* quals_out, float* probs_out, float* logits_out, int64_t* ticket);
int dcb_wait(dcb_engine* e, int64_t ticket);

/* The first stage of stitch_utils.stitch_to_fastq for a batch of reads -- get_full_sequence + remove_gaps
 * (stitch_utils.py:51-98) -- on the device: the windows [zmw_start[z], zmw_start[z+1]) of `bases` / `quals`
 * ([n_windows, L] bytes exactly as dcb_forward writes them, sorted by window position) are concatenated and the gap
 * character ' ' is dropped together with the quality character under it.  Read z is written at offset
 * zmw_start[z] * L of seq_out / qual_out (each n_windows * L bytes) and len_out[z] receives its length.  zmw_start is a
 * host array of n_zmw + 1 non-decreasing window indices.  flags: DCB_ROWS_ON_DEVICE => bases/quals are device
 * pointers (e.g. the DCB_OUT_ON_DEVICE outputs of dcb_forward); DCB_OUT_ON_DEVICE => seq_out/qual_out/len_out are
 * device pointers.  The missing-window check and the empty / quality / length filters stay with the caller
 * (deepconsensus_b200/stitch_gpu.py), which has the window positions and read names. */
int dcb_stitch(dcb_engine* e, const uint8_t* bases, const uint8_t* quals, int32_t n_windows, int32_t L,
               const int32_t* zmw_start, int32_t n_zmw, uint32_t flags,
               uint8_t* seq_out, uint8_t* qual_out, int32_t* len_out);

/* ---- the rest of the post-model stage on the device (SURVEY.md section 8(f)2) ------------------------------------------
 * dcb_stitch_fastq = stitch_utils.stitch_to_fastq for a batch of reads (stitch_utils.py:131-189): dcb_stitch, then per
 * read the missing-window check of get_full_sequence (window i must not start beyond i * L, stitch_utils.py:60-78), the
 * only-gaps check, the quality filter round(avg_phred(quals), 5) >= min_quality (utils.py:88-106,
 * stitch_utils.py:101-109), the length filter, and for the reads that pass the FASTQ record
 * '@' name '\n' sequence "\n+\n" quality '\n' (stitch_utils.py:112-119) written at rec_off[z] of fastq_out.
 *   window_pos [n_windows]   DCModelOutput.window_pos of every window (sorted within a read)
 *   names / name_off         the read names, concatenated; read z is names[name_off[z] .. name_off[z+1])
 *   fastq_out, fastq_cap     caller-sized; names + 2 * n_windows * L + 6 * n_zmw bytes always suffice
 *   rec_off [n_zmw + 1]      byte offset of every read's record (rec_off[n_zmw] = total bytes written)
 *   outcome [n_zmw]          DCB_READ_* -- the OutcomeCounter field the reference would bump
 *   avg_q [n_zmw]            the read's average Phred (float64)
 * bases / quals are host arrays, or device arrays with DCB_ROWS_ON_DEVICE (e.g. dcb_forward's DCB_OUT_ON_DEVICE
 * outputs); every output is a host array.  A read whose average quality lies within 1e-7 of the filter threshold is
 * reported with DCB_READ_BORDERLINE or-ed in (its record IS written): the caller re-evaluates that read with the
 * reference's own float64 expression, because NumPy's pairwise sum and the histogram sum used here may differ in the
 * last bits (deepconsensus_b200/stitch_gpu.py does). */
#define DCB_READ_OK 0
#define DCB_READ_EMPTY 1          /* OutcomeCounter.empty_sequence (a window is missing) */
#define DCB_READ_ONLY_GAPS 2      /* OutcomeCounter.only_gaps */
#define DCB_READ_LOW_QUALITY 3    /* OutcomeCounter.failed_quality_filter */
#define DCB_READ_TOO_SHORT 4      /* OutcomeCounter.failed_length_filter */
#define DCB_READ_BORDERLINE 0x80  /* flag: quality within 1e-7 of the threshold, caller decides */
int dcb_stitch_fastq(dcb_engine* e, const uint8_t* bases, const uint8_t* quals, int32_t n_windows, int32_t L,
                     const int32_t* zmw_start, int32_t n_zmw, const int32_t* window_pos,
                     const uint8_t* names, const int32_t* name_off, double min_quality, int32_t min_length,
                     uint32_t flags, uint8_t* fastq_out, int64_t fastq_cap, int64_t* rec_off, int32_t* outcome,
                     double* avg_q);

/* dcb_stitch_fastq for windows of their own width (CCS smart windows, dcb_prep_set_smart_windows): window w is the bytes
 * [window_off[w], window_off[w + 1]) of bases / quals -- max_length bytes for a scored window, W bytes for an overflow
 * window -- laid out back to back in sorted order; window_off int64 [n_windows + 1], non-decreasing.  L (max_length)
 * still drives the missing-window check: window i of a read must not start beyond i * L, whatever the widths of the
 * windows before it (stitch_utils.py:60-78).  fastq_out: names + 2 * window_off[n_windows] + 6 * n_zmw bytes suffice.
 * Everything else as dcb_stitch_fastq. */
int dcb_stitch_fastq_ragged(dcb_engine* e, const uint8_t* bases, const uint8_t* quals, int32_t n_windows,
                            const int64_t* window_off, int32_t L, const int32_t* zmw_start, int32_t n_zmw,
                            const int32_t* window_pos, const uint8_t* names, const int32_t* name_off, double min_quality,
                            int32_t min_length, uint32_t flags, uint8_t* fastq_out, int64_t fastq_cap, int64_t* rec_off,
                            int32_t* outcome, double* avg_q);

/* The skip decision of inference_on_n_zmws (quick_inference.py:663-672) for a batch of windows:
 * mask[w] = avg_phred(ccs_bq[w, :]) > skip_windows_above (entries < 0 are spacing and are dropped, utils.py:88-106);
 * 2 = within 1e-7 of the threshold, caller decides.  ccs_bq: host int16 [n_windows, L]. */
int dcb_skip_mask(dcb_engine* e, const int16_t* ccs_bq, int32_t n_windows, int32_t L, double skip_windows_above,
                  uint8_t* mask_out, double* avg_out /* nullable */);

/* process_skipped_window (quick_inference.py:567-594) for k windows that bypass the model: window j adopts the CCS
 * bases (ccs_ids, host u8 [k, L], ids 0..4 -> ' ATCG') and the CCS base qualities (ccs_bq, host int16 [k, L]) after
 * calibrate_quality_scores (calibration_lib.py:77-99; float64) / min(., max_base_quality) / int32 truncation / +33,
 * and is written to row dst_window[j] of bases / quals ([*, L]; device arrays with DCB_OUT_ON_DEVICE -- e.g. the arrays
 * dcb_forward filled for the scored windows, so that dcb_stitch_fastq can run on them without a host round trip). */
int dcb_fill_skipped(dcb_engine* e, const uint8_t* ccs_ids, const int16_t* ccs_bq, const int32_t* dst_window, int32_t k,
                     int32_t L, int32_t calibration_enabled, double calibration_threshold, double calibration_w,
                     double calibration_b, uint32_t flags, uint8_t* bases, uint8_t* quals);
/* dcb_fill_skipped for windows of their own width (an overflow window keeps all W columns, quick_inference.py:567-594):
 * window j is the entries [src_off[j], src_off[j + 1]) of ccs_ids (u8) / ccs_bq (int16), src_off int64 [k + 1] with
 * src_off[0] = 0, and lands at byte dst_off[j] (int64 [k]) of bases / quals. */
int dcb_fill_skipped_ragged(dcb_engine* e, const uint8_t* ccs_ids, const int16_t* ccs_bq, const int64_t* src_off,
                            const int64_t* dst_off, int32_t k, int32_t calibration_enabled, double calibration_threshold,
                            double calibration_w, double calibration_b, uint32_t flags, uint8_t* bases, uint8_t* quals);

/* ---- feature construction from BAM (SURVEY.md section 8(f)3; host C++, htslib-free, needs no GPU) -----------------------
 * What `deepconsensus run` does in front of the model: stream the subreads-to-CCS BAM ZMW by ZMW (SubreadGrouper,
 * pre_lib.py:50-91), expand / clip / indent every subread (expand_clip_indent with trim_insertions, :1061-1239), fetch
 * the CCS read (:966-998,1322-1330), space all reads out (space_out_subreads, :1242-1276), cut windows of max_length
 * columns (DcExample.iter_examples, :625-697) and lay the feature rows out (extract_features, :704-744) -- as float32
 * rows and / or directly as packed rows.  Errors: negative return code, message from dcb_prep_last_error(). */
typedef struct dcb_prep dcb_prep;
typedef struct dcb_zmw_info {
  int32_t n_windows;          /* windows of this ZMW (examples without any CCS position are dropped, as the reference does) */
  int32_t n_subreads;         /* mapped subreads in the BAM (the first max_passes are used) */
  const char* name;           /* CCS read name = reference name of the subread alignments; valid until the next call */
  int32_t has_ec, has_np, has_rq;
  float ec, rq;               /* aux tags of the CCS read (construct_ccs_read) */
  int32_t np_num_passes;
  const char* rg;             /* RG tag or NULL */
  int32_t ccs_length, spaced_width;
} dcb_zmw_info;
int dcb_prep_open(const char* subreads_to_ccs_bam, const char* ccs_bam, int32_t max_passes, int32_t max_length,
                  int32_t use_ccs_bq, int32_t ins_trim, dcb_prep** out);
/* Process ZMWs on n_threads worker threads plus one BAM-decoding thread (results still come out in file order); call
 * before the first dcb_prep_next_zmw.  n_threads <= 0: everything on the calling thread. */
int dcb_prep_set_threads(dcb_prep* p, int32_t n_threads);
/* CCS smart windows (`deepconsensus run --use_ccs_smart_windows`, pre_lib.py:625-650,1329-1331): enable != 0 cuts every
 * ZMW into windows whose widths, in CCS bases, come from the CCS record's `wl` tag (a B array of any integer subtype)
 * instead of into max_length columns.  A window's spaced width W (its columns once space_out_subreads has opened gap
 * columns) may exceed max_length: such an overflow window bypasses the model and keeps all W columns.  A CCS record
 * without an integer `wl` array, or whose `wl` does not partition the CCS read exactly, is an error (DCB_ERR_INVALID,
 * message names the read).  Call before the first dcb_prep_next_zmw; off by default. */
int dcb_prep_set_smart_windows(dcb_prep* p, int32_t enable);
int dcb_prep_next_zmw(dcb_prep* p, dcb_zmw_info* info);   /* 1 = a ZMW is loaded, 0 = end of file, < 0 = error */
/* The windows of the loaded ZMW; every output may be NULL.  rows float32 [n, R, L]; packed [n, dcb_packed_window_bytes];
 * window_pos / num_passes int32 [n]; overflow u8 [n] (1 = spaced width > max_length, smart windows only); ccs_bq int16
 * [n, L] (-1 at gaps and padding).  An overflow window holds its first L columns here (never scored). */
int dcb_prep_get_windows(dcb_prep* p, float* rows, uint8_t* packed, int32_t* window_pos, uint8_t* overflow,
                         int16_t* ccs_bq, int32_t* num_passes);
/* widths int32 [n]: the spaced width W of every window of the loaded ZMW (max_length for fixed-width windows). */
int dcb_prep_get_window_widths(dcb_prep* p, int32_t* widths);
/* The overflow windows of the loaded ZMW in full, in window order, ragged (each window's W columns back to back, S = the
 * sum of their widths); every output may be NULL.  rows float32 [R, W] per window (S * R floats in all); ccs_ids u8 [S]
 * (CCS base ids 0..4); ccs_bq int16 [S] (-1 at gaps). */
int dcb_prep_get_overflow_windows(dcb_prep* p, float* rows, uint8_t* ccs_ids, int16_t* ccs_bq);
const char* dcb_prep_ccs_header(dcb_prep* p);             /* SAM header text of the CCS BAM */
void dcb_prep_close(dcb_prep* p);
const char* dcb_prep_last_error(void);
/* Unaligned BAM output as quick_inference.py:742-760,892-897 writes it (flag 4, mapq 255, tags ec:f np:i rq:f RG:Z zm:i). */
typedef struct dcb_bamw dcb_bamw;
int dcb_bamw_open(const char* path, const char* header_text, dcb_bamw** out);
int dcb_bamw_write(dcb_bamw* w, const char* name, const uint8_t* seq, const uint8_t* qual_phred33, int32_t len,
                   int32_t has_ec, float ec, int32_t np_num_passes, float rq, const char* rg);
int dcb_bamw_close(dcb_bamw* w);

/* Device time of the last dcb_forward (milliseconds, CUDA events on the engine's stream). */
int dcb_last_forward_ms(dcb_engine* e, float* ms);
/* Number of engine kernels launched by the last dcb_forward. */
int dcb_last_forward_launches(dcb_engine* e, int32_t* n);

/* Per-kernel timing of the dominant kernel (the fused FFN, or the whole encoder stack when it runs
 * in one launch): when enabled, every ffn_pair_kernel / stack_pair_kernel launch is bracketed by
 * CUDA events on the engine's stream; dcb_get_profile returns the accumulated device time, launch
 * count and tokens processed since dcb_set_profile. */
int dcb_set_profile(dcb_engine* e, int32_t enabled);
int dcb_get_profile(dcb_engine* e, float* ffn_ms_total, int32_t* ffn_launches, int64_t* ffn_tokens);
/* Device time (ms) and launch count per kernel class since dcb_set_profile: [0] embed, [1] row GEMM
 * (condenser / unfused out-proj), [2] QKV GEMM, [3] attention, [4] FFN (+ fused out-proj), [5] head;
 * *fused_oproj = 1 when the attention out-projection runs inside the FFN kernel. */
int dcb_get_profile_kernels(dcb_engine* e, float* ms6, int32_t* n6, int32_t* fused_oproj);

/* Pinned host memory helpers (for callers that want async H2D/D2H). */
int dcb_alloc_host(size_t bytes, void** out);
int dcb_free_host(void* p);
/* Device memory helpers so a host language can keep inputs resident (bench `value`). */
int dcb_alloc_device(dcb_engine* e, size_t bytes, void** out);
int dcb_free_device(dcb_engine* e, void* p);
int dcb_memcpy_h2d(dcb_engine* e, void* dst_dev, const void* src_host, size_t bytes);
int dcb_memcpy_d2h(dcb_engine* e, void* dst_host, const void* src_dev, size_t bytes);
int dcb_synchronize(dcb_engine* e);

const char* dcb_last_error(const dcb_engine* e); /* e may be NULL: last create() error */
const char* dcb_version(void);
void dcb_destroy(dcb_engine* e);

#ifdef __cplusplus
}
#endif
#endif /* DCB200_H_ */

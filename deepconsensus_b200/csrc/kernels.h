// Launchers of the dcb200 device kernels (definitions in kernels.cu).
#pragma once
#include <cuda_runtime.h>

#include "common.h"

namespace dcb {

cudaError_t kernels_init();

size_t embed_smem_bytes(int R, int echunks, int table_elems);
void launch_embed(const float* rows, int R, int L, int Lw, int M, int ntiles, int echunks,
                  const EmbedCol* cols, const EmbedRow* rowmeta, const __nv_bfloat16* tables,
                  int table_elems, __nv_bfloat16* emb, int* status, cudaStream_t st);
// D = A * B^T with the 288-wide row epilogue (condenser + pos-enc, attention out-proj).
void launch_gemm_row(const __nv_bfloat16* a_img, const __nv_bfloat16* b_img, int ksteps, int ntiles,
                     const RowEpi& epi, cudaStream_t st);
// fused q/k/v projection: A [tile][36][128][8] -> qkv image [tile][108][128][8]
void launch_gemm_qkv(const __nv_bfloat16* a_img, const __nv_bfloat16* b_img, int ntiles,
                     __nv_bfloat16* qkv_img, cudaStream_t st);
// fused embedding + condenser (+pos-enc, residual image, next operand); false if it does not fit smem
size_t embed_condense_smem_bytes(int R, int echunks, int table_elems, int packed_stride);
// `packed` != null: read the packed rows (include/dcb200.h) instead of `rows`; only when embed_condense_reads_packed().
bool embed_condense_reads_packed(int L, int Lw);
bool launch_embed_condense(const float* rows, const uint8_t* packed, const PackedLayout& pl, int R, int L, int Lw, int M,
                           int ntiles, int echunks, const EmbedCol* cols,
                           const EmbedRow* rowmeta, const __nv_bfloat16* tables, int table_elems,
                           const __nv_bfloat16* wc_img, const RowEpi& epi, int* status, cudaStream_t st);
void launch_unpack_rows(const uint8_t* packed, const PackedLayout& pl, int nwindows, float* rows, cudaStream_t st);
// fused QKV projection + banded attention on window-aligned tiles (Lw == 128); w_img: per (head, rank)
// [18 k-steps][2][216][8] with rows = [q|k|v] halves
void launch_qkv_attn(const __nv_bfloat16* a_img, const uint8_t* w_img, int ntiles, int L, int win,
                     __nv_bfloat16* att, cudaStream_t st);
void launch_attention(const __nv_bfloat16* qkv, __nv_bfloat16* att, int L, int Lw, int win, int nwindows,
                      cudaStream_t st);
// fused FFN on CTA pairs (cta_group::2); w2img is the per-rank half-chunk weight image.
// With wo2img != null the attention out-projection (+ residual, + pre-norm `mid_ln_*` or identity) is
// fused in front: a_img is then the attention operand image and epi.x the residual before the
// attention sub-layer.
void launch_ffn_pair(const __nv_bfloat16* a_img, const uint8_t* w2img, const float* b1, int ff, int ntiles,
                     const RowEpi& epi, cudaStream_t st, const uint8_t* wo2img = nullptr,
                     const float* mid_ln_g = nullptr, const float* mid_ln_b = nullptr);
// The whole encoder stack in one launch (window-aligned tiles, attn_win_size in [1,16]): x is the fp32 residual
// image written by the embedding kernel.  hp.bases != null: the head (final LayerNorm, fc1, softmax, argmax, Phred,
// calibration, ASCII) runs in the kernel's tail and x is not written back; otherwise x returns the output of the last
// layer for launch_head.
void launch_stack(float* x, int ntiles, int L, int win, const StackParams& p, const HeadParams& hp, cudaStream_t st);
int read_ffn_trace(unsigned long long* out, int n);
void launch_head(const HeadParams& p, int ntiles, cudaStream_t st);
// per-read window concatenation + gap compaction; read z = windows [zmw_start[z], zmw_start[z+1]) (device pointers)
// read z spans bytes [read_off[z], read_off[z + 1]) of bases / quals (and of seq_out / qual_out); int64 offsets
void launch_stitch(const uint8_t* bases, const uint8_t* quals, const int64_t* read_off, int n_zmw,
                   uint8_t* seq_out, uint8_t* qual_out, int32_t* len_out, cudaStream_t st);


// ---- post-model stage on the device (post_kernels.cu); outcome codes: DCB_READ_* of include/dcb200.h
void launch_read_outcome(const uint8_t* qual, const int32_t* len, const int64_t* read_off, const int32_t* zmw_start,
                         const int32_t* window_pos, int L, int n_zmw, const double* p10, double min_quality, int min_length, int32_t* outcome,
                         double* avg_q, cudaStream_t st);
void launch_fastq(const uint8_t* seq, const uint8_t* qual, const int32_t* len, const int64_t* read_off, int n_zmw,
                  const int32_t* outcome, const uint8_t* names, const int32_t* name_off, int64_t* rec_off, uint8_t* fastq,
                  int64_t cap, cudaStream_t st);
void launch_skip_mask(const int16_t* ccs_bq, int n_windows, int L, const double* p10, double thr, uint8_t* mask,
                      double* avg_out, cudaStream_t st);
// skipped window j: source bytes [src_off[j], src_off[j + 1]) of ccs_ids / ccs_bq -> bytes from dst_off[j] of bases / quals
void launch_fill_skipped(const uint8_t* ccs_ids, const int16_t* ccs_bq, const int64_t* src_off, const int64_t* dst_off, int k,
                         int calib_enabled,
                         double thr, double cw, double cb, int max_q, uint8_t* bases, uint8_t* quals, int* status,
                         cudaStream_t st);

// ---- strict-fp32 path (strict_kernels.cu): row-major float32 activations, windows packed back to back
void launch_strict_embed(const float* rows, int R, int L, int E, int nwindows, const StrictEmbedRow* meta,
                         const float* tables, float* emb, int* status, cudaStream_t st);
void launch_strict_gemm(const float* A, const float* B, float* C, int M, int N, int K, const StrictEpi& ep,
                        cudaStream_t st);
void launch_strict_layernorm(const float* x, float* y, int M, const float* g, const float* b, cudaStream_t st);
void launch_strict_attention(const float* q, const float* k, const float* v, float* o, int nwindows, int L, int win,
                             cudaStream_t st);
void launch_strict_head(const float* x, int M, const HeadParams& hp, cudaStream_t st);

}  // namespace dcb

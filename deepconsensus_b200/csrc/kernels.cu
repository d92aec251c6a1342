// dcb200 device kernels (sm_100a).
//
//   embed_rows_kernel   rows f32 [B,R,L] -> concatenated embeddings, bf16 operand image
//                       (format_rows clip + OnDeviceEmbedding gathers + concat + cast;
//                        data_providers.py:151-162, networks.py:42-63,457-507)
//   gemm_kernel         persistent, warp-specialised tcgen05 GEMM: bulk-copy (TMA) producer
//                       warp, single-thread UMMA issuer, 4 epilogue warps reading TMEM.
//                       Used for the condenser (+pos-enc), fused QKV, attention out-proj.
//   embed_condense_kernel  embedding + condenser GEMM in one pass (CTA pairs); the bf16
//                       embedding never goes to HBM
//   ffn_pair_kernel     fused FFN on CTA pairs: relu(x W1 + b1) W2 + b2 with the [128 x 2048]
//                       hidden activation living only in TMEM/SMEM (ffn_layer.py:83-86),
//                       optionally behind the attention out-projection
//   band_attention_kernel  banded multi-head softmax attention (attention_layer.py:198-214)
//   qkv_attn_pair_kernel   fused QKV projection + banded attention on window-aligned tiles
//   stack_pair_kernel   the whole encoder stack (+ head) in one launch (stack_kernel.cuh)
//   head_kernel         final LayerNorm -> fc1 -> softmax -> argmax -> Phred -> ASCII
//                       (encoder_stack.py:197, networks.py:342,238, quick_inference.py:377-414)
//   unpack_rows_kernel  packed rows -> float32 [B, R, L] rows
//   stitch_kernel       per-read window concatenation + gap compaction (stitch_utils.py:51-98)
#include "kernels.h"

#include <cuda_bf16.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include "head_finish.cuh"
#include "sm100.cuh"

namespace dcb {

// cycle-trace hooks (-DDCB_TRACE) and the device buffer scripts/gpu_trace*.py read back
__device__ unsigned long long g_ffn_trace[256 * 16];
#ifdef DCB_TRACE
#define TRACE_T0() long long _t0 = clock64()
#define TRACE_ADD(var) do { long long _t1 = clock64(); (var) += _t1 - _t0; _t0 = _t1; } while (0)
#else
#define TRACE_T0() do {} while (0)
#define TRACE_ADD(var) do {} while (0)
#endif


// =====================================================================================
// embed
// =====================================================================================
// One CTA per 128-token tile.  Phase 1 turns the tile's R x 128 input values into table ids
// (clip -> shift -> truncate -> range check) in shared memory with coalesced loads along L;
// phase 2 assembles 16-byte K-chunks of the operand image from the shared-memory tables.
__global__ void __launch_bounds__(256)
embed_rows_kernel(const float* __restrict__ rows, int R, int L, int Lw, int M, int echunks,
                  const EmbedCol* __restrict__ cols, const EmbedRow* __restrict__ rowmeta,
                  const __nv_bfloat16* __restrict__ tables, int table_elems,
                  __nv_bfloat16* __restrict__ emb, int* __restrict__ status) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __nv_bfloat16* s_tab = reinterpret_cast<__nv_bfloat16*>(smem);
  const int tab_bytes = (table_elems * 2 + 15) & ~15;
  EmbedCol* s_cols = reinterpret_cast<EmbedCol*>(smem + tab_bytes);
  const int cols_bytes = (echunks * 8 * (int)sizeof(EmbedCol) + 15) & ~15;
  uint16_t* s_ids = reinterpret_cast<uint16_t*>(smem + tab_bytes + cols_bytes);  // [R][128]
  const int tile = blockIdx.x;
  for (int i = threadIdx.x; i < table_elems; i += blockDim.x) s_tab[i] = tables[i];
  for (int i = threadIdx.x; i < echunks * 8; i += blockDim.x) s_cols[i] = cols[i];
  for (int idx = threadIdx.x; idx < R * kTileM; idx += blockDim.x) {
    const int rr = idx / kTileM, r = idx % kTileM;
    const int tok = tile * kTileM + r;
    int id = 0;
    if (tok < M) {
      const int b = tok / Lw, l = tok - b * Lw;
      const EmbedRow m = rowmeta[rr];
      float f = l < L ? __ldg(rows + ((size_t)b * R + rr) * L + l) : 0.f;   // window padding rows embed to id 0
      if (m.clip_hi > 0.f) f = fminf(fmaxf(f, 0.f), m.clip_hi);  // format_rows (data_providers.py:151-162)
      f += (float)m.shift;                                         // networks.py:495
      id = (int)f;  // truncation toward zero == tf.cast(float32 -> int32)
      if (id < 0 || id >= m.vocab) {
        atomicOr(status, 1);  // TF's CPU gather raises here; flag and clamp
        id = id < 0 ? 0 : m.vocab - 1;
      }
    }
    s_ids[idx] = (uint16_t)id;
  }
  __syncthreads();
  const int total = echunks * kTileM;
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int kc = idx / kTileM;
    const int r = idx % kTileM;
    uint4 val;
    const EmbedCol c0 = s_cols[kc * 8];
    if (c0.width == 8 && c0.col == 0 && c0.src_row >= 0) {
      // fast path: the whole 16-byte chunk is one width-8 embedding row (bases/pw/ip/ccs/bq/sn)
      const int id = s_ids[c0.src_row * kTileM + r];
      val = *reinterpret_cast<const uint4*>(s_tab + c0.table_off + id * 8);
    } else {
      uint32_t packed[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t pr = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const EmbedCol c = s_cols[kc * 8 + 2 * j + h];
          uint32_t bits = 0;
          if (c.src_row >= 0) {
            const int id = s_ids[c.src_row * kTileM + r];
            bits = __bfloat16_as_ushort(s_tab[c.table_off + id * c.width + c.col]);
          }
          pr |= bits << (16 * h);
        }
        packed[j] = pr;
      }
      val = make_uint4(packed[0], packed[1], packed[2], packed[3]);
    }
    uint4* dst = reinterpret_cast<uint4*>(emb + ((size_t)tile * echunks + kc) * kTileM * 8) + r;
    *dst = val;
  }
}

// =====================================================================================
// row epilogue shared by the d-wide GEMMs (thread == token row)
// =====================================================================================
// acc is read from TMEM columns [tmem_row_base, +288) of this thread's lane.
// Returns after the last TMEM read has completed (caller then releases the accumulator).
template <bool kSecondPassOnly>
__device__ __forceinline__ void row_epilogue_pass2(const RowEpi& e, int tile, int r, float mean,
                                                   float rstd) {
  // LayerNorm normalisation pass: re-read x_new (this thread's own writes) from global.
  const float4* xrow = reinterpret_cast<const float4*>(e.x + (size_t)tile * x_image_elems()) + r;
  uint4* xbrow = reinterpret_cast<uint4*>(e.xb + (size_t)tile * act_image_elems(kDP)) + r;
#pragma unroll 1
  for (int cb = 0; cb < kDP / 8; ++cb) {
    float v[8];
    const float4 a = xrow[(size_t)(cb * 2) * kTileM];
    const float4 b = xrow[(size_t)(cb * 2 + 1) * kTileM];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = cb * 8 + j;
      v[j] = col < kD ? (v[j] - mean) * rstd * __ldg(e.ln_g + col) + __ldg(e.ln_b + col) : 0.f;
    }
    xbrow[(size_t)cb * kTileM] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                            pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  }
}

struct RowStats {
  float mean, rstd;
};

// x_old prefetch for the row epilogue: kRowPF column blocks of 16 floats in flight per thread.
constexpr int kRowPF = 4;
struct RowPrefetch {
  float4 buf[kRowPF][4];
};

__device__ __forceinline__ void row_prefetch_issue(const RowEpi& e, int tile, int r, int cb,
                                                   float4 (&dst)[4]) {
  const float4* xrow = reinterpret_cast<const float4*>(e.x + (size_t)tile * x_image_elems()) + r;
#pragma unroll
  for (int i = 0; i < 4; ++i) dst[i] = xrow[(size_t)(cb * 4 + i) * kTileM];
}

// Issue the first kRowPF blocks (call before waiting for the accumulator).
__device__ __forceinline__ void row_prefetch_start(const RowEpi& e, int tile, int r, RowPrefetch& pf) {
  if (e.has_xold) {
#pragma unroll
    for (int k = 0; k < kRowPF; ++k) row_prefetch_issue(e, tile, r, k, pf.buf[k]);
  } else if (e.pe) {
    // no residual input (the condenser GEMM): the registers carry the token's positional-encoding row instead
    if (e.pe_img) {
      const float4* pi = reinterpret_cast<const float4*>(e.pe_img) + r;
#pragma unroll
      for (int k = 0; k < kRowPF; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) pf.buf[k][i] = __ldg(pi + (size_t)(k * 4 + i) * kTileM);
    } else {
      const int l = (tile * kTileM + r) % e.L;
      const float4* pr = reinterpret_cast<const float4*>(e.pe + (size_t)l * kDP);
#pragma unroll
      for (int k = 0; k < kRowPF; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) pf.buf[k][i] = __ldg(pr + k * 4 + i);
    }
  }
}

__device__ __forceinline__ RowStats row_epilogue_pass1(const RowEpi& e, uint32_t tmem_row_base,
                                                       int tile, int r, RowPrefetch& pf,
                                                       long long* t_ldtm = nullptr) {
  const int tok = tile * kTileM + r;
  const int l = tok % e.L;
  float4* xrow = reinterpret_cast<float4*>(e.x + (size_t)tile * x_image_elems()) + r;
  uint4* xbrow = e.xb ? reinterpret_cast<uint4*>(e.xb + (size_t)tile * act_image_elems(kDP)) + r
                      : nullptr;
  const bool ln = e.ln_g != nullptr;
  float s1 = 0.f, s2 = 0.f, shift = 0.f;
  // Compact loop on purpose: fully unrolled (18 blocks x every predicated residual / pos-enc / bias / LayerNorm variant)
  // this function was thousands of straight-line instructions and its warps stalled on instruction fetch (ncu:
  // stall_no_inst).  Groups of kRowPF blocks keep the prefetch-buffer indices static.
  static_assert(kRowPF == 4, "the block loop is unrolled by the prefetch depth");
#pragma unroll 1
  for (int cg = 0; cg < kDP / 16; cg += kRowPF) {
#pragma unroll
  for (int cj = 0; cj < kRowPF; ++cj) {
    const int cb = cg + cj;
    if (cb >= kDP / 16) break;
    uint32_t acc[16];
#ifdef DCB_TRACE
    const long long _tl0 = clock64();
#endif
    tmem_ld16(tmem_row_base + cb * 16, acc);
    float v[16];
    if (e.has_xold) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 t = pf.buf[cj][i];
        v[4 * i + 0] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
      }
      if (cb + kRowPF < kDP / 16) row_prefetch_issue(e, tile, r, cb + kRowPF, pf.buf[cj]);
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = 0.f;
    }
    tmem_ld_wait();
#ifdef DCB_TRACE
    if (t_ldtm) *t_ldtm += clock64() - _tl0;
#endif
    float pev[16];
    if (e.pe) {
      // one token's 16 positional values are 64 contiguous bytes: 4 x 128-bit loads (rows differ per lane, so every
      // load is its own L2 round trip).  Without a residual to read (the embedding GEMM) the RowPrefetch registers
      // carry the positional rows instead, kRowPF blocks ahead (row_prefetch_start).
      const float4* pr = reinterpret_cast<const float4*>(e.pe + (size_t)l * kDP + cb * 16);
      if (!e.has_xold) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 t = pf.buf[cj][i];
          pev[4 * i + 0] = t.x; pev[4 * i + 1] = t.y; pev[4 * i + 2] = t.z; pev[4 * i + 3] = t.w;
        }
        if (cb + kRowPF < kDP / 16) {
          if (e.pe_img) {
            const float4* pi = reinterpret_cast<const float4*>(e.pe_img) + r;
#pragma unroll
            for (int i = 0; i < 4; ++i) pf.buf[cj][i] = __ldg(pi + (size_t)((cb + kRowPF) * 4 + i) * kTileM);
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) pf.buf[cj][i] = __ldg(pr + kRowPF * 4 + i);
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 t = __ldg(pr + i);
          pev[4 * i + 0] = t.x; pev[4 * i + 1] = t.y; pev[4 * i + 2] = t.z; pev[4 * i + 3] = t.w;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int col = cb * 16 + i;
      float t = v[i] + __uint_as_float(acc[i]);
      if (e.bias) t += __ldg(e.bias + col);
      if (e.pe) t += pev[i];
      v[i] = col < kD ? t : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
      xrow[(size_t)(cb * 4 + i) * kTileM] =
          make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    if (ln) {
      if (cb == 0) shift = v[0];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float dlt = (cb * 16 + i < kD) ? v[i] - shift : 0.f;
        s1 += dlt;
        s2 += dlt * dlt;
      }
    } else if (xbrow) {
      xbrow[(size_t)(cb * 2) * kTileM] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                                    pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      xbrow[(size_t)(cb * 2 + 1) * kTileM] =
          make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]),
                     pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
    }
  }
  }
  RowStats st;
  const float m1 = s1 * (1.f / kD);
  const float var = fmaxf(s2 * (1.f / kD) - m1 * m1, 0.f);
  st.mean = shift + m1;
  st.rstd = rsqrtf(var + 1e-6f);
  return st;
}

// Lean form of the row epilogue for the embedding / condenser GEMM in front of the one-kernel stack: no residual
// input, no bias, no LayerNorm, no bf16 operand image -- x = acc + positional table (image order), nothing else.
// A small loop body (the general function carries every predicated variant and stalls on instruction fetch).
// The 288 accumulator columns come from two 144-column TMEM regions (col0: columns 0..143, col1: 144..287); `free0` is
// arrived on (one lane per warp) as soon as the first region has been read, so the next tile's UMMAs may overwrite it
// while the second half of this tile is still being stored.
__device__ __forceinline__ void row_epilogue_embed_lean(const RowEpi& e, uint32_t tmem_row_base, int tile, int r,
                                                        uint32_t col0, uint32_t col1, uint64_t* free0) {
  float4* xrow = reinterpret_cast<float4*>(e.x + (size_t)tile * x_image_elems()) + r;
  const float4* pi = reinterpret_cast<const float4*>(e.pe_img) + r;
  // two register buffers: the tcgen05.ld and the positional rows of block cb + 1 are in flight while block cb is stored
  uint32_t a[16], b[16];
  float4 pa[4], pb[4];
  auto fetch = [&](uint32_t (&acc)[16], float4 (&p)[4], int cb) {
    tmem_ld16(tmem_row_base + (cb < kNC / 16 ? col0 + cb * 16 : col1 + (cb - kNC / 16) * 16), acc);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#ifdef DCB_EXP_NOPE
      p[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#else
      p[i] = __ldg(pi + (size_t)(cb * 4 + i) * kTileM);
#endif
  };
  auto emit = [&](const uint32_t (&acc)[16], const float4 (&p)[4], int cb) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int col = cb * 16 + 4 * i;
      float4 o;
      o.x = col + 0 < kD ? __uint_as_float(acc[4 * i + 0]) + p[i].x : 0.f;
      o.y = col + 1 < kD ? __uint_as_float(acc[4 * i + 1]) + p[i].y : 0.f;
      o.z = col + 2 < kD ? __uint_as_float(acc[4 * i + 2]) + p[i].z : 0.f;
      o.w = col + 3 < kD ? __uint_as_float(acc[4 * i + 3]) + p[i].w : 0.f;
#ifdef DCB_EXP_NOSTORE
      if (o.x == 123.456f)
#endif
      xrow[(size_t)(cb * 4 + i) * kTileM] = o;
    }
  };
  static_assert((kDP / 16) % 2 == 0, "block pairs");
  fetch(a, pa, 0);
#pragma unroll 1
  for (int cb = 0; cb < kDP / 16; cb += 2) {
    tmem_ld_wait();
    if (cb == kNC / 16 - 1) {             // block 8 = the last one of the first region is in registers
      tc_fence_before();
      __syncwarp();
      if ((threadIdx.x & 31) == 0) mbar_arrive(free0);
    }
    fetch(b, pb, cb + 1);
    emit(a, pa, cb);
    tmem_ld_wait();
    if (cb + 2 < kDP / 16) fetch(a, pa, cb + 2);
    emit(b, pb, cb + 1);
  }
  static_assert((kNC / 16 - 1) % 2 == 0, "the first region ends on an even block");
}

// =====================================================================================
// generic persistent tcgen05 GEMM
// =====================================================================================
// D[128 x (NCH*144)] = A[128 x K] * B^T, A image [tile][K/8][128][8], B image per n-group
// [K/8][NCH*144][8].  One work item = (tile, n-group).
//
// EPI_QKV : store bf16 into the qkv operand image (column offset group*NCH*144)
// EPI_ROW : row epilogue (residual / bias / pos-enc / LayerNorm), NCH must be 2
enum { EPI_QKV = 0, EPI_ROW = 1 };

template <int NCH>
struct GemmCfg {
  static constexpr int kNItem = NCH * kNC;
  static constexpr int kSK = 2;                                  // k-steps per stage
  static constexpr int kABytesPerK = 2 * kTileM * 16;            // 4096
  static constexpr int kBBytesPerK = 2 * kNItem * 16;
  static constexpr int kStageBytes = kSK * (kABytesPerK + kBBytesPerK);
  static constexpr int kStages = 4;
  static constexpr int kTmemCols = 512;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024;
};

template <int NCH, int EPI>
__global__ void __launch_bounds__(192, 1)
gemm_kernel(const __nv_bfloat16* __restrict__ a_img, const __nv_bfloat16* __restrict__ b_img,
            int ksteps, int ntiles, int ngroups, __nv_bfloat16* __restrict__ out_img,
            int out_chunks, RowEpi epi) {
  using Cfg = GemmCfg<NCH>;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* stage_base = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* full = bars;                      // [kStages]
  uint64_t* empty = bars + Cfg::kStages;      // [kStages]
  uint64_t* acc_full = bars + 2 * Cfg::kStages;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(acc_empty + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < Cfg::kStages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 128);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_holder, Cfg::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  const int nitems = ntiles * ngroups;
  const int kstages = (ksteps + Cfg::kSK - 1) / Cfg::kSK;
  const size_t a_tile_bytes = (size_t)ksteps * Cfg::kABytesPerK;
  const size_t b_group_bytes = (size_t)ksteps * Cfg::kBBytesPerK;

  if (warp == 0) {
    // ------------------------------------------------------------- producer
    if (lane == 0) {
      uint32_t slot = 0, phase = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int tile = item / ngroups, grp = item % ngroups;
        const uint8_t* a_src = reinterpret_cast<const uint8_t*>(a_img) + tile * a_tile_bytes;
        const uint8_t* b_src = reinterpret_cast<const uint8_t*>(b_img) + grp * b_group_bytes;
        for (int s = 0; s < kstages; ++s) {
          const int kh = min(Cfg::kSK, ksteps - s * Cfg::kSK);
          mbar_wait(&empty[slot], phase ^ 1);
          uint8_t* sa = stage_base + slot * Cfg::kStageBytes;
          uint8_t* sb = sa + Cfg::kSK * Cfg::kABytesPerK;
          mbar_arrive_expect_tx(&full[slot], kh * (Cfg::kABytesPerK + Cfg::kBBytesPerK));
          bulk_g2s(sa, a_src + (size_t)s * Cfg::kSK * Cfg::kABytesPerK, kh * Cfg::kABytesPerK,
                   &full[slot]);
          bulk_g2s(sb, b_src + (size_t)s * Cfg::kSK * Cfg::kBBytesPerK, kh * Cfg::kBBytesPerK,
                   &full[slot]);
          if (++slot == Cfg::kStages) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------- MMA issuer (whole warp; the elected lane issues)
    {
      constexpr uint32_t idesc = make_idesc_bf16(kTileM, kNC);
      uint32_t slot = 0, phase = 0, it = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
        mbar_wait(acc_empty, (it & 1) ^ 1);
        tc_fence_after();
        for (int s = 0; s < kstages; ++s) {
          const int kh = min(Cfg::kSK, ksteps - s * Cfg::kSK);
          mbar_wait(&full[slot], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(stage_base + slot * Cfg::kStageBytes);
          const uint32_t sb = sa + Cfg::kSK * Cfg::kABytesPerK;
          for (int kk = 0; kk < kh; ++kk) {
            const uint64_t adesc = make_kc16_desc(sa + kk * Cfg::kABytesPerK, kTileM * 16, 128);
#pragma unroll
            for (int j = 0; j < NCH; ++j) {
              const uint64_t bdesc = make_kc16_desc(sb + kk * Cfg::kBBytesPerK + j * kNC * 16,
                                                    Cfg::kNItem * 16, 128);
              umma_bf16_ss_warp(tmem_base + j * kNC, adesc, bdesc, idesc, (s | kk) != 0);
            }
          }
          umma_commit_warp(&empty[slot]);
          if (++slot == Cfg::kStages) { slot = 0; phase ^= 1; }
        }
        umma_commit_warp(acc_full);
      }
    }
  } else {
    // ------------------------------------------------------------- epilogue (4 warps)
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;       // token row within the tile
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t it = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
      const int tile = item / ngroups, grp = item % ngroups;
      RowPrefetch pf;
      if constexpr (EPI == EPI_ROW) row_prefetch_start(epi, tile, r, pf);
      mbar_wait(acc_full, it & 1);
      tc_fence_after();
      if constexpr (EPI == EPI_QKV) {
        uint4* orow = reinterpret_cast<uint4*>(out_img + (size_t)tile * kTileM * out_chunks * 8) + r;
#pragma unroll 1
        for (int cb = 0; cb < Cfg::kNItem / 16; ++cb) {
          uint32_t acc[16];
          tmem_ld16(tmem_row + cb * 16, acc);
          tmem_ld_wait();
          float v[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(acc[i]);
          const int kc = (grp * Cfg::kNItem + cb * 16) / 8;
          orow[(size_t)kc * kTileM] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                                 pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
          orow[(size_t)(kc + 1) * kTileM] =
              make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]),
                         pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
        }
        tc_fence_before();
        mbar_arrive(acc_empty);
      } else {
        static_assert(EPI != EPI_ROW || NCH == 2, "row epilogue needs the full 288-wide row");
        const RowStats st = row_epilogue_pass1(epi, tmem_row, tile, r, pf);
        tc_fence_before();
        mbar_arrive(acc_empty);   // accumulator free: next item's MMAs overlap the LN pass
        if (epi.ln_g && epi.xb) row_epilogue_pass2<false>(epi, tile, r, st.mean, st.rstd);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// =====================================================================================
// fused embedding + condenser
// =====================================================================================
// Builds the concatenated-embedding operand (networks.py:457-507) straight into shared memory, K-slab
// by K-slab, and multiplies it with the condenser weights (networks.py:426-434) -- the [tokens x E]
// bf16 embedding never goes to HBM.  Roles: warp 0 streams condenser-weight slabs (bulk copies), warp 1
// issues the UMMAs, warps 2-9 turn the tile's R x 128 input values into table ids (format_rows clip,
// shift, truncate, range check) and then assemble 16-byte K-chunks of each slab from the shared-memory
// tables, warps 10-13 run the row epilogue (+positional encoding, fp32 residual image, next sub-layer's
// bf16 operand / LayerNorm).
struct EmbCfg {
  static constexpr int kSlabK = 5;                                   // k-steps per A slab / B stage
  static constexpr int kASlabBytes = kSlabK * 2 * kTileM * 16;       // 20480
  static constexpr int kBSlabBytes = kSlabK * 2 * kDP * 16;          // 46080
  static constexpr int kBuilders = 384;  // builder threads (12 warps: their id / slab phases are latency-bound, 0.3 IPC per
                                         // scheduler with 8 warps -- more warps, not more work per warp, is what helps)
  static constexpr int kChunkGroups = kBuilders / kTileM;              // 3: thread = (row, chunk group)
  static constexpr int kItems = (2 * kSlabK + kChunkGroups - 1) / kChunkGroups;   // 4 chunks per thread and slab at most
  static constexpr int kThreads = 128 + kBuilders + 128;   // {producer, UMMA, 2 service warps}, builders, row epilogue
  static constexpr int kTmemCols = 512;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(EmbCfg::kThreads, 1)
embed_condense_kernel(const float* __restrict__ rows, const uint8_t* __restrict__ packed, PackedLayout pl, int R, int L,
                      int Lw, int M, int ntiles, int echunks,
                      const EmbedCol* __restrict__ cols, const EmbedRow* __restrict__ rowmeta,
                      const __nv_bfloat16* __restrict__ tables, int table_elems,
                      const __nv_bfloat16* __restrict__ wc_img, RowEpi epi, int* __restrict__ status) {
  using C = EmbCfg;
  extern __shared__ __align__(1024) uint8_t smem[];
#ifdef DCB_TRACE
  const long long t_entry = clock64();
#endif
  const int tab_bytes = (table_elems * 2 + 127) & ~127;
  const int cols_only = (echunks * 8 * (int)sizeof(EmbedCol) + 15) & ~15;
  const int cols_bytes = (cols_only + echunks * 8 + 127) & ~127;          // + one 8-byte descriptor per K-chunk
  const int ids_bytes = (R * kTileM * 2 + 127) & ~127;
  __nv_bfloat16* s_tab = reinterpret_cast<__nv_bfloat16*>(smem);
  EmbedCol* s_cols = reinterpret_cast<EmbedCol*>(smem + tab_bytes);
  // per 16-byte K-chunk: .x = source row | kind << 16 | width << 24, .y = table offset (elements).  kind 0: zeros,
  // 1: one row of a width-8 table, 3: 8 / width consecutive rows of one width-2 / width-4 table, 2: anything else
  uint2* s_chunk = reinterpret_cast<uint2*>(smem + tab_bytes + cols_only);
  uint16_t* s_ids = reinterpret_cast<uint16_t*>(smem + tab_bytes + cols_bytes);
  // packed rows: the next window's bytes are staged here by one bulk copy while the current tile's slabs are built, so
  // the id phase reads shared memory instead of waiting on dependent batches of global loads
  const int raw_bytes = packed ? ((pl.stride + 127) & ~127) : 0;
  uint8_t* s_raw = smem + tab_bytes + cols_bytes + ids_bytes;
  uint8_t* sAslab = smem + ((tab_bytes + cols_bytes + ids_bytes + raw_bytes + 1023) & ~1023);
  uint8_t* sB = sAslab + 2 * C::kASlabBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + 2 * C::kBSlabBytes);
  uint64_t* a_full = bars;          // [2] builders -> MMA
  uint64_t* a_empty = bars + 2;     // [2] MMA -> builders
  uint64_t* b_full = bars + 4;      // [2]
  uint64_t* b_empty = bars + 6;     // [2]
  uint64_t* acc_full = bars + 8;
  uint64_t* acc_empty = bars + 9;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 10);
  uint64_t* raw_full = bars + 11;   // bulk copy -> builders
  uint64_t* raw_empty = bars + 12;  // builders -> copy issuer
  // Accumulator: three 144-column TMEM regions; a tile's two column halves take regions (2 it) % 3 and (2 it + 1) % 3 of
  // the CTA's it-th tile, so the region the epilogue reads LAST is not needed by the next tile and the one it reads FIRST is
  // released half way through -- the next tile's UMMAs start under the second half of the epilogue (lean epilogue only;
  // the general row epilogue keeps regions 0 and 1 and releases both at its end).
  uint64_t* reg_free = bars + 13;   // [3] epilogue -> UMMA issuer
  const bool lean = !epi.has_xold && epi.pe_img && !epi.bias && !epi.ln_g && !epi.xb;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ksteps = echunks / 2;
  const int nslabs = (ksteps + C::kSlabK - 1) / C::kSlabK;
  // CTA pairs share the condenser-weight stream: each CTA fetches half of every slab and multicasts it to both (an SM
  // ingests only 30-50 B/cycle from L2, and 322 KB of weights per 128-token tile made that the pace of the slab loop).
  // Both CTAs of a pair therefore run the same number of rounds; a CTA whose tile index falls past the end rebuilds the
  // last tile and drops the result.
  const uint32_t rank = cluster_ctarank();
  const int rounds = (ntiles + (int)gridDim.x - 1) / (int)gridDim.x;
  auto tile_of = [&](int ti) { return min(ti * (int)gridDim.x + (int)blockIdx.x, ntiles - 1); };
  auto tile_valid = [&](int ti) { return ti * (int)gridDim.x + (int)blockIdx.x < ntiles; };

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_full[i], C::kBuilders / 32);     // one arrive per builder warp
      mbar_init(&a_empty[i], 1);
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 2);    // the UMMA warps of both CTAs of the pair
    }
    mbar_init(raw_full, 1);
    mbar_init(raw_empty, 1);
    mbar_init(acc_full, 1);
    for (int i = 0; i < 3; ++i) mbar_init(&reg_free[i], 4);   // one arrive per epilogue warp
    mbar_fence_init();
  }
  // tables (the blob is padded to 8 elements per table, the device allocation is 256-byte aligned) and column
  // descriptors with wide copies
  {
    const int nvec = table_elems / 8;
    const uint4* tv = reinterpret_cast<const uint4*>(tables);
    for (int i = threadIdx.x; i < nvec; i += blockDim.x) reinterpret_cast<uint4*>(s_tab)[i] = __ldg(tv + i);
    for (int i = nvec * 8 + threadIdx.x; i < table_elems; i += blockDim.x) s_tab[i] = tables[i];
    // column descriptors: 8 per K-chunk = 160 bytes = ten 16-byte words (the device allocation is 256-byte aligned)
    static_assert((8 * sizeof(EmbedCol)) % 16 == 0, "EmbedCol is copied in 16-byte words");
    const uint4* cv = reinterpret_cast<const uint4*>(cols);
    const int nw = echunks * (int)(8 * sizeof(EmbedCol) / 16);
    for (int i = threadIdx.x; i < nw; i += blockDim.x) reinterpret_cast<uint4*>(s_cols)[i] = __ldg(cv + i);
  }
  __shared__ EmbedRow s_meta[160];                 // per input row: clip / shift / vocabulary (R <= 160: max_passes <= 38)
  const EmbedRow* __restrict__ rmeta = R <= 160 ? s_meta : rowmeta;
  if (R <= 160) for (int i = threadIdx.x; i < R; i += blockDim.x) s_meta[i] = rowmeta[i];
  if (warp == 1) tmem_alloc(tmem_holder, C::kTmemCols);
  __syncthreads();
  for (int kc = threadIdx.x; kc < echunks; kc += blockDim.x) {
    const EmbedCol* cc = s_cols + kc * 8;
    const EmbedCol c0 = cc[0];
    uint32_t kind = 2;
    bool none = true;
    for (int j = 0; j < 8; ++j) none = none && cc[j].src_row < 0;
    if (none) kind = 0;
    else if (c0.src_row >= 0 && c0.col == 0 && c0.width == 8) kind = 1;
    else if (c0.src_row >= 0 && c0.col == 0 && (c0.width == 2 || c0.width == 4)) {
      bool ok = true;
      for (int j = 0; j < 8; ++j)
        ok = ok && cc[j].src_row == c0.src_row + j / c0.width && cc[j].col == j % c0.width && cc[j].width == c0.width &&
             cc[j].table_off == c0.table_off;
      if (ok) kind = 3;
    }
    s_chunk[kc] = make_uint2((uint32_t)(uint16_t)c0.src_row | (kind << 16) | ((uint32_t)c0.width << 24), (uint32_t)c0.table_off);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();               // the partner's barriers are initialised before any multicast lands
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp < 4) {
   setmaxnreg_dec<56>();
   if (warp == 0) {
    // ------------------------------------------------------------- condenser-weight producer
    if (lane == 0) {
      uint32_t n = 0;
      for (int ti = 0; ti < rounds; ++ti)
        for (int sl = 0; sl < nslabs; ++sl, ++n) {
          const uint32_t b = n & 1;
          const int kh = min(C::kSlabK, ksteps - sl * C::kSlabK);
          const uint32_t half = (uint32_t)kh * kDP * 16;           // this CTA's half of the slab (multiple of 16 bytes)
          mbar_wait(&b_empty[b], ((n >> 1) & 1) ^ 1);              // slot free in BOTH CTAs
          mbar_arrive_expect_tx(&b_full[b], 2 * half);
          bulk_g2s_multicast(sB + b * C::kBSlabBytes + rank * half,
                             reinterpret_cast<const uint8_t*>(wc_img) + (size_t)sl * C::kBSlabBytes + rank * half, half,
                             &b_full[b], (uint16_t)3);
        }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------- UMMA issuer (whole warp, elected lane issues)
    {
      constexpr uint32_t idesc = make_idesc_bf16(kTileM, kNC);
      uint32_t n = 0, it = 0, par = 0;      // par: bit r = parity of region r's acquisitions
      for (int ti = 0; ti < rounds; ++ti, ++it) {
        const uint32_t rot = lean ? it : 0u;
        const uint32_t jr[2] = {(2 * rot) % 3, (2 * rot + 1) % 3};
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          mbar_wait(&reg_free[jr[j]], ((par >> jr[j]) & 1) ^ 1);
          par ^= 1u << jr[j];
        }
        tc_fence_after();
        for (int sl = 0; sl < nslabs; ++sl, ++n) {
          const uint32_t b = n & 1;
          const int kh = min(C::kSlabK, ksteps - sl * C::kSlabK);
          mbar_wait(&a_full[b], (n >> 1) & 1);
          mbar_wait(&b_full[b], (n >> 1) & 1);
          tc_fence_after();
          const uint32_t sa = smem_u32(sAslab + b * C::kASlabBytes);
          const uint32_t sb = smem_u32(sB + b * C::kBSlabBytes);
          for (int kk = 0; kk < kh; ++kk) {
            const uint64_t adesc = make_kc16_desc(sa + kk * 4096, kTileM * 16, 128);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              const uint64_t bdesc = make_kc16_desc(sb + kk * (2 * kDP * 16) + j * kNC * 16, kDP * 16, 128);
              umma_bf16_ss_warp(tmem_base + jr[j] * kNC, adesc, bdesc, idesc, (sl | kk) != 0);
            }
          }
          umma_commit_warp(&a_empty[b]);
          umma_commit_multicast_warp(&b_empty[b], (uint16_t)3);
        }
        umma_commit_warp(acc_full);
      }
    }
   } else {
    // warps 2-3 (otherwise idle): pull the NEXT tile's input rows into L2 -- the builders' id phase is a chain of
    // dependent global-load batches and runs at L2 instead of HBM latency that way.  One tile ahead (paced by acc_full).
    const int pt = threadIdx.x - 64;   // 0..63
    uint32_t it = 0;
    if (packed) {
      // one bulk copy per round, a round ahead: window of round ti goes out as soon as the id phase of round ti - 1 is over
      if (pt == 0)
        for (int ti = 0; ti < rounds; ++ti) {
          if (ti > 0) mbar_wait(raw_empty, (ti - 1) & 1);
          mbar_arrive_expect_tx(raw_full, (uint32_t)pl.stride);
          bulk_g2s(s_raw, packed + (size_t)tile_of(ti) * pl.stride, (uint32_t)pl.stride, raw_full);
        }
    } else
    for (int ti = 0; ti < rounds; ++ti, ++it) {
      const int nxt = (ti + 1) * (int)gridDim.x + (int)blockIdx.x;
      if (nxt < ntiles) {
        const int w_lo = (nxt * kTileM) / Lw;
        int w_hi = (nxt * kTileM + kTileM - 1) / Lw;
        const int nwin = (M + Lw - 1) / Lw;
        if (w_hi > nwin - 1) w_hi = nwin - 1;
        const uint8_t* base = reinterpret_cast<const uint8_t*>(rows + (size_t)w_lo * R * L);
        const size_t bytes = (size_t)(w_hi - w_lo + 1) * R * L * sizeof(float);
        for (size_t off = (size_t)pt * 128; off < bytes; off += 64 * 128)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
      }
      mbar_wait(acc_full, it & 1);
    }
   }
  } else if (warp < 4 + C::kBuilders / 32) {
    setmaxnreg_dec<80>();
    // ------------------------------------------------------------- builders (384 threads)
    const int bt = threadIdx.x - 128;   // 0..255
    uint32_t n = 0;
    long long t_ids = 0, t_aempty = 0, t_build = 0;
    const long long t_begin = clock64();
    for (int ti = 0; ti < rounds; ++ti) {
      const int tile = tile_of(ti);
      TRACE_T0();
      // every slab of the previous tile has been built (program order), but its last reads of s_ids
      // happen in other builder threads: synchronise the builders before overwriting the ids
      asm volatile("bar.sync 1, %0;" ::"n"(C::kBuilders) : "memory");
      if (packed) {
        // Packed rows (include/dcb200.h; launcher guarantees Lw == kTileM and L % 4 == 0): the window is
        // [3P+1+bq][L] bytes + four SN floats.  Item = (plane row pr, 4 consecutive positions) = one 32-bit load; a
        // warp reads 128 contiguous bytes.  Ids are what tf.cast(format_rows(value)) would give for the float32 rows
        // the packed form stands for (data_providers.py:151-162, networks.py:457-507).
        const bool wvalid = (size_t)tile * kTileM < (size_t)M;
        mbar_wait(raw_full, ti & 1);                     // this round's window is in shared memory
        const uint8_t* wbase = s_raw;
        const uint32_t* base32 = reinterpret_cast<const uint32_t*>(wbase);
        const int P = pl.P, PR = 3 * P + 1 + pl.bq, L4 = L >> 2;
        const int nitems = (PR * 32 + C::kBuilders - 1) / C::kBuilders;
        auto load_item = [&](int k) -> uint32_t {
          const int item = bt + k * C::kBuilders;
          const int pr = item >> 5, g = item & 31;
          if (k < nitems && pr < PR && wvalid && g < L4) return base32[pr * L4 + g];
          return 0u;
        };
        uint32_t f0 = load_item(0), f1 = load_item(1), f2 = load_item(2);
#pragma unroll 1
        for (int k = 0; k < nitems; ++k) {
          const uint32_t cur = f0;
          f0 = f1; f1 = f2; f2 = load_item(k + 3);
          const int item = bt + k * C::kBuilders;
          const int pr = item >> 5, g = item & 31;
          if (pr < PR) {
            // reference row this plane feeds (a base|strand byte feeds two)
            const int ru = pr < 3 * P ? pr : (pr == 3 * P ? 4 * P : 4 * P + 1);
            // (shared-memory copy of the row descriptors whenever it exists: a plain LDS instead of a generic load)
            const EmbedRow m = R <= 160 ? s_meta[ru] : rowmeta[ru];
            // the item's four bytes at once (byte-wise SIMD): clip, range check, clamp, then widen to 16-bit ids
            const uint32_t vmax = (uint32_t)min(m.vocab - 1, 255) * 0x01010101u;
            uint32_t idv, bad;
            if (pr < P) {
              const int sv = R <= 160 ? s_meta[3 * P + pr].vocab : rowmeta[3 * P + pr].vocab;
              const uint32_t svmax = (uint32_t)min(sv - 1, 255) * 0x01010101u;
              uint32_t sidv = (cur >> 3) & 0x03030303u;
              idv = cur & 0x07070707u;
              bad = (cur & 0xe0e0e0e0u) | __vcmpgtu4(idv, vmax) | __vcmpgtu4(sidv, svmax);
              sidv = __vminu4(sidv, svmax);
              *reinterpret_cast<uint2*>(&s_ids[(3 * P + pr) * kTileM + 4 * g]) =
                  make_uint2(__byte_perm(sidv, 0u, 0x4140), __byte_perm(sidv, 0u, 0x4342));
            } else {
              const uint32_t hi4 = (m.clip_hi > 0.f ? (uint32_t)min((int)m.clip_hi, 255) : 255u) * 0x01010101u;
              idv = __vminu4(cur, hi4);
              bad = __vcmpgtu4(idv, vmax);
            }
            idv = __vminu4(idv, vmax);
            if (bad) atomicOr(status, 1);
            *reinterpret_cast<uint2*>(&s_ids[ru * kTileM + 4 * g]) =
                make_uint2(__byte_perm(idv, 0u, 0x4140), __byte_perm(idv, 0u, 0x4342));
          }
        }
        if (bt < 128) {
          // the four SN rows: one value per window, repeated along L (pre_lib.py:741-742)
          const int ri = bt >> 5, g = bt & 31, ru = R - 4 + ri;
          uint32_t id = 0;
          if (wvalid && g < L4) {
            const EmbedRow m = rmeta[ru];
            float v = reinterpret_cast<const float*>(wbase + pl.sn_off)[ri];
            if (m.clip_hi > 0.f) v = fminf(fmaxf(v, 0.f), m.clip_hi);
            v += (float)m.shift;
            int iv = (int)v;
            if (iv < 0 || iv >= m.vocab) { atomicOr(status, 1); iv = iv < 0 ? 0 : m.vocab - 1; }
            id = (uint32_t)iv;
          }
          *reinterpret_cast<uint2*>(&s_ids[ru * kTileM + 4 * g]) = make_uint2(id | (id << 16), id | (id << 16));
        }
      } else if (Lw == kTileM && (L & 3) == 0) {
        // window-aligned layout (tile == window): the tile's input is one contiguous [R][L] block.  Item = (row ru,
        // 4 consecutive positions): all of a thread's ~11 float4 loads are issued before the first is used (one
        // exposed memory latency instead of six dependent batches), a warp reads 512 contiguous bytes.
        const bool wvalid = (size_t)tile * kTileM < (size_t)M;
        const float4* base4 = reinterpret_cast<const float4*>(rows + (size_t)(wvalid ? tile : 0) * R * L);
        const int nitems = (R * 32 + C::kBuilders - 1) / C::kBuilders;
        auto load_item = [&](int k) -> float4 {
          const int item = bt + k * C::kBuilders;
          const int ru = item >> 5, g = item & 31;
          if (k < nitems && ru < R && wvalid && 4 * g < L) return __ldg(base4 + ((size_t)ru * L + 4 * g) / 4);
          return make_float4(0.f, 0.f, 0.f, 0.f);
        };
        // Compact loop with the loads of the next three items in flight.  (A fully unrolled variant with all ~11 loads
        // issued up front had the shorter id phase, 12.0 k vs 14.2 k cycles per tile, but the larger kernel: 0.147 vs
        // 0.127 ms -- its instruction footprint slowed every other phase of the kernel.)
        float4 f0 = load_item(0), f1 = load_item(1), f2 = load_item(2);
#pragma unroll 1
        for (int k = 0; k < nitems; ++k) {
          const float4 cur = f0;
          f0 = f1; f1 = f2; f2 = load_item(k + 3);
          const int item = bt + k * C::kBuilders;
          const int ru = item >> 5, g = item & 31;
          if (ru < R) {
            const EmbedRow m = rmeta[ru];
            const float vals[4] = {cur.x, cur.y, cur.z, cur.w};
            uint32_t ids[4];
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              int id = 0;
              if (wvalid && 4 * g + q4 < L) {
                float v = vals[q4];
                if (m.clip_hi > 0.f) v = fminf(fmaxf(v, 0.f), m.clip_hi);  // format_rows (data_providers.py:151-162)
                v += (float)m.shift;                                         // networks.py:495
                id = (int)v;                                                 // tf.cast(float32 -> int32) truncates
                if (id < 0 || id >= m.vocab) {
                  atomicOr(status, 1);
                  id = id < 0 ? 0 : m.vocab - 1;
                }
              }
              ids[q4] = (uint32_t)id;
            }
            *reinterpret_cast<uint2*>(&s_ids[ru * kTileM + 4 * g]) = make_uint2(ids[0] | (ids[1] << 16), ids[2] | (ids[3] << 16));
          }
        }
      } else {
        // thread = (token r, input rows rr0, rr0 + G, ...; G = 3 row groups): 8 independent global loads in flight per batch
        constexpr int G = C::kChunkGroups;
        const int r = bt & (kTileM - 1), rr0 = bt >> 7;
        const int tok = tile * kTileM + r;
        const int bw0 = tok / Lw, l0 = tok - bw0 * Lw;
        const bool tvalid = tok < M && l0 < L;      // layout padding (l >= L) embeds to id 0 everywhere
        const int bw = tvalid ? bw0 : 0, l = tvalid ? l0 : 0;
        const float* base = rows + (size_t)bw * R * L + l;
        for (int rr = rr0; rr < R; rr += 8 * G) {
          float f[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int ru = rr + G * u;
            f[u] = (tvalid && ru < R) ? __ldg(base + (size_t)ru * L) : 0.f;
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int ru = rr + G * u;
            if (ru < R) {
              int id = 0;
              if (tvalid) {
                const EmbedRow m = rmeta[ru];
                float v = f[u];
                if (m.clip_hi > 0.f) v = fminf(fmaxf(v, 0.f), m.clip_hi);  // format_rows (data_providers.py:151-162)
                v += (float)m.shift;                                         // networks.py:495
                id = (int)v;                                                 // tf.cast(float32 -> int32) truncates
                if (id < 0 || id >= m.vocab) {
                  atomicOr(status, 1);
                  id = id < 0 ? 0 : m.vocab - 1;
                }
              }
              s_ids[ru * kTileM + r] = (uint16_t)id;
            }
          }
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(C::kBuilders) : "memory");
      if (packed && bt == 0) mbar_arrive(raw_empty);     // every builder is past its reads of the staged window
      TRACE_ADD(t_ids);
      for (int sl = 0; sl < nslabs; ++sl, ++n) {
        const uint32_t b = n & 1;
        const int kh = min(C::kSlabK, ksteps - sl * C::kSlabK);
        mbar_wait(&a_empty[b], ((n >> 1) & 1) ^ 1);
        TRACE_ADD(t_aempty);
        uint4* dst = reinterpret_cast<uint4*>(sAslab + b * C::kASlabBytes);
        // A thread builds up to four of the slab's 2 kh 16-byte chunks for its row (chunk kcl = 3 j + bt / 128, row r =
        // bt % 128).  The three dependent shared-memory reads (column descriptor -> id -> table row) are
        // issued for all of its items before any is used, so their latencies overlap instead of adding up.
        {
          const int r = bt & (kTileM - 1), kc0 = bt >> 7;
          uint2 cd[C::kItems];
          uint32_t id[C::kItems];
          uint4 val[C::kItems];
#pragma unroll
          for (int j = 0; j < C::kItems; ++j)
            if (C::kChunkGroups * j + kc0 < 2 * kh) cd[j] = s_chunk[sl * C::kSlabK * 2 + C::kChunkGroups * j + kc0];
#pragma unroll
          for (int j = 0; j < C::kItems; ++j) {
            id[j] = 0;
            if (C::kChunkGroups * j + kc0 < 2 * kh && ((cd[j].x >> 16) & 0xff) == 1) id[j] = s_ids[(cd[j].x & 0xffff) * kTileM + r];
          }
#pragma unroll
          for (int j = 0; j < C::kItems; ++j) {
            if (C::kChunkGroups * j + kc0 < 2 * kh) {
              const uint32_t kind = (cd[j].x >> 16) & 0xff, src = cd[j].x & 0xffff, off = cd[j].y;
              if (kind == 1) {
                val[j] = *reinterpret_cast<const uint4*>(s_tab + off + id[j] * 8);
              } else if (kind == 3) {
                if ((cd[j].x >> 24) == 2) {
                  uint32_t w[4];
#pragma unroll
                  for (int q = 0; q < 4; ++q)
                    w[q] = *reinterpret_cast<const uint32_t*>(s_tab + off + (uint32_t)s_ids[(src + q) * kTileM + r] * 2);
                  val[j] = make_uint4(w[0], w[1], w[2], w[3]);
                } else {
                  const uint2 lo = *reinterpret_cast<const uint2*>(s_tab + off + (uint32_t)s_ids[src * kTileM + r] * 4);
                  const uint2 hi = *reinterpret_cast<const uint2*>(s_tab + off + (uint32_t)s_ids[(src + 1) * kTileM + r] * 4);
                  val[j] = make_uint4(lo.x, lo.y, hi.x, hi.y);
                }
              } else if (kind == 0) {
                val[j] = make_uint4(0u, 0u, 0u, 0u);
              } else {
                const int kc = sl * C::kSlabK * 2 + C::kChunkGroups * j + kc0;
                uint32_t packed[4];
#pragma unroll 1
                for (int jj = 0; jj < 4; ++jj) {
                  uint32_t pr = 0;
#pragma unroll
                  for (int h = 0; h < 2; ++h) {
                    const EmbedCol c = s_cols[kc * 8 + 2 * jj + h];
                    uint32_t bits = 0;
                    if (c.src_row >= 0) {
                      const int idd = s_ids[c.src_row * kTileM + r];
                      bits = __bfloat16_as_ushort(s_tab[c.table_off + idd * c.width + c.col]);
                    }
                    pr |= bits << (16 * h);
                  }
                  packed[jj] = pr;
                }
                val[j] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
              }
            }
          }
#pragma unroll
          for (int j = 0; j < C::kItems; ++j)
            if (C::kChunkGroups * j + kc0 < 2 * kh) dst[(size_t)(C::kChunkGroups * j + kc0) * kTileM + r] = val[j];
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[b]);      // 256 arrivals on one shared-memory word serialise: one per warp
        TRACE_ADD(t_build);
      }
    }
#ifdef DCB_TRACE
    if (bt == 0 && blockIdx.x < 256) {
      unsigned long long* tr = g_ffn_trace + blockIdx.x * 16;
      tr[0] = clock64() - t_begin; tr[1] = t_ids; tr[2] = t_aempty; tr[3] = t_build; tr[6] = t_begin - t_entry;
    }
#endif
  } else {
    setmaxnreg_inc<184>();   // 640 threads start with 96 registers: the service warps release 128 x 40, the builders 384 x 16 = 128 x 88
    // ------------------------------------------------------------- row epilogue (4 warps)
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t it = 0;
    long long t_accfull = 0, t_epi = 0;
    for (int ti = 0; ti < rounds; ++ti, ++it) {
      const int tile = tile_of(ti);
      const bool valid = tile_valid(ti);
      const uint32_t rot = lean ? it : 0u;
      const uint32_t j0 = (2 * rot) % 3, j1 = (2 * rot + 1) % 3;
      RowPrefetch pf;
      if (!lean && valid) row_prefetch_start(epi, tile, r, pf);   // positional rows in flight while the GEMM finishes
      TRACE_T0();
      mbar_wait(acc_full, it & 1);
      TRACE_ADD(t_accfull);
      tc_fence_after();
      RowStats st{0.f, 1.f};
      bool first_released = false;
      if (!valid) {}                                             // the pair's filler round: nothing to store
      else if (lean) { row_epilogue_embed_lean(epi, tmem_row, tile, r, j0 * kNC, j1 * kNC, &reg_free[j0]); first_released = true; }
      else st = row_epilogue_pass1(epi, tmem_row, tile, r, pf);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (!first_released) mbar_arrive(&reg_free[j0]);
        mbar_arrive(&reg_free[j1]);
      }
      TRACE_ADD(t_epi);
#ifdef DCB_TRACE
      if (q == 0 && lane == 0 && blockIdx.x < 256) { unsigned long long* tr = g_ffn_trace + blockIdx.x * 16; tr[4] = t_accfull; tr[5] = t_epi; }
#endif
      if (valid && epi.ln_g && epi.xb) row_epilogue_pass2<false>(epi, tile, r, st.mean, st.rstd);
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();               // no multicast or remote arrive is still under way towards a CTA that exits
#ifdef DCB_TRACE
  if (threadIdx.x == 128 && blockIdx.x < 256) g_ffn_trace[blockIdx.x * 16 + 7] = clock64() - t_entry;
#endif
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

size_t embed_condense_smem_bytes(int R, int echunks, int table_elems, int packed_stride) {
  const size_t tab = (table_elems * 2 + 127) & ~127;
  const size_t colsb = ((((size_t)echunks * 8 * sizeof(EmbedCol) + 15) & ~(size_t)15) + (size_t)echunks * 8 + 127) & ~(size_t)127;
  const size_t ids = ((size_t)R * kTileM * 2 + 127) & ~(size_t)127;
  const size_t raw = ((size_t)packed_stride + 127) & ~(size_t)127;      // 0 for float32 rows
  return ((tab + colsb + ids + raw + 1023) & ~(size_t)1023) + 2 * EmbCfg::kASlabBytes + 2 * EmbCfg::kBSlabBytes + 256;
}

// =====================================================================================
// fused FFN on CTA pairs (tcgen05 cta_group::2)
// =====================================================================================
// Two CTAs (a cluster of 2 = one TPC's SM pair) process two 128-token tiles together with M=256
// UMMAs issued by the leader (cluster rank 0).  Each CTA keeps its own x tile, hidden chunk and
// accumulators (rows of D split across the two TMEMs) but holds only HALF of every weight chunk
// (N/2 rows of B), so per SM the weight bytes pulled from L2 and written to / re-read from shared
// memory are halved and every MMA instruction carries twice the work.
//
// Per-rank weight image (w2img): for ff chunk c and rank r at offset (2c + r) * 73728 B:
//   [W1 half: 36 k-chunks x 64 hidden rows x 16 B][W2 half: 16 k-chunks x 144 output rows x 16 B]
// W1 half r holds hidden units c*128 + r*64 + [0,64); W2 half r holds, for each 144-wide N chunk j,
// output rows j*144 + r*72 + [0,72).
//
// Cross-CTA protocol (leader L, peer P):
//   full[slot] (L): local producer arrive.expect_tx + P's relay thread arrives remotely once P's own
//                   copy of the stage has landed (count 2).      full[slot] (P): local only.
//   empty[slot], a_empty, h_full, hs_free[2], y_full: tcgen05.commit multicast to both CTAs.
//   a_full (L): local expect_tx + remote arrive from P's relay (count 2).
//   h_free, hs_full[2], y_empty (L): one arrive per epilogue warp of BOTH CTAs (P's remotely).
struct Ffn2Cfg {
  static constexpr int kABytes = (kDP / 8) * kTileM * 16;            // 73728
  static constexpr int kHBytes = (kFFChunk / 8) * kTileM * 16;       // 32768
  static constexpr int kSlotBytes = 18432;
  static constexpr int kSlots = 4;
  static constexpr int kW1Rows = kFFChunk / 2;                       // 64 hidden rows per CTA
  static constexpr int kW1StageK = 9;
  static constexpr int kW1Stages = 2;
  static constexpr int kW1StageBytes = kW1StageK * 2 * kW1Rows * 16; // 18432
  static constexpr int kW2Rows = kDP / 2;                            // 144 output rows per CTA
  static constexpr int kW2StageK = 4;
  static constexpr int kW2Stages = 2;
  static constexpr int kW2StageBytes = kW2StageK * 2 * kW2Rows * 16; // 18432
  static constexpr int kHalfChunkBytes = kW1Stages * kW1StageBytes + kW2Stages * kW2StageBytes;  // 73728
  static constexpr int kWoStageK = 3;                                // attention out-proj: k-steps per stage
  static constexpr int kWoStages = (kDP / 16) / kWoStageK;           // 6
  static constexpr int kWoStageBytes = kWoStageK * 2 * kW2Rows * 16; // 13824
  static constexpr int kTmemY = 0;
  static constexpr int kTmemH = kDP;
  static constexpr int kTmemCols = 512;
  static constexpr int kMaxFF = 2048;
  static constexpr int kOffA = 0;
  static constexpr int kOffH = kABytes;
  static constexpr int kOffRing = kOffH + 2 * kHBytes;
  static constexpr int kOffB1 = kOffRing + kSlots * kSlotBytes;
  static constexpr int kOffBars = kOffB1 + kMaxFF * 4;
  static constexpr int kSmemBytes = kOffBars + 256;
};
static_assert(Ffn2Cfg::kSmemBytes <= 232448, "FFN pair shared memory budget");
static_assert(Ffn2Cfg::kW1Stages * Ffn2Cfg::kW1StageK == kDP / 16 && Ffn2Cfg::kW2Stages * Ffn2Cfg::kW2StageK == kFFChunk / 16, "stages");

// Four warpgroups: WG0 = {bulk-copy producer, two UMMA issuers (leader) or the relay thread (peer), 1 idle warp};
// WG1+WG2 = hidden-chunk epilogue (two warps share each TMEM lane quarter and split the chunk's columns, halving the
// G1 -> epilogue -> G1 dependency chain); WG3 = row epilogue of the finished tile, which thereby overlaps the next
// tile's GEMMs (its residual loads are software-prefetched).  setmaxnreg moves registers from WG0-2 to WG3, whose
// fully unrolled prefetching loop needs ~200.
constexpr int kFfnThreads = 512;

// kFuse: the attention output projection (attention_layer.py:218) + its residual / pre-norm
// (encoder_stack.py:72-93) run in front of the FFN on the same tile: a_img is then the attention
// operand image, Y <- x_old + att*Wo (out-proj UMMAs accumulate onto the residual already in TMEM),
// the row warps turn Y (= x_mid, never written to HBM) into the FFN's bf16 operand tile in shared
// memory (`mid`: identity for ReZero, LayerNorm otherwise), then the FFN proceeds as before.
template <bool kFuse>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFfnThreads, 1)
ffn_pair_kernel(const __nv_bfloat16* __restrict__ a_img, const uint8_t* __restrict__ w2img,
                const float* __restrict__ b1, int ff, int ntiles, RowEpi epi, int stagger_cycles,
                const uint8_t* __restrict__ wo2img, const float* __restrict__ mid_ln_g,
                const float* __restrict__ mid_ln_b) {
  using C = Ffn2Cfg;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem + C::kOffA;
  uint8_t* sH = smem + C::kOffH;
  uint8_t* sRing = smem + C::kOffRing;
  float* sB1 = reinterpret_cast<float*>(smem + C::kOffB1);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kOffBars);
  uint64_t* full = bars;                   // [kSlots]
  uint64_t* empty = bars + C::kSlots;      // [kSlots]
  uint64_t* a_full = bars + 2 * C::kSlots;
  uint64_t* a_empty = a_full + 1;
  uint64_t* h_full = a_full + 2;
  uint64_t* h_free = a_full + 3;
  uint64_t* hs_full = a_full + 4;          // [2]
  uint64_t* hs_free = a_full + 6;          // [2]
  uint64_t* y_full = a_full + 8;
  uint64_t* y_empty = a_full + 9;
  uint64_t* ymid_full = a_full + 10;       // out-proj UMMAs done: Y holds x_mid (kFuse)
  uint64_t* a2_full = a_full + 11;         // both CTAs' row warps wrote the FFN operand tile (kFuse, leader)
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(a_full + 12);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int nchunks = ff / kFFChunk;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int npairs = (int)gridDim.x >> 1;
  const int pair = (int)blockIdx.x >> 1;
  const int tile_pairs = (ntiles + 1) >> 1;
  const int rounds = (tile_pairs + npairs - 1) / npairs;

  if (threadIdx.x == 0) {
    for (int i = 0; i < C::kSlots; ++i) {
      mbar_init(&full[i], leader ? 2 : 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(a_full, leader ? 2 : 1);
    mbar_init(a_empty, 1);
    mbar_init(h_full, 1);
    mbar_init(h_free, 16);         // 8 hidden-epilogue warps x 2 CTAs (used in the leader only)
    mbar_init(&hs_full[0], 16);
    mbar_init(&hs_full[1], 16);
    mbar_init(&hs_free[0], 1);
    mbar_init(&hs_free[1], 1);
    mbar_init(y_full, 1);
    mbar_init(y_empty, 8);         // 4 row-epilogue warps x 2 CTAs (leader only)
    mbar_init(ymid_full, 1);
    mbar_init(a2_full, 8);
    mbar_fence_init();
  }
  for (int i = threadIdx.x; i < ff; i += blockDim.x) sB1[i] = b1[i];
  if (warp == 1) tmem_alloc_pair(tmem_holder, C::kTmemCols);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  // a tile index for this CTA in round ti (clamped: an out-of-range CTA recomputes the last tile)
  auto tile_of = [&](int ti) { return ((ti * npairs + pair) << 1) + (int)rank; };

  // De-synchronise the pairs: in lock step every CTA hits its residual read / write burst at the
  // same moment and HBM (not the tensor pipe) sets the pace; a start offset spreads the bursts.
  if (stagger_cycles > 0) {
    const long long t0 = clock64();
    const long long wait = (long long)(pair & 7) * stagger_cycles;
    while (clock64() - t0 < wait) {
    }
  }

  if (warp < 4) {
   setmaxnreg_dec<64>();
   if (warp == 0) {
    // ------------------------------------------------------------- producer (both CTAs, own halves)
    if (lane == 0) {
      uint32_t slot = 0, phase = 0;
      auto push = [&](const uint8_t* src, uint32_t bytes) {
        mbar_wait(&empty[slot], phase ^ 1);
#ifdef DCB_EXP_NOW   // timing experiment only (wrong results): no weight bytes move, stages "land" immediately
        mbar_arrive(&full[slot]);
#else
        mbar_arrive_expect_tx(&full[slot], bytes);
        bulk_g2s(sRing + slot * C::kSlotBytes, src, bytes, &full[slot]);
#endif
        if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
      };
      auto half = [&](int c) { return w2img + ((size_t)c * 2 + rank) * C::kHalfChunkBytes; };
      auto push_w1 = [&](int c) {
        for (int s = 0; s < C::kW1Stages; ++s) push(half(c) + s * C::kW1StageBytes, C::kW1StageBytes);
      };
      auto push_w2 = [&](int c) {
        const uint8_t* src = half(c) + C::kW1Stages * C::kW1StageBytes;
        for (int s = 0; s < C::kW2Stages; ++s) push(src + s * C::kW2StageBytes, C::kW2StageBytes);
      };
      for (int ti = 0; ti < rounds; ++ti) {
        const int tile = min(tile_of(ti), ntiles - 1);
        mbar_wait(a_empty, (ti & 1) ^ 1);
        mbar_arrive_expect_tx(a_full, C::kABytes);
        bulk_g2s(sA, reinterpret_cast<const uint8_t*>(a_img) + (size_t)tile * C::kABytes, C::kABytes, a_full);
        if constexpr (kFuse) {
          const uint8_t* wo = wo2img + (size_t)rank * C::kWoStages * C::kWoStageBytes;
          for (int s = 0; s < C::kWoStages; ++s) push(wo + s * C::kWoStageBytes, C::kWoStageBytes);
        }
        push_w1(0);
        for (int c = 0; c < nchunks; ++c) {
          if (c + 1 < nchunks) push_w1(c + 1);
          push_w2(c);
        }
      }
    }
   } else if (warp == 1 || warp == 2) {
    if (leader || lane == 0) {   // leader: whole warp walks the issue program (elected lane issues); peer: relay thread
      if (leader) {
        // ----------------------------------------------------------- UMMA issuers (leader only)
        // Two issuing threads share the tensor pipe: warp 1 issues the out-proj and every GEMM1,
        // warp 2 every GEMM2.  (One thread alone spends ~70 cycles per UMMA on descriptor set-up,
        // barrier polls and commits and cannot keep the pipe fed with 64-72-cycle instructions.)
        // Both walk the same global sequence of ring stages and act only on their own.
        constexpr uint32_t idesc_h = make_idesc_bf16(2 * kTileM, kFFChunk);
        constexpr uint32_t idesc_y = make_idesc_bf16(2 * kTileM, kNC);
        constexpr uint16_t kBoth = 3;
        const bool g1 = warp == 1;
        const uint32_t a_addr = smem_u32(sA);
        uint32_t slot = 0, phase = 0, n = 0;
        long long t_hfree = 0, t_full = 0, t_hsfull = 0, t_issue = 0, t_afull = 0, t_yempty = 0, t_oproj = 0, t_a2full = 0;
        const long long t_begin = clock64();
        auto skip = [&](int count) {
          for (int s = 0; s < count; ++s)
            if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
        };
        auto gemm1 = [&](uint32_t nn) {
          TRACE_T0();
          mbar_wait(h_free, (nn & 1) ^ 1);
          TRACE_ADD(t_hfree);
          tc_fence_after();
          for (int s = 0; s < C::kW1Stages; ++s) {
            mbar_wait(&full[slot], phase);
            TRACE_ADD(t_full);
            tc_fence_after();
            const uint32_t sb = smem_u32(sRing + slot * C::kSlotBytes);
#pragma unroll
            for (int kk = 0; kk < C::kW1StageK; ++kk) {
              const int kstep = s * C::kW1StageK + kk;
              const uint64_t adesc = make_kc16_desc(a_addr + kstep * 4096, kTileM * 16, 128);
              const uint64_t bdesc = make_kc16_desc(sb + kk * (2 * C::kW1Rows * 16), C::kW1Rows * 16, 128);
              umma_bf16_ss_pair_warp(tmem_base + C::kTmemH, adesc, bdesc, idesc_h, kstep != 0);
            }
            umma_commit_pair_warp(&empty[slot], kBoth);
            if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
            TRACE_ADD(t_issue);
          }
          umma_commit_pair_warp(h_full, kBoth);
        };
        auto gemm2 = [&](uint32_t nn) {
          const uint32_t b = nn & 1;
          TRACE_T0();
          mbar_wait(&hs_full[b], (nn >> 1) & 1);
          TRACE_ADD(t_hsfull);
          tc_fence_after();
          const uint32_t h_addr = smem_u32(sH + b * C::kHBytes);
          for (int s = 0; s < C::kW2Stages; ++s) {
            mbar_wait(&full[slot], phase);
            TRACE_ADD(t_full);
            tc_fence_after();
            const uint32_t sb = smem_u32(sRing + slot * C::kSlotBytes);
#pragma unroll
            for (int kk = 0; kk < C::kW2StageK; ++kk) {
              const int kstep = s * C::kW2StageK + kk;
              const uint64_t adesc = make_kc16_desc(h_addr + kstep * 4096, kTileM * 16, 128);
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const uint64_t bdesc = make_kc16_desc(sb + kk * (2 * C::kW2Rows * 16) + j * (kNC / 2) * 16,
                                                      C::kW2Rows * 16, 128);
                umma_bf16_ss_pair_warp(tmem_base + C::kTmemY + j * kNC, adesc, bdesc, idesc_y, true);
              }
            }
            umma_commit_pair_warp(&empty[slot], kBoth);
            if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
            TRACE_ADD(t_issue);
          }
          umma_commit_pair_warp(&hs_free[b], kBoth);
        };
        for (int ti = 0; ti < rounds; ++ti) {
          if (g1) {
            { TRACE_T0(); mbar_wait(a_full, ti & 1); TRACE_ADD(t_afull); }
            tc_fence_after();
            if constexpr (kFuse) {
              // Y (= x_old, stored by the row warps) += att * Wo^T
              TRACE_T0();
              mbar_wait(y_empty, ti & 1);
              TRACE_ADD(t_yempty);
              tc_fence_after();
              for (int s = 0; s < C::kWoStages; ++s) {
                mbar_wait(&full[slot], phase);
                tc_fence_after();
                const uint32_t sb = smem_u32(sRing + slot * C::kSlotBytes);
#pragma unroll
                for (int kk = 0; kk < C::kWoStageK; ++kk) {
                  const int kstep = s * C::kWoStageK + kk;
                  const uint64_t adesc = make_kc16_desc(a_addr + kstep * 4096, kTileM * 16, 128);
#pragma unroll
                  for (int j = 0; j < 2; ++j) {
                    const uint64_t bdesc = make_kc16_desc(sb + kk * (2 * C::kW2Rows * 16) + j * (kNC / 2) * 16,
                                                          C::kW2Rows * 16, 128);
                    umma_bf16_ss_pair_warp(tmem_base + C::kTmemY + j * kNC, adesc, bdesc, idesc_y, true);
                  }
                }
                umma_commit_pair_warp(&empty[slot], kBoth);
                if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
              }
              umma_commit_pair_warp(ymid_full, kBoth);
              TRACE_ADD(t_oproj);
              mbar_wait(a2_full, ti & 1);   // FFN operand tile written by both CTAs' row warps
              TRACE_ADD(t_a2full);
              tc_fence_after();
            }
            gemm1(n);
            for (int c = 0; c < nchunks; ++c) {
              if (c + 1 < nchunks) gemm1(n + c + 1);
              else umma_commit_pair_warp(a_empty, kBoth);   // every UMMA that reads sA has been issued
              skip(C::kW2Stages);
            }
          } else {
            if constexpr (kFuse) skip(C::kWoStages);
            skip(C::kW1Stages);
            for (int c = 0; c < nchunks; ++c) {
              if (c + 1 < nchunks) skip(C::kW1Stages);
              if (!kFuse && c == 0) {
                mbar_wait(y_empty, ti & 1);   // "Y holds x_old": both CTAs' row warps initialised it
                tc_fence_after();
              }
              gemm2(n + c);
            }
            umma_commit_pair_warp(y_full, kBoth);
          }
          n += nchunks;
        }
#ifdef DCB_TRACE
        if (g1 && lane == 0 && blockIdx.x < 256) {
          unsigned long long* tr = g_ffn_trace + blockIdx.x * 16;
          tr[0] = clock64() - t_begin; tr[1] = t_hfree; tr[2] = t_full; tr[3] = t_hsfull;
          tr[4] = t_issue; tr[5] = t_afull; tr[6] = t_yempty; tr[7] = t_a2full; tr[15] = t_oproj;
        }
#endif
      } else if (warp == 1) {
        // ----------------------------------------------------------- relay (peer): forward "my half
        // of this stage / my x tile has landed" to the leader's barriers, in consumption order
        uint32_t slot = 0, phase = 0;
        auto relay_stages = [&](int count) {
          for (int s = 0; s < count; ++s) {
            mbar_wait(&full[slot], phase);
            mbar_arrive_cluster(&full[slot], 0);
            if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
          }
        };
        for (int ti = 0; ti < rounds; ++ti) {
          mbar_wait(a_full, ti & 1);
          mbar_arrive_cluster(a_full, 0);
          if constexpr (kFuse) relay_stages(C::kWoStages);
          relay_stages(C::kW1Stages);
          for (int c = 0; c < nchunks; ++c) {
            if (c + 1 < nchunks) relay_stages(C::kW1Stages);
            relay_stages(C::kW2Stages);
          }
        }
      }
    }
   }
  } else {
    // ------------------------------------------------------------- epilogue warps (both CTAs)
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
    auto arrive_leader = [&](uint64_t* bar) {   // one arrive per warp on the leader's barrier
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(bar); else mbar_arrive_cluster(bar, 0);
      }
    };
    if (warp < 12) {
      setmaxnreg_dec<96>();
      const int half = (warp - 4) >> 2;
      uint32_t n = 0;
      long long t_hfull = 0, t_hsfree = 0, t_body = 0;
      for (int ti = 0; ti < rounds; ++ti) {
        for (int c = 0; c < nchunks; ++c, ++n) {
          const uint32_t b = n & 1;
          TRACE_T0();
          mbar_wait(h_full, n & 1);
          TRACE_ADD(t_hfull);
          tc_fence_after();
          mbar_wait(&hs_free[b], ((n >> 1) & 1) ^ 1);
          TRACE_ADD(t_hsfree);
          uint4* hrow = reinterpret_cast<uint4*>(sH + b * C::kHBytes) + r;
          const float* bias = sB1 + c * kFFChunk + half * (kFFChunk / 2);
          // all four 16-column TMEM loads in flight, one wait, then release the accumulator
          // immediately so GEMM1 of the next chunk overlaps the math + smem stores below
          uint32_t acc[kFFChunk / 32][16];
#pragma unroll
          for (int cc = 0; cc < kFFChunk / 32; ++cc)
            tmem_ld16(tmem_row + C::kTmemH + (half * (kFFChunk / 32) + cc) * 16, acc[cc]);
          tmem_ld_wait();
          tc_fence_before();
          arrive_leader(h_free);
#pragma unroll
          for (int cc = 0; cc < kFFChunk / 32; ++cc) {
            const int cb = half * (kFFChunk / 32) + cc;
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = fmaxf(__uint_as_float(acc[cc][i]) + bias[cc * 16 + i], 0.f);
#ifdef DCB_EXP_NOHST   // timing experiment only (wrong results): the hidden tile is not written to shared memory
            if (v[0] + v[5] + v[9] + v[15] == 12345.678f)
#endif
            {
            hrow[(size_t)(cb * 2) * kTileM] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                                         pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
            hrow[(size_t)(cb * 2 + 1) * kTileM] =
                make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]),
                           pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
            }
          }
          fence_proxy_async_smem();
          arrive_leader(&hs_full[b]);
          TRACE_ADD(t_body);
        }
      }
#ifdef DCB_TRACE
      if (warp == 4 && lane == 0 && blockIdx.x < 256) {
        unsigned long long* tr = g_ffn_trace + blockIdx.x * 16;
        tr[8] = t_hfull; tr[9] = t_hsfree; tr[10] = t_body;
      }
#endif
    } else {
      setmaxnreg_inc<216>();
      long long t_yfull = 0, t_row1 = 0, t_ldtm = 0, t_phaseA = 0;
      const float4* xbase = reinterpret_cast<const float4*>(epi.x) + r;
      auto xrow_of = [&](int tile) { return xbase + (size_t)tile * (x_image_elems() / 4); };
      // ---- first tile: Y <- x_old (residual-in-accumulator), two batches of 9 column blocks
      {
#ifdef DCB_TRACE
        const long long _ta0 = clock64();
#endif
        const float4* xrow = xrow_of(min(tile_of(0), ntiles - 1));
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float4 buf[9][4];
#pragma unroll
          for (int kq = 0; kq < 9; ++kq)
#pragma unroll
            for (int i = 0; i < 4; ++i) buf[kq][i] = xrow[(size_t)((half * 9 + kq) * 4 + i) * kTileM];
#pragma unroll
          for (int kq = 0; kq < 9; ++kq) {
            uint32_t v[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              v[4 * i + 0] = __float_as_uint(buf[kq][i].x); v[4 * i + 1] = __float_as_uint(buf[kq][i].y);
              v[4 * i + 2] = __float_as_uint(buf[kq][i].z); v[4 * i + 3] = __float_as_uint(buf[kq][i].w);
            }
            tmem_st16(tmem_row + C::kTmemY + (half * 9 + kq) * 16, v);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        arrive_leader(y_empty);
#ifdef DCB_TRACE
        t_phaseA += clock64() - _ta0;
#endif
      }
      for (int ti = 0; ti < rounds; ++ti) {
        const int tile_raw = tile_of(ti);
        const bool valid = tile_raw < ntiles;
        const bool has_next = ti + 1 < rounds;
        const float4* xnext = xrow_of(min(tile_of(ti + 1), ntiles - 1));
        if constexpr (kFuse) {
          // mid epilogue: Y = x_mid after the out-proj.  Produce the FFN's bf16 operand tile in sA
          // (the attention tile there has been consumed: ymid_full follows the out-proj UMMAs).
          mbar_wait(ymid_full, ti & 1);
          tc_fence_after();
          float mean = 0.f, rstd = 1.f;
          if (mid_ln_g) {
            float s1 = 0.f, s2 = 0.f, shift = 0.f;
#pragma unroll 2
            for (int cb = 0; cb < kDP / 16; ++cb) {
              uint32_t acc[16];
              tmem_ld16(tmem_row + C::kTmemY + cb * 16, acc);
              tmem_ld_wait();
              if (cb == 0) shift = __uint_as_float(acc[0]);
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float dlt = (cb * 16 + i < kD) ? __uint_as_float(acc[i]) - shift : 0.f;
                s1 += dlt;
                s2 += dlt * dlt;
              }
            }
            const float m1 = s1 * (1.f / kD);
            mean = shift + m1;
            rstd = rsqrtf(fmaxf(s2 * (1.f / kD) - m1 * m1, 0.f) + 1e-6f);
          }
          uint4* arow = reinterpret_cast<uint4*>(sA) + r;
#pragma unroll 2
          for (int cb = 0; cb < kDP / 16; ++cb) {
            uint32_t acc[16];
            tmem_ld16(tmem_row + C::kTmemY + cb * 16, acc);
            tmem_ld_wait();
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int col = cb * 16 + i;
              float t = __uint_as_float(acc[i]);
              if (mid_ln_g) t = (t - mean) * rstd * __ldg(mid_ln_g + col) + __ldg(mid_ln_b + col);
              v[i] = col < kD ? t : 0.f;
            }
            arow[(size_t)(cb * 2) * kTileM] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                                         pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
            arow[(size_t)(cb * 2 + 1) * kTileM] =
                make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]),
                           pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
          }
          tc_fence_before();
          fence_proxy_async_smem();
          arrive_leader(a2_full);
        }
        // The row warps now idle for the 16 hidden chunks: pull the next tile's residual into L2 so the
        // hand-over pass below reads it at L2 latency instead of HBM latency (8 rows share a 128-byte line:
        // thread r fetches the lines of chunks c == r (mod 8)).
        if (has_next) {
#pragma unroll
          for (int c = 0; c < kXChunks / 8; ++c)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(xnext + (size_t)(c * 8 + (r & 7)) * kTileM));
        }
        // ---- drain the finished tile AND re-initialise Y with the next tile's residual in the same
        // pass: each 16-column block is read out (x_new = Y + b2 -> global) and immediately
        // overwritten with x_old of the next tile, whose loads were issued kRowPF blocks ahead.
        RowPrefetch pf;
        if (has_next) {
#pragma unroll
          for (int kq = 0; kq < kRowPF; ++kq)
#pragma unroll
            for (int i = 0; i < 4; ++i) pf.buf[kq][i] = xnext[(size_t)(kq * 4 + i) * kTileM];
        }
        TRACE_T0();
        mbar_wait(y_full, ti & 1);
        TRACE_ADD(t_yfull);
        tc_fence_after();
        {
          const int tile_st = min(tile_raw, ntiles - 1);
          float4* xrow = reinterpret_cast<float4*>(epi.x + (size_t)tile_st * x_image_elems()) + r;
          uint4* xbrow = epi.xb ? reinterpret_cast<uint4*>(epi.xb + (size_t)tile_st * act_image_elems(kDP)) + r : nullptr;
          const bool ln = epi.ln_g != nullptr;
          float s1 = 0.f, s2 = 0.f, shift = 0.f;
#pragma unroll
          for (int cb = 0; cb < kDP / 16; ++cb) {
            uint32_t acc[16];
            tmem_ld16(tmem_row + C::kTmemY + cb * 16, acc);
            tmem_ld_wait();
            if (has_next) {
              uint32_t nx[16];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 t = pf.buf[cb % kRowPF][i];
                nx[4 * i + 0] = __float_as_uint(t.x); nx[4 * i + 1] = __float_as_uint(t.y);
                nx[4 * i + 2] = __float_as_uint(t.z); nx[4 * i + 3] = __float_as_uint(t.w);
              }
              tmem_st16(tmem_row + C::kTmemY + cb * 16, nx);
              if (cb + kRowPF < kDP / 16) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  pf.buf[cb % kRowPF][i] = xnext[(size_t)((cb + kRowPF) * 4 + i) * kTileM];
              }
            }
            if (valid) {
              float v[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const int col = cb * 16 + i;
                float t = __uint_as_float(acc[i]);
                if (epi.bias) t += __ldg(epi.bias + col);
                v[i] = col < kD ? t : 0.f;
              }
#pragma unroll
              for (int i = 0; i < 4; ++i)
                xrow[(size_t)(cb * 4 + i) * kTileM] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
              if (ln) {
                if (cb == 0) shift = v[0];
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                  const float dlt = (cb * 16 + i < kD) ? v[i] - shift : 0.f;
                  s1 += dlt;
                  s2 += dlt * dlt;
                }
              } else if (xbrow) {
                xbrow[(size_t)(cb * 2) * kTileM] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]),
                                                              pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
                xbrow[(size_t)(cb * 2 + 1) * kTileM] =
                    make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]),
                               pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
              }
            }
          }
          if (has_next) {
            tmem_st_wait();
            tc_fence_before();
            arrive_leader(y_empty);      // "Y holds x_old" of the next tile
          }
          TRACE_ADD(t_row1);
          if (valid && ln && epi.xb) {
            const float m1 = s1 * (1.f / kD);
            const float mean = shift + m1;
            const float rstd = rsqrtf(fmaxf(s2 * (1.f / kD) - m1 * m1, 0.f) + 1e-6f);
            row_epilogue_pass2<false>(epi, tile_raw, r, mean, rstd);
          }
        }
        tc_fence_before();
      }
#ifdef DCB_TRACE
      if (warp == 12 && lane == 0 && blockIdx.x < 256) {
        unsigned long long* tr = g_ffn_trace + blockIdx.x * 16;
        tr[11] = t_yfull; tr[12] = t_row1; tr[13] = t_ldtm; tr[14] = t_phaseA;
      }
#endif
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, C::kTmemCols);
  }
}

// =====================================================================================
// banded attention (mma.sync m16n8k16 bf16, online softmax over 16-key tiles)
// =====================================================================================
// One CTA per (window, head).  K and V rows of the window are staged in shared memory
// (row stride 152 bf16 = 304 B: conflict-free for the 32-bit K-fragment loads and for
// ldmatrix.trans on V); Q fragments are read straight from the global operand image.
// FLOP share of this kernel is ~1-4 % of the model, so the legacy warp-level MMA path
// is used here on purpose (SURVEY.md section 7, "Window/tile alignment for attention").
constexpr int kAttStride = 144;              // dense rows; 16-byte chunks are rotated by the row index
constexpr int kAttChunks = kDHP / 8;         // 18 chunks per row

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0,
                                               uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t& r0, uint32_t& r1, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];"
               : "=r"(r0), "=r"(r1)
               : "r"(addr));
}

// element (token, col) of a bf16 operand image with `chunks` 8-wide chunks per row
__device__ __forceinline__ size_t img_off(int tok, int col, int chunks) {
  const int tile = tok / kTileM, r = tok % kTileM;
  return (((size_t)tile * chunks + (col >> 3)) * kTileM + r) * 8 + (col & 7);
}

// Shared-memory K/V rows are dense (288 B) with the 18 16-byte chunks of row r rotated by r
// (physical chunk = (c + r) mod 18): 8 consecutive rows then hit 8 distinct 16-byte bank groups
// (48 r mod 128 is a permutation of the multiples of 16), which keeps both the 32-bit K-fragment
// loads and ldmatrix.trans on V conflict-free without padding -- 73.7 KB per CTA, 3 CTAs per SM.
__device__ __forceinline__ int att_rot(int chunk, int rowmod) {
  const int t = chunk + rowmod;
  return t >= kAttChunks ? t - kAttChunks : t;
}

__global__ void __launch_bounds__(128, 3)
band_attention_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ att,
                      int L, int Lw, int win, int nwindows) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int w = blockIdx.x >> 1;
  const int head = blockIdx.x & 1;
  if (w >= nwindows) return;
  const int Lp = (L + 15) & ~15;  // key rows padded to a multiple of 16 (zero filled)
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(smem);
  __nv_bfloat16* sV = sK + (size_t)Lp * kAttStride;
  constexpr int qkv_chunks = kQKVN / 8;  // 108
  const int kcol = (2 + head) * kDHP, vcol = (4 + head) * kDHP, qcol = head * kDHP;
  const int tok0 = w * Lw;   // windows start every Lw tokens in the flattened layout (Lw >= L)
#ifdef DCB_TRACE
  const long long _t_start = clock64();
#endif

  // stage K, V with cp.async: thread = row (coalesced 16 B chunks across the warp), no divisions
  for (int row = threadIdx.x; row < Lp; row += blockDim.x) {
    const int rm = row % kAttChunks;
    __nv_bfloat16* dk = sK + (size_t)row * kAttStride;
    __nv_bfloat16* dv = sV + (size_t)row * kAttStride;
    if (row < L) {
      const int tok = tok0 + row;
      const size_t base = ((size_t)(tok / kTileM) * qkv_chunks) * kTileM * 8 + (size_t)(tok % kTileM) * 8;
      const __nv_bfloat16* gk = qkv + base + (size_t)(kcol >> 3) * kTileM * 8;
      const __nv_bfloat16* gv = qkv + base + (size_t)(vcol >> 3) * kTileM * 8;
#pragma unroll
      for (int ch = 0; ch < kAttChunks; ++ch) {
        const int pc = att_rot(ch, rm) * 8;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dk + pc)),
                     "l"(gk + (size_t)ch * kTileM * 8) : "memory");
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dv + pc)),
                     "l"(gv + (size_t)ch * kTileM * 8) : "memory");
      }
    } else {
#pragma unroll
      for (int ch = 0; ch < kAttChunks; ++ch) {
        *reinterpret_cast<uint4*>(dk + ch * 8) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(dv + ch * 8) = make_uint4(0, 0, 0, 0);
      }
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int band = win > 0 ? win : L;  // attn_win_size None/0 => full attention
  constexpr float kLog2e = 1.4426950408889634f;

  // Q fragments for 9 k-steps: rows i0+g, i0+g+8 (zero beyond L), straight from global.
  // In the operand image a row's k-chunks are kTileM*8 elements apart, so every fragment address is
  // the row base plus a compile-time constant (no per-load index arithmetic).
  constexpr int kChunkElems = kTileM * 8;
  uint32_t qa[kDHP / 16][4];
  auto load_q = [&](int qb) {
    const int r0 = qb * 16 + g, r1 = r0 + 8;
    const __nv_bfloat16* q0 = qkv + img_off(tok0 + (r0 < L ? r0 : 0), qcol + 2 * t, qkv_chunks);
    const __nv_bfloat16* q1 = qkv + img_off(tok0 + (r1 < L ? r1 : 0), qcol + 2 * t, qkv_chunks);
#pragma unroll
    for (int ks = 0; ks < kDHP / 16; ++ks) {
      const uint32_t v0 = __ldg(reinterpret_cast<const uint32_t*>(q0 + (2 * ks) * kChunkElems));
      const uint32_t v1 = __ldg(reinterpret_cast<const uint32_t*>(q1 + (2 * ks) * kChunkElems));
      const uint32_t v2 = __ldg(reinterpret_cast<const uint32_t*>(q0 + (2 * ks + 1) * kChunkElems));
      const uint32_t v3 = __ldg(reinterpret_cast<const uint32_t*>(q1 + (2 * ks + 1) * kChunkElems));
      qa[ks][0] = r0 < L ? v0 : 0u;
      qa[ks][1] = r1 < L ? v1 : 0u;
      qa[ks][2] = r0 < L ? v2 : 0u;
      qa[ks][3] = r1 < L ? v3 : 0u;
    }
  };
  if (warp * 16 < L) load_q(warp);
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
#ifdef DCB_TRACE
  const long long _t_staged = clock64();
#endif

  for (int qb = warp; qb * 16 < L; qb += 4) {
    const int i0 = qb * 16;
    const int r0 = i0 + g, r1 = i0 + g + 8;
    if (qb != warp) load_q(qb);
    float o[kDHP / 8][4];
#pragma unroll
    for (int nt = 0; nt < kDHP / 8; ++nt) { o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f; }
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

    int jlo = i0 - band; if (jlo < 0) jlo = 0; jlo &= ~15;
    int jhi = i0 + 15 + band + 1; if (jhi > L) jhi = L;
    for (int j0 = jlo; j0 < jhi; j0 += 16) {
      // S tile 16 x 16 = two n-tiles of 8 keys; two partial accumulators per n-tile shorten the
      // dependent HMMA chains (4 independent chains instead of 2)
      float s[2][4], s2[2][4];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        s2[nt][0] = s2[nt][1] = s2[nt][2] = s2[nt][3] = 0.f;
      }
      const int krow0 = j0 + g, krow1 = j0 + 8 + g;
      const __nv_bfloat16* kr0 = sK + (size_t)krow0 * kAttStride + 2 * t;
      const __nv_bfloat16* kr1 = sK + (size_t)krow1 * kAttStride + 2 * t;
      const int km0 = krow0 % kAttChunks, km1 = krow1 % kAttChunks;
#pragma unroll
      for (int ks = 0; ks < kDHP / 16; ++ks) {
        const uint32_t a0 = *reinterpret_cast<const uint32_t*>(kr0 + att_rot(2 * ks, km0) * 8);
        const uint32_t a1 = *reinterpret_cast<const uint32_t*>(kr0 + att_rot(2 * ks + 1, km0) * 8);
        const uint32_t c0 = *reinterpret_cast<const uint32_t*>(kr1 + att_rot(2 * ks, km1) * 8);
        const uint32_t c1 = *reinterpret_cast<const uint32_t*>(kr1 + att_rot(2 * ks + 1, km1) * 8);
        if (ks & 1) {
          mma_bf16_16816(s2[0], qa[ks], a0, a1);
          mma_bf16_16816(s2[1], qa[ks], c0, c1);
        } else {
          mma_bf16_16816(s[0], qa[ks], a0, a1);
          mma_bf16_16816(s[1], qa[ks], c0, c1);
        }
      }
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) s[nt][e] += s2[nt][e];
      // mask: |i - j| <= band and j < L  (tf.where(mask, logits, -1e9): exp underflows to 0)
      float tmax0 = -INFINITY, tmax1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int i = (e < 2) ? r0 : r1;
          const int j = j0 + nt * 8 + 2 * t + (e & 1);
          const int dlt = i - j;
          const bool ok = (j < L) && (dlt <= band) && (dlt >= -band);
          s[nt][e] = ok ? s[nt][e] : -INFINITY;
        }
        tmax0 = fmaxf(tmax0, fmaxf(s[nt][0], s[nt][1]));
        tmax1 = fmaxf(tmax1, fmaxf(s[nt][2], s[nt][3]));
      }
      tmax0 = fmaxf(tmax0, __shfl_xor_sync(0xffffffffu, tmax0, 1));
      tmax0 = fmaxf(tmax0, __shfl_xor_sync(0xffffffffu, tmax0, 2));
      tmax1 = fmaxf(tmax1, __shfl_xor_sync(0xffffffffu, tmax1, 1));
      tmax1 = fmaxf(tmax1, __shfl_xor_sync(0xffffffffu, tmax1, 2));
      const float mn0 = fmaxf(m0, tmax0), mn1 = fmaxf(m1, tmax1);
      // rows with no valid key yet keep m = -inf; use 0 as the subtraction base there
      const float base0 = mn0 == -INFINITY ? 0.f : mn0, base1 = mn1 == -INFINITY ? 0.f : mn1;
      const float sc0 = exp2f((m0 - base0) * kLog2e), sc1 = exp2f((m1 - base1) * kLog2e);
      m0 = mn0; m1 = mn1;
      float ps0 = 0.f, ps1 = 0.f;
      uint32_t pa[4];
      {
        float p[2][4];
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          p[nt][0] = exp2f((s[nt][0] - base0) * kLog2e);
          p[nt][1] = exp2f((s[nt][1] - base0) * kLog2e);
          p[nt][2] = exp2f((s[nt][2] - base1) * kLog2e);
          p[nt][3] = exp2f((s[nt][3] - base1) * kLog2e);
          ps0 += p[nt][0] + p[nt][1];
          ps1 += p[nt][2] + p[nt][3];
        }
        // C fragments of the two n-tiles form the A fragment of one 16-key k-step
        pa[0] = pack_bf16x2(p[0][0], p[0][1]);
        pa[1] = pack_bf16x2(p[0][2], p[0][3]);
        pa[2] = pack_bf16x2(p[1][0], p[1][1]);
        pa[3] = pack_bf16x2(p[1][2], p[1][3]);
      }
      l0 = l0 * sc0 + ps0;
      l1 = l1 * sc1 + ps1;
      // O = O * scale + P V
      const int vrow = j0 + (lane & 15);
      const int vm = vrow % kAttChunks;
      const uint32_t vbase = smem_u32(sV + (size_t)vrow * kAttStride);
#pragma unroll
      for (int nt = 0; nt < kDHP / 8; ++nt) {
        o[nt][0] *= sc0; o[nt][1] *= sc0; o[nt][2] *= sc1; o[nt][3] *= sc1;
        uint32_t b0, b1;
        ldmatrix_x2_trans(b0, b1, vbase + att_rot(nt, vm) * 16);
        mma_bf16_16816(o[nt], pa, b0, b1);
      }
    }
    // normalise (row sums live in the quad) and store bf16 to the attention operand image
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float inv0 = 1.f / l0, inv1 = 1.f / l1;
    __nv_bfloat16* o0 = att + img_off(tok0 + (r0 < L ? r0 : 0), head * kDHP + 2 * t, kDP / 8);
    __nv_bfloat16* o1 = att + img_off(tok0 + (r1 < L ? r1 : 0), head * kDHP + 2 * t, kDP / 8);
#pragma unroll
    for (int nt = 0; nt < kDHP / 8; ++nt) {
      if (r0 < L)
        *reinterpret_cast<uint32_t*>(o0 + nt * kChunkElems) = pack_bf16x2(o[nt][0] * inv0, o[nt][1] * inv0);
      if (r1 < L)
        *reinterpret_cast<uint32_t*>(o1 + nt * kChunkElems) = pack_bf16x2(o[nt][2] * inv1, o[nt][3] * inv1);
    }
  }
#ifdef DCB_TRACE
  if (threadIdx.x == 0 && blockIdx.x < 256) {
    unsigned long long* tr = g_ffn_trace + blockIdx.x * 16;
    unsigned int smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    tr[13] = _t_staged - _t_start; tr[14] = clock64() - _t_staged; tr[15] = smid;
  }
#endif
}

// =====================================================================================
// fused q/k/v projection + banded attention (window-aligned tiles, CTA pairs)
// =====================================================================================
// One 128-row tile = one window (engine layout Lw == 128).  A CTA pair handles two windows with
// M=256 UMMAs (each CTA holds half of every weight k-step).  Per head: Q|K|V = X * [Wq|Wk|Wv]_h
// (54 UMMAs, N=144) land in TMEM, 8 worker warps move them as bf16 into shared memory (rows of
// 288 B, 16-byte chunks rotated by the row index -- the layout band_attention_kernel stages into),
// then each worker warp runs the banded softmax attention of one 16-query block straight from
// shared memory (mma.sync) while the tensor core already computes the next head's projections.
// q, k and v never touch HBM (-516 KB per window and layer through the SM's L2 port).
struct QaCfg {
  static constexpr int kABytes = (kDP / 8) * kTileM * 16;            // 73728
  static constexpr int kStride = 152;                                // padded row (304 B): conflict-free, no index rotation
  static constexpr int kMatBytes = kTileM * kStride * 2;             // 38912: q, k or v of one head
  static constexpr int kRows = 3 * (kDHP / 2);                       // 216 weight rows per CTA per k-step
  static constexpr int kStageBytes = 2 * kRows * 16;                 // 6912: one k-step
  static constexpr int kSlots = 6;
  static constexpr int kHeadBytes = (kDP / 16) * kStageBytes;        // 124416 per (head, rank)
  static constexpr int kOffA = 0;
  static constexpr int kOffQ = kABytes;
  static constexpr int kOffRing = kOffQ + 3 * kMatBytes;
  static constexpr int kOffBars = kOffRing + kSlots * kStageBytes;
  static constexpr int kSmemBytes = kOffBars + 256;
  static constexpr int kThreads = 384;   // WG0 = {producer, UMMA issuer / relay, 2 idle}, WG1-2 = 8 worker warps
  static constexpr int kTmemCols = 512;
};
static_assert(QaCfg::kSmemBytes <= 232448, "qkv+attention shared memory budget");

// kTwoPass: attn_win_size <= 16, i.e. every 16-query block sees at most 3 key tiles (two-pass softmax);
// otherwise the general online-softmax loop (any band, incl. full attention).
template <bool kTwoPass>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(QaCfg::kThreads, 1)
qkv_attn_pair_kernel(const __nv_bfloat16* __restrict__ a_img, const uint8_t* __restrict__ w_img, int ntiles,
                     int L, int win, __nv_bfloat16* __restrict__ att) {
  using C = QaCfg;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem + C::kOffA;
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem + C::kOffQ);
  constexpr int kS = C::kStride;
  __nv_bfloat16* sK = sQ + kTileM * kS;
  __nv_bfloat16* sV = sK + kTileM * kS;
  uint8_t* sRing = smem + C::kOffRing;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kOffBars);
  uint64_t* full = bars;                    // [kSlots]
  uint64_t* empty = bars + C::kSlots;       // [kSlots]
  uint64_t* a_full = bars + 2 * C::kSlots;
  uint64_t* a_empty = a_full + 1;
  uint64_t* acc_full = a_full + 2;
  uint64_t* acc_free = a_full + 3;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(a_full + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int npairs = (int)gridDim.x >> 1, pair = (int)blockIdx.x >> 1;
  const int tile_pairs = (ntiles + 1) >> 1;
  const int rounds = (tile_pairs + npairs - 1) / npairs;
  auto tile_of = [&](int ti) { return ((ti * npairs + pair) << 1) + (int)rank; };

  if (threadIdx.x == 0) {
    for (int i = 0; i < C::kSlots; ++i) { mbar_init(&full[i], leader ? 2 : 1); mbar_init(&empty[i], 1); }
    mbar_init(a_full, leader ? 2 : 1);
    mbar_init(a_empty, 1);
    mbar_init(acc_full, 1);
    mbar_init(acc_free, 16);     // 8 worker warps x 2 CTAs (leader only)
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_holder, C::kTmemCols);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;

  if (warp < 4) {
   setmaxnreg_dec<40>();
   if (warp == 0) {
    if (lane == 0) {
      uint32_t slot = 0, phase = 0;
      for (int ti = 0; ti < rounds; ++ti) {
        const int tile = min(tile_of(ti), ntiles - 1);
        mbar_wait(a_empty, (ti & 1) ^ 1);
        mbar_arrive_expect_tx(a_full, C::kABytes);
        bulk_g2s(sA, reinterpret_cast<const uint8_t*>(a_img) + (size_t)tile * C::kABytes, C::kABytes, a_full);
        for (int h = 0; h < kHeads; ++h) {
          const uint8_t* src = w_img + ((size_t)h * 2 + rank) * C::kHeadBytes;
          for (int ks = 0; ks < kDP / 16; ++ks) {
            mbar_wait(&empty[slot], phase ^ 1);
            mbar_arrive_expect_tx(&full[slot], C::kStageBytes);
            bulk_g2s(sRing + slot * C::kStageBytes, src + (size_t)ks * C::kStageBytes, C::kStageBytes, &full[slot]);
            if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader || lane == 0) {   // leader: whole warp, elected lane issues; peer: relay thread
      uint32_t slot = 0, phase = 0;
      if (leader) {
        constexpr uint32_t idesc = make_idesc_bf16(2 * kTileM, kNC);
        constexpr uint16_t kBoth = 3;
        const uint32_t a_addr = smem_u32(sA);
        uint32_t hi = 0;
        long long t_afull = 0, t_accfree = 0, t_full = 0, t_issue = 0;
        const long long t_begin = clock64();
        for (int ti = 0; ti < rounds; ++ti) {
          { TRACE_T0(); mbar_wait(a_full, ti & 1); TRACE_ADD(t_afull); }
          tc_fence_after();
          for (int h = 0; h < kHeads; ++h, ++hi) {
            TRACE_T0();
            mbar_wait(acc_free, (hi & 1) ^ 1);
            TRACE_ADD(t_accfree);
            tc_fence_after();
            for (int ks = 0; ks < kDP / 16; ++ks) {
              mbar_wait(&full[slot], phase);
              TRACE_ADD(t_full);
              tc_fence_after();
              const uint32_t sb = smem_u32(sRing + slot * C::kStageBytes);
              const uint64_t adesc = make_kc16_desc(a_addr + ks * 4096, kTileM * 16, 128);
#pragma unroll
              for (int m = 0; m < 3; ++m) {
                const uint64_t bdesc = make_kc16_desc(sb + m * (kDHP / 2) * 16, C::kRows * 16, 128);
                umma_bf16_ss_pair_warp(tmem_base + m * kDHP, adesc, bdesc, idesc, ks != 0);
              }
              umma_commit_pair_warp(&empty[slot], kBoth);
              if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
              TRACE_ADD(t_issue);
            }
            umma_commit_pair_warp(acc_full, kBoth);
          }
          umma_commit_pair_warp(a_empty, kBoth);
        }
#ifdef DCB_TRACE
        if (lane == 0 && blockIdx.x < 108) {
          unsigned long long* tr = g_ffn_trace + (blockIdx.x % 108 + 148) * 16;
          tr[0] = clock64() - t_begin; tr[1] = t_afull; tr[2] = t_accfree; tr[3] = t_full; tr[4] = t_issue; tr[7] = rounds;
        }
#endif
      } else {
        for (int ti = 0; ti < rounds; ++ti) {
          mbar_wait(a_full, ti & 1);
          mbar_arrive_cluster(a_full, 0);
          for (int s = 0; s < kHeads * (kDP / 16); ++s) {
            mbar_wait(&full[slot], phase);
            mbar_arrive_cluster(&full[slot], 0);
            if (++slot == C::kSlots) { slot = 0; phase ^= 1; }
          }
        }
      }
    }
   } else {
    // warps 2-3 (otherwise idle): pull the NEXT tile's operand image into L2 so its bulk load, which can
    // only be issued once this tile's UMMAs have released sA, completes at L2 latency
    const int pt = threadIdx.x - 64;   // 0..63
    for (int ti = 0; ti + 1 < rounds; ++ti) {
      const int tile = min(tile_of(ti + 1), ntiles - 1);
      const uint8_t* base = reinterpret_cast<const uint8_t*>(a_img) + (size_t)tile * C::kABytes;
      for (int ln = pt; ln < C::kABytes / 128; ln += 64)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (size_t)ln * 128));
      // pace: one tile ahead is enough -- wait until this round's tile has been consumed
      mbar_wait(a_empty, ti & 1);
    }
   }
  } else {
    setmaxnreg_inc<232>();
    // ------------------------------------------------------------- workers (8 warps)
    const int ew = warp - 4;
    const int q = warp & 3;
    const int r = q * 32 + lane;                 // token row this thread moves out of TMEM
    const int halfsel = ew >> 2;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
    const int g = lane >> 2, t = lane & 3;
    const int band = win > 0 ? win : L;
    constexpr float kLog2e = 1.4426950408889634f;
    constexpr int kChunkElems = kTileM * 8;
    uint32_t hi = 0;
    long long t_accfull = 0, t_epi = 0, t_att = 0;
    for (int ti = 0; ti < rounds; ++ti) {
      const int tile_raw = tile_of(ti);
      const bool valid = tile_raw < ntiles;
      for (int h = 0; h < kHeads; ++h, ++hi) {
        TRACE_T0();
        mbar_wait(acc_full, hi & 1);
        TRACE_ADD(t_accfull);
        tc_fence_after();
        // ---- TMEM -> bf16 -> shared memory (27 column blocks of 16: q 0-8, k 9-17, v 18-26)
        const int cb0 = halfsel ? 14 : 0, cb1 = halfsel ? 27 : 14;
#pragma unroll 2
        for (int cb = cb0; cb < cb1; ++cb) {
          uint32_t acc[16];
          tmem_ld16(tmem_row + cb * 16, acc);
          tmem_ld_wait();
          const int m = cb / 9, j = cb - m * 9;
          __nv_bfloat16* dst = sQ + (size_t)m * kTileM * kS + (size_t)r * kS;
          float v[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(acc[i]);
          *reinterpret_cast<uint4*>(dst + (2 * j) * 8) =
              make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
          *reinterpret_cast<uint4*>(dst + (2 * j + 1) * 8) =
              make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { if (leader) mbar_arrive(acc_free); else mbar_arrive_cluster(acc_free, 0); }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        TRACE_ADD(t_epi);

        // ---- banded attention of query block `ew` (rows 16*ew .. +15) from shared memory
        {
          const int i0 = ew * 16;
          const int r0 = i0 + g, r1 = r0 + 8;
          const __nv_bfloat16* q0 = sQ + (size_t)r0 * kS + 2 * t;
          const __nv_bfloat16* q1 = sQ + (size_t)r1 * kS + 2 * t;
          uint32_t qa[kDHP / 16][4];
#pragma unroll
          for (int ks = 0; ks < kDHP / 16; ++ks) {
            qa[ks][0] = *reinterpret_cast<const uint32_t*>(q0 + ks * 16);
            qa[ks][1] = *reinterpret_cast<const uint32_t*>(q1 + ks * 16);
            qa[ks][2] = *reinterpret_cast<const uint32_t*>(q0 + ks * 16 + 8);
            qa[ks][3] = *reinterpret_cast<const uint32_t*>(q1 + ks * 16 + 8);
          }
          float o[kDHP / 8][4];
#pragma unroll
          for (int nt = 0; nt < kDHP / 8; ++nt) { o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f; }
          float l0 = 0.f, l1 = 0.f;
          int jlo = i0 - band; if (jlo < 0) jlo = 0; jlo &= ~15;
          int jhi = i0 + 15 + band + 1; if (jhi > L) jhi = L;
          const int nkt = (jhi - jlo + 15) >> 4;
          constexpr int kMaxKT = 3;
          if constexpr (kTwoPass) {
            // ---- band fits in <= 3 key tiles (attn_win_size <= 16): two-pass softmax.  All score tiles
            // are computed first (independent HMMA chains), one row maximum, one exponentiation, then
            // P*V accumulates without any rescaling.
            float sc[kMaxKT][2][4];
#pragma unroll
            for (int kt = 0; kt < kMaxKT; ++kt)
#pragma unroll
              for (int nt = 0; nt < 2; ++nt) sc[kt][nt][0] = sc[kt][nt][1] = sc[kt][nt][2] = sc[kt][nt][3] = 0.f;
#pragma unroll
            for (int kt = 0; kt < kMaxKT; ++kt) {
              if (kt < nkt) {
                const int krow0 = jlo + kt * 16 + g, krow1 = krow0 + 8;
                const __nv_bfloat16* kr0 = sK + (size_t)krow0 * kS + 2 * t;
                const __nv_bfloat16* kr1 = sK + (size_t)krow1 * kS + 2 * t;
#pragma unroll
                for (int ks = 0; ks < kDHP / 16; ++ks) {
                  const uint32_t a0 = *reinterpret_cast<const uint32_t*>(kr0 + ks * 16);
                  const uint32_t a1 = *reinterpret_cast<const uint32_t*>(kr0 + ks * 16 + 8);
                  const uint32_t c0 = *reinterpret_cast<const uint32_t*>(kr1 + ks * 16);
                  const uint32_t c1 = *reinterpret_cast<const uint32_t*>(kr1 + ks * 16 + 8);
                  mma_bf16_16816(sc[kt][0], qa[ks], a0, a1);
                  mma_bf16_16816(sc[kt][1], qa[ks], c0, c1);
                }
              }
            }
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int kt = 0; kt < kMaxKT; ++kt)
#pragma unroll
              for (int nt = 0; nt < 2; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const int i = (e < 2) ? r0 : r1;
                  const int j = jlo + kt * 16 + nt * 8 + 2 * t + (e & 1);
                  const int dlt = i - j;
                  const bool ok = (kt < nkt) && (j < L) && (dlt <= band) && (dlt >= -band);
                  const float v = ok ? sc[kt][nt][e] : -INFINITY;
                  sc[kt][nt][e] = v;
                  if (e < 2) mx0 = fmaxf(mx0, v); else mx1 = fmaxf(mx1, v);
                }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
            const float base0 = mx0 == -INFINITY ? 0.f : mx0 * kLog2e, base1 = mx1 == -INFINITY ? 0.f : mx1 * kLog2e;
            uint32_t pa[kMaxKT][4];
#pragma unroll
            for (int kt = 0; kt < kMaxKT; ++kt) {
              float p[2][4];
#pragma unroll
              for (int nt = 0; nt < 2; ++nt) {
                p[nt][0] = exp2f(fmaf(sc[kt][nt][0], kLog2e, -base0));
                p[nt][1] = exp2f(fmaf(sc[kt][nt][1], kLog2e, -base0));
                p[nt][2] = exp2f(fmaf(sc[kt][nt][2], kLog2e, -base1));
                p[nt][3] = exp2f(fmaf(sc[kt][nt][3], kLog2e, -base1));
                l0 += p[nt][0] + p[nt][1];
                l1 += p[nt][2] + p[nt][3];
              }
              pa[kt][0] = pack_bf16x2(p[0][0], p[0][1]);
              pa[kt][1] = pack_bf16x2(p[0][2], p[0][3]);
              pa[kt][2] = pack_bf16x2(p[1][0], p[1][1]);
              pa[kt][3] = pack_bf16x2(p[1][2], p[1][3]);
            }
#pragma unroll
            for (int kt = 0; kt < kMaxKT; ++kt) {
              if (kt < nkt) {
                const int vrow = jlo + kt * 16 + (lane & 15);
                const uint32_t vbase = smem_u32(sV + (size_t)vrow * kS);
#pragma unroll
                for (int nt = 0; nt < kDHP / 8; ++nt) {
                  uint32_t b0, b1;
                  ldmatrix_x2_trans(b0, b1, vbase + nt * 16);
                  mma_bf16_16816(o[nt], pa[kt], b0, b1);
                }
              }
            }
          } else {
          // ---- general band (incl. full attention): online softmax over 16-key tiles
          float m0 = -INFINITY, m1 = -INFINITY;
          for (int j0 = jlo; j0 < jhi; j0 += 16) {
            float sc[2][4], sc2[2][4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
              sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
              sc2[nt][0] = sc2[nt][1] = sc2[nt][2] = sc2[nt][3] = 0.f;
            }
            const int krow0 = j0 + g, krow1 = j0 + 8 + g;
            const __nv_bfloat16* kr0 = sK + (size_t)krow0 * kS + 2 * t;
            const __nv_bfloat16* kr1 = sK + (size_t)krow1 * kS + 2 * t;
#pragma unroll
            for (int ks = 0; ks < kDHP / 16; ++ks) {
              const uint32_t a0 = *reinterpret_cast<const uint32_t*>(kr0 + ks * 16);
              const uint32_t a1 = *reinterpret_cast<const uint32_t*>(kr0 + ks * 16 + 8);
              const uint32_t c0 = *reinterpret_cast<const uint32_t*>(kr1 + ks * 16);
              const uint32_t c1 = *reinterpret_cast<const uint32_t*>(kr1 + ks * 16 + 8);
              if (ks & 1) {
                mma_bf16_16816(sc2[0], qa[ks], a0, a1);
                mma_bf16_16816(sc2[1], qa[ks], c0, c1);
              } else {
                mma_bf16_16816(sc[0], qa[ks], a0, a1);
                mma_bf16_16816(sc[1], qa[ks], c0, c1);
              }
            }
            float tmax0 = -INFINITY, tmax1 = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int i = (e < 2) ? r0 : r1;
                const int j = j0 + nt * 8 + 2 * t + (e & 1);
                const int dlt = i - j;
                const bool ok = (j < L) && (dlt <= band) && (dlt >= -band);
                sc[nt][e] = ok ? sc[nt][e] + sc2[nt][e] : -INFINITY;
              }
              tmax0 = fmaxf(tmax0, fmaxf(sc[nt][0], sc[nt][1]));
              tmax1 = fmaxf(tmax1, fmaxf(sc[nt][2], sc[nt][3]));
            }
            tmax0 = fmaxf(tmax0, __shfl_xor_sync(0xffffffffu, tmax0, 1));
            tmax0 = fmaxf(tmax0, __shfl_xor_sync(0xffffffffu, tmax0, 2));
            tmax1 = fmaxf(tmax1, __shfl_xor_sync(0xffffffffu, tmax1, 1));
            tmax1 = fmaxf(tmax1, __shfl_xor_sync(0xffffffffu, tmax1, 2));
            const float mn0 = fmaxf(m0, tmax0), mn1 = fmaxf(m1, tmax1);
            const float base0 = mn0 == -INFINITY ? 0.f : mn0, base1 = mn1 == -INFINITY ? 0.f : mn1;
            const float f0 = exp2f((m0 - base0) * kLog2e), f1 = exp2f((m1 - base1) * kLog2e);
            m0 = mn0; m1 = mn1;
            float ps0 = 0.f, ps1 = 0.f;
            uint32_t pa[4];
            {
              float p[2][4];
#pragma unroll
              for (int nt = 0; nt < 2; ++nt) {
                p[nt][0] = exp2f((sc[nt][0] - base0) * kLog2e);
                p[nt][1] = exp2f((sc[nt][1] - base0) * kLog2e);
                p[nt][2] = exp2f((sc[nt][2] - base1) * kLog2e);
                p[nt][3] = exp2f((sc[nt][3] - base1) * kLog2e);
                ps0 += p[nt][0] + p[nt][1];
                ps1 += p[nt][2] + p[nt][3];
              }
              pa[0] = pack_bf16x2(p[0][0], p[0][1]);
              pa[1] = pack_bf16x2(p[0][2], p[0][3]);
              pa[2] = pack_bf16x2(p[1][0], p[1][1]);
              pa[3] = pack_bf16x2(p[1][2], p[1][3]);
            }
            l0 = l0 * f0 + ps0;
            l1 = l1 * f1 + ps1;
            const int vrow = j0 + (lane & 15);
            const uint32_t vbase = smem_u32(sV + (size_t)vrow * kS);
#pragma unroll
            for (int nt = 0; nt < kDHP / 8; ++nt) {
              o[nt][0] *= f0; o[nt][1] *= f0; o[nt][2] *= f1; o[nt][3] *= f1;
              uint32_t b0, b1;
              ldmatrix_x2_trans(b0, b1, vbase + nt * 16);
              mma_bf16_16816(o[nt], pa, b0, b1);
            }
          }
          }
          l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
          l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
          l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
          l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
          const float inv0 = 1.f / l0, inv1 = 1.f / l1;
          if (valid) {
            __nv_bfloat16* obase = att + ((size_t)tile_raw * (kDP / 8) + h * kAttChunks) * kChunkElems + 2 * t;
#pragma unroll
            for (int nt = 0; nt < kDHP / 8; ++nt) {
              if (r0 < L)
                *reinterpret_cast<uint32_t*>(obase + (size_t)nt * kChunkElems + r0 * 8) = pack_bf16x2(o[nt][0] * inv0, o[nt][1] * inv0);
              if (r1 < L)
                *reinterpret_cast<uint32_t*>(obase + (size_t)nt * kChunkElems + r1 * 8) = pack_bf16x2(o[nt][2] * inv1, o[nt][3] * inv1);
            }
          }
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // q/k/v of this head fully consumed
        TRACE_ADD(t_att);
      }
    }
#ifdef DCB_TRACE
    if (warp == 4 && lane == 0 && blockIdx.x < 108) {
      unsigned long long* tr = g_ffn_trace + (blockIdx.x % 108 + 148) * 16;
      tr[8] = t_accfull; tr[9] = t_epi; tr[10] = t_att;
    }
#endif
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, C::kTmemCols);
  }
}

#include "stack_kernel.cuh"

// =====================================================================================
// head: final LayerNorm -> fc1 -> softmax -> argmax / Phred / ASCII
// =====================================================================================
__global__ void __launch_bounds__(128)
head_kernel(HeadParams p) {
  // logits_j = sum_c ((x_c - mean) * rstd * g_c + b_c) * W_cj + bfc_j
  //          = rstd * (sum_c y_c * (g_c W_cj) - mean_y * A_j) + B_j + bfc_j,   y = x - shift, A_j = sum_c g_c W_cj,
  //            B_j = sum_c b_c W_cj
  // so ONE pass over the row accumulates sum y, sum y^2 and the five sums y * gW_j (the residual image is read once).
  __shared__ __align__(16) float sGW[kD * 8];
  __shared__ float sA[kVocab], sBj[kVocab];
  for (int i = threadIdx.x; i < kD * 2; i += blockDim.x)
    reinterpret_cast<float4*>(sGW)[i] = __ldg(reinterpret_cast<const float4*>(p.gw8) + i);
  if (threadIdx.x < kVocab) { sA[threadIdx.x] = p.ab[threadIdx.x]; sBj[threadIdx.x] = p.ab[8 + threadIdx.x]; }
  __syncthreads();
  const int tile = blockIdx.x, r = threadIdx.x;
  const int tok = tile * kTileM + r;
  if (tok >= p.M) return;
  const int wdw = tok / p.Lw, pos = tok - wdw * p.Lw;
  if (pos >= p.L) return;                       // layout padding row
  const size_t oidx = (size_t)wdw * p.L + pos;  // outputs are dense [B, L]
  const float4* xrow = reinterpret_cast<const float4*>(p.x + (size_t)tile * x_image_elems()) + r;
  // mean / variance are biased, eps = 1e-6 (encoder_stack.py:131-133); 10 loads in flight per batch
  float s1 = 0.f, s2 = 0.f;
  float t[kVocab];
#pragma unroll
  for (int j = 0; j < kVocab; ++j) t[j] = 0.f;
  const float shift = xrow[0].x;
  constexpr int kHB = 10;
  static_assert((kD / 4) % kHB == 0, "head batch");
#pragma unroll 1
  for (int c0 = 0; c0 < kD / 4; c0 += kHB) {
    float4 v[kHB];
#pragma unroll
    for (int u = 0; u < kHB; ++u) v[u] = xrow[(size_t)(c0 + u) * kTileM];
#pragma unroll
    for (int u = 0; u < kHB; ++u) {
      const float ys[4] = {v[u].x - shift, v[u].y - shift, v[u].z - shift, v[u].w - shift};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int col = (c0 + u) * 4 + i;
        s1 += ys[i];
        s2 = fmaf(ys[i], ys[i], s2);
        const float4 w0 = *reinterpret_cast<const float4*>(&sGW[col * 8]);       // two 16-byte broadcast reads per element
        const float w4 = sGW[col * 8 + 4];
        t[0] = fmaf(ys[i], w0.x, t[0]); t[1] = fmaf(ys[i], w0.y, t[1]); t[2] = fmaf(ys[i], w0.z, t[2]);
        t[3] = fmaf(ys[i], w0.w, t[3]); t[4] = fmaf(ys[i], w4, t[4]);
      }
    }
  }
  const float m1 = s1 * (1.f / kD);             // mean of y
  const float rstd = rsqrtf(fmaxf(s2 * (1.f / kD) - m1 * m1, 0.f) + 1e-6f);
  float lg[kVocab];
#pragma unroll
  for (int j = 0; j < kVocab; ++j) lg[j] = rstd * (t[j] - m1 * sA[j]) + sBj[j];   // + fc1 bias in head_finish (networks.py:342)
  head_finish(p, lg, oidx);
}

// =====================================================================================
// launchers
// =====================================================================================
// Environment switches exist only in the developer build (-DDCB_DEV_SWITCHES, libdcb200_dev.so).
static const char* dev_env(const char* name) {
#ifdef DCB_DEV_SWITCHES
  return getenv(name);
#else
  (void)name;
  return nullptr;
#endif
}

static int g_num_sms = 0;
static int num_sms() {
  if (!g_num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

cudaError_t kernels_init() {
  cudaError_t e;
  e = cudaFuncSetAttribute(gemm_kernel<3, EPI_QKV>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           GemmCfg<3>::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(gemm_kernel<2, EPI_ROW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           GemmCfg<2>::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(ffn_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Ffn2Cfg::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(ffn_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Ffn2Cfg::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(stack_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, StackCfg::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(stack_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, StackCfg::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(qkv_attn_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, QaCfg::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(qkv_attn_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, QaCfg::kSmemBytes);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(embed_condense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024);   // + 2 KB static
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(embed_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(band_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           2 * 256 * kAttStride * 2);
  return e;
}

size_t embed_smem_bytes(int R, int echunks, int table_elems) {
  return (size_t)((table_elems * 2 + 15) & ~15) + ((echunks * 8 * sizeof(EmbedCol) + 15) & ~(size_t)15) +
         (size_t)R * kTileM * 2;
}

void launch_embed(const float* rows, int R, int L, int Lw, int M, int ntiles, int echunks,
                  const EmbedCol* cols, const EmbedRow* rowmeta, const __nv_bfloat16* tables,
                  int table_elems, __nv_bfloat16* emb, int* status, cudaStream_t st) {
  embed_rows_kernel<<<ntiles, 256, embed_smem_bytes(R, echunks, table_elems), st>>>(
      rows, R, L, Lw, M, echunks, cols, rowmeta, tables, table_elems, emb, status);
}

void launch_gemm_row(const __nv_bfloat16* a_img, const __nv_bfloat16* b_img, int ksteps, int ntiles,
                     const RowEpi& epi, cudaStream_t st) {
  const int grid = ntiles < num_sms() ? ntiles : num_sms();
  gemm_kernel<2, EPI_ROW><<<grid, 192, GemmCfg<2>::kSmemBytes, st>>>(a_img, b_img, ksteps, ntiles, 1,
                                                                     nullptr, 0, epi);
}

void launch_gemm_qkv(const __nv_bfloat16* a_img, const __nv_bfloat16* b_img, int ntiles,
                     __nv_bfloat16* qkv_img, cudaStream_t st) {
  const int items = ntiles * 2;
  const int grid = items < num_sms() ? items : num_sms();
  RowEpi none{};
  gemm_kernel<3, EPI_QKV><<<grid, 192, GemmCfg<3>::kSmemBytes, st>>>(a_img, b_img, kDP / 16, ntiles, 2,
                                                                     qkv_img, kQKVN / 8, none);
}

bool embed_condense_reads_packed(int L, int Lw) { return Lw == kTileM && (L & 3) == 0; }

bool launch_embed_condense(const float* rows, const uint8_t* packed, const PackedLayout& pl, int R, int L, int Lw, int M,
                           int ntiles, int echunks, const EmbedCol* cols,
                           const EmbedRow* rowmeta, const __nv_bfloat16* tables, int table_elems,
                           const __nv_bfloat16* wc_img, const RowEpi& epi, int* status, cudaStream_t st) {
  const size_t smem = embed_condense_smem_bytes(R, echunks, table_elems, packed ? pl.stride : 0);
  if (smem > 225 * 1024) return false;
  if (packed && !embed_condense_reads_packed(L, Lw)) return false;
  int grid = ntiles < num_sms() ? ntiles : num_sms();
  grid = (grid + 1) & ~1;           // CTA pairs (the kernel's cluster dimension)
  if (grid > (num_sms() & ~1)) grid = num_sms() & ~1;
  embed_condense_kernel<<<grid, EmbCfg::kThreads, smem, st>>>(rows, packed, pl, R, L, Lw, M, ntiles, echunks, cols, rowmeta,
                                                              tables, table_elems, wc_img, epi, status);
  return true;
}

// packed rows -> the float32 [B, R, L] rows they stand for (paths that do not read the packed form directly: strict
// fp32, L > 128 / L % 4 != 0, the developer build's unfused kernels)
__global__ void __launch_bounds__(256)
unpack_rows_kernel(const uint8_t* __restrict__ packed, PackedLayout pl, int nwindows, float* __restrict__ rows) {
  const int b = blockIdx.x;
  const uint8_t* w = packed + (size_t)b * pl.stride;
  float* out = rows + (size_t)b * pl.R * pl.L;
  for (int i = threadIdx.x; i < pl.R * pl.L; i += blockDim.x) {
    const int r = i / pl.L, l = i - r * pl.L;
    out[i] = packed_value(pl, w, r, l);
  }
}

void launch_unpack_rows(const uint8_t* packed, const PackedLayout& pl, int nwindows, float* rows, cudaStream_t st) {
  if (nwindows > 0) unpack_rows_kernel<<<nwindows, 256, 0, st>>>(packed, pl, nwindows, rows);
}

void launch_qkv_attn(const __nv_bfloat16* a_img, const uint8_t* w_img, int ntiles, int L, int win,
                     __nv_bfloat16* att, cudaStream_t st) {
  static int max_pairs = 0;
  cudaLaunchConfig_t cfg{};
  cfg.blockDim = dim3(QaCfg::kThreads);
  cfg.dynamicSmemBytes = QaCfg::kSmemBytes;
  cfg.stream = st;
  if (!max_pairs) {
    cfg.gridDim = dim3(num_sms() / 2 * 2);
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, qkv_attn_pair_kernel<true>, &cfg) != cudaSuccess || nc <= 0) nc = num_sms() / 2;
    max_pairs = nc;
  }
  int pairs = (ntiles + 1) / 2;
  if (pairs > max_pairs) pairs = max_pairs;
  cfg.gridDim = dim3(pairs * 2);
  if (win > 0 && win <= 16) cudaLaunchKernelEx(&cfg, qkv_attn_pair_kernel<true>, a_img, w_img, ntiles, L, win, att);
  else cudaLaunchKernelEx(&cfg, qkv_attn_pair_kernel<false>, a_img, w_img, ntiles, L, win, att);
}

void launch_stack(float* x, int ntiles, int L, int win, const StackParams& p, const HeadParams& hp, cudaStream_t st) {
  static int max_pairs = 0;
  cudaLaunchConfig_t cfg{};
  cfg.blockDim = dim3(StackCfg::kThreads);
  cfg.dynamicSmemBytes = StackCfg::kSmemBytes;
  cfg.stream = st;
  if (!max_pairs) {
    cfg.gridDim = dim3(num_sms() / 2 * 2);
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, stack_pair_kernel<false>, &cfg) != cudaSuccess || nc <= 0) nc = num_sms() / 2;
    max_pairs = nc;
    if (dev_env("DCB_VERBOSE")) fprintf(stderr, "[dcb200] stack kernel: %d co-resident CTA pairs\n", nc);
  }
  int pairs = (ntiles + 1) / 2;
  if (pairs > max_pairs) pairs = max_pairs;
  cfg.gridDim = dim3(pairs * 2);
  if (L > kTileM) cudaLaunchKernelEx(&cfg, stack_pair_kernel<true>, x, ntiles, L, win, p, hp);   // one window per CTA pair
  else cudaLaunchKernelEx(&cfg, stack_pair_kernel<false>, x, ntiles, L, win, p, hp);
}

void launch_attention(const __nv_bfloat16* qkv, __nv_bfloat16* att, int L, int Lw, int win, int nwindows,
                      cudaStream_t st) {
  const int Lp = (L + 15) & ~15;
  const size_t smem = (size_t)2 * Lp * kAttStride * 2;
  band_attention_kernel<<<nwindows * 2, 128, smem, st>>>(qkv, att, L, Lw, win, nwindows);
}

void launch_ffn_pair(const __nv_bfloat16* a_img, const uint8_t* w2img, const float* b1, int ff, int ntiles,
                     const RowEpi& epi, cudaStream_t st, const uint8_t* wo2img, const float* mid_ln_g,
                     const float* mid_ln_b) {
  static int max_pairs = 0;
  cudaLaunchConfig_t cfg{};
  cfg.blockDim = dim3(kFfnThreads);
  cfg.dynamicSmemBytes = Ffn2Cfg::kSmemBytes;
  cfg.stream = st;
  if (!max_pairs) {
    cfg.gridDim = dim3(num_sms() / 2 * 2);
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, ffn_pair_kernel<false>, &cfg) != cudaSuccess || nc <= 0) nc = num_sms() / 2;
    max_pairs = nc;
    if (const char* env = dev_env("DCB_FFN_MAX_PAIRS")) { const int v = atoi(env); if (v > 0 && v < max_pairs) max_pairs = v; }
    if (dev_env("DCB_VERBOSE")) fprintf(stderr, "[dcb200] ffn pair kernel: %d co-resident CTA pairs\n", nc);
  }
  int pairs = (ntiles + 1) / 2;
  if (pairs > max_pairs) pairs = max_pairs;
  cfg.gridDim = dim3(pairs * 2);
  static int stagger = -1;
  if (stagger < 0) { const char* env = dev_env("DCB_FFN_STAGGER"); stagger = env ? atoi(env) : 0; }
  if (wo2img)
    cudaLaunchKernelEx(&cfg, ffn_pair_kernel<true>, a_img, w2img, b1, ff, ntiles, epi, stagger, wo2img, mid_ln_g, mid_ln_b);
  else
    cudaLaunchKernelEx(&cfg, ffn_pair_kernel<false>, a_img, w2img, b1, ff, ntiles, epi, stagger, wo2img, mid_ln_g, mid_ln_b);
}

int read_ffn_trace(unsigned long long* out, int n) {
  if (n > 256 * 16) n = 256 * 16;
  return cudaMemcpyFromSymbol(out, g_ffn_trace, (size_t)n * sizeof(unsigned long long)) == cudaSuccess ? 0 : -1;
}

// =====================================================================================
// stitch: per-read concatenation of windows + gap compaction (stitch_utils.py:51-98)
// =====================================================================================
// One CTA per read (ZMW).  Its windows are contiguous in the batch, so the read's input is one span of bytes
// [read_off[z], read_off[z + 1]) in `bases` / `quals` (windows of max_length bytes, or of their own width when CCS smart
// windows overflow); the gap character ' ' and the quality character under it are dropped (order preserving:
// ballot-free block prefix sum over 1024-character tiles) and the compacted read is written at the same offset of
// seq_out / qual_out.  Offsets are int64 (a batch may exceed 2 GiB of window bytes); one read stays below 2^31 bytes.  Integer / byte work only: bit-exact against the reference's string loops.
__global__ void __launch_bounds__(256)
stitch_kernel(const uint8_t* __restrict__ bases, const uint8_t* __restrict__ quals,
              const int64_t* __restrict__ read_off, uint8_t* __restrict__ seq_out, uint8_t* __restrict__ qual_out,
              int32_t* __restrict__ len_out) {
  __shared__ int s_warp[8];
  __shared__ int s_total;
  const int z = blockIdx.x;
  const int64_t off = read_off[z];
  const int n = (int)(read_off[z + 1] - off);
  const uint8_t* in_b = bases + off;
  const uint8_t* in_q = quals + off;
  uint8_t* out_b = seq_out + off;
  uint8_t* out_q = qual_out + off;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int running = 0;
  for (int t0 = 0; t0 < n; t0 += 1024) {
    uint8_t b[4], q[4];
    int cnt = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int idx = t0 + threadIdx.x * 4 + k;
      b[k] = idx < n ? in_b[idx] : (uint8_t)' ';
      q[k] = idx < n ? in_q[idx] : (uint8_t)0;
      cnt += b[k] != (uint8_t)' ';
    }
    // inclusive scan inside the warp, then across the 8 warps
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
      int acc = 0;
      for (int w = 0; w < 8; ++w) { const int v = s_warp[w]; s_warp[w] = acc; acc += v; }
      s_total = acc;
    }
    __syncthreads();
    int pos = running + s_warp[warp] + incl - cnt;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (b[k] != (uint8_t)' ') {
        out_b[pos] = b[k];
        out_q[pos] = q[k];
        ++pos;
      }
    }
    running += s_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) len_out[z] = running;
}

void launch_stitch(const uint8_t* bases, const uint8_t* quals, const int64_t* read_off, int n_zmw,
                   uint8_t* seq_out, uint8_t* qual_out, int32_t* len_out, cudaStream_t st) {
  if (n_zmw > 0) stitch_kernel<<<n_zmw, 256, 0, st>>>(bases, quals, read_off, seq_out, qual_out, len_out);
}

void launch_head(const HeadParams& p, int ntiles, cudaStream_t st) {
  head_kernel<<<ntiles, 128, 0, st>>>(p);
}

}  // namespace dcb

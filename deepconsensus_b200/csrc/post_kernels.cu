// Post-model stage of the path on the device (SURVEY.md section 8(f)2): what `stitch_utils.stitch_to_fastq` and the
// skip branch of `inference_on_n_zmws` do per read / per window after the model, as integer / byte kernels.
//
//   read_outcome_kernel   per read: missing-window check of get_full_sequence (stitch_utils.py:60-78), only-gaps check,
//                         avg-Phred quality filter (utils.py:88-106, stitch_utils.py:101-109) and length filter
//                         (stitch_utils.py:131-189) on the compacted read dcb_stitch's kernel wrote -> outcome code
//   fastq_layout_kernel   exclusive scan of the record lengths of the reads that pass -> byte offsets
//   fastq_write_kernel    '@' name '\n' sequence "\n+\n" quality '\n' (format_as_fastq, stitch_utils.py:112-119)
//   skip_mask_kernel      avg_phred(ccs_base_quality_scores) > skip_windows_above (quick_inference.py:663-672)
//   fill_skipped_kernel   process_skipped_window (quick_inference.py:567-594): skipped windows adopt the CCS bases and
//                         the (calibrated, capped) CCS base qualities, written straight into the output arrays
//
// avg_phred is -10 log10(mean 10^(-q/10)) in float64.  The qualities are small integers, so the mean is formed from an
// exact integer histogram times a table of 10^(-q/10) (the table comes from the host's libm `pow`, the function NumPy
// calls).  NumPy sums the per-base terms pairwise instead, so the two float64 means can differ in the last bits; every
// decision that lies within 1e-7 of its threshold is therefore flagged DCB_READ_BORDERLINE / mask value 2 and the host
// re-evaluates it with the reference's NumPy expression (deepconsensus_b200/stitch_gpu.py) -- decisions are identical
// to the reference's by construction, and the byte work is bit-exact.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/dcb200.h"
#include "kernels.h"

namespace dcb {

__global__ void __launch_bounds__(256)
read_outcome_kernel(const uint8_t* __restrict__ qual, const int32_t* __restrict__ len, const int64_t* __restrict__ read_off,
                    const int32_t* __restrict__ zmw_start, const int32_t* __restrict__ window_pos, int L, const double* __restrict__ p10, double min_quality,
                    int min_length, int32_t* __restrict__ outcome, double* __restrict__ avg_q_out) {
  __shared__ int s_hist[256];
  __shared__ int s_missing;
  const int z = blockIdx.x;
  const int w0 = zmw_start[z], w1 = zmw_start[z + 1];
  s_hist[threadIdx.x] = 0;
  if (threadIdx.x == 0) s_missing = 0;
  __syncthreads();
  // get_full_sequence: window i of the read must not start beyond i * max_length (a window is missing otherwise) --
  // whatever the widths of the windows before it (stitch_utils.py:60-78 advances by max_length per window)
  for (int i = threadIdx.x; i < w1 - w0; i += blockDim.x)
    if (window_pos[w0 + i] > i * L) s_missing = 1;
  const int n = len[z];
  const uint8_t* q = qual + read_off[z];
  for (int i = threadIdx.x; i < n; i += blockDim.x) atomicAdd(&s_hist[q[i]], 1);   // integer atomics: exact
  __syncthreads();
  if (threadIdx.x != 0) return;
  int code;
  double avg_q = 0.0;
  if (s_missing || w1 == w0 || read_off[z + 1] == read_off[z]) code = DCB_READ_EMPTY;   // `not full_seq`
  else if (n == 0) code = DCB_READ_ONLY_GAPS;
  else {
    // quality_string_to_array subtracts 33; entries < 0 are dropped by avg_phred (none can be: chars >= '!')
    int nonzero = 0, cnt = 0;
    double s = 0.0;
    for (int c = 33; c < 256; ++c)
      if (s_hist[c]) { cnt += s_hist[c]; if (c > 33) nonzero = 1; s += (double)s_hist[c] * p10[c - 33]; }
    if (nonzero && cnt > 0) avg_q = -10.0 * log10(s / (double)cnt);
    const double thr = min_quality - 5e-6;                 // round(avg_q, 5) >= min_quality
    // within 1e-7 of the threshold the host re-evaluates with the reference's NumPy expression: the read is treated
    // as passing the quality filter here (its record is written) and flagged
    const bool border = fabs(avg_q - thr) < 1e-7;
    const bool pass_q = border || avg_q >= thr;
    code = !pass_q ? DCB_READ_LOW_QUALITY : (n < min_length ? DCB_READ_TOO_SHORT : DCB_READ_OK);
    if (border) code |= DCB_READ_BORDERLINE;
  }
  outcome[z] = code;
  avg_q_out[z] = avg_q;
}

// one block: record length of every read that is written (OK, possibly borderline), exclusive scan -> offsets
__global__ void __launch_bounds__(1024)
fastq_layout_kernel(const int32_t* __restrict__ len, const int32_t* __restrict__ outcome, const int32_t* __restrict__ name_off,
                    int n_zmw, int64_t* __restrict__ rec_off) {
  __shared__ long long s_part[1024];
  const int per = (n_zmw + 1023) / 1024;
  const int lo = threadIdx.x * per, hi = min(n_zmw, lo + per);
  long long local = 0;
  for (int z = lo; z < hi; ++z) {
    const bool ok = (outcome[z] & 0x7f) == DCB_READ_OK;
    local += ok ? (long long)(name_off[z + 1] - name_off[z]) + 2ll * len[z] + 6 : 0;   // '@' '\n' '\n' '+' '\n' '\n'
  }
  s_part[threadIdx.x] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long acc = 0;
    for (int i = 0; i < 1024; ++i) { const long long v = s_part[i]; s_part[i] = acc; acc += v; }
    rec_off[n_zmw] = acc;
  }
  __syncthreads();
  long long off = s_part[threadIdx.x];
  for (int z = lo; z < hi; ++z) {
    rec_off[z] = off;
    const bool ok = (outcome[z] & 0x7f) == DCB_READ_OK;
    off += ok ? (long long)(name_off[z + 1] - name_off[z]) + 2ll * len[z] + 6 : 0;
  }
}

__global__ void __launch_bounds__(256)
fastq_write_kernel(const uint8_t* __restrict__ seq, const uint8_t* __restrict__ qual, const int32_t* __restrict__ len,
                   const int64_t* __restrict__ read_off, const int32_t* __restrict__ outcome,
                   const uint8_t* __restrict__ names, const int32_t* __restrict__ name_off,
                   const int64_t* __restrict__ rec_off, uint8_t* __restrict__ fastq, int64_t cap) {
  const int z = blockIdx.x;
  if ((outcome[z] & 0x7f) != DCB_READ_OK) return;
  const int n = len[z], nl = name_off[z + 1] - name_off[z];
  const int64_t o = rec_off[z];
  if (o + nl + 2ll * n + 6 > cap) return;                  // caller sized the buffer too small: rec_off[n_zmw] tells
  const uint8_t* s = seq + read_off[z];
  const uint8_t* q = qual + read_off[z];
  const uint8_t* nm = names + name_off[z];
  uint8_t* out = fastq + o;
  if (threadIdx.x == 0) {
    out[0] = '@'; out[1 + nl] = '\n'; out[2 + nl + n] = '\n'; out[3 + nl + n] = '+'; out[4 + nl + n] = '\n';
    out[5 + nl + 2 * n] = '\n';
  }
  for (int i = threadIdx.x; i < nl; i += blockDim.x) out[1 + i] = nm[i];
  for (int i = threadIdx.x; i < n; i += blockDim.x) { out[2 + nl + i] = s[i]; out[5 + nl + n + i] = q[i]; }
}

// one warp per window: avg_phred of the window's CCS base qualities (-1 entries dropped) > threshold
__global__ void __launch_bounds__(256)
skip_mask_kernel(const int16_t* __restrict__ ccs_bq, int n_windows, int L, const double* __restrict__ p10, double thr,
                 uint8_t* __restrict__ mask, double* __restrict__ avg_out) {
  const int w = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= n_windows) return;
  const int16_t* q = ccs_bq + (size_t)w * L;
  double s = 0.0;
  int cnt = 0, nonzero = 0;
  for (int i = lane; i < L; i += 32) {
    const int v = q[i];
    if (v >= 0) { ++cnt; nonzero |= v != 0; s += p10[v > 255 ? 255 : v]; }
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {               // fixed butterfly order: deterministic
    s += __shfl_xor_sync(0xffffffffu, s, d);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
    nonzero |= __shfl_xor_sync(0xffffffffu, nonzero, d);
  }
  if (lane) return;
  const double avg = (nonzero && cnt) ? -10.0 * log10(s / (double)cnt) : 0.0;
  mask[w] = fabs(avg - thr) < 1e-7 ? 2 : (avg > thr ? 1 : 0);
  if (avg_out) avg_out[w] = avg;
}

// process_skipped_window for k windows, one warp per window: window j (source bytes [src_off[j], src_off[j + 1]), max_length
// of them, or its own width for an overflow window) goes to the output bytes from dst_off[j]
__global__ void __launch_bounds__(256)
fill_skipped_kernel(const uint8_t* __restrict__ ccs_ids, const int16_t* __restrict__ ccs_bq,
                    const int64_t* __restrict__ src_off, const int64_t* __restrict__ dst_off,
                    int k, int calib_enabled, double thr, double cw, double cb, int max_q,
                    uint8_t* __restrict__ bases, uint8_t* __restrict__ quals, int* __restrict__ status) {
  const char vocab[5] = {' ', 'A', 'T', 'C', 'G'};
  const int j = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (j >= k) return;
  const int64_t s0 = src_off[j], width = src_off[j + 1] - s0, d0 = dst_off[j];
  for (int64_t l = threadIdx.x & 31; l < width; l += 32) {
    const int64_t i = s0 + l;
    int id = ccs_ids[i];
    if (id > 4) { atomicOr(status, 1); id = 4; }
    const int qraw = ccs_bq[i];
    int qi;
    if (calib_enabled) {
      // calibrate_quality_scores on an integer array: float64 throughout (calibration_lib.py:89-99)
      double qd = (double)qraw;
      if (thr == 0.0) qd = qd * cw + cb;
      else { const bool above = qd > thr; qd = qd * (above ? cw : 1.0) + (above ? cb : 0.0); }
      qd = fmin(qd, (double)max_q);                    // np.minimum
      qi = (int)qd;                                     // astype(int32): truncation
    } else {
      qi = qraw < max_q ? qraw : max_q;
    }
    const int64_t o = d0 + l;
    bases[o] = (uint8_t)vocab[id];
    quals[o] = (uint8_t)(qi + 33);                      // quality_scores_to_string (utils.py:60-62)
  }
}

void launch_read_outcome(const uint8_t* qual, const int32_t* len, const int64_t* read_off, const int32_t* zmw_start,
                         const int32_t* window_pos, int L, int n_zmw, const double* p10, double min_quality,
                         int min_length, int32_t* outcome, double* avg_q, cudaStream_t st) {
  if (n_zmw > 0)
    read_outcome_kernel<<<n_zmw, 256, 0, st>>>(qual, len, read_off, zmw_start, window_pos, L, p10, min_quality, min_length,
                                               outcome, avg_q);
}

void launch_fastq(const uint8_t* seq, const uint8_t* qual, const int32_t* len, const int64_t* read_off, int n_zmw,
                  const int32_t* outcome, const uint8_t* names, const int32_t* name_off, int64_t* rec_off, uint8_t* fastq,
                  int64_t cap, cudaStream_t st) {
  if (n_zmw <= 0) return;
  fastq_layout_kernel<<<1, 1024, 0, st>>>(len, outcome, name_off, n_zmw, rec_off);
  fastq_write_kernel<<<n_zmw, 256, 0, st>>>(seq, qual, len, read_off, outcome, names, name_off, rec_off, fastq, cap);
}

void launch_skip_mask(const int16_t* ccs_bq, int n_windows, int L, const double* p10, double thr, uint8_t* mask,
                      double* avg_out, cudaStream_t st) {
  if (n_windows > 0) skip_mask_kernel<<<(n_windows + 7) / 8, 256, 0, st>>>(ccs_bq, n_windows, L, p10, thr, mask, avg_out);
}

void launch_fill_skipped(const uint8_t* ccs_ids, const int16_t* ccs_bq, const int64_t* src_off, const int64_t* dst_off, int k,
                         int calib_enabled, double thr, double cw, double cb, int max_q, uint8_t* bases, uint8_t* quals,
                         int* status, cudaStream_t st) {
  if (k <= 0) return;
  fill_skipped_kernel<<<(k + 7) / 8, 256, 0, st>>>(ccs_ids, ccs_bq, src_off, dst_off, k, calib_enabled, thr, cw, cb, max_q,
                                                    bases, quals, status);
}

}  // namespace dcb

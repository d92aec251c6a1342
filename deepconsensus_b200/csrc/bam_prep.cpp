// Feature construction from BAM, htslib-free (SURVEY.md section 8(f)3 + the producer half of 8(f)1): the part of
// `deepconsensus run` that sits in front of the model path, as host C++ behind the C ABI (include/dcb200.h "dcb_prep_*",
// "dcb_bamw_*").
//
//   BGZF / BAM reader            what pysam.AlignmentFile does for pre_lib.py:50-91,1279-1367 (SAM/BAM spec v1.6 section 4)
//   SubreadGrouper               pre_lib.py:50-91     mapped subreads of one ZMW (`zm` tag), in file order
//   trim_insertions              pre_lib.py:1061-1125 insertions longer than ins_trim removed from seq / cigar / pw / ip
//   expand_clip_indent           pre_lib.py:1128-1239 gaps at deletions, soft clips removed, indent to the CCS start,
//                                                     pw / ip reversed for reverse-strand alignments
//   construct_ccs_read           pre_lib.py:966-998
//   space_out_subreads           pre_lib.py:1242-1276 columns opened in every read wherever any read has an insertion
//   DcExample.iter_examples /    pre_lib.py:625-744   windows of max_length columns (or of the CCS record's `wl` widths),
//                                                     padding, the [R, L] feature rows --
//   extract_features                                  written as float32 rows AND as packed rows (dcb_pack_rows' format)
//   unaligned BAM writer         quick_inference.py:740-760,892-897  (ec, np, rq, RG, zm tags; the CCS BAM's header)
//
// Pinned against the reference's own fixture: the windows built here from testdata/human_1m/{subreads_to_ccs,ccs}.bam
// equal, value for value, the 1 593 examples of testdata/human_1m/tf_examples/inference/inference.tfrecord.gz that the
// reference's preprocess wrote from the same BAMs (tests/test_bam_prep.py).
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <zlib.h>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/dcb200.h"
#include "common.h"

namespace {

thread_local std::string g_prep_error;

int pfail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_prep_error = buf;
  return code;
}

// ----------------------------------------------------------------------------------------------- BGZF reader
struct Bgzf {
  FILE* f = nullptr;
  std::vector<uint8_t> block;   // inflated current block
  size_t pos = 0;
  bool fail = false;
  ~Bgzf() { if (f) fclose(f); }
  bool next_block() {
    uint8_t h[12];
    size_t n = fread(h, 1, 12, f);
    if (n == 0) return false;                       // clean EOF
    if (n != 12 || h[0] != 31 || h[1] != 139 || h[2] != 8 || !(h[3] & 4)) { fail = true; return false; }
    const int xlen = h[10] | (h[11] << 8);
    std::vector<uint8_t> extra(xlen);
    if (fread(extra.data(), 1, xlen, f) != (size_t)xlen) { fail = true; return false; }
    int bsize = -1;
    for (int i = 0; i + 4 <= xlen;) {
      const int slen = extra[i + 2] | (extra[i + 3] << 8);
      if (extra[i] == 'B' && extra[i + 1] == 'C' && slen == 2) bsize = extra[i + 4] | (extra[i + 5] << 8);
      i += 4 + slen;
    }
    if (bsize < 0) { fail = true; return false; }
    const int clen = bsize - xlen - 19;
    if (clen < 0) { fail = true; return false; }
    std::vector<uint8_t> comp(clen + 8);
    if (fread(comp.data(), 1, clen + 8, f) != (size_t)clen + 8) { fail = true; return false; }
    const uint32_t isize = comp[clen + 4] | (comp[clen + 5] << 8) | (comp[clen + 6] << 16) | ((uint32_t)comp[clen + 7] << 24);
    block.resize(isize);
    pos = 0;
    if (isize == 0) return true;                    // the EOF marker block (or an empty block)
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) { fail = true; return false; }
    zs.next_in = comp.data(); zs.avail_in = clen;
    zs.next_out = block.data(); zs.avail_out = isize;
    const int rc = inflate(&zs, Z_FINISH);
    inflateEnd(&zs);
    if (rc != Z_STREAM_END || zs.total_out != isize) { fail = true; return false; }
    const uint32_t crc = comp[clen] | (comp[clen + 1] << 8) | (comp[clen + 2] << 16) | ((uint32_t)comp[clen + 3] << 24);
    if ((uint32_t)crc32(0, block.data(), isize) != crc) { fail = true; return false; }
    return true;
  }
  // 1 = ok, 0 = clean EOF before any byte, -1 = error / truncated
  int read(void* dst, size_t n) {
    uint8_t* d = static_cast<uint8_t*>(dst);
    size_t got = 0;
    while (got < n) {
      if (pos == block.size()) {
        if (!next_block()) return (got == 0 && !fail) ? 0 : -1;
        continue;
      }
      const size_t take = std::min(n - got, block.size() - pos);
      memcpy(d + got, block.data() + pos, take);
      pos += take; got += take;
    }
    return 1;
  }
};

struct Tag { char type = 0, sub = 0; const uint8_t* p = nullptr; size_t count = 0; };

struct BamRecord {
  std::string qname, seq;
  int32_t refid = -1, pos = -1;
  uint16_t flag = 0;
  std::vector<uint32_t> cigar;        // len << 4 | op
  std::vector<uint8_t> qual, aux;
  bool find(const char* name, Tag* t) const {
    size_t i = 0;
    const size_t n = aux.size();
    while (i + 3 <= n) {
      const bool hit = aux[i] == (uint8_t)name[0] && aux[i + 1] == (uint8_t)name[1];
      const char ty = (char)aux[i + 2];
      i += 3;
      size_t len = 0, cnt = 1;
      char sub = 0;
      switch (ty) {
        case 'A': case 'c': case 'C': len = 1; break;
        case 's': case 'S': len = 2; break;
        case 'i': case 'I': case 'f': len = 4; break;
        case 'Z': case 'H': { size_t j = i; while (j < n && aux[j]) ++j; len = j - i + 1; break; }
        case 'B': {
          if (i + 5 > n) return false;
          sub = (char)aux[i];
          cnt = aux[i + 1] | (aux[i + 2] << 8) | (aux[i + 3] << 16) | ((size_t)aux[i + 4] << 24);
          const size_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
          i += 5; len = es * cnt; break;
        }
        default: return false;
      }
      if (i + len > n) return false;
      if (hit) { t->type = ty; t->sub = sub; t->p = aux.data() + i; t->count = cnt; return true; }
      i += len;
    }
    return false;
  }
  static double scalar(const Tag& t) {
    switch (t.type) {
      case 'c': return (int8_t)t.p[0];
      case 'C': return t.p[0];
      case 's': { int16_t v; memcpy(&v, t.p, 2); return v; }
      case 'S': { uint16_t v; memcpy(&v, t.p, 2); return v; }
      case 'i': { int32_t v; memcpy(&v, t.p, 4); return v; }
      case 'I': { uint32_t v; memcpy(&v, t.p, 4); return v; }
      case 'f': { float v; memcpy(&v, t.p, 4); return v; }
      default: return 0;
    }
  }
  static double element(const Tag& t, size_t i) {
    switch (t.sub) {
      case 'c': return (int8_t)t.p[i];
      case 'C': return t.p[i];
      case 's': { int16_t v; memcpy(&v, t.p + 2 * i, 2); return v; }
      case 'S': { uint16_t v; memcpy(&v, t.p + 2 * i, 2); return v; }
      case 'i': { int32_t v; memcpy(&v, t.p + 4 * i, 4); return v; }
      case 'I': { uint32_t v; memcpy(&v, t.p + 4 * i, 4); return v; }
      case 'f': { float v; memcpy(&v, t.p + 4 * i, 4); return v; }
      default: return 0;
    }
  }
};

struct BamReader {
  Bgzf z;
  std::string header_text;
  std::vector<std::string> refs;
  std::vector<int32_t> ref_len;
  int open(const char* path) {
    z.f = fopen(path, "rb");
    if (!z.f) return pfail(DCB_ERR_INVALID, "cannot open %s", path);
    char magic[4];
    int32_t l_text, n_ref;
    if (z.read(magic, 4) != 1 || memcmp(magic, "BAM\1", 4) || z.read(&l_text, 4) != 1 || l_text < 0)
      return pfail(DCB_ERR_INVALID, "%s: not a BAM file", path);
    header_text.resize(l_text);
    if (l_text && z.read(&header_text[0], l_text) != 1) return pfail(DCB_ERR_INVALID, "%s: truncated header", path);
    while (!header_text.empty() && header_text.back() == '\0') header_text.pop_back();
    if (z.read(&n_ref, 4) != 1 || n_ref < 0) return pfail(DCB_ERR_INVALID, "%s: truncated header", path);
    for (int i = 0; i < n_ref; ++i) {
      int32_t l_name, l_ref;
      if (z.read(&l_name, 4) != 1 || l_name <= 0) return pfail(DCB_ERR_INVALID, "%s: bad reference list", path);
      std::string nm(l_name, '\0');
      if (z.read(&nm[0], l_name) != 1 || z.read(&l_ref, 4) != 1) return pfail(DCB_ERR_INVALID, "%s: bad reference list", path);
      nm.resize(strlen(nm.c_str()));
      refs.push_back(nm);
      ref_len.push_back(l_ref);
    }
    return DCB_OK;
  }
  // 1 = record, 0 = EOF, < 0 = error
  int next(BamRecord* r) {
    int32_t bs;
    const int rc = z.read(&bs, 4);
    if (rc == 0) return 0;
    if (rc < 0 || bs < 32) return pfail(DCB_ERR_INVALID, "truncated BAM record");
    if (bs > (64 << 20)) return pfail(DCB_ERR_INVALID, "implausible BAM record size %d", bs);
    std::vector<uint8_t> b(bs);
    if (z.read(b.data(), bs) != 1) return pfail(DCB_ERR_INVALID, "truncated BAM record");
    int32_t l_seq;
    uint16_t n_cig;
    memcpy(&r->refid, &b[0], 4);
    memcpy(&r->pos, &b[4], 4);
    const int l_name = b[8];
    memcpy(&n_cig, &b[12], 2);
    memcpy(&r->flag, &b[14], 2);
    memcpy(&l_seq, &b[16], 4);
    if (l_seq < 0) return pfail(DCB_ERR_INVALID, "corrupt BAM record");
    size_t o = 32;
    if (o + l_name + 4ull * n_cig + (l_seq + 1) / 2 + l_seq > (size_t)bs) return pfail(DCB_ERR_INVALID, "corrupt BAM record");
    r->qname.assign(reinterpret_cast<const char*>(&b[o]), l_name ? l_name - 1 : 0);
    o += l_name;
    r->cigar.resize(n_cig);
    if (n_cig) memcpy(r->cigar.data(), &b[o], 4ull * n_cig);
    o += 4ull * n_cig;
    static const char kNt[] = "=ACMGRSVTWYHKDBN";
    r->seq.resize(l_seq);
    for (int i = 0; i < l_seq; ++i) r->seq[i] = kNt[(b[o + i / 2] >> (i & 1 ? 0 : 4)) & 15];
    o += (l_seq + 1) / 2;
    r->qual.assign(b.begin() + o, b.begin() + o + l_seq);
    o += l_seq;
    r->aux.assign(b.begin() + o, b.end());
    return 1;
  }
};

// ----------------------------------------------------------------------------------------------- Read (pre_lib.py:111-421)
constexpr uint8_t kCMatch = 0, kCIns = 1, kCDel = 2, kCRefSkip = 3, kCSoft = 4, kCHard = 5, kCPad = 6, kCEq = 7, kCDiff = 8;
constexpr char kGap = ' ';

struct Read {
  std::string name;
  std::vector<char> bases;
  std::vector<uint8_t> cigar, pw, ip;
  float sn[4] = {0, 0, 0, 0};
  int strand = 0;                       // dc_constants.Strand: 0 unknown, 1 forward, 2 reverse
  std::vector<int32_t> ccs_idx;
  std::vector<int32_t> bq;              // base_quality_scores (CCS read only)
  bool bq_any = false;                  // `base_quality_scores.any()`: spacing only applies then (pre_lib.py:247-250)
  // spacing state (pre_lib.py:176-216)
  std::vector<int32_t> seq_indices;
  size_t idx_seq = 0;
  int32_t idx_spaced = 0;
  bool done = false;
};

// pysam get_aligned_pairs(): (query index | -1, reference index | -1) per alignment column; H and P give no column
void aligned_pairs(const std::vector<uint32_t>& cigar, int32_t pos, std::vector<int32_t>* qidx, std::vector<int32_t>* ridx) {
  int32_t q = 0, r = pos;
  for (uint32_t c : cigar) {
    const int op = c & 15;
    const int len = (int)(c >> 4);
    switch (op) {
      case kCMatch: case kCEq: case kCDiff: for (int i = 0; i < len; ++i) { qidx->push_back(q++); ridx->push_back(r++); } break;
      case kCIns: case kCSoft: for (int i = 0; i < len; ++i) { qidx->push_back(q++); ridx->push_back(-1); } break;
      case kCDel: case kCRefSkip: for (int i = 0; i < len; ++i) { qidx->push_back(-1); ridx->push_back(r++); } break;
      default: break;
    }
  }
}

// trim_insertions (pre_lib.py:1061-1125), literally: an insertion longer than ins_trim disappears from the sequence, the
// cigar and the kinetics; every other operation except a deletion advances the sequence position by its length
void trim_insertions(BamRecord* r, std::vector<double>* pw, std::vector<double>* ip, int ins_trim) {
  if (ins_trim <= 0) return;
  std::vector<uint32_t> cig;
  std::string seq;
  std::vector<char> mask(r->seq.size(), 1);
  size_t sp = 0;
  for (uint32_t c : r->cigar) {
    const int op = c & 15;
    const size_t len = c >> 4;
    if (op == kCIns && (int)len > ins_trim) {
      for (size_t i = sp; i < sp + len && i < mask.size(); ++i) mask[i] = 0;
      sp += len;
    } else {
      cig.push_back(c);
      if (op != kCDel) {
        seq += r->seq.substr(std::min(sp, r->seq.size()), len);
        sp += len;
      }
    }
  }
  const bool rev = r->flag & 16;
  auto filter = [&](std::vector<double>* v) {
    if (v->empty()) return;
    std::vector<double> out;
    const size_t n = mask.size();
    for (size_t i = 0; i < v->size() && i < n; ++i)
      if (rev ? mask[n - 1 - i] : mask[i]) out.push_back((*v)[i]);
    v->swap(out);
  };
  filter(pw);
  filter(ip);
  r->seq = seq;
  r->cigar = cig;
}

int expand_clip_indent(BamRecord* rec, int ins_trim, Read* out) {
  Tag t;
  std::vector<double> pw, ip;
  if (rec->find("pw", &t) && t.type == 'B') { pw.resize(t.count); for (size_t i = 0; i < t.count; ++i) pw[i] = BamRecord::element(t, i); }
  if (rec->find("ip", &t) && t.type == 'B') { ip.resize(t.count); for (size_t i = 0; i < t.count; ++i) ip[i] = BamRecord::element(t, i); }
  {
    // sanity before anything is sized from the record: alignments to a CCS read span at most a few hundred kilobases
    uint64_t cols = 0;
    for (uint32_t c : rec->cigar) cols += c >> 4;
    if (cols > (1u << 24) || rec->pos < 0 || rec->pos > (1 << 24))
      return pfail(DCB_ERR_INVALID, "%s: implausible alignment (cigar / position)", rec->qname.c_str());
  }
  trim_insertions(rec, &pw, &ip, ins_trim);
  std::vector<int32_t> read_idx, ccs_idx;
  aligned_pairs(rec->cigar, rec->pos, &read_idx, &ccs_idx);
  const size_t aln = read_idx.size();
  std::vector<char> seq(aln, kGap);
  std::vector<uint8_t> npw(aln, 0), nip(aln, 0);
  const bool rev = rec->flag & 16;
  if (rev) { std::reverse(pw.begin(), pw.end()); std::reverse(ip.begin(), ip.end()); }
  size_t nq = 0;
  for (size_t i = 0; i < aln; ++i) nq += read_idx[i] >= 0;
  if (nq != rec->seq.size()) return pfail(DCB_ERR_INVALID, "%s: cigar covers %zu query bases, sequence has %zu", rec->qname.c_str(), nq, rec->seq.size());
  if (pw.size() != nq || ip.size() != nq) return pfail(DCB_ERR_INVALID, "%s: pw / ip tags do not match the sequence length", rec->qname.c_str());
  {
    size_t k = 0;
    for (size_t i = 0; i < aln; ++i)
      if (read_idx[i] >= 0) { seq[i] = rec->seq[k]; npw[i] = (uint8_t)pw[k]; nip[i] = (uint8_t)ip[k]; ++k; }   // uint8 arrays (pre_lib.py:1166-1167)
  }
  if (!rec->find("sn", &t) || t.type != 'B' || t.count < 4) return pfail(DCB_ERR_INVALID, "%s: no sn tag", rec->qname.c_str());
  for (int i = 0; i < 4; ++i) out->sn[i] = (float)BamRecord::element(t, i);
  std::vector<uint8_t> cig;
  size_t lead_soft = 0, trail_soft = 0;
  for (size_t ci = 0; ci < rec->cigar.size(); ++ci) {
    const int op = rec->cigar[ci] & 15;
    const size_t len = rec->cigar[ci] >> 4;
    if (op != kCHard) cig.insert(cig.end(), len, (uint8_t)op);
  }
  {
    // query_alignment_start / _end: query bases outside leading / trailing soft clips
    size_t i = 0;
    while (i < rec->cigar.size() && (rec->cigar[i] & 15) == kCHard) ++i;
    if (i < rec->cigar.size() && (rec->cigar[i] & 15) == kCSoft) lead_soft = rec->cigar[i] >> 4;
    size_t j = rec->cigar.size();
    while (j > 0 && (rec->cigar[j - 1] & 15) == kCHard) --j;
    if (j > 0 && (rec->cigar[j - 1] & 15) == kCSoft && j - 1 != i) trail_soft = rec->cigar[j - 1] >> 4;
  }
  if (cig.size() != aln) return pfail(DCB_ERR_INVALID, "%s: unsupported cigar operation (pad)", rec->qname.c_str());
  bool any_soft = false;
  for (uint8_t c : cig) any_soft |= c == kCSoft;
  size_t qs = 0, qe = aln;
  if (any_soft) {
    for (size_t i = 0; i < aln; ++i) if (cig[i] == kCSoft) seq[i] = kGap;
    const int32_t qstart = (int32_t)lead_soft, qlast = (int32_t)rec->seq.size() - (int32_t)trail_soft - 1;
    bool f1 = false, f2 = false;
    for (size_t i = 0; i < aln; ++i) {
      if (!f1 && read_idx[i] == qstart) { qs = i; f1 = true; }
      if (!f2 && read_idx[i] == qlast) { qe = i + 1; f2 = true; }
    }
    if (!f1 || !f2 || qe < qs) return pfail(DCB_ERR_INVALID, "%s: cannot locate the aligned part", rec->qname.c_str());
  }
  const size_t indent = rec->pos > 0 ? (size_t)rec->pos : 0;
  const size_t n = indent + (qe - qs);
  out->name = rec->qname;
  out->bases.assign(n, kGap);
  out->cigar.assign(n, kCRefSkip);
  out->pw.assign(n, 0);
  out->ip.assign(n, 0);
  out->ccs_idx.assign(n, -1);
  for (size_t i = qs; i < qe; ++i) {
    const size_t o = indent + (i - qs);
    out->bases[o] = seq[i]; out->cigar[o] = cig[i]; out->pw[o] = npw[i]; out->ip[o] = nip[i]; out->ccs_idx[o] = ccs_idx[i];
  }
  out->strand = rev ? 2 : 1;
  return DCB_OK;
}

void construct_ccs_read(const BamRecord& rec, Read* out) {
  const size_t n = rec.seq.size();
  out->name = rec.qname;
  out->bases.assign(rec.seq.begin(), rec.seq.end());
  out->cigar.assign(n, kCMatch);
  out->pw.assign(n, 0);
  out->ip.assign(n, 0);
  out->strand = 0;
  out->ccs_idx.resize(n);
  out->bq.resize(n);
  out->bq_any = false;
  for (size_t i = 0; i < n; ++i) { out->ccs_idx[i] = (int32_t)i; out->bq[i] = rec.qual[i]; out->bq_any |= rec.qual[i] != 0; }
}

// space_out_subreads (pre_lib.py:1242-1276) for inference reads (no label)
void space_out(std::vector<Read>& reads) {
  for (Read& r : reads) { r.seq_indices.assign(r.bases.size(), 0); r.idx_seq = 0; r.idx_spaced = 0; r.done = false; }
  auto next_is_ins = [](const Read& r) { return r.idx_seq < r.cigar.size() && r.cigar[r.idx_seq] == kCIns; };
  for (;;) {
    bool all_done = true;
    for (const Read& r : reads) all_done &= r.done;
    if (all_done) break;
    bool any_ins = false;
    for (const Read& r : reads) {
      if (r.done) continue;
      if (next_is_ins(r)) { any_ins = true; break; }
    }
    for (Read& r : reads) {
      if (r.done) continue;
      if (any_ins && !next_is_ins(r)) {
        ++r.idx_spaced;                                        // add_gap
      } else {
        if (r.idx_seq < r.bases.size()) { r.seq_indices[r.idx_seq] = r.idx_spaced; ++r.idx_seq; ++r.idx_spaced; }   // move
        if (r.idx_seq >= r.bases.size()) r.done = true;
      }
    }
  }
  int32_t max_len = 0;
  for (const Read& r : reads) max_len = std::max(max_len, r.idx_spaced);
  for (Read& r : reads) {                                      // put_spacing
    std::vector<char> b(max_len, kGap);
    std::vector<uint8_t> pw(max_len, 0), ip(max_len, 0);
    std::vector<int32_t> ci(max_len, -1), bq;
    if (r.bq_any) bq.assign(max_len, -1);
    for (size_t i = 0; i < r.bases.size(); ++i) {
      const int32_t o = r.seq_indices[i];
      b[o] = r.bases[i]; pw[o] = r.pw[i]; ip[o] = r.ip[i]; ci[o] = r.ccs_idx[i];
      if (r.bq_any) bq[o] = r.bq[i];
    }
    r.bases.swap(b); r.pw.swap(pw); r.ip.swap(ip); r.ccs_idx.swap(ci);
    if (r.bq_any) r.bq.swap(bq);
  }
}

inline float encode_base(char c) {          // dc_constants.SEQ_VOCAB = ' ATCG'
  switch (c) { case 'A': return 1.f; case 'T': return 2.f; case 'C': return 3.f; case 'G': return 4.f; default: return 0.f; }
}

// Everything derived from one ZMW (what a DcExample holds after space_out_subreads + the window list)
struct ZmwState {
  std::vector<Read> reads;        // subreads..., ccs (spaced)
  std::string name, rg;
  float ec = 0, rq = 0;
  int has_ec = 0, has_np = 0, has_rq = 0, has_rg = 0;
  int32_t np_passes = 0, n_subreads = 0, ccs_length = 0;
  std::vector<int32_t> win_start; // column of every emitted window
  std::vector<int32_t> win_width; // its spaced width (max_length for fixed-width windows)
  int rc = DCB_OK;                // error of the processing step (message in `error`)
  std::string error;
};

struct ZmwJob {
  std::vector<BamRecord> group;
  BamRecord ccs;
  std::string name;
};

struct PrepCfg { int P = 0, L = 0, bq = 0, ins_trim = 0, R = 0, smart = 0; dcb::PackedLayout pl{}; };

// DcExample.calculate_windows with window_widths (pre_lib.py:625-650): the `wl` tag of the CCS record gives every
// window's width in CCS bases; walking the spaced CCS row, window i ends once wl[i] non-gap columns are behind it.
// The reference raises where the tag is missing (KeyError), where sum(wl) walks past the row (IndexError) and where the
// spaced widths do not add up to ccs_width (assert); those cases are errors here too.
int smart_window_widths(const BamRecord& c, const Read& ccs, int ccs_width, std::vector<int32_t>* widths) {
  Tag t;
  if (!c.find("wl", &t)) return pfail(DCB_ERR_INVALID, "%s: no wl tag (needed for CCS smart windows)", c.qname.c_str());
  if (t.type != 'B' || !t.sub || !strchr("cCsSiI", t.sub))
    return pfail(DCB_ERR_INVALID, "%s: the wl tag is not an integer array", c.qname.c_str());
  const int64_t width = (int64_t)ccs.bases.size();
  int64_t last = 0;
  for (size_t i = 0; i < t.count; ++i) {
    const int64_t want = (int64_t)BamRecord::element(t, i);
    int64_t orig = 0, spaced = 0;
    while (orig < want) {
      if (last + spaced >= width)
        return pfail(DCB_ERR_INVALID, "%s: the wl tag covers more than the CCS read's %zu bases", c.qname.c_str(), c.seq.size());
      if (ccs.bases[last + spaced] != kGap) ++orig;
      ++spaced;
    }
    widths->push_back((int32_t)spaced);
    last += spaced;
  }
  if (last != ccs_width)
    return pfail(DCB_ERR_INVALID, "%s: the wl tag's windows span %lld columns, the spaced CCS read %d", c.qname.c_str(),
                 (long long)last, ccs_width);
  return DCB_OK;
}

// CPU-heavy part, no I/O: expand_clip_indent per subread, construct_ccs_read, space_out_subreads, window list
void process_zmw(const PrepCfg& cfg, ZmwJob* job, ZmwState* st) {
  st->name = job->name;
  st->n_subreads = (int32_t)job->group.size();
  st->reads.clear();
  st->reads.resize(job->group.size() + 1);
  for (size_t i = 0; i < job->group.size(); ++i) {
    const int rc = expand_clip_indent(&job->group[i], cfg.ins_trim, &st->reads[i]);
    if (rc) { st->rc = rc; st->error = g_prep_error; return; }
  }
  const BamRecord& c = job->ccs;
  construct_ccs_read(c, &st->reads.back());
  Tag t;
  st->has_ec = c.find("ec", &t); if (st->has_ec) st->ec = (float)BamRecord::scalar(t);
  st->has_np = c.find("np", &t); if (st->has_np) st->np_passes = (int32_t)BamRecord::scalar(t);
  st->has_rq = c.find("rq", &t); if (st->has_rq) st->rq = (float)BamRecord::scalar(t);
  st->has_rg = c.find("RG", &t) && t.type == 'Z'; if (st->has_rg) st->rg = reinterpret_cast<const char*>(t.p);
  st->ccs_length = (int32_t)c.seq.size();
  space_out(st->reads);
  // DcExample.iter_examples (pre_lib.py:625-697): windows of max_length columns, or of the widths the wl tag gives
  const Read& ccs = st->reads.back();
  const int width = (int)ccs.bases.size();
  int ccs_width = width;
  while (ccs_width > 0 && (ccs.bases[ccs_width - 1] == ' ' || ccs.bases[ccs_width - 1] == '\t' || ccs.bases[ccs_width - 1] == '\n')) --ccs_width;
  std::vector<int32_t> widths;
  if (cfg.smart) {
    if (smart_window_widths(c, ccs, ccs_width, &widths)) { st->rc = DCB_ERR_INVALID; st->error = g_prep_error; return; }
  } else {
    widths.assign((ccs_width + cfg.L - 1) / cfg.L, cfg.L);
  }
  st->win_start.clear();
  st->win_width.clear();
  int start = 0;
  for (const int32_t ww : widths) {
    if (start > ccs_width) break;
    const int s0 = start;
    start += ww;
    bool any = false;
    for (int i = s0; i < std::min(s0 + ww, width); ++i) any |= ccs.ccs_idx[i] >= 0;
    if (!any) continue;                                         // n_examples_no_ccs_idx
    st->win_start.push_back(s0);
    st->win_width.push_back(ww);                                // overflow: ww > max_length
  }
}

// extract_features (pre_lib.py:704-744) of the columns [s, s + n) into float32 rows [R, Wo]; columns n..Wo-1 are padding
void write_rows(const ZmwState& st, const PrepCfg& cf, int s, int n, int Wo, float* d) {
  const int P = cf.P, R = cf.R;
  const int keep = (int)std::min<size_t>(P, st.reads.size() - 1);
  const Read& ccs = st.reads.back();
  memset(d, 0, sizeof(float) * (size_t)R * Wo);
  for (int k = 0; k < keep; ++k) {
    const Read& r = st.reads[k];
    for (int i = 0; i < n; ++i) {
      d[(size_t)k * Wo + i] = encode_base(r.bases[s + i]);
      d[(size_t)(P + k) * Wo + i] = (float)r.pw[s + i];
      d[(size_t)(2 * P + k) * Wo + i] = (float)r.ip[s + i];
    }
    for (int i = 0; i < Wo; ++i) d[(size_t)(3 * P + k) * Wo + i] = (float)r.strand;   // repeated over the whole width
  }
  for (int i = 0; i < n; ++i) d[(size_t)4 * P * Wo + i] = encode_base(ccs.bases[s + i]);
  if (cf.bq)
    for (int i = 0; i < Wo; ++i) d[(size_t)(4 * P + 1) * Wo + i] = (i < n && ccs.bq_any) ? (float)ccs.bq[s + i] : -1.f;
  for (int j = 0; j < 4; ++j)
    for (int i = 0; i < Wo; ++i) d[(size_t)(R - 4 + j) * Wo + i] = st.reads[0].sn[j];
}

}  // namespace

struct dcb_prep {
  BamReader sub, ccs;
  PrepCfg cfg;
  bool have_pending = false, sub_eof = false;
  BamRecord pending;
  int64_t pending_zm = 0;
  ZmwState cur;                   // the ZMW handed out by the last dcb_prep_next_zmw
  // optional worker pool (dcb_prep_set_threads): one reader thread decodes and groups, n workers process, results are
  // handed out in file order
  int n_threads = 0;
  bool started = false, stop = false;
  std::thread reader;
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv_job, cv_res, cv_space;
  std::deque<std::pair<int64_t, ZmwJob>> jobs;
  std::map<int64_t, ZmwState> results;
  int64_t next_seq = 0, total = -1;   // total: number of ZMWs once the reader hit the end (or an error)
  int reader_rc = DCB_OK;
  std::string reader_error;
};

namespace {

// Sequential I/O: the next group of mapped subreads with one zm (SubreadGrouper, pre_lib.py:50-91) and its CCS record
// (pre_lib.py:1322-1330).  1 = job filled, 0 = end of file, < 0 = error.
int read_job(dcb_prep* p, ZmwJob* job) {
  std::vector<BamRecord>& group = job->group;
  group.clear();
  int64_t zm = 0;
  bool have_zm = false;
  auto zm_of = [&](const BamRecord& r, int64_t* v) {
    Tag t;
    if (!r.find("zm", &t)) return false;
    *v = (int64_t)BamRecord::scalar(t);
    return true;
  };
  // consecutive records with the same zm; unmapped records are dropped, but the very first record of the file sets the
  // first group's zm even when it is unmapped
  if (p->have_pending) { group.push_back(p->pending); zm = p->pending_zm; have_zm = true; p->have_pending = false; }
  while (!p->sub_eof) {
    BamRecord r;
    const int rc = p->sub.next(&r);
    if (rc < 0) return rc;
    if (rc == 0) { p->sub_eof = true; break; }
    int64_t rz;
    if (!zm_of(r, &rz)) return pfail(DCB_ERR_INVALID, "%s: no zm tag", r.qname.c_str());
    if (!have_zm) { zm = rz; have_zm = true; if (!(r.flag & 4)) group.push_back(r); continue; }
    if (r.flag & 4) continue;
    if (rz == zm) { group.push_back(r); continue; }
    if (!group.empty()) { p->pending = r; p->pending_zm = rz; p->have_pending = true; break; }
    group.push_back(r); zm = rz;
  }
  if (group.empty()) return 0;
  const int32_t refid = group[0].refid;
  if (refid < 0 || refid >= (int32_t)p->sub.refs.size()) return pfail(DCB_ERR_INVALID, "%s: no reference name", group[0].qname.c_str());
  job->name = p->sub.refs[refid];
  for (;;) {
    const int rc = p->ccs.next(&job->ccs);
    if (rc < 0) return rc;
    if (rc == 0) return pfail(DCB_ERR_INVALID, "ccs bam does not contain %s", job->name.c_str());
    if (job->ccs.qname == job->name) break;
  }
  return 1;
}

void reader_main(dcb_prep* p) {
  int64_t seq = 0;
  for (;;) {
    ZmwJob job;
    const int rc = read_job(p, &job);
    std::unique_lock<std::mutex> lk(p->mu);
    if (rc <= 0) {
      if (rc < 0) { p->reader_rc = rc; p->reader_error = g_prep_error; }
      p->total = seq;
      p->cv_job.notify_all();
      p->cv_res.notify_all();
      return;
    }
    p->cv_space.wait(lk, [&] { return p->stop || (int64_t)(p->jobs.size() + p->results.size()) < 4ll * p->n_threads + 4; });
    if (p->stop) return;
    p->jobs.emplace_back(seq++, std::move(job));
    p->cv_job.notify_one();
  }
}

void worker_main(dcb_prep* p) {
  for (;;) {
    std::pair<int64_t, ZmwJob> item;
    {
      std::unique_lock<std::mutex> lk(p->mu);
      p->cv_job.wait(lk, [&] { return p->stop || !p->jobs.empty() || p->total >= 0; });
      if (p->stop) return;
      if (p->jobs.empty()) return;                 // reader finished and nothing left
      item = std::move(p->jobs.front());
      p->jobs.pop_front();
    }
    ZmwState st;
    process_zmw(p->cfg, &item.second, &st);
    {
      std::lock_guard<std::mutex> lk(p->mu);
      p->results.emplace(item.first, std::move(st));
    }
    p->cv_res.notify_all();
  }
}

void stop_threads(dcb_prep* p) {
  if (!p->started) return;
  {
    std::lock_guard<std::mutex> lk(p->mu);
    p->stop = true;
  }
  p->cv_job.notify_all(); p->cv_res.notify_all(); p->cv_space.notify_all();
  if (p->reader.joinable()) p->reader.join();
  for (auto& w : p->workers) if (w.joinable()) w.join();
  p->started = false;
}

}  // namespace

extern "C" {

const char* dcb_prep_last_error(void) { return g_prep_error.c_str(); }

int dcb_prep_open(const char* subreads_to_ccs_bam, const char* ccs_bam, int32_t max_passes, int32_t max_length,
                  int32_t use_ccs_bq, int32_t ins_trim, dcb_prep** out) {
  if (!subreads_to_ccs_bam || !ccs_bam || !out || max_passes <= 0 || max_length <= 0) return pfail(DCB_ERR_INVALID, "dcb_prep_open: bad argument");
  dcb_prep* p = new dcb_prep();
  PrepCfg& c = p->cfg;
  c.P = max_passes; c.L = max_length; c.bq = use_ccs_bq ? 1 : 0; c.ins_trim = ins_trim;
  c.R = 4 * max_passes + 5 + c.bq;
  c.pl = dcb::make_packed_layout(max_passes, max_length, c.bq);
  int rc = p->sub.open(subreads_to_ccs_bam);
  if (!rc) rc = p->ccs.open(ccs_bam);
  if (rc) { delete p; return rc; }
  *out = p;
  return DCB_OK;
}

// Process ZMWs on `n_threads` worker threads (plus one thread that decodes the BAMs); results still come out of
// dcb_prep_next_zmw in file order.  Call before the first dcb_prep_next_zmw; n_threads <= 0 keeps everything on the caller.
int dcb_prep_set_threads(dcb_prep* p, int32_t n_threads) {
  if (!p) return pfail(DCB_ERR_INVALID, "dcb_prep_set_threads: null handle");
  if (p->started || p->next_seq) return pfail(DCB_ERR_STATE, "dcb_prep_set_threads: the stream has already started");
  p->n_threads = n_threads > 0 ? std::min(n_threads, 256) : 0;
  return DCB_OK;
}

// Windows from the CCS record's `wl` tag instead of max_length columns (--use_ccs_smart_windows, pre_lib.py:1329-1331).
int dcb_prep_set_smart_windows(dcb_prep* p, int32_t enable) {
  if (!p) return pfail(DCB_ERR_INVALID, "dcb_prep_set_smart_windows: null handle");
  if (p->started || p->next_seq) return pfail(DCB_ERR_STATE, "dcb_prep_set_smart_windows: the stream has already started");
  p->cfg.smart = enable ? 1 : 0;
  return DCB_OK;
}

void dcb_prep_close(dcb_prep* p) {
  if (!p) return;
  stop_threads(p);
  delete p;
}

// Advances to the next ZMW that has mapped subreads.  Returns 1 and fills `info`, 0 at the end of the file, < 0 on error.
int dcb_prep_next_zmw(dcb_prep* p, dcb_zmw_info* info) {
  if (!p || !info) return pfail(DCB_ERR_INVALID, "dcb_prep_next_zmw: null argument");
  if (p->n_threads > 0) {
    if (!p->started) {
      p->started = true;
      p->reader = std::thread(reader_main, p);
      for (int i = 0; i < p->n_threads; ++i) p->workers.emplace_back(worker_main, p);
    }
    std::unique_lock<std::mutex> lk(p->mu);
    p->cv_res.wait(lk, [&] { return p->results.count(p->next_seq) || (p->total >= 0 && p->next_seq >= p->total); });
    auto it = p->results.find(p->next_seq);
    if (it == p->results.end()) {
      if (p->reader_rc) { g_prep_error = p->reader_error; return p->reader_rc; }
      return 0;
    }
    p->cur = std::move(it->second);
    p->results.erase(it);
    ++p->next_seq;
    lk.unlock();
    p->cv_space.notify_all();
  } else {
    ZmwJob job;
    const int rc = read_job(p, &job);
    if (rc <= 0) return rc;
    p->cur = ZmwState();
    process_zmw(p->cfg, &job, &p->cur);
    ++p->next_seq;
  }
  if (p->cur.rc) { g_prep_error = p->cur.error; return p->cur.rc; }
  const ZmwState& st = p->cur;
  memset(info, 0, sizeof *info);
  info->n_windows = (int32_t)st.win_start.size();
  info->n_subreads = st.n_subreads;
  info->name = st.name.c_str();
  info->has_ec = st.has_ec; info->ec = st.ec;
  info->has_np = st.has_np; info->np_num_passes = st.np_passes;
  info->has_rq = st.has_rq; info->rq = st.rq;
  info->rg = st.has_rg ? st.rg.c_str() : nullptr;
  info->ccs_length = st.ccs_length;
  info->spaced_width = (int32_t)st.reads.back().bases.size();
  return 1;
}

// The windows of the current ZMW (DcExample.extract_features / to_features_dict, pre_lib.py:704-762).  Every output may
// be NULL.  rows: float32 [n, R, L]; packed: [n, packed_window_bytes]; window_pos / num_passes: [n]; overflow: [n]
// (always 0 with fixed-width windows); ccs_bq: int16 [n, L] (-1 at gaps and padding).  An overflow window (smart
// windows wider than max_length) appears here with its first L columns; dcb_prep_get_overflow_windows has all of it.
int dcb_prep_get_windows(dcb_prep* p, float* rows, uint8_t* packed, int32_t* window_pos, uint8_t* overflow,
                         int16_t* ccs_bq, int32_t* num_passes) {
  if (!p) return pfail(DCB_ERR_INVALID, "dcb_prep_get_windows: null handle");
  const ZmwState& st = p->cur;
  if (st.reads.empty()) return pfail(DCB_ERR_STATE, "dcb_prep_get_windows: no ZMW loaded");
  const PrepCfg& cf = p->cfg;
  const int L = cf.L, P = cf.P, R = cf.R;
  const size_t nsub = st.reads.size() - 1;
  const int keep = (int)std::min<size_t>(P, nsub);
  const Read& ccs = st.reads.back();
  const int width = (int)ccs.bases.size();
  for (size_t w = 0; w < st.win_start.size(); ++w) {
    const int s = st.win_start[w], ww = st.win_width[w];
    const int nw = std::min(ww, width - s);                   // columns of the window
    const int n = std::min(L, nw);                             // of those, the ones in the first L; the rest is padding
    if (rows) write_rows(st, cf, s, n, L, rows + w * (size_t)R * L);
    if (packed) {
      uint8_t* o = packed + w * (size_t)cf.pl.stride;
      memset(o, 0, cf.pl.stride);
      for (int k = 0; k < keep; ++k) {
        const Read& r = st.reads[k];
        for (int i = 0; i < L; ++i) {
          const int base = i < n ? (int)encode_base(r.bases[s + i]) : 0;
          o[k * L + i] = (uint8_t)(base | (r.strand << 3));
        }
        for (int i = 0; i < n; ++i) { o[(P + k) * L + i] = r.pw[s + i]; o[(2 * P + k) * L + i] = r.ip[s + i]; }
      }
      for (int i = 0; i < n; ++i) o[3 * P * L + i] = (uint8_t)encode_base(ccs.bases[s + i]);
      if (cf.bq)
        for (int i = 0; i < L; ++i) o[(3 * P + 1) * L + i] = (uint8_t)(((i < n && ccs.bq_any) ? ccs.bq[s + i] : -1) + 1);
      memcpy(o + cf.pl.sn_off, st.reads[0].sn, 16);
    }
    if (window_pos) {
      int32_t mn = 0;
      bool found = false;
      for (int i = 0; i < nw; ++i) {
        const int32_t v = ccs.ccs_idx[s + i];
        if (v >= 0 && (!found || v < mn)) { mn = v; found = true; }
      }
      window_pos[w] = mn;                                       // ccs_bounds.start
    }
    if (overflow) overflow[w] = ww > L;
    if (num_passes) num_passes[w] = keep;
    if (ccs_bq)
      for (int i = 0; i < L; ++i) ccs_bq[w * (size_t)L + i] = (int16_t)((i < n && ccs.bq_any) ? ccs.bq[s + i] : -1);
  }
  return DCB_OK;
}

int dcb_prep_get_window_widths(dcb_prep* p, int32_t* widths) {
  if (!p || !widths) return pfail(DCB_ERR_INVALID, "dcb_prep_get_window_widths: null argument");
  if (p->cur.reads.empty()) return pfail(DCB_ERR_STATE, "dcb_prep_get_window_widths: no ZMW loaded");
  std::copy(p->cur.win_width.begin(), p->cur.win_width.end(), widths);
  return DCB_OK;
}

// The overflow windows of the current ZMW in full, ragged: window after window, W columns each.
int dcb_prep_get_overflow_windows(dcb_prep* p, float* rows, uint8_t* ccs_ids, int16_t* ccs_bq) {
  if (!p) return pfail(DCB_ERR_INVALID, "dcb_prep_get_overflow_windows: null handle");
  const ZmwState& st = p->cur;
  if (st.reads.empty()) return pfail(DCB_ERR_STATE, "dcb_prep_get_overflow_windows: no ZMW loaded");
  const PrepCfg& cf = p->cfg;
  const Read& ccs = st.reads.back();
  size_t off = 0;
  for (size_t w = 0; w < st.win_start.size(); ++w) {
    const int s = st.win_start[w], ww = st.win_width[w];
    if (ww <= cf.L) continue;
    const int n = std::min(ww, (int)ccs.bases.size() - s);
    if (rows) write_rows(st, cf, s, n, ww, rows + off * cf.R);
    for (int i = 0; i < ww; ++i) {
      if (ccs_ids) ccs_ids[off + i] = (uint8_t)(i < n ? encode_base(ccs.bases[s + i]) : 0);
      if (ccs_bq) ccs_bq[off + i] = (int16_t)((i < n && ccs.bq_any) ? ccs.bq[s + i] : -1);
    }
    off += ww;
  }
  return DCB_OK;
}

// Header text of the CCS BAM (the output BAM reuses it, quick_inference.py:894-897).
const char* dcb_prep_ccs_header(dcb_prep* p) { return p ? p->ccs.header_text.c_str() : ""; }

}  // extern "C"

// ----------------------------------------------------------------------------------------------- BAM writer
struct dcb_bamw {
  FILE* f = nullptr;
  std::vector<uint8_t> buf;
  bool failed = false;
  void flush_block(bool force_empty = false) {
    if (buf.empty() && !force_empty) return;
    const uLong src = (uLong)buf.size();
    std::vector<uint8_t> comp(compressBound(src) + 64);
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (deflateInit2(&zs, Z_DEFAULT_COMPRESSION, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) { failed = true; return; }
    zs.next_in = buf.data(); zs.avail_in = (uInt)src;
    zs.next_out = comp.data(); zs.avail_out = (uInt)comp.size();
    const int rc = deflate(&zs, Z_FINISH);
    const size_t clen = zs.total_out;
    deflateEnd(&zs);
    if (rc != Z_STREAM_END) { failed = true; return; }
    const uint32_t bsize = (uint32_t)(clen + 25);              // 18 header + data + 8 trailer - 1
    uint8_t h[18] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0, (uint8_t)(bsize & 255), (uint8_t)(bsize >> 8)};
    const uint32_t crc = (uint32_t)crc32(0, buf.data(), (uInt)src), isz = (uint32_t)src;
    uint8_t t[8] = {(uint8_t)crc, (uint8_t)(crc >> 8), (uint8_t)(crc >> 16), (uint8_t)(crc >> 24),
                    (uint8_t)isz, (uint8_t)(isz >> 8), (uint8_t)(isz >> 16), (uint8_t)(isz >> 24)};
    if (fwrite(h, 1, 18, f) != 18 || fwrite(comp.data(), 1, clen, f) != clen || fwrite(t, 1, 8, f) != 8) failed = true;
    buf.clear();
  }
  void put(const void* p, size_t n) {
    const uint8_t* s = static_cast<const uint8_t*>(p);
    while (n) {
      const size_t room = 0xff00 - buf.size();
      const size_t take = std::min(room, n);
      buf.insert(buf.end(), s, s + take);
      s += take; n -= take;
      if (buf.size() >= 0xff00) flush_block();
    }
  }
};

extern "C" {

int dcb_bamw_open(const char* path, const char* header_text, dcb_bamw** out) {
  if (!path || !out) return pfail(DCB_ERR_INVALID, "dcb_bamw_open: bad argument");
  dcb_bamw* w = new dcb_bamw();
  w->f = fopen(path, "wb");
  if (!w->f) { delete w; return pfail(DCB_ERR_INVALID, "cannot create %s", path); }
  const std::string text = header_text ? header_text : "";
  const int32_t l_text = (int32_t)text.size(), n_ref = 0;
  w->put("BAM\1", 4);
  w->put(&l_text, 4);
  w->put(text.data(), text.size());
  w->put(&n_ref, 4);
  w->flush_block();
  *out = w;
  return DCB_OK;
}

// One unaligned record as quick_inference.py:742-760 writes it: flag 4, mapq 255, tags ec:f (-1 when absent), np:i, rq:f,
// RG:Z, zm:i (the ZMW number parsed from the name "movie/zmw/ccs").
int dcb_bamw_write(dcb_bamw* w, const char* name, const uint8_t* seq, const uint8_t* qual_phred33, int32_t len, int32_t has_ec,
                   float ec, int32_t np_num_passes, float rq, const char* rg) {
  if (!w || !name || !seq || !qual_phred33 || len < 0) return pfail(DCB_ERR_INVALID, "dcb_bamw_write: bad argument");
  const size_t l_name = strlen(name) + 1;
  if (l_name > 255) return pfail(DCB_ERR_INVALID, "read name too long");
  int64_t zm = 0;
  {
    const char* a = strchr(name, '/');
    if (!a) return pfail(DCB_ERR_INVALID, "%s: cannot parse the ZMW number", name);
    zm = strtoll(a + 1, nullptr, 10);
  }
  std::vector<uint8_t> rec;
  auto put32 = [&](int32_t v) { const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); rec.insert(rec.end(), p, p + 4); };
  put32(-1);                                                   // refID
  put32(-1);                                                   // pos
  rec.push_back((uint8_t)l_name);
  rec.push_back(255);                                          // mapq
  rec.push_back(4680 & 255); rec.push_back(4680 >> 8);         // bin of an unmapped read (reg2bin(-1, 0))
  rec.push_back(0); rec.push_back(0);                          // n_cigar_op
  rec.push_back(4); rec.push_back(0);                          // flag 4
  put32(len);
  put32(-1); put32(-1); put32(0);                              // next refID, next pos, tlen
  rec.insert(rec.end(), name, name + l_name);
  static int8_t code[256];
  static bool init = false;
  if (!init) { memset(code, 15, sizeof code); const char* nt = "=ACMGRSVTWYHKDBN"; for (int i = 0; i < 16; ++i) code[(uint8_t)nt[i]] = (int8_t)i; init = true; }
  for (int i = 0; i < len; i += 2) {
    const int hi = code[seq[i]], lo = i + 1 < len ? code[seq[i + 1]] : 0;
    rec.push_back((uint8_t)((hi << 4) | lo));
  }
  for (int i = 0; i < len; ++i) rec.push_back((uint8_t)(qual_phred33[i] - 33));
  auto tagf = [&](const char* n, float v) { rec.push_back(n[0]); rec.push_back(n[1]); rec.push_back('f'); const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); rec.insert(rec.end(), p, p + 4); };
  auto tagi = [&](const char* n, int32_t v) { rec.push_back(n[0]); rec.push_back(n[1]); rec.push_back('i'); put32(v); };
  tagf("ec", (has_ec && ec != 0.f) ? ec : -1.f);               // `ec or -1`
  tagi("np", np_num_passes);
  tagf("rq", rq);
  if (rg) { rec.push_back('R'); rec.push_back('G'); rec.push_back('Z'); rec.insert(rec.end(), rg, rg + strlen(rg) + 1); }
  tagi("zm", (int32_t)zm);
  const int32_t bs = (int32_t)rec.size();
  w->put(&bs, 4);
  w->put(rec.data(), rec.size());
  return w->failed ? pfail(DCB_ERR_INVALID, "write failed") : DCB_OK;
}

int dcb_bamw_close(dcb_bamw* w) {
  if (!w) return DCB_OK;
  w->flush_block();
  w->flush_block(true);                                        // the BGZF end-of-file marker: an empty block
  const bool bad = w->failed || fclose(w->f) != 0;
  delete w;
  return bad ? pfail(DCB_ERR_INVALID, "closing the BAM failed") : DCB_OK;
}

}  // extern "C"

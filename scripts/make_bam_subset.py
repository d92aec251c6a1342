"""Cut the reference's subread BAM fixture down to a subset of its ZMWs, so that the stored file stays under 1 MB.

  python scripts/make_bam_subset.py SUBREADS_TO_CCS_BAM

SUBREADS_TO_CCS_BAM is the reference's testdata/human_1m/subreads_to_ccs.bam (10 ZMWs, 4.6 MB of BAM records).  The
header and every record of the ZMWs in KEEP are written, in file order, as BGZF to tests/golden/human_1m/
subreads_to_ccs.bam; records are not changed.  Windows are built per ZMW, so the windows of the kept ZMWs are exactly
the ones the reference's preprocess made from the whole file: tests/test_bam_prep.py compares them with their entries
of tests/golden/human_1m/inference_digest.json (scripts/make_bam_golden.py), which keeps all 1 593.  ccs.bam stays
whole: the reader skips CCS reads that have no subreads.
The first two ZMWs are kept because tests/test_bam_prep.py corrupts the records of the first ~300 KB.
"""
import gzip
import os
import struct
import sys
import zlib

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(REPO, "tests", "golden", "human_1m")
KEEP = (4194375, 4194376, 4194377, 4194379, 4194381, 4194387, 4194388)
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_members(raw):
  pos = 0
  while pos < len(raw):
    bsize = raw[pos + 16] | (raw[pos + 17] << 8)
    yield raw[pos:pos + bsize + 1]
    pos += bsize + 1


def bgzf(data):
  out = bytearray()
  for i in range(0, len(data), 0xff00):
    blk = data[i:i + 0xff00]
    c = zlib.compressobj(9, zlib.DEFLATED, -15)
    comp = c.compress(blk) + c.flush()
    bs = len(comp) + 25
    out += bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, bs & 255, bs >> 8]) + comp
    out += struct.pack("<II", zlib.crc32(blk), len(blk))
  return bytes(out) + BGZF_EOF


def main(src):
  with open(src, "rb") as f:
    plain = b"".join(gzip.decompress(m) for m in bgzf_members(f.read()))
  pos = 8 + struct.unpack_from("<i", plain, 4)[0]                      # magic, l_text, text
  n_ref = struct.unpack_from("<i", plain, pos)[0]
  pos += 4
  for _ in range(n_ref):
    pos += 4 + struct.unpack_from("<i", plain, pos)[0] + 4
  out, kept = bytearray(plain[:pos]), set()
  while pos < len(plain):
    size = 4 + struct.unpack_from("<i", plain, pos)[0]
    l_name = plain[pos + 12]
    zmw = int(plain[pos + 36:pos + 35 + l_name].decode().split("/")[1])  # movie/zmw/start_end
    if zmw in KEEP:
      out += plain[pos:pos + size]
      kept.add(zmw)
    pos += size
  assert kept == set(KEEP), sorted(set(KEEP) - kept)
  with open(os.path.join(OUT, "subreads_to_ccs.bam"), "wb") as f:
    f.write(bgzf(bytes(out)))
  print(len(KEEP), "ZMWs ->", os.path.join(OUT, "subreads_to_ccs.bam"))


if __name__ == "__main__":
  main(sys.argv[1])

"""Feature construction from BAM (csrc/bam_prep.cpp, deepconsensus_b200/preprocess.py; SURVEY.md section 8(f)3) -- no GPU.

THE pin: inference_digest.json is a digest of the 1 593 examples the reference's own `deepconsensus preprocess` wrote
from its BAM fixtures testdata/human_1m/{subreads_to_ccs,ccs}.bam (10 ZMWs; tf_examples/inference/inference.tfrecord.gz;
scripts/make_bam_golden.py).  tests/golden/human_1m/ccs.bam is a byte copy; subreads_to_ccs.bam holds the unchanged
records of 7 of the 10 ZMWs (KEPT_ZMWS, scripts/make_bam_subset.py), which keeps it under 1 MB.  Windows are built per
ZMW, so the 958 windows rebuilt here must equal their digest entries, value for value: names, window positions, pass
counts, all 85 x 100 float32 feature values, the CCS base qualities.  That covers BGZF / BAM decoding, SubreadGrouper,
trim_insertions (ins_trim=5), expand_clip_indent, construct_ccs_read, space_out_subreads, iter_examples and
extract_features.
"""
import hashlib
import json
import os

import numpy as np
import pytest

from deepconsensus_b200 import engine, params as params_lib, preprocess

KEPT_ZMWS = ("4194375", "4194376", "4194377", "4194379", "4194381", "4194387", "4194388")   # in file order


@pytest.fixture(scope="module")
def bam_dir(golden_dir):
  return os.path.join(golden_dir, "human_1m")


def _sha(a, dt):
  return hashlib.sha1(np.ascontiguousarray(a, dt).tobytes()).hexdigest()


def test_windows_equal_the_reference_preprocess_output(bam_dir):
  with open(os.path.join(bam_dir, "inference_digest.json")) as f:
    gold = json.load(f)
  assert gold["summary"]["ins_trim"] == "5" and gold["summary"]["n_examples"] == len(gold["windows"]) == 1593
  want = [g for g in gold["windows"] if g["name"].split("/")[1] in KEPT_ZMWS]
  stream = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"),
                                       max_passes=20, max_length=100, use_ccs_bq=False, ins_trim=5)
  assert "@HD" in stream.ccs_header or "@RG" in stream.ccs_header
  k, zmws = 0, 0
  p = params_lib.synthetic_params(20, 100)
  for z in stream.__iter__():
    zmws += 1
    n = len(z["window_pos"])
    assert z["rows"].shape == (n, 85, 100)
    if zmws == 1:
      assert abs(z["ec"] - 5.64211) < 1e-4 and z["np_num_passes"] == 5 and abs(z["rq"] - 0.994656) < 1e-5 and z["rg"] == "231b5401"
    packed = None
    for i in range(n):
      g = want[k]
      assert (z["name"], int(z["window_pos"][i]), int(z["num_passes"][i])) == (g["name"], g["window_pos"], g["num_passes"]), k
      assert _sha(z["rows"][i], "<f4") == g["rows_sha1"], (k, g["name"], g["window_pos"])
      assert _sha(z["ccs_bq"][i].astype(np.int64), "<i8") == g["bq_sha1"], k
      assert not z["overflow"][i]
      k += 1
    # the packed producer writes exactly what dcb_pack_rows makes of the float32 rows
    np.testing.assert_array_equal(engine.pack_rows(p, z["rows"]), _packed_of(stream, z, bam_dir, zmws))
  assert k == len(want) == 958 and zmws == len(KEPT_ZMWS)
  stream.close()


_packed_cache = {}


def _packed_of(stream, z, bam_dir, zmw_index):
  """Packed rows of the same ZMW from a second stream that asks for packed output only."""
  if "stream" not in _packed_cache:
    _packed_cache["stream"] = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"),
                                                          os.path.join(bam_dir, "ccs.bam"), 20, 100, False, 5)
  s2 = _packed_cache["stream"]
  z2 = s2.next_zmw(want_rows=False, want_packed=True)
  assert z2["name"] == z["name"] and "rows" not in z2
  return z2["packed"]


def test_feature_dicts_have_the_reference_keys(bam_dir):
  zmws = list(preprocess.stream_zmw_windows(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"),
                                            20, 100, limit=2))
  assert len(zmws) == 2
  fd = zmws[0][0]
  assert sorted(fd) == sorted(["subreads", "subreads/num_passes", "name", "window_pos", "ccs_base_quality_scores",
                               "overflow", "ec", "np_num_passes", "rq", "rg"])       # DcExample.to_features_dict
  assert fd["subreads"].shape == (85, 100, 1) and fd["subreads"].dtype == np.float32
  assert fd["ccs_base_quality_scores"].shape == (100,) and fd["overflow"] is False


def test_ccs_bq_row_and_other_geometries(bam_dir):
  """use_ccs_bq adds the row 4P+1 = the CCS base qualities (-1 at gaps / padding); other max_passes / max_length
  re-window the same spaced alignment."""
  a = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"), 20, 100, False, 5)
  b = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"), 20, 100, True, 5)
  c = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"), 5, 120, True, 5)
  za, zb, zc = a.next_zmw(), b.next_zmw(want_packed=True), c.next_zmw()
  assert zb["rows"].shape[1] == 86 and zc["rows"].shape[1:] == (26, 120)
  np.testing.assert_array_equal(zb["rows"][:, :81], za["rows"][:, :81])
  np.testing.assert_array_equal(zb["rows"][:, 82:], za["rows"][:, 81:])
  np.testing.assert_array_equal(zb["rows"][:, 81], zb["ccs_bq"].astype(np.float32))
  assert (zb["rows"][:, 81][zb["rows"][:, 80] == 0] == -1).all()                      # gap columns carry -1
  p = params_lib.synthetic_params(20, 100, use_ccs_bq=True)
  np.testing.assert_array_equal(engine.pack_rows(p, zb["rows"]), zb["packed"])
  assert int(zc["num_passes"].max()) <= 5
  # the CCS row, gaps removed and windows concatenated, is the CCS sequence
  ccs = np.concatenate([w[80][w[80] > 0] for w in za["rows"]])
  assert len(ccs) > 1000
  for s in (a, b, c):
    s.close()


def test_bam_writer_round_trip(tmp_path, bam_dir):
  """Records written by BamWriter come back through the same BAM reader (as a CCS BAM) with sequence, qualities and
  tags intact; the file ends with the BGZF EOF marker."""
  src = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"), 20, 100)
  header = src.ccs_header
  z = src.next_zmw()
  src.close()
  name = z["name"]
  seq = "ACGTTGCAAC" * 7000 + "GATTACA"                         # > 64 KB: several BGZF blocks
  qual = "".join(chr(33 + (i * 7) % 94) for i in range(len(seq)))
  out = str(tmp_path / "out.bam")
  w = preprocess.BamWriter(out, header)
  w.write_fastq_record("@%s\n%s\n+\n%s\n" % (name, seq, qual), ec=z["ec"], np_num_passes=z["np_num_passes"], rq=z["rq"], rg=z["rg"])
  w.write_fastq_record("@%s\n%s\n+\n%s\n" % (name.replace("/ccs", "/other"), "ACGT", "!!I~"), ec=None, np_num_passes=3, rq=0.5, rg="x")
  w.close()
  raw = open(out, "rb").read()
  assert raw[:4] == b"\x1f\x8b\x08\x04" and raw.endswith(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
  # read it back: use it as the "CCS BAM" of the fixture's first ZMW
  back = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), out, 20, 100, True)
  assert back.ccs_header == header
  with pytest.raises(preprocess.PrepError):
    # the CCS sequence now has another length than the alignments refer to -> windows still build, but names must match:
    # second ZMW is not in this one-read "CCS BAM"
    back.next_zmw()
    back.next_zmw()
  back.close()
  import gzip
  plain = b"".join(gzip.decompress(m) for m in _members(raw))
  assert plain[:4] == b"BAM\x01" and name.encode() in plain and b"zm" in plain and b"RGZ" in plain
  i = plain.index(b"ecf")
  assert abs(np.frombuffer(plain[i + 3:i + 7], "<f4")[0] - z["ec"]) < 1e-6
  j = plain.rindex(b"ecf")
  assert np.frombuffer(plain[j + 3:j + 7], "<f4")[0] == -1.0      # `ec or -1`


def _members(raw):
  """Split a BGZF file into its gzip members (BSIZE in the BC extra field)."""
  pos = 0
  while pos < len(raw):
    bsize = raw[pos + 16] | (raw[pos + 17] << 8)
    yield raw[pos:pos + bsize + 1]
    pos += bsize + 1


def test_errors_are_reported(tmp_path, bam_dir):
  with pytest.raises(preprocess.PrepError, match="cannot open"):
    preprocess.BamFeatureStream(str(tmp_path / "missing.bam"), os.path.join(bam_dir, "ccs.bam"), 20, 100)
  bad = tmp_path / "bad.bam"
  bad.write_bytes(b"not a bam file at all, not even gzip")
  with pytest.raises(preprocess.PrepError, match="not a BAM"):
    preprocess.BamFeatureStream(str(bad), os.path.join(bam_dir, "ccs.bam"), 20, 100)
  trunc = tmp_path / "trunc.bam"
  raw = open(os.path.join(bam_dir, "subreads_to_ccs.bam"), "rb").read()
  trunc.write_bytes(raw[:len(raw) // 3])
  s = preprocess.BamFeatureStream(str(trunc), os.path.join(bam_dir, "ccs.bam"), 20, 100)
  with pytest.raises(preprocess.PrepError):
    for _ in s:
      pass


def test_threaded_stream_equals_the_serial_one(bam_dir):
  """dcb_prep_set_threads: worker threads process ZMWs out of order, results come back in file order and identical."""
  a = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"), 20, 100, True, 5)
  b = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"), 20, 100, True, 5,
                                  threads=4)
  n = 0
  while True:
    za, zb = a.next_zmw(want_packed=True), b.next_zmw(want_packed=True)
    assert (za is None) == (zb is None)
    if za is None:
      break
    n += 1
    assert za["name"] == zb["name"] and za["ec"] == zb["ec"] and za["rg"] == zb["rg"]
    for k in ("rows", "packed", "window_pos", "ccs_bq", "num_passes", "overflow"):
      np.testing.assert_array_equal(za[k], zb[k])
  assert n == len(KEPT_ZMWS)
  a.close()
  # closing a threaded stream that was only partly consumed must not hang
  c = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, "ccs.bam"), 20, 100, False, 5,
                                  threads=3)
  assert c.next_zmw() is not None
  c.close()
  b.close()
  # errors surface in order from the threaded stream too
  raw = open(os.path.join(bam_dir, "subreads_to_ccs.bam"), "rb").read()
  import tempfile
  with tempfile.TemporaryDirectory() as d:
    path = os.path.join(d, "trunc.bam")
    open(path, "wb").write(raw[:len(raw) // 3])
    s = preprocess.BamFeatureStream(path, os.path.join(bam_dir, "ccs.bam"), 20, 100, threads=2)
    with pytest.raises(preprocess.PrepError):
      for _ in s:
        pass
    s.close()


def test_corrupted_bams_fail_cleanly(tmp_path, bam_dir):
  """The BAM decoder parses untrusted bytes: random corruption of the record stream (re-compressed as valid BGZF) must
  end in PrepError or in a normal result, never in a crash or a hang (serial and threaded streams)."""
  import gzip, random, struct, zlib
  raw = open(os.path.join(bam_dir, "subreads_to_ccs.bam"), "rb").read()
  plain = b"".join(gzip.decompress(m) for m in _members(raw))
  pos = 4
  pos += 4 + struct.unpack_from("<i", plain, pos)[0]
  n_ref = struct.unpack_from("<i", plain, pos)[0]
  pos += 4
  for _ in range(n_ref):
    pos += 4 + struct.unpack_from("<i", plain, pos)[0] + 4
  while pos < 300000:                                   # a record boundary ~300 KB in (two ZMWs)
    pos += 4 + struct.unpack_from("<i", plain, pos)[0]
  base = plain[:pos]

  def bgzf(data):
    out = bytearray()
    for i in range(0, len(data), 0xff00):
      blk = data[i:i + 0xff00]
      c = zlib.compressobj(1, zlib.DEFLATED, -15)
      comp = c.compress(blk) + c.flush()
      bs = len(comp) + 25
      out += bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, bs & 255, bs >> 8]) + comp
      out += struct.pack("<II", zlib.crc32(blk), len(blk))
    return bytes(out) + bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")

  rng = random.Random(7)
  ok = err = 0
  for it in range(40):
    b = bytearray(base)
    for _ in range(rng.choice([1, 1, 2, 5, 20])):
      b[rng.randrange(4, len(b))] = rng.randrange(256)
    if rng.random() < 0.2:
      b = b[:rng.randrange(100, len(b))]
    path = str(tmp_path / "f.bam")
    open(path, "wb").write(bgzf(bytes(b)))
    try:
      s = preprocess.BamFeatureStream(path, os.path.join(bam_dir, "ccs.bam"), 20, 100, True, 5, threads=rng.choice([0, 2]))
      for z in s:
        assert z["rows"].shape[1:] == (86, 100)
      s.close()
      ok += 1
    except preprocess.PrepError:
      err += 1
  assert ok + err == 40 and err >= 5 and ok >= 5

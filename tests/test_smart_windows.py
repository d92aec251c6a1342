"""CCS smart windows (`--use_ccs_smart_windows`): window widths from the CCS records' `wl` tag, overflow windows wider
than max_length, and the ragged post-model stage they need.

The pin: smart_windows_digest.json holds, per window, what the reference's own pre_lib (create_proc_feeder with
use_ccs_smart_windows, iter_examples, to_features_dict) builds from subreads_to_ccs.bam + ccs_wl.bam, a copy of ccs.bam
whose records carry a seeded `wl` tag (scripts/make_smart_windows_golden.py).  CPU tests check feature construction
against it; GPU tests check the ragged device entries against the host mirrors and the whole run against the reference
flow on per-window objects.
"""
import gzip
import hashlib
import itertools
import json
import os
import shutil
import struct
import zlib

import numpy as np
import pytest

from deepconsensus_b200 import calibration, engine, inference, params as params_lib, preprocess, stitch_utils

P, L = 20, 100
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


@pytest.fixture(scope="module")
def bam_dir(golden_dir):
  return os.path.join(golden_dir, "human_1m")


@pytest.fixture(scope="module")
def digest(bam_dir):
  with open(os.path.join(bam_dir, "smart_windows_digest.json")) as f:
    return json.load(f)


def _stream(bam_dir, bq, ccs="ccs_wl.bam", **kw):
  return preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), os.path.join(bam_dir, ccs), P, L, bq, 5,
                                     **kw)


def _window_hash(name, pos, overflow, width, num_passes, rows, bq):
  h = hashlib.sha1(("%s|%d|%d|%d|%d|%s" % (name, pos, overflow, width, num_passes, tuple(rows.shape))).encode())
  h.update(np.ascontiguousarray(rows, "<f4").tobytes())
  h.update(np.ascontiguousarray(bq, "<i8").tobytes())
  return h.hexdigest()[:16]


def _wide(z, R):
  """Per window of a next_zmw bundle: (rows [R, max(W, L)], ccs_bq [max(W, L)]) as to_features_dict has them."""
  out, off = [], 0
  for i in range(len(z["window_pos"])):
    if z["overflow"][i]:
      w = int(z["widths"][i])
      out.append((z["wide_rows"][off * R:(off + w) * R].reshape(R, w), z["wide_ccs_bq"][off:off + w]))
      off += w
    else:
      out.append((z["rows"][i], z["ccs_bq"][i]))
  assert off == len(z["wide_ccs_bq"]) == len(z["wide_ccs_ids"])
  return out


@pytest.mark.parametrize("use_ccs_bq", [False, True])
def test_windows_equal_the_reference_smart_windows(bam_dir, digest, use_ccs_bq):
  gold = [[name] + e for name, z in digest["geometries"]["use_ccs_bq=%d" % use_ccs_bq].items() for e in z]
  s = _stream(bam_dir, use_ccs_bq, use_ccs_smart_windows=True)
  p = params_lib.synthetic_params(P, L, use_ccs_bq=use_ccs_bq)
  R = s.total_rows
  k = n_over = 0
  while True:
    z = s.next_zmw(want_packed=True)
    if z is None:
      break
    for i, (rows, bq) in enumerate(_wide(z, R)):
      g = gold[k]
      got = (z["name"], int(z["window_pos"][i]), bool(z["overflow"][i]), int(z["widths"][i]), int(z["num_passes"][i]))
      assert got == (g[0], g[1], bool(g[2]), g[3], g[4]), k
      assert _window_hash(*got, rows, bq.astype(np.int64)) == g[5], (k, got)
      if z["overflow"][i]:
        # the [n, L] arrays hold the window's first L columns; the CCS ids are the CCS row of the wide rows
        np.testing.assert_array_equal(z["rows"][i], rows[:, :L])
        n_over += 1
      k += 1
    fit = z["overflow"] == 0
    np.testing.assert_array_equal(engine.pack_rows(p, z["rows"][fit]), z["packed"][fit])
    ccs = np.concatenate([r[4 * P] for (r, _), o in zip(_wide(z, R), z["overflow"]) if o] or [np.zeros(0)])
    np.testing.assert_array_equal(z["wide_ccs_ids"], ccs.astype(np.uint8))
  s.close()
  assert k == len(gold) and n_over == sum(g[2] for g in gold) > 100
  assert max(g[3] for g in gold) > 200


def test_smart_windows_off_ignores_the_wl_tag(bam_dir):
  """Without the switch, ccs_wl.bam gives exactly the windows of the reference's fixed-width preprocess output."""
  with open(os.path.join(bam_dir, "inference_digest.json")) as f:
    gold = json.load(f)
  kept = {"4194375", "4194376", "4194377", "4194379", "4194381", "4194387", "4194388"}
  want = [g for g in gold["windows"] if g["name"].split("/")[1] in kept]
  s = _stream(bam_dir, False)
  k = 0
  for z in s:
    assert (z["widths"] == L).all() and not z["overflow"].any() and len(z["wide_ccs_ids"]) == 0
    for i in range(len(z["window_pos"])):
      g = want[k]
      assert (z["name"], int(z["window_pos"][i]), int(z["num_passes"][i])) == (g["name"], g["window_pos"], g["num_passes"])
      assert hashlib.sha1(np.ascontiguousarray(z["rows"][i], "<f4").tobytes()).hexdigest() == g["rows_sha1"], k
      assert hashlib.sha1(z["ccs_bq"][i].astype("<i8").tobytes()).hexdigest() == g["bq_sha1"], k
      k += 1
  s.close()
  assert k == len(want) == 958


def test_threaded_smart_stream_equals_the_serial_one(bam_dir):
  a = _stream(bam_dir, True, use_ccs_smart_windows=True)
  b = _stream(bam_dir, True, use_ccs_smart_windows=True, threads=4)
  n = 0
  while True:
    za, zb = a.next_zmw(want_packed=True), b.next_zmw(want_packed=True)
    assert (za is None) == (zb is None)
    if za is None:
      break
    n += 1
    for key in ("rows", "packed", "window_pos", "ccs_bq", "num_passes", "overflow", "widths", "wide_rows", "wide_ccs_ids",
                "wide_ccs_bq"):
      np.testing.assert_array_equal(za[key], zb[key])
  assert n == 7
  a.close()
  b.close()


def test_stream_zmw_windows_has_the_reference_shapes(bam_dir):
  zmws = list(preprocess.stream_zmw_windows(os.path.join(bam_dir, "subreads_to_ccs.bam"),
                                            os.path.join(bam_dir, "ccs_wl.bam"), P, L, use_ccs_smart_windows=True))
  over = [w for z in zmws for w in z if w["overflow"]]
  fit = [w for z in zmws for w in z if not w["overflow"]]
  assert over and fit
  for w in over:
    W = w["subreads"].shape[1]
    assert W > L and w["subreads"].shape == (85, W, 1) and w["ccs_base_quality_scores"].shape == (W,)
  assert all(w["subreads"].shape == (85, L, 1) and w["ccs_base_quality_scores"].shape == (L,) for w in fit)


# ------------------------------------------------------------------------------------------- wl tag errors / subtypes
def _bam_records(path):
  plain = gzip.open(path, "rb").read()
  pos = 4
  pos += 4 + struct.unpack_from("<i", plain, pos)[0]
  n_ref = struct.unpack_from("<i", plain, pos)[0]
  pos += 4
  for _ in range(n_ref):
    pos += 4 + struct.unpack_from("<i", plain, pos)[0] + 4
  header, recs = plain[:pos], []
  while pos < len(plain):
    bs = struct.unpack_from("<i", plain, pos)[0]
    recs.append(plain[pos + 4:pos + 4 + bs])
    pos += 4 + bs
  return header, recs


def _bgzf(data):
  out = bytearray()
  for i in range(0, len(data), 0xff00):
    blk = data[i:i + 0xff00]
    c = zlib.compressobj(1, zlib.DEFLATED, -15)
    comp = c.compress(blk) + c.flush()
    bs = len(comp) + 25
    out += bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, bs & 255, bs >> 8]) + comp
    out += struct.pack("<II", zlib.crc32(blk), len(blk))
  return bytes(out) + EOF_BLOCK


def _split_wl(rec):
  """(record without its trailing wl:B:S tag, the wl values); the fixture appends wl as the last tag."""
  i = rec.rindex(b"wlBS")
  n = struct.unpack_from("<I", rec, i + 4)[0]
  assert i + 8 + 2 * n == len(rec)
  return rec[:i], list(struct.unpack_from("<%dH" % n, rec, i + 8))


def _with_first_wl(bam_dir, tmp_path, make_tag):
  """ccs_wl.bam with the first record's wl tag replaced by make_tag(wl values) (b"" removes it)."""
  header, recs = _bam_records(os.path.join(bam_dir, "ccs_wl.bam"))
  base, wl = _split_wl(recs[0])
  recs[0] = base + make_tag(wl)
  path = str(tmp_path / "ccs_edit.bam")
  with open(path, "wb") as f:
    f.write(_bgzf(header + b"".join(struct.pack("<i", len(r)) + r for r in recs)))
  return path


def _first_zmw(ccs_path, bam_dir, threads=0):
  s = preprocess.BamFeatureStream(os.path.join(bam_dir, "subreads_to_ccs.bam"), ccs_path, P, L, True, 5, threads=threads,
                                  use_ccs_smart_windows=True)
  try:
    return s.next_zmw(want_packed=True)
  finally:
    s.close()


def _int_array(sub, vals):
  fmt = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I"}[sub]
  return b"wlB" + sub.encode() + struct.pack("<I%d%s" % (len(vals), fmt), len(vals), *vals)


@pytest.mark.parametrize("threads", [0, 2])
def test_wl_tag_errors_name_the_read(bam_dir, tmp_path, threads):
  name = "m54238_180901_011437/4194375/ccs"
  cases = {
      "no wl tag": lambda wl: b"",
      "not an integer array": lambda wl: b"wlBf" + struct.pack("<I%df" % len(wl), len(wl), *wl),
      "covers more than": lambda wl: _int_array("S", wl[:-1] + [wl[-1] + 1]),
      "span": lambda wl: _int_array("S", wl[:-1] + [wl[-1] - 1]),
  }
  for msg, make in cases.items():
    path = _with_first_wl(bam_dir, tmp_path, make)
    with pytest.raises(preprocess.PrepError, match=msg) as e:
      _first_zmw(path, bam_dir, threads)
    assert name in str(e.value)


def test_wl_integer_subtypes_parse_alike(bam_dir, tmp_path):
  ref = _first_zmw(os.path.join(bam_dir, "ccs_wl.bam"), bam_dir)
  for sub in ("i", "I"):
    z = _first_zmw(_with_first_wl(bam_dir, tmp_path, lambda wl: _int_array(sub, wl)), bam_dir)
    for key in ("rows", "packed", "window_pos", "widths", "overflow", "wide_rows", "wide_ccs_bq"):
      np.testing.assert_array_equal(ref[key], z[key])


# ------------------------------------------------------------------------------------------- host mirror
def _options(min_quality=0, skip_windows_above=45, ccs_cal="skip"):
  return inference.InferenceOptions(max_length=L, example_height=85, max_passes=P, min_quality=min_quality, min_length=0,
                                    batch_size=256, use_ccs_bq=False, cpus=0, skip_windows_above=skip_windows_above,
                                    use_saved_model=False, max_base_quality=93,
                                    dc_calibration_values=calibration.parse_calibration_string("skip"),
                                    ccs_calibration_values=calibration.parse_calibration_string(ccs_cal))


def test_host_mirror_stitches_wide_windows(bam_dir):
  """split_skipped_windows + process_skipped_window + stitch_to_fastq take W-wide windows as the reference does: the
  read of a ZMW whose windows are all skipped is its CCS (gaps removed), unless a window wider than L columns made a
  later window start beyond i * L (empty_sequence)."""
  zmws = list(preprocess.stream_zmw_windows(os.path.join(bam_dir, "subreads_to_ccs.bam"),
                                            os.path.join(bam_dir, "ccs_wl.bam"), P, L, use_ccs_smart_windows=True))
  opts = _options(skip_windows_above=1)                           # every window skipped: no model needed
  for_model, skipped = inference.split_skipped_windows(zmws, opts)
  assert not for_model and any(len(o.sequence) > L for o in skipped)
  cnt = stitch_utils.OutcomeCounter()
  recs = {}
  for name, grp in itertools.groupby(sorted(skipped, key=lambda o: (o.molecule_name, o.window_pos)),
                                     lambda o: o.molecule_name):
    recs[name] = stitch_utils.stitch_to_fastq(name, list(grp), L, 0, 0, cnt)
  assert cnt.success + cnt.empty_sequence == 7 and cnt.empty_sequence > 0 and cnt.success > 0
  for z in zmws:
    if recs[z[0]["name"]] is not None:
      ccs = "".join(" ATCG"[int(v)] for w in z for v in w["subreads"][80, :, 0]).replace(" ", "")
      assert recs[z[0]["name"]].splitlines()[1] == ccs


# ------------------------------------------------------------------------------------------- GPU
def _ragged_batch(rng, n_reads, widths_of, gap_frac=0.3, L=L):
  """Seeded reads of windows with given widths: per-window DCModelOutputs (sorted) + the flat byte layout."""
  outs, names = [], []
  for r in range(n_reads):
    name = "m/%d/ccs" % r
    widths = widths_of(r)
    pos = 0
    for i, w in enumerate(widths):
      b = rng.choice(np.frombuffer(b"ATCG", np.uint8), w)
      b[rng.random(w) < gap_frac] = ord(" ")
      q = rng.integers(33, 33 + 60, w).astype(np.uint8)
      wp = pos if not (r % 7 == 3 and i == 1) else pos + L + 1            # every 7th read misses a window
      outs.append(stitch_utils.DCModelOutput(molecule_name=name, window_pos=wp, ec=0, np_num_passes=0, rq=0, rg="",
                                             sequence=b.tobytes().decode(), quality_string=q.tobytes().decode()))
      pos += min(w, L)
  outs.sort(key=lambda o: (o.molecule_name, o.window_pos))
  return outs


def _host_records(outs, min_quality, min_length, L=L):
  cnt, recs = stitch_utils.OutcomeCounter(), []
  for name, grp in itertools.groupby(outs, lambda o: o.molecule_name):
    recs.append(stitch_utils.stitch_to_fastq(name, list(grp), L, min_quality, min_length, cnt))
  return recs, cnt


def _device_records(model, outs, min_quality, min_length, ragged, L=L):
  from deepconsensus_b200 import stitch_gpu
  names = [o.molecule_name for o in outs]
  pos = [int(o.window_pos) for o in outs]
  cnt = stitch_utils.OutcomeCounter()
  if ragged:
    b = np.frombuffer("".join(o.sequence for o in outs).encode(), np.uint8)
    q = np.frombuffer("".join(o.quality_string for o in outs).encode(), np.uint8)
    off = np.concatenate([[0], np.cumsum([len(o.sequence) for o in outs])]).astype(np.int64)
    recs = stitch_gpu.stitch_batch_to_fastq(model, b, q, names, pos, L, min_quality, min_length, cnt, window_off=off)
  else:
    b = np.stack([np.frombuffer(o.sequence.encode(), np.uint8) for o in outs])
    q = np.stack([np.frombuffer(o.quality_string.encode(), np.uint8) for o in outs])
    recs = stitch_gpu.stitch_batch_to_fastq(model, b, q, names, pos, L, min_quality, min_length, cnt)
  return recs, cnt


@pytest.fixture(scope="module")
def tiny_model():
  from deepconsensus_b200 import weights as weights_lib
  p = params_lib.synthetic_params(P, L, num_hidden_layers=1)
  model = engine.B200Model(p, weights_lib.init_weights(p, seed=1), max_batch=4)
  yield model
  model.close()


@pytest.mark.gpu
def test_ragged_stitch_with_all_widths_L_equals_the_fixed_entry(tiny_model):
  rng = np.random.default_rng(5)
  outs = _ragged_batch(rng, 40, lambda r: [L] * (1 + r % 5))
  for mq, ml in ((0, 0), (20, 0), (0, 150)):
    fixed = _device_records(tiny_model, outs, mq, ml, ragged=False)
    ragged = _device_records(tiny_model, outs, mq, ml, ragged=True)
    assert fixed[0] == ragged[0] and fixed[1] == ragged[1]


@pytest.mark.gpu
def test_ragged_stitch_matches_stitch_to_fastq(tiny_model):
  """Mixed widths incl. W > 1024 (several stitch tiles per window), one-window reads, gap-only reads, missing-window
  reads, and reads within 1e-7 of min_quality."""
  rng = np.random.default_rng(11)
  widths = lambda r: [int(rng.choice([L, L, 37, 160, 1500, 2100])) for _ in range(1 + r % 4)]
  outs = _ragged_batch(rng, 60, widths)
  gaps = _ragged_batch(rng, 2, lambda r: [L, 300], gap_frac=1.0)                # reads of gaps only
  for o in gaps:
    o.molecule_name = "g" + o.molecule_name
  outs = sorted(outs + gaps, key=lambda o: (o.molecule_name, o.window_pos))
  # borderline reads: every base Q20 -> avg_phred 20 up to rounding, threshold 20
  border = _ragged_batch(rng, 3, lambda r: [L, 1200][:1 + r % 2])
  for o in border:
    o.molecule_name = "b" + o.molecule_name
    o.quality_string = chr(33 + 20) * len(o.quality_string)
  outs = sorted(outs + border, key=lambda o: (o.molecule_name, o.window_pos))
  for mq, ml in ((0, 0), (20, 0), (20, 400), (25, 0)):
    want = _host_records(outs, mq, ml)
    got = _device_records(tiny_model, outs, mq, ml, ragged=True)
    assert got[0] == want[0], (mq, ml)
    assert got[1] == want[1], (mq, ml)
  cnt = _host_records(outs, 0, 0)[1]
  assert cnt.empty_sequence > 0 and cnt.only_gaps > 0 and cnt.success > 0


@pytest.mark.gpu
@pytest.mark.parametrize("cal", ["skip", "0,1.1,-0.5", "20,0.9,1.5"])
def test_ragged_fill_skipped_matches_process_skipped_window(tiny_model, cal):
  rng = np.random.default_rng(3)
  widths = [L, 37, 260, 1500, L, 101]
  opts = _options(ccs_cal=cal)
  ids = [rng.integers(0, 5, w).astype(np.uint8) for w in widths]
  bqs = [rng.integers(-1, 94, w).astype(np.int16) for w in widths]
  for b, i in zip(bqs, ids):
    b[i == 0] = -1
  src_off = np.concatenate([[0], np.cumsum(widths)]).astype(np.int64)
  perm = rng.permutation(len(widths))                                           # scattered destinations
  dst_widths = np.array(widths)[perm]
  dst_at = np.concatenate([[0], np.cumsum(dst_widths)]).astype(np.int64)
  dst_off = np.empty(len(widths), np.int64)
  dst_off[perm] = dst_at[:-1]
  bases, quals = np.zeros(int(src_off[-1]), np.uint8), np.zeros(int(src_off[-1]), np.uint8)
  tiny_model.fill_skipped_ragged(np.concatenate(ids), np.concatenate(bqs), src_off, dst_off, bases, quals,
                                 calibration=opts.ccs_calibration_values)
  rows_of = params_lib.get_indices(P, False)[4][0]
  for j, w in enumerate(widths):
    rows = np.zeros((85, w, 1), np.float32)
    rows[rows_of, :, 0] = ids[j]
    want = inference.process_skipped_window(dict(subreads=rows, ccs_base_quality_scores=bqs[j].astype(np.int64),
                                                 window_pos=0, name="x", ec=0, np_num_passes=0, rq=0, rg=""), opts)
    a = int(dst_off[j])
    assert bases[a:a + w].tobytes().decode() == want.sequence
    assert quals[a:a + w].tobytes().decode() == want.quality_string
  # all widths L: byte-identical to the fixed entry
  k = 8
  ids_f, bq_f = rng.integers(0, 5, (k, L)).astype(np.uint8), rng.integers(0, 94, (k, L)).astype(np.int16)
  dst = rng.permutation(k).astype(np.int32)
  fb, fq = np.zeros((k, L), np.uint8), np.zeros((k, L), np.uint8)
  tiny_model.fill_skipped(ids_f, bq_f, dst, fb, fq, calibration=opts.ccs_calibration_values)
  rb, rq = np.zeros(k * L, np.uint8), np.zeros(k * L, np.uint8)
  tiny_model.fill_skipped_ragged(ids_f, bq_f, np.arange(k + 1, dtype=np.int64) * L, dst.astype(np.int64) * L, rb, rq,
                                 calibration=opts.ccs_calibration_values)
  np.testing.assert_array_equal(fb.reshape(-1), rb)
  np.testing.assert_array_equal(fq.reshape(-1), rq)


@pytest.mark.gpu
def test_run_with_smart_windows_end_to_end(golden_dir, tmp_path):
  """run(use_ccs_smart_windows=True) on subreads_to_ccs.bam + ccs_wl.bam gives the records and counters of the
  reference flow on per-window objects; inference_on_zmw_windows agrees."""
  from deepconsensus_b200 import run as run_lib, weights as weights_lib
  d = os.path.join(golden_dir, "human_1m")
  ck = tmp_path / "model"
  shutil.copytree(os.path.join(golden_dir, "ckpt", "model"), ck)
  args = dict(subreads_to_ccs=os.path.join(d, "subreads_to_ccs.bam"), ccs_bam=os.path.join(d, "ccs_wl.bam"),
              checkpoint=str(ck / "checkpoint-1"), batch_zmws=4, batch_size=256, min_quality=0, random_weights=3,
              use_ccs_smart_windows=True)
  fq = str(tmp_path / "out.fastq")
  cnt = run_lib.run(output=fq, **args)
  bam = str(tmp_path / "out.bam")
  cnt2 = run_lib.run(output=bam, **args)
  assert cnt.__dict__ == cnt2.__dict__
  got = open(fq).read()
  p = params_lib.read_params_from_json(str(ck / "checkpoint-1"))
  opts = _options()
  opts.dc_calibration_values = calibration.parse_calibration_string(p.get("dc_calibration", "skip"))
  params_lib.modify_params(p, max_length=L)
  model, p = inference.initialize_model("", p, opts, weights=weights_lib.init_weights(p, seed=3))
  zmws = list(preprocess.stream_zmw_windows(args["subreads_to_ccs"], args["ccs_bam"], P, L, use_ccs_smart_windows=True))
  for_model, skipped = inference.split_skipped_windows(zmws, opts)
  preds = sorted(inference.run_model_on_examples(for_model, model, p, opts) + skipped,
                 key=lambda dc: (dc.molecule_name, dc.window_pos))
  want, want_cnt = [], stitch_utils.OutcomeCounter()
  want_cnt_overflow_pass = False
  for name, grp in itertools.groupby(preds, lambda dc: dc.molecule_name):
    grp = list(grp)
    rec = stitch_utils.stitch_to_fastq(name, grp, L, 0, 0, want_cnt)
    if rec:
      want.append(rec)
      if any(len(o.sequence) > L for o in grp):
        want_cnt_overflow_pass = True
  assert sorted(got.split("@")[1:]) == sorted("".join(want).split("@")[1:])
  assert cnt.__dict__ == want_cnt.__dict__
  assert any(len(o.sequence) > L for o in skipped) and want_cnt_overflow_pass and cnt.empty_sequence > 0
  # the same windows through inference_on_zmw_windows and through run_model_and_stitch
  c3 = stitch_utils.OutcomeCounter()
  recs = inference.inference_on_zmw_windows(zmws, model, p, opts, c3)
  assert sorted(r for r in recs if r) == sorted(want) and c3.__dict__ == want_cnt.__dict__
  c4 = stitch_utils.OutcomeCounter()
  recs = inference.run_model_and_stitch(for_model, model, p, opts, c4, skipped_outputs=skipped)
  assert sorted(r for r in recs if r) == sorted(want) and c4.__dict__ == want_cnt.__dict__
  model.close()
  raw = open(bam, "rb").read()
  plain, pos = b"", 0
  while pos < len(raw):
    bs = raw[pos + 16] | (raw[pos + 17] << 8)
    plain += gzip.decompress(raw[pos:pos + bs + 1])
    pos += bs + 1
  for rec in want:
    name, seq, _, qual = rec.splitlines()
    assert name[1:].encode() + b"\0" in plain
    assert bytes(ord(c) - 33 for c in qual[:50]) in plain

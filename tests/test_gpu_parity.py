"""Parity of the CUDA engine (through the C-ABI / ctypes binding) against the oracle.  -m gpu.

BASELINE.json north_star: outputs "must match the reference TF-CPU path on the same input windows within fp32 logit
tolerance (identical argmax bases)".  Two arithmetic modes are checked, with the tolerances written here:

STRICT (dcb_config.precision = DCB_PRECISION_FP32 / DCB_STRICT_FP32): float32 operands and accumulation, the
reference's own arithmetic; differs from the oracle / the reference-code goldens by summation order only.
  * |logit - oracle_fp32| <= STRICT_LOGIT_TOL (2e-4 absolute; measured ~2e-5),
  * bases identical on EVERY position whose fp32 top-2 logit margin exceeds STRICT_MARGIN = 1e-3,
  * quality characters within +-1 everywhere (a 1e-5 probability change can cross a rounding boundary of the integer
    Phred score), exact on >= STRICT_QV_EXACT of the positions.

DEFAULT (bf16 tensor-core operands, fp32 accumulation; DESIGN.md section 4): the operand rounding moves logits by
0.02-0.1 on these random-weight models (gates = ~1.2x the largest value measured over all cases):
  * max |logit - oracle_fp32| <= LOGIT_TOL_FP32, RMS <= LOGIT_RMS_FP32, |logit - oracle_bf16| <= LOGIT_TOL_EMU,
  * bases identical on >= BASES_MIN of ALL positions and on every position with fp32 margin > MARGIN,
  * quality characters exact on >= QV_EXACT_MIN of all positions, within +-1 outside the margin.

BOTH: the device epilogue (argmax / 1-p / -10 log10 / calibration / cap / round / ASCII) is bit-exact integer/byte work
given the device's own probabilities -- np.array_equal against an independent NumPy evaluation of the same definition
(float32 throughout, correctly rounded float32 log10; oracle.postprocess log10="exact"), and equal to the reference's
literal `np.log10` form up to the platform libm's last-ulp differences (none on this image).
"""
import ast
import os

import numpy as np
import pytest

from deepconsensus_b200 import calibration, parity, params as params_lib, synthetic, weights as weights_lib
from oracle import model as omodel, postprocess as opost

pytestmark = pytest.mark.gpu

STRICT_LOGIT_TOL = 2e-4
STRICT_MARGIN = 1e-3
STRICT_QV_EXACT = 0.995
LOGIT_TOL_FP32 = 0.12
LOGIT_RMS_FP32 = 0.02
LOGIT_TOL_EMU = 0.12
MARGIN = 0.25
BASES_MIN = 0.99
BASES_MIN_POSITIONS = 2000       # below this one near-tie is 0.05 % or more: the count gate applies instead
QV_EXACT_MIN = 0.96
CAL = "0,1.197654,-0.99781"


@pytest.fixture(scope="module")
def engine_mod():
  from deepconsensus_b200 import engine
  engine.load_library()
  return engine


def _cal_tuple(cal):
  return (cal.threshold, cal.w, cal.b) if cal.enabled else None


def _epilogue_exact(out, cal):
  """The device epilogue on the device's own probabilities: bit-exact."""
  yy, qq = opost.quality_from_probs(out["probs"], 93, _cal_tuple(cal), log10="exact")
  sb, sq = opost.to_ascii(yy, qq)
  assert np.array_equal(sb, out["bases"])
  assert np.array_equal(sq, out["quals"])
  y2, q2 = opost.quality_from_probs(out["probs"], 93, _cal_tuple(cal))           # the reference's literal np.log10 form
  assert (opost.to_ascii(y2, q2)[1] != out["quals"]).mean() <= 1e-4


def _ref_dict(logits, probs, cal):
  y, q = opost.quality_from_probs(probs, 93, _cal_tuple(cal))
  rb, rq = opost.to_ascii(y, q)
  return dict(bases=rb, quals=rq, logits=logits)


def _assert_strict(out, ref, what=""):
  st = parity.compare(out, ref, margin=STRICT_MARGIN)
  assert st["max_logit_err"] <= STRICT_LOGIT_TOL, (what, st)
  assert st["base_mismatches_outside_margin"] == 0, (what, st)
  assert st["max_dq"] <= 1 and st["qv_exact_pct"] >= 100 * STRICT_QV_EXACT, (what, st)
  return st


def _assert_default(out, ref, what=""):
  st = parity.compare(out, ref, margin=MARGIN)
  assert st["max_logit_err"] <= LOGIT_TOL_FP32 and st["rms_logit_err"] <= LOGIT_RMS_FP32, (what, st)
  assert st["base_mismatches_outside_margin"] == 0, (what, st)
  # share of identical calls: 99 % on samples large enough for a percentage to mean something; on every sample the
  # mismatch count must be what the measured logit error predicts from the reference's own margins (parity.compare)
  assert st["positions"] < BASES_MIN_POSITIONS or st["bases_identical_pct"] >= 100 * BASES_MIN, (what, st)
  assert st["base_mismatches"] <= 3 * st["expected_flips"] + 3, (what, st)
  assert st["qv_exact_pct"] >= 100 * QV_EXACT_MIN and st["max_dq_outside_margin"] <= 1, (what, st)
  return st


def _check(engine_mod, p, w, rows, cal_str=CAL, chunk_tiles=0, max_batch=None):
  cal = calibration.parse_calibration_string(cal_str)
  model = engine_mod.B200Model(p, w, max_batch=max_batch or rows.shape[0], calibration=cal, chunk_tiles=chunk_tiles)
  out = model.forward(rows, want_probs=True, want_logits=True)           # strict_input: any id out of range raises
  launches = model.last_launches
  strict = model.forward(rows, want_probs=True, want_logits=True, strict=True)
  strict_launches = model.last_launches
  model.close()
  assert launches > 0 and strict_launches > launches
  ref = omodel.forward(rows, p, w)
  emu = omodel.forward(rows, p, w, emulate="bf16")
  refd = _ref_dict(ref["logits"], ref["probs"], cal)
  for o in (out, strict):
    assert np.isfinite(o["logits"]).all() and np.abs(o["probs"].sum(-1) - 1).max() < 1e-5
    _epilogue_exact(o, cal)
  _assert_strict(strict, refd)
  assert np.abs(strict["probs"] - ref["probs"]).max() < 2e-5
  _assert_default(out, refd)
  assert np.abs(out["logits"] - emu["logits"]).max() <= LOGIT_TOL_EMU
  # the default path against the strict path (both on the device): same gates
  _assert_default(out, strict)
  return out


def test_c2_shape_rezero(engine_mod):
  p = params_lib.synthetic_params(20, 120)
  _check(engine_mod, p, weights_lib.init_weights(p, seed=1), synthetic.make_rows(p, 9, seed=2))


def test_layernorm_bq_5_layers_L100(engine_mod):
  p = params_lib.synthetic_params(20, 100, use_ccs_bq=True, num_hidden_layers=5, rezero=False)
  _check(engine_mod, p, weights_lib.init_weights(p, seed=3), synthetic.make_rows(p, 7, seed=4), cal_str="10,0.9,1.5")


def test_prelayernorm_rows_whose_mean_runs_away(engine_mod):
  """Deferred LayerNorm of the stack kernel (operands rounded around the row's previous mean): sub-layer outputs with a
  large common-mode component move the mean by many standard deviations per sub-layer.  The kernel's guard re-centres
  those rows; without it the logit error is 0.09 on this case (oracle emulation with the guard off,
  tests/test_oracle_model.py), with it the usual 0.02-0.03."""
  p = params_lib.synthetic_params(20, 100, use_ccs_bq=True, num_hidden_layers=3, rezero=False)
  w = synthetic.mean_drift_weights(p, weights_lib.init_weights(p, seed=5))
  rows = synthetic.make_rows(p, 6, seed=6)
  cal = calibration.parse_calibration_string(CAL)
  model = engine_mod.B200Model(p, w, max_batch=6, calibration=cal)
  out = model.forward(rows, want_probs=True, want_logits=True)
  strict = model.forward(rows, want_probs=True, want_logits=True, strict=True)
  model.close()
  ref = omodel.forward(rows, p, w)
  emu = omodel.forward(rows, p, w, emulate="bf16")
  refd = _ref_dict(ref["logits"], ref["probs"], cal)
  _epilogue_exact(out, cal)
  # float32 itself is coarser here (row means of ~175 against a spread of ~2): the strict path's summation order shows
  assert np.abs(strict["logits"] - ref["logits"]).max() < 2e-3
  _assert_default(out, refd, "mean drift, default vs fp32 oracle")
  assert np.abs(out["logits"] - ref["logits"]).max() < 0.05
  assert np.abs(out["logits"] - emu["logits"]).max() < 0.04


def test_c5_shape_P32_L200(engine_mod):
  p = params_lib.synthetic_params(32, 200)
  _check(engine_mod, p, weights_lib.init_weights(p, seed=5), synthetic.make_rows(p, 5, seed=6), cal_str="skip")


def test_full_attention_when_no_window(engine_mod):
  p = params_lib.synthetic_params(20, 100, attn_win_size=None, num_hidden_layers=2)
  _check(engine_mod, p, weights_lib.init_weights(p, seed=7), synthetic.make_rows(p, 3, seed=8))


def test_real_windows_from_reference_fixture(engine_mod, golden_dir):
  rows = np.load(os.path.join(golden_dir, "real_windows_human_1m.npz"))["rows"]
  p = params_lib.synthetic_params(20, 100)
  _check(engine_mod, p, weights_lib.init_weights(p, seed=9), rows)


def test_ragged_batches_chunks_and_determinism(engine_mod):
  p = params_lib.synthetic_params(20, 120, num_hidden_layers=2)
  w = weights_lib.init_weights(p, seed=10)
  rows = synthetic.make_rows(p, 37, seed=11)
  whole = _check(engine_mod, p, w, rows)
  model = engine_mod.B200Model(p, w, max_batch=16, chunk_tiles=3,     # 3 engine calls, several chunks each
                               calibration=calibration.parse_calibration_string(CAL))
  split = model.forward(rows, want_logits=True)
  again = model.forward(rows, want_logits=True)
  one = model.forward(rows[:1], want_logits=True)
  model.close()
  assert np.array_equal(split["logits"], again["logits"])             # deterministic
  assert np.array_equal(split["bases"], whole["bases"]) and np.array_equal(split["quals"], whole["quals"])
  assert np.array_equal(split["logits"], whole["logits"])             # windows are independent units
  assert np.array_equal(one["logits"][0], whole["logits"][0])         # batch of 1


def test_out_of_range_input_is_flagged(engine_mod):
  p = params_lib.synthetic_params(20, 100, num_hidden_layers=1)
  w = weights_lib.init_weights(p, seed=12)
  rows = synthetic.make_rows(p, 2, seed=13)
  rows[0, 0, 5, 0] = 7.0                                               # base id 7 does not exist
  model = engine_mod.B200Model(p, w, max_batch=2)
  with pytest.raises(engine_mod.DcbError) as ei:
    model.forward(rows)
  assert ei.value.code == -5
  model.close()


def test_empty_batch_and_bad_shapes(engine_mod):
  p = params_lib.synthetic_params(20, 100, num_hidden_layers=1)
  model = engine_mod.B200Model(p, weights_lib.init_weights(p, seed=1), max_batch=4)
  out = model.forward(np.zeros((0, 85, 100, 1), np.float32))
  assert out["bases"].shape == (0, 100)
  with pytest.raises(ValueError):
    model.forward(np.zeros((1, 86, 100, 1), np.float32))
  model.close()


def test_run_model_on_examples_and_stitch(engine_mod, golden_dir):
  """The reference-facing call: feature dicts in, DCModelOutput list out, FASTQ via stitch_utils."""
  from deepconsensus_b200 import inference, stitch_utils
  z = np.load(os.path.join(golden_dir, "real_windows_human_1m.npz"))
  rows, names, pos = z["rows"], z["names"], z["window_pos"]
  p = params_lib.synthetic_params(20, 100)
  w = weights_lib.init_weights(p, seed=14)
  cal = calibration.parse_calibration_string(CAL)
  opts = inference.InferenceOptions(max_length=100, example_height=85, max_passes=20, min_quality=0, min_length=0,
                                    batch_size=24, use_ccs_bq=False, cpus=0, skip_windows_above=45,
                                    use_saved_model=False, max_base_quality=93, dc_calibration_values=cal,
                                    ccs_calibration_values=calibration.parse_calibration_string("skip"))
  model, p = inference.initialize_model("", p, opts, weights=w)
  fds = [dict(subreads=rows[i][..., None], **{"subreads/num_passes": 3}, window_pos=int(pos[i]), name=str(names[i]),
              ccs_base_quality_scores=np.zeros(100), ec=1.0, np_num_passes=3, rq=0.99, rg="rg") for i in range(len(rows))]
  preds = inference.run_model_on_examples(fds, model, p, opts)
  # fast path: the same windows, grouped by read and sorted by position, straight to FASTQ records with the byte work
  # on the device -- must equal stitch_to_fastq over the per-window objects, read for read
  order = sorted(range(len(fds)), key=lambda i: (fds[i]["name"], fds[i]["window_pos"]))
  cnt_fast = stitch_utils.OutcomeCounter()
  fast = inference.run_model_and_stitch([fds[i] for i in order], model, p, opts, cnt_fast)
  cnt_ref, slow, i = stitch_utils.OutcomeCounter(), [], 0
  while i < len(order):
    j = i
    while j < len(order) and fds[order[j]]["name"] == fds[order[i]]["name"]:
      j += 1
    slow.append(stitch_utils.stitch_to_fastq(fds[order[i]]["name"], [preds[k] for k in order[i:j]], 100, 0, 0, cnt_ref))
    i = j
  assert fast == slow and cnt_fast.__dict__ == cnt_ref.__dict__
  model.close()
  assert len(preds) == len(rows) and all(len(o.sequence) == 100 and len(o.quality_string) == 100 for o in preds)
  ref = omodel.forward(rows, p, w)
  y, q = opost.quality_from_probs(ref["probs"], 93, (cal.threshold, cal.w, cal.b))
  agree = np.mean([np.mean(np.frombuffer(o.sequence.encode(), np.uint8) == opost.to_ascii(y[i], q[i])[0]) for i, o in enumerate(preds)])
  assert agree > 0.98
  # windows of one ZMW, re-indexed contiguously, stitch into a FASTQ record
  first = str(names[0])
  mine = [o for o in preds if o.molecule_name == first]
  for k, o in enumerate(sorted(mine, key=lambda o: o.window_pos)):
    o.window_pos = k * 100
  cnt = stitch_utils.OutcomeCounter()
  fq = stitch_utils.stitch_to_fastq(first, sorted(mine, key=lambda o: o.window_pos), 100, 0, 0, cnt)
  assert fq is not None and fq.startswith("@" + first + "\n") and cnt.success == 1


def test_run_model_and_stitch_merges_skipped_windows(engine_mod, golden_dir):
  """The reference concatenates predictions_from_model + predictions_for_skipped_windows, sorts by (name, window_pos)
  and stitches per read (quick_inference.py:657-686,721-736); skip_windows_above=45 is the default and overflow
  windows always bypass the model.  run_model_and_stitch(..., skipped_outputs=...) must give the same FASTQ records as
  that flow built from per-window objects, read for read -- including reads that consist only of skipped windows."""
  import itertools
  from deepconsensus_b200 import inference, stitch_utils
  z = np.load(os.path.join(golden_dir, "real_windows_human_1m.npz"))
  rows, names, pos = z["rows"], z["names"], z["window_pos"]
  p = params_lib.synthetic_params(20, 100, num_hidden_layers=2)
  w = weights_lib.init_weights(p, seed=15)
  cal = calibration.parse_calibration_string(CAL)
  opts = inference.InferenceOptions(max_length=100, example_height=85, max_passes=20, min_quality=0, min_length=0,
                                    batch_size=16, use_ccs_bq=False, cpus=0, skip_windows_above=45,
                                    use_saved_model=False, max_base_quality=93, dc_calibration_values=cal,
                                    ccs_calibration_values=calibration.parse_calibration_string("skip"))
  model, p = inference.initialize_model("", p, opts, weights=w)
  rng = np.random.default_rng(3)
  by_zmw = {}
  keep_real = set(sorted(set(str(n) for n in names))[-2:])
  for i in range(len(rows)):
    kind = rng.integers(0, 4)                      # 0: overflow, 1: high-quality CCS (skipped), 2-3: scored
    bq = np.full(100, 60 if kind == 1 else 20, np.int64)
    # window_pos re-indexed contiguously per read (get_full_sequence advances by max_length per window,
    # stitch_utils.py:60-78); two reads keep their real CCS coordinates and therefore stitch to "missing window"
    name = str(names[i])
    k = len(by_zmw.get(name, []))
    wp = int(pos[i]) if name in keep_real else k * 100
    fd = dict(subreads=rows[i][..., None], **{"subreads/num_passes": 3}, window_pos=wp, name=name,
              ccs_base_quality_scores=bq, ec=1.0, np_num_passes=3, rq=0.99, rg="rg", overflow=bool(kind == 0))
    by_zmw.setdefault(name, []).append(fd)
  first = sorted(by_zmw)[0]
  for fd in by_zmw[first]:                         # one read made of skipped windows only
    fd["overflow"] = True
  for_model, skipped = inference.split_skipped_windows(by_zmw.values(), opts)
  assert skipped and for_model and len(skipped) + len(for_model) == len(rows)
  # the reference flow on per-window objects
  preds = inference.run_model_on_examples(for_model, model, p, opts) + skipped
  preds = sorted(preds, key=lambda dc: (dc.molecule_name, dc.window_pos))
  want, want_cnt = [], stitch_utils.OutcomeCounter()
  for name, grp in itertools.groupby(preds, lambda dc: dc.molecule_name):
    want.append(stitch_utils.stitch_to_fastq(name, list(grp), 100, 0, 0, want_cnt))
  got_cnt = stitch_utils.OutcomeCounter()
  got = inference.run_model_and_stitch(for_model, model, p, opts, got_cnt, skipped_outputs=skipped)
  assert got == want and got_cnt.__dict__ == want_cnt.__dict__
  assert sum(r is not None for r in got) >= 3 and got_cnt.empty_sequence >= 1
  # dropping the skipped windows (the round-1 behaviour) is NOT equivalent
  lost_cnt = stitch_utils.OutcomeCounter()
  lost = inference.run_model_and_stitch(for_model, model, p, opts, lost_cnt)
  assert lost != want
  model.close()


@pytest.mark.parametrize("ccs_cal,min_q,min_len", [("skip", 0, 0), ("0,1.1,-0.5", 20, 0), ("30,0.9,2.0", 0, 450)])
def test_device_post_model_stage_equals_reference_flow(engine_mod, golden_dir, ccs_cal, min_q, min_len):
  """SURVEY.md 8(f)2 on the device: skip decision (dcb_skip_mask), process_skipped_window (dcb_fill_skipped), sort,
  stitch + filters + FASTQ bytes (dcb_stitch_fastq) == the reference flow on per-window Python objects
  (split_skipped_windows -> run_model_on_examples -> sorted -> stitch_to_fastq), read for read, counter for counter."""
  import itertools
  from deepconsensus_b200 import inference, stitch_utils
  z = np.load(os.path.join(golden_dir, "real_windows_human_1m.npz"))
  rows, names, pos = z["rows"], z["names"], z["window_pos"]
  p = params_lib.synthetic_params(20, 100, num_hidden_layers=2)
  w = weights_lib.init_weights(p, seed=25)
  opts = inference.InferenceOptions(max_length=100, example_height=85, max_passes=20, min_quality=min_q, min_length=min_len,
                                    batch_size=32, use_ccs_bq=False, cpus=0, skip_windows_above=45,
                                    use_saved_model=False, max_base_quality=93,
                                    dc_calibration_values=calibration.parse_calibration_string(CAL),
                                    ccs_calibration_values=calibration.parse_calibration_string(ccs_cal))
  model, p = inference.initialize_model("", p, opts, weights=w)
  rng = np.random.default_rng(8)
  by_zmw = {}
  for i in range(len(rows)):
    name = str(names[i])
    k = len(by_zmw.get(name, []))
    kind = rng.integers(0, 5)
    ccs = rows[i][80]
    bq = np.where(ccs == 0, -1, rng.integers(50 if kind == 1 else 5, 94 if kind == 1 else 60, size=100)).astype(np.int64)
    if kind == 2:
      bq[:] = np.where(ccs == 0, -1, 45)                      # average exactly at the threshold: not skipped (> 45)
    fd = dict(subreads=rows[i][..., None], **{"subreads/num_passes": 3}, window_pos=k * 100, name=name,
              ccs_base_quality_scores=bq, ec=1.0, np_num_passes=3, rq=0.99, rg="rg", overflow=bool(kind == 0))
    by_zmw.setdefault(name, []).append(fd)
  zmws = [by_zmw[k] for k in sorted(by_zmw)]
  zmws[1][3]["window_pos"] += 100                             # a missing window in one read
  for_model, skipped = inference.split_skipped_windows(zmws, opts)
  assert len(skipped) >= 8 and len(for_model) >= 8
  assert sum(not fd["overflow"] for zz in zmws for fd in zz) > len(for_model)      # some skipped by quality, not overflow
  preds = sorted(inference.run_model_on_examples(for_model, model, p, opts) + skipped,
                 key=lambda dc: (dc.molecule_name, dc.window_pos))
  want, want_cnt = [], stitch_utils.OutcomeCounter()
  for name, grp in itertools.groupby(preds, lambda dc: dc.molecule_name):
    want.append(stitch_utils.stitch_to_fastq(name, list(grp), 100, min_q, min_len, want_cnt))
  got_cnt = stitch_utils.OutcomeCounter()
  got = inference.inference_on_zmw_windows(zmws, model, p, opts, got_cnt)
  assert got == want and got_cnt.__dict__ == want_cnt.__dict__
  assert got_cnt.empty_sequence >= 1
  if min_q or min_len:
    assert got_cnt.failed_quality_filter + got_cnt.failed_length_filter >= 1
  else:
    assert got_cnt.success >= 1
  # the device predicate alone, against the NumPy expression, incl. all-gap and all-zero windows
  bq = np.stack([np.asarray(fd["ccs_base_quality_scores"]) for zz in zmws for fd in zz]).astype(np.int16)
  bq[0, :] = -1
  bq[1, :] = 0
  mask, avg = model.skip_mask(bq, 45)
  from deepconsensus_b200 import utils as u
  ref_avg = np.array([u.avg_phred(r) for r in bq])
  assert np.abs(avg - ref_avg).max() < 1e-9
  exact = mask != 2
  assert np.array_equal(mask[exact].astype(bool), (ref_avg > 45)[exact]) and (mask == 2).sum() >= 1
  model.close()


def test_run_from_bam_fixtures_end_to_end(engine_mod, golden_dir, tmp_path):
  """BASELINE configs[0] (plumbing): `deepconsensus run` on the reference's own BAM fixtures (testdata/human_1m; the
  stored subread BAM keeps 7 of its 10 ZMWs, 958 windows) -- BAM -> features (C++) -> skip / model / fill / stitch
  (CUDA) -> FASTQ and BAM.  The fixture model directory ships without its data shard, so the variables are seeded; the
  check is that the whole native flow gives the records the reference flow on per-window Python objects gives, and that
  FASTQ and BAM outputs agree."""
  import gzip, itertools, shutil
  from deepconsensus_b200 import inference, preprocess, run as run_lib, stitch_utils
  d = os.path.join(golden_dir, "human_1m")
  ck = tmp_path / "model"
  shutil.copytree(os.path.join(golden_dir, "ckpt", "model"), ck)
  args = dict(subreads_to_ccs=os.path.join(d, "subreads_to_ccs.bam"), ccs_bam=os.path.join(d, "ccs.bam"),
              checkpoint=str(ck / "checkpoint-1"), batch_zmws=4, batch_size=256, min_quality=0, random_weights=3)
  fq = str(tmp_path / "out.fastq")
  cnt = run_lib.run(output=fq, **args)
  bam = str(tmp_path / "out.bam")
  cnt2 = run_lib.run(output=bam, **args)
  assert cnt.__dict__ == cnt2.__dict__ and cnt.success + cnt.failed_quality_filter + cnt.empty_sequence + cnt.only_gaps == 7
  got = open(fq).read()
  # reference flow from per-window objects
  p = params_lib.read_params_from_json(str(ck / "checkpoint-1"))
  opts = inference.InferenceOptions(max_length=100, example_height=85, max_passes=20, min_quality=0, min_length=0,
                                    batch_size=256, use_ccs_bq=False, cpus=0, skip_windows_above=45, use_saved_model=False,
                                    max_base_quality=93,
                                    dc_calibration_values=calibration.parse_calibration_string(p.get("dc_calibration", "skip")),
                                    ccs_calibration_values=calibration.parse_calibration_string("skip"))
  params_lib.modify_params(p, max_length=100)
  model, p = inference.initialize_model("", p, opts, weights=weights_lib.init_weights(p, seed=3))
  zmws = list(preprocess.stream_zmw_windows(args["subreads_to_ccs"], args["ccs_bam"], 20, 100))
  for_model, skipped = inference.split_skipped_windows(zmws, opts)
  preds = sorted(inference.run_model_on_examples(for_model, model, p, opts) + skipped,
                 key=lambda dc: (dc.molecule_name, dc.window_pos))
  model.close()
  want, want_cnt = [], stitch_utils.OutcomeCounter()
  for name, grp in itertools.groupby(preds, lambda dc: dc.molecule_name):
    rec = stitch_utils.stitch_to_fastq(name, list(grp), 100, 0, 0, want_cnt)
    if rec:
      want.append(rec)
  # the run processes ZMWs in batches of 4 in file order and sorts within a batch; compare as sets of records
  assert sorted(got.split("@")[1:]) == sorted("".join(want).split("@")[1:])
  assert cnt.__dict__ == want_cnt.__dict__ and cnt.success >= 5
  # BAM output: same names / sequences / qualities as the FASTQ
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


def test_pipeline_survives_errors_and_mixed_use(engine_mod):
  """(1) a wait() that raises (out-of-range id) must not leave the younger submission in flight: the next call works;
  (2) a blocking forward() between two submit()s must not collide with the slot of the outstanding handle."""
  from deepconsensus_b200 import inference
  p = params_lib.synthetic_params(20, 100, num_hidden_layers=1)
  w = weights_lib.init_weights(p, seed=16)
  model = engine_mod.B200Model(p, w, max_batch=8)
  good = synthetic.make_rows(p, 8, seed=17)
  bad = good.copy()
  bad[0, 0, 0] = 9.0
  want = model.forward(good)
  with pytest.raises(engine_mod.DcbError):
    list(model.forward_batches([bad, good, good]))
  again = list(model.forward_batches([good, good[:3]]))
  assert np.array_equal(again[0]["bases"], want["bases"]) and np.array_equal(again[1]["quals"], want["quals"][:3])
  fds = [dict(subreads=r[..., None] if r.ndim == 2 else r, **{"subreads/num_passes": 3}, window_pos=0, name="m/%d/ccs" % i,
              ccs_base_quality_scores=np.zeros(100), ec=1.0, np_num_passes=3, rq=0.99, rg="rg")
         for i, r in enumerate(np.concatenate([bad, good, good]))]
  opts = inference.InferenceOptions(max_length=100, example_height=85, max_passes=20, min_quality=0, min_length=0,
                                    batch_size=8, use_ccs_bq=False, cpus=0, skip_windows_above=0, use_saved_model=False,
                                    max_base_quality=93, dc_calibration_values=calibration.parse_calibration_string("skip"),
                                    ccs_calibration_values=calibration.parse_calibration_string("skip"))
  with pytest.raises(engine_mod.DcbError):
    inference.run_model_on_examples(fds, model, p, opts)
  assert len(inference.run_model_on_examples(fds[8:], model, p, opts)) == 16
  h0 = model.submit(good)
  mid = model.forward(good[:2])                     # consumes a ticket while h0 is outstanding
  h1 = model.submit(good[:5])
  o0, o1 = model.wait(h0), model.wait(h1)
  assert np.array_equal(o0["bases"], want["bases"]) and np.array_equal(o1["bases"], want["bases"][:5])
  assert np.array_equal(mid["quals"], want["quals"][:2])
  model.close()


@pytest.mark.parametrize("P,L,bq,layers", [(20, 120, False, 2), (20, 100, True, 2), (32, 200, False, 1), (5, 40, True, 1)])
def test_packed_rows_give_bit_identical_results(engine_mod, P, L, bq, layers):
  """dcb_forward_packed (SURVEY.md 8(f)1): packed rows read inside the embedding kernel (L <= 128) or unpacked on the
  device (L = 200, strict path) -> exactly the outputs of dcb_forward on the float32 rows, ~5.5x fewer H2D bytes."""
  p = params_lib.synthetic_params(P, L, use_ccs_bq=bq, num_hidden_layers=layers)
  w = weights_lib.init_weights(p, seed=80 + L)
  rows = synthetic.make_rows(p, 23, seed=81 + L)
  model = engine_mod.B200Model(p, w, max_batch=16)            # 23 windows: two engine calls, ragged second one
  packed = model.pack_rows(rows)
  assert packed.shape[1] * 4 < rows[0].size * 4
  for strict in (False, True):
    a = model.forward(rows, want_probs=True, want_logits=True, strict=strict)
    b = model.forward_packed(packed, want_probs=True, want_logits=True, strict=strict)
    for k in ("bases", "quals", "probs", "logits"):
      assert np.array_equal(a[k], b[k]), (k, strict)
  # device-resident packed rows + device-side outputs
  B = 16
  dp = model.alloc_device(packed[:B].nbytes)
  model.memcpy_h2d(dp, packed[:B])
  db, dq = model.alloc_device(B * L), model.alloc_device(B * L)
  t = model.submit_packed_raw(dp, B, engine_mod.DCB_ROWS_ON_DEVICE | engine_mod.DCB_OUT_ON_DEVICE, db, dq)
  model.wait_raw(t)
  hb = np.empty((B, L), np.uint8)
  model.memcpy_d2h(hb, db)
  assert np.array_equal(hb, a["bases"][:B]) or np.array_equal(hb, model.forward(rows[:B])["bases"])
  # an out-of-vocabulary byte is flagged by the device exactly like the float path
  bad = packed[:2].copy()
  bad[1, 3] = 6                                               # base id 6
  with pytest.raises(engine_mod.DcbError) as ei:
    model.forward_packed(bad)
  assert ei.value.code == -5
  for d in (dp, db, dq):
    model.free_device(d)
  model.close()


def test_initialize_model_from_a_tf_checkpoint(engine_mod, tmp_path):
  """quick_inference.initialize_model restores a TF2 checkpoint (quick_inference.py:515-529): here read without
  TensorFlow (tf_checkpoint) from prefix / directory, and the engine scores exactly as with the same arrays passed in."""
  from deepconsensus_b200 import inference, tf_checkpoint
  p = params_lib.synthetic_params(20, 100, use_ccs_bq=True, rezero=False, num_hidden_layers=2)
  w = weights_lib.init_weights(p, seed=90)
  tf_checkpoint.write_checkpoint(str(tmp_path / "checkpoint-4"), w)
  opts = inference.InferenceOptions(max_length=100, example_height=86, max_passes=20, min_quality=0, min_length=0,
                                    batch_size=8, use_ccs_bq=True, cpus=0, skip_windows_above=0, use_saved_model=False,
                                    max_base_quality=93, dc_calibration_values=calibration.parse_calibration_string(CAL),
                                    ccs_calibration_values=calibration.parse_calibration_string("skip"))
  rows = synthetic.make_rows(p, 5, seed=91)
  m0, _ = inference.initialize_model("", p.copy(), opts, weights=w)
  want = m0.forward(rows, want_logits=True)
  m0.close()
  for path in (str(tmp_path / "checkpoint-4"), str(tmp_path)):
    m, _ = inference.initialize_model(path, p.copy(), opts)
    got = m.forward(rows, want_logits=True)
    m.close()
    assert np.array_equal(got["logits"], want["logits"]) and np.array_equal(got["quals"], want["quals"])
  del w["model/fc1/bias"]
  tf_checkpoint.write_checkpoint(str(tmp_path / "checkpoint-5"), w)
  with pytest.raises(Exception):
    inference.initialize_model(str(tmp_path / "checkpoint-5"), p.copy(), opts)


def test_unfused_fallback_paths_agree_with_fused(engine_mod):
  """DCB_STACK / DCB_FUSE_HEAD / DCB_FUSE_OPROJ / DCB_FUSE_EMBED / DCB_FUSE_QA / DCB_ALIGN select measured alternatives
  of the same math.  They exist only in the developer build (libdcb200_dev.so, -DDCB_DEV_SWITCHES) and
  are read when an engine is created; the product library ignores the environment (checked first)."""
  p = params_lib.synthetic_params(20, 120, num_hidden_layers=2)
  w = weights_lib.init_weights(p, seed=21)
  rows = synthetic.make_rows(p, 5, seed=22)
  ref = omodel.forward(rows, p, w)["logits"]
  dev = engine_mod.load_dev_library()
  outs = {}
  for name, env in (("fused", {}),                                     # default: whole stack in one kernel
                    ("per_layer", {"DCB_STACK": "0"}),                  # QKV+attention and out-proj+FFN kernels per layer
                    ("separate_head", {"DCB_FUSE_HEAD": "0"}),          # head_kernel after the stack instead of its fused tail
                    ("unfused", {"DCB_FUSE_OPROJ": "0", "DCB_FUSE_EMBED": "0", "DCB_FUSE_QA": "0"}),
                    ("packed", {"DCB_ALIGN": "0"})):                    # windows packed back to back, separate QKV / attention
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
      model = engine_mod.B200Model(p, w, max_batch=8, library=dev)
      outs[name] = model.forward(rows, want_logits=True)["logits"]
      launches = model.last_launches
      model.close()
      if name == "per_layer":
        prod = engine_mod.B200Model(p, w, max_batch=8)              # product library: the switch is ignored
        prod.forward(rows)
        assert prod.last_launches == 2 and launches > 2
        prod.close()
    finally:
      for k, v in old.items():
        if v is None:
          os.environ.pop(k, None)
        else:
          os.environ[k] = v
    assert np.abs(outs[name] - ref).max() <= LOGIT_TOL_FP32, name
  assert np.abs(outs["fused"] - outs["per_layer"]).max() < 0.05
  assert np.abs(outs["fused"] - outs["separate_head"]).max() < 1e-3
  assert np.abs(outs["fused"] - outs["unfused"]).max() < 0.05
  assert np.abs(outs["fused"] - outs["packed"]).max() < 0.05


@pytest.mark.parametrize("name", ["rezero_p20", "layernorm_p20", "rezero_p20_bq", "layernorm_p20_bq", "rezero_p5_win3",
                                  "c2_p20_l120", "c5_p32_l200", "c5_p32_l200_ln_bq"])
def test_engine_against_reference_code_goldens(engine_mod, golden_dir, name):
  """CUDA paths vs outputs of the reference's OWN model code (tests/golden/ref_model_*.npz, generated by
  scripts/make_model_golden.py) -- no oracle in between.  Includes the BASELINE configs[1] (P=20, L=120) and
  configs[4] (P=32, L=200) shapes."""
  z = np.load(os.path.join(golden_dir, "ref_model_%s.npz" % name))
  p = params_lib.get_config(str(z["config"]))
  for k, v in ast.literal_eval(str(z["overrides"])).items():
    p[k] = v
  params_lib.modify_params(p, max_length=int(z["max_length"]))
  w = weights_lib.init_weights(p, seed=int(z["seed"]))
  rows = z["rows"]
  cal = calibration.parse_calibration_string("skip")
  model = engine_mod.B200Model(p, w, max_batch=rows.shape[0])
  out = model.forward(rows, want_probs=True, want_logits=True)
  strict = model.forward(rows, want_probs=True, want_logits=True, strict=True)
  model.close()
  refd = _ref_dict(z["logits"], z["probs"], cal)
  _assert_strict(strict, refd, name)
  assert np.abs(strict["probs"] - z["probs"]).max() < 2e-5
  _assert_default(out, refd, name)
  assert np.abs(out["probs"] - z["probs"]).max() < 0.03


def test_strict_precision_engine_and_per_call_override(engine_mod):
  """dcb_config.precision = DCB_PRECISION_FP32 makes strict the default of the engine; DCB_FAST_BF16 / DCB_STRICT_FP32
  override per call; both flags at once are refused; ragged batches, chunking (batch > strict chunk) and determinism."""
  p = params_lib.synthetic_params(20, 120, num_hidden_layers=2)
  w = weights_lib.init_weights(p, seed=71)
  rows = synthetic.make_rows(p, 150, seed=72)                # 150 x 120 tokens > the 16 k-token strict chunk
  cal = calibration.parse_calibration_string(CAL)
  ms = engine_mod.B200Model(p, w, max_batch=150, calibration=cal, precision="fp32")
  mf = engine_mod.B200Model(p, w, max_batch=150, calibration=cal)
  a = ms.forward(rows, want_logits=True, want_probs=True)
  b = mf.forward(rows, want_logits=True, want_probs=True, strict=True)
  assert np.array_equal(a["logits"], b["logits"]) and np.array_equal(a["quals"], b["quals"])
  again = ms.forward(rows, want_logits=True)
  assert np.array_equal(a["logits"], again["logits"])
  sub = ms.forward(rows[140:147], want_logits=True)
  assert np.array_equal(sub["logits"], a["logits"][140:147])          # windows are independent units
  fast_on_strict = ms.forward(rows, want_logits=True, strict=False)
  fast = mf.forward(rows, want_logits=True)
  assert np.array_equal(fast_on_strict["logits"], fast["logits"])
  piped = list(ms.forward_batches([rows[:150], rows[:33]], want_logits=True))
  assert np.array_equal(piped[0]["logits"], a["logits"]) and np.array_equal(piped[1]["logits"], a["logits"][:33])
  with pytest.raises(engine_mod.DcbError):
    ms.forward_raw(rows.ctypes.data, 1, engine_mod.DCB_STRICT_FP32 | engine_mod.DCB_FAST_BF16,
                   a["bases"].ctypes.data, a["quals"].ctypes.data)
  ref = omodel.forward(rows[:16], p, w)
  _assert_strict({k: v[:16] for k, v in a.items()}, _ref_dict(ref["logits"], ref["probs"], cal))
  _epilogue_exact(a, cal)
  bad = rows[:2].copy()
  bad[1, 0, 3] = 9.0
  with pytest.raises(engine_mod.DcbError) as ei:
    ms.forward(bad)
  assert ei.value.code == -5
  ms.close()
  mf.close()


@pytest.mark.parametrize("cfg", ["c3_b4096", "c5_b8192"])
def test_full_size_default_vs_strict_on_device(engine_mod, cfg):
  """BASELINE configs[2] (checkpoint config: L=100, CCS-BQ, 5 pre-LN layers; batch 4096) and configs[4] (P=32, L=200,
  batch 8192) at FULL size.  The oracle cannot score thousands of windows in test time, so: (1) the default path is
  compared with the strict-fp32 path ON THE DEVICE over 512 windows spread over the whole batch (first / middle / last
  CTA rounds and chunks), (2) the strict path is pinned to the oracle on 8 of those windows, (3) sub-batch
  reproducibility and the exact epilogue hold over the full batch."""
  if cfg == "c3_b4096":
    p = params_lib.synthetic_params(20, 100, use_ccs_bq=True, num_hidden_layers=5, rezero=False)
    B, seed = 4096, 301
  else:
    p = params_lib.synthetic_params(32, 200)
    B, seed = 8192, 302
  w = weights_lib.init_weights(p, seed=seed)
  rows = synthetic.make_rows(p, B, seed=seed + 1)
  cal = calibration.parse_calibration_string(CAL)
  model = engine_mod.B200Model(p, w, max_batch=B, calibration=cal)
  full = model.forward(rows, want_probs=True, want_logits=True)
  _epilogue_exact(full, cal)
  assert np.isfinite(full["logits"]).all()
  idx = np.unique(np.concatenate([np.arange(0, 64), np.arange(B // 2 - 32, B // 2 + 32), np.arange(B - 64, B),
                                  np.random.default_rng(5).choice(B, 320, replace=False)]))
  sub = model.forward(rows[idx], want_probs=True, want_logits=True)
  assert np.array_equal(sub["logits"], full["logits"][idx])              # windows are independent units
  strict = model.forward(rows[idx], want_probs=True, want_logits=True, strict=True)
  model.close()
  st = _assert_default(sub, strict, cfg)
  print(cfg, "default vs strict on %d windows:" % len(idx), parity.summary(st))
  pick = idx[:: max(1, len(idx) // 8)][:8]
  ref = omodel.forward(rows[pick], p, w)
  sel = np.searchsorted(idx, pick)
  _assert_strict({k: v[sel] for k, v in strict.items()}, _ref_dict(ref["logits"], ref["probs"], cal), cfg)


def test_pipelined_submit_wait_matches_blocking_forward(engine_mod):
  """dcb_submit / dcb_wait (two batches in flight, H2D of batch i+1 under the kernels of batch i) returns exactly what
  dcb_forward returns, keeps order, reports per-ticket input errors and refuses a third outstanding submission."""
  p = params_lib.synthetic_params(20, 120)
  w = weights_lib.init_weights(p, seed=31)
  model = engine_mod.B200Model(p, w, max_batch=16)
  batches = [synthetic.make_rows(p, n, seed=40 + i) for i, n in enumerate((16, 7, 16, 1, 12))]
  blocking = [model.forward(b, want_probs=True) for b in batches]
  piped = list(model.forward_batches(batches, want_probs=True))
  assert len(piped) == len(blocking)
  for a, b in zip(blocking, piped):
    assert np.array_equal(a["bases"], b["bases"]) and np.array_equal(a["quals"], b["quals"])
    assert np.array_equal(a["probs"], b["probs"])
  # a bad batch between two good ones: only its own ticket reports the range error
  bad = batches[1].copy()
  bad[0, 0, 0] = 9.0
  h0 = model.submit(batches[0])
  h1 = model.submit(bad)
  with pytest.raises(engine_mod.DcbError):
    model.submit(batches[2])                      # two already in flight
  o0 = model.wait(h0)
  with pytest.raises(engine_mod.DcbError):
    model.wait(h1)
  with pytest.raises(engine_mod.DcbError):
    model.wait(h1)                                # not in flight any more
  h2 = model.submit(batches[2])
  o2 = model.wait(h2)
  assert np.array_equal(o0["bases"], blocking[0]["bases"]) and np.array_equal(o2["quals"], blocking[2]["quals"])
  model.close()


def test_full_size_properties_c2_batch_1024(engine_mod):
  """BASELINE configs[1] at its full size (1024 windows, 20 x 120, 6 layers): too big for the oracle in test time, so the
  CUDA path is checked through size-independent properties -- windows are independent units, hence
  (a) permuting the batch permutes the outputs bit-exactly, (b) any sub-batch reproduces its rows of the full batch
  bit-exactly (different tile -> SM assignment, different pairing), (c) probabilities sum to one, (d) the device epilogue
  (argmax / Phred / calibration / ASCII) is exact integer work on the device's own probabilities, (e) a 16-window slice
  agrees with the oracle."""
  p = params_lib.synthetic_params(20, 120)
  w = weights_lib.init_weights(p, seed=101)
  B = 1024
  rows = synthetic.make_rows(p, B, seed=102)
  cal = calibration.parse_calibration_string(CAL)
  model = engine_mod.B200Model(p, w, max_batch=B, calibration=cal)
  full = model.forward(rows, want_probs=True)
  again = model.forward(rows, want_probs=True)
  assert np.array_equal(full["probs"], again["probs"]) and np.array_equal(full["quals"], again["quals"])
  rng = np.random.default_rng(7)
  perm = rng.permutation(B)
  permuted = model.forward(rows[perm], want_probs=True)
  assert np.array_equal(permuted["probs"], full["probs"][perm])
  assert np.array_equal(permuted["bases"], full["bases"][perm]) and np.array_equal(permuted["quals"], full["quals"][perm])
  for lo, hi in ((0, 1), (5, 12), (300, 811), (1023, 1024)):
    sub = model.forward(rows[lo:hi], want_probs=True)
    assert np.array_equal(sub["probs"], full["probs"][lo:hi]), (lo, hi)
    assert np.array_equal(sub["bases"], full["bases"][lo:hi]) and np.array_equal(sub["quals"], full["quals"][lo:hi])
  assert np.isfinite(full["probs"]).all() and np.abs(full["probs"].sum(-1) - 1).max() < 1e-5
  _epilogue_exact(full, cal)
  # every one of the 1024 windows: default path against the strict-fp32 path, both on the device
  fl = model.forward(rows, want_probs=True, want_logits=True)
  assert np.array_equal(fl["probs"], full["probs"])
  strict = model.forward(rows, want_probs=True, want_logits=True, strict=True)
  st = _assert_default(fl, strict, "c2 b1024")
  print("C2 B=1024 default vs strict:", parity.summary(st))
  ref = omodel.forward(rows[500:516], p, w)
  refd = _ref_dict(ref["logits"], ref["probs"], cal)
  _assert_strict({k: v[500:516] for k, v in strict.items()}, refd, "c2 b1024 strict")
  _assert_default({k: v[500:516] for k, v in fl.items()}, refd, "c2 b1024 default")
  model.close()
  m2 = engine_mod.B200Model(p, w, max_batch=16, calibration=cal)
  o16 = m2.forward(rows[500:516], want_probs=True, want_logits=True)
  m2.close()
  assert np.array_equal(o16["probs"], full["probs"][500:516])


@pytest.mark.parametrize("layers,ff,rezero,win,L,B", [
    (1, 128, True, 12, 120, 3),      # one layer, one hidden chunk: the FFN stage program never reaches the tail slots
    (3, 640, False, 16, 128, 4),     # pre-LN, band at the two-pass limit, window exactly one tile
    (8, 256, True, 1, 64, 5),        # deepest stack the one-kernel path takes, narrowest band, short windows
    (9, 256, True, 12, 100, 2),      # deeper than kMaxLayers: falls back to the per-layer kernels
])
def test_stack_kernel_corner_shapes(engine_mod, layers, ff, rezero, win, L, B):
  p = params_lib.synthetic_params(20, L, num_hidden_layers=layers, rezero=rezero, attn_win_size=win)
  p.filter_size = ff
  w = weights_lib.init_weights(p, seed=50 + layers)
  rows = synthetic.make_rows(p, B, seed=60 + layers)
  model = engine_mod.B200Model(p, w, max_batch=B)
  out = model.forward(rows, want_logits=True)
  launches = model.last_launches
  model.close()
  assert launches == (2 if layers <= 8 else 2 + 2 * layers)
  ref = omodel.forward(rows, p, w)
  assert np.isfinite(out["logits"]).all()
  # these are structural tests of the kernel's stage programs; the bf16 rounding error grows with depth (measured
  # 0.22 at 8 layers with the narrowest band), so the 8- and 9-layer cases get a proportionally wider gate
  assert np.abs(out["logits"] - ref["logits"]).max() <= (LOGIT_TOL_FP32 if layers <= 6 else 0.30)


@pytest.mark.parametrize("L,win,rezero,layers,B", [
    (200, 12, True, 6, 5),       # BASELINE configs[4] shape
    (129, 12, True, 2, 3),       # one valid row in the second tile
    (144, 16, False, 2, 4),      # pre-LN, band at the two-pass limit: the halo tile is fully used
    (256, 1, True, 3, 2),        # both tiles full, narrowest band
    (136, 8, False, 1, 1),       # single window
])
def test_wide_windows_on_the_one_kernel_stack(engine_mod, L, win, rezero, layers, B):
  """128 < L <= 256: one window per CTA pair (Lw = 256), the attention band crosses the pair through remote
  shared-memory fragment loads.  Same two launches as the L <= 128 path; parity gates as everywhere else."""
  p = params_lib.synthetic_params(20, L, num_hidden_layers=layers, rezero=rezero, attn_win_size=win)
  w = weights_lib.init_weights(p, seed=400 + L)
  rows = synthetic.make_rows(p, B, seed=401 + L)
  cal = calibration.parse_calibration_string(CAL)
  model = engine_mod.B200Model(p, w, max_batch=B, calibration=cal)
  out = model.forward(rows, want_probs=True, want_logits=True)
  assert model.last_launches == 2
  again = model.forward(rows, want_logits=True)
  assert np.array_equal(out["logits"], again["logits"])
  one = model.forward(rows[B - 1:], want_logits=True)
  assert np.array_equal(one["logits"][0], out["logits"][B - 1])
  strict = model.forward(rows, want_probs=True, want_logits=True, strict=True)
  model.close()
  ref = omodel.forward(rows, p, w)
  refd = _ref_dict(ref["logits"], ref["probs"], cal)
  _assert_strict(strict, refd)
  _assert_default(out, refd)
  _epilogue_exact(out, cal)
  # the positions next to the cut (112..143) are the ones that use the partner's rows: check them on their own
  cut = slice(112, min(L, 144))
  assert np.abs(out["logits"][:, cut] - ref["logits"][:, cut]).max() <= LOGIT_TOL_FP32


# ----------------------------------------------------------------------------------------------------------------
# SURVEY section 8(f) "next": stitching.  dcb_stitch does get_full_sequence + remove_gaps on the device (bytes: exact).
def _tiny_model(engine_mod, L=100):
  p = params_lib.synthetic_params(20, L, num_hidden_layers=1)
  return engine_mod.B200Model(p, weights_lib.init_weights(p, seed=1), max_batch=4), p


def test_device_stitch_against_executed_reference(engine_mod, golden_dir):
  """All 120 cases produced by executing the reference's stitch_utils (tests/golden/ref_stitch.json), stitched in
  batches on the device: FASTQ records and outcome counters must be identical, read for read."""
  import json
  from deepconsensus_b200 import stitch_gpu, stitch_utils
  with open(os.path.join(golden_dir, "ref_stitch.json")) as f:
    cases = json.load(f)["cases"]
  model, _ = _tiny_model(engine_mod)
  groups = {}
  for c in cases:
    groups.setdefault((c["max_length"], c["min_quality"], c["min_length"]), []).append(c)
  checked = 0
  for (L, min_q, min_len), cs in groups.items():
    bases, quals, names, pos = [], [], [], []
    for i, c in enumerate(cs):
      for w in c["windows"]:
        if w["dropped"]:
          continue
        assert len(w["sequence"]) == L and len(w["quality_string"]) == L
        bases.append(np.frombuffer(w["sequence"].encode("latin-1"), np.uint8))
        quals.append(np.frombuffer(w["quality_string"].encode("latin-1"), np.uint8))
        names.append("%s#%d" % (c["name"], i))          # reads with equal names in different cases stay separate
        pos.append(w["window_pos"])
    cnt = stitch_utils.OutcomeCounter()
    got = stitch_gpu.stitch_batch_to_fastq(model, np.stack(bases), np.stack(quals), names, pos, L, min_q, min_len, cnt)
    want_cnt = stitch_utils.OutcomeCounter()
    j = 0
    for i, c in enumerate(cs):
      if not any(not w["dropped"] for w in c["windows"]):
        continue                                          # a read with no windows at all never reaches the batch
      want = c["fastq"]
      if want is not None:
        want = want.replace("@" + c["name"] + "\n", "@%s#%d\n" % (c["name"], i), 1)
      assert got[j] == want, (c["name"], i)
      for k, v in c["counter"].items():
        setattr(want_cnt, k, getattr(want_cnt, k) + v)
      j += 1
      checked += 1
    assert j == len(got)
    assert cnt.__dict__ == want_cnt.__dict__
  assert checked >= 100
  model.close()


def test_device_stitch_chain_from_forward_outputs(engine_mod):
  """forward (outputs left on the device) -> dcb_stitch on those device buffers == forward to host -> Python mirror
  of stitch_to_fastq, for reads of ragged window counts, including one with a missing window and empty inputs."""
  from deepconsensus_b200 import stitch_gpu, stitch_utils
  model, p = _tiny_model(engine_mod, L=100)
  model.close()
  p = params_lib.synthetic_params(20, 100, num_hidden_layers=2)
  w = weights_lib.init_weights(p, seed=77)
  B, L = 37, 100
  model = engine_mod.B200Model(p, w, max_batch=B)
  rows = synthetic.make_rows(p, B, seed=78)
  host = model.forward(rows)
  counts = [1, 5, 2, 9, 3, 7, 10]
  assert sum(counts) == B
  names, pos = [], []
  for z, n in enumerate(counts):
    for i in range(n):
      names.append("m/%d/ccs" % z)
      pos.append(i * L if not (z == 3 and i >= 4) else (i + 1) * L)     # read 3 misses its 5th window
  # device chain
  dev_rows = model.alloc_device(rows.nbytes)
  model.memcpy_h2d(dev_rows, rows[..., 0])
  db, dq = model.alloc_device(B * L), model.alloc_device(B * L)
  model.forward_raw(dev_rows, B, engine_mod.DCB_ROWS_ON_DEVICE | engine_mod.DCB_OUT_ON_DEVICE, db, dq)
  cnt = stitch_utils.OutcomeCounter()
  got = stitch_gpu.stitch_batch_to_fastq(model, db, dq, names, pos, L, 0, 0, cnt, n_windows=B, on_device=True)
  # Python mirror, read by read
  want, want_cnt, k = [], stitch_utils.OutcomeCounter(), 0
  for z, n in enumerate(counts):
    preds = []
    for i in range(n):
      o = stitch_utils.DCModelOutput(names[k], pos[k], 1.0, 3, 0.99, "rg")
      o.sequence = host["bases"][k].tobytes().decode("ascii")
      o.quality_string = host["quals"][k].tobytes().decode("ascii")
      preds.append(o)
      k += 1
    want.append(stitch_utils.stitch_to_fastq(names[k - 1], preds, L, 0, 0, want_cnt))
  assert got == want and cnt.__dict__ == want_cnt.__dict__
  assert want[3] is None and cnt.empty_sequence == 1 and cnt.success >= 5
  # degenerate inputs
  s, q, l = model.stitch(np.zeros((0, L), np.uint8), np.zeros((0, L), np.uint8), np.array([0], np.int32))
  assert l.shape == (0,)
  allgap = np.full((2, L), ord(" "), np.uint8)
  s, q, l = model.stitch(allgap, allgap, np.array([0, 2], np.int32))
  assert l.tolist() == [0]
  for d in (dev_rows, db, dq):
    model.free_device(d)
  model.close()

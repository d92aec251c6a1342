"""Host driver pieces of `deepconsensus run` that touch the model (mirror of the hot-path part of
`deepconsensus/inference/quick_inference.py`).

  InferenceOptions        quick_inference.py:238-275 (same field names)
  batch_examples          quick_inference.py:304-338
  run_model_on_examples   quick_inference.py:341-415   <- the drop-in: same signature, same return
  initialize_model        quick_inference.py:485-532   (weights come from an .npz / dict instead of a
                                                         TF checkpoint; see INTEGRATION.md)

`run_model_on_examples` hands the stacked rows to the CUDA engine, which returns the per-position
base and quality characters directly (the device epilogue does argmax / Phred / calibration /
clip / round, quick_inference.py:377-389); the host only slices bytes into `DCModelOutput`s.
"""
from __future__ import annotations

import dataclasses
from typing import Any, Dict, Iterable, Iterator, List, Optional, Tuple, Union

import numpy as np

from deepconsensus_b200 import calibration as calibration_lib
from deepconsensus_b200 import constants
from deepconsensus_b200 import engine as engine_lib
from deepconsensus_b200 import params as params_lib
from deepconsensus_b200 import stitch_utils
from deepconsensus_b200 import utils
from deepconsensus_b200 import weights as weights_lib


@dataclasses.dataclass
class InferenceOptions:
  """Options used across the inference stages (quick_inference.py:238-275)."""
  max_length: int
  example_height: int
  max_passes: int
  min_quality: int
  min_length: int
  batch_size: int
  use_ccs_bq: bool
  cpus: int
  skip_windows_above: int
  use_saved_model: bool
  max_base_quality: int
  dc_calibration_values: calibration_lib.QualityCalibrationValues
  ccs_calibration_values: calibration_lib.QualityCalibrationValues


def format_rows(subreads: np.ndarray, params: params_lib.Params) -> np.ndarray:
  """Shape check only: the PW/IP/SN clipping of data_providers.format_rows (:128-184) runs on the
  device inside the embedding kernel, so rows are passed through unmodified."""
  rows = np.asarray(subreads, dtype=constants.NP_DATA_TYPE)
  if rows.ndim == 2:
    rows = rows[..., None]
  if rows.shape != (params.total_rows, params.max_length, 1):
    raise ValueError("expected subreads of shape %s, got %s" %
                     ((params.total_rows, params.max_length, 1), rows.shape))
  return rows


def process_feature_dict(features: Dict[str, Any], params: params_lib.Params) -> Dict[str, Any]:
  """data_providers.process_feature_dict (:187-223) without TensorFlow."""
  return {
      "rows": format_rows(features["subreads"], params),
      "label": np.array([]),
      "num_passes": features["subreads/num_passes"],
      "window_pos": features["window_pos"],
      "name": features["name"],
      "ccs_base_quality_scores": features["ccs_base_quality_scores"],
      "ec": features["ec"],
      "np_num_passes": features["np_num_passes"],
      "rq": features["rq"],
      "rg": features["rg"],
  }


def batch_examples(feature_dicts: List[Dict[str, Any]], model_params: params_lib.Params,
                   options: InferenceOptions) -> Iterator[Dict[str, Any]]:
  """Stack values for each feature, `options.batch_size` windows at a time (quick_inference.py:304-338)."""
  processed = [process_feature_dict(fd, model_params) for fd in feature_dicts]
  for i in range(0, len(processed), options.batch_size):
    one_batch = processed[i:i + options.batch_size]
    yield {key: np.stack([x[key] for x in one_batch]) for key in constants.DC_FEATURES}


def run_model_on_examples(feature_dicts: List[Dict[str, Any]], model: engine_lib.B200Model,
                          model_params: params_lib.Params,
                          options: InferenceOptions) -> List[stitch_utils.DCModelOutput]:
  """Runs the model over windows and returns one DCModelOutput per window (quick_inference.py:341-415)."""
  predictions: List[stitch_utils.DCModelOutput] = []

  def collect(data, out):
    bases, quals = out["bases"], out["quals"]
    for i in range(bases.shape[0]):
      predictions.append(stitch_utils.DCModelOutput(
          window_pos=data["window_pos"][i], molecule_name=data["name"][i], ec=data["ec"][i],
          np_num_passes=data["np_num_passes"][i], rq=data["rq"][i], rg=data["rg"][i],
          sequence=bases[i].tobytes().decode("ascii"),
          quality_string=quals[i].tobytes().decode("ascii")))

  _pipelined(model, batch_examples(feature_dicts, model_params, options), collect)
  return predictions


def _pipelined(model: engine_lib.B200Model, batches: Iterable[Dict[str, Any]], collect) -> None:
  """Two batches in flight: while the device scores batch i, batch i+1 is stacked and copied (dcb_submit / dcb_wait).
  If a wait raises (e.g. DCB_ERR_INPUT_RANGE), the younger submission is retired too, so the model stays usable."""
  pending = None
  try:
    for data in batches:
      handle = model.submit(data["rows"])
      prev, pending = pending, (data, handle)
      if prev is not None:
        collect(prev[0], model.wait(prev[1]))
    if pending is not None:
      last, pending = pending, None
      collect(last[0], model.wait(last[1]))
  finally:
    if pending is not None:
      model.drain(pending[1])


def process_skipped_window(feature_dict: Dict[str, Any], options: InferenceOptions) -> stitch_utils.DCModelOutput:
  """A window that is not sent to the model adopts the CCS bases and (calibrated, capped) CCS base qualities
  (quick_inference.py:567-594)."""
  rows = feature_dict["subreads"]
  ccs_index = params_lib.get_indices(options.max_passes, options.use_ccs_bq)[4]
  ccs = rows[ccs_index[0], :, 0]
  ccs_seq = utils.encoded_sequence_to_string(ccs)
  ccs_quality_scores = feature_dict["ccs_base_quality_scores"]
  if options.ccs_calibration_values.enabled:
    ccs_quality_scores = calibration_lib.calibrate_quality_scores(ccs_quality_scores, options.ccs_calibration_values)
  ccs_quality_scores = np.minimum(ccs_quality_scores, options.max_base_quality)
  ccs_quality_scores = ccs_quality_scores.astype(dtype=np.int32)
  return stitch_utils.DCModelOutput(
      window_pos=feature_dict["window_pos"], molecule_name=feature_dict["name"], sequence=ccs_seq,
      quality_string=utils.quality_scores_to_string(ccs_quality_scores), ec=feature_dict["ec"],
      np_num_passes=feature_dict["np_num_passes"], rq=feature_dict["rq"], rg=feature_dict["rg"])


def split_skipped_windows(feature_dicts_for_zmws: Iterable[Iterable[Dict[str, Any]]], options: InferenceOptions
                          ) -> Tuple[List[Dict[str, Any]], List[stitch_utils.DCModelOutput]]:
  """The skip decision of `inference_on_n_zmws` (quick_inference.py:657-676): overflowing windows, and windows whose
  CCS already averages above `skip_windows_above`, bypass the model and adopt the CCS call."""
  for_model, skipped = [], []
  for one_zmw in feature_dicts_for_zmws:
    for window in one_zmw:
      skip_example = False
      if window["overflow"]:
        skipped.append(process_skipped_window(window, options))
        skip_example = True
      if options.skip_windows_above and not skip_example:
        if utils.avg_phred(window["ccs_base_quality_scores"]) > options.skip_windows_above:
          skipped.append(process_skipped_window(window, options))
          skip_example = True
      if not skip_example:
        for_model.append(window)
  return for_model, skipped


def run_model_and_stitch(feature_dicts: List[Dict[str, Any]], model: engine_lib.B200Model,
                         model_params: params_lib.Params, options: InferenceOptions,
                         outcome_counter: stitch_utils.OutcomeCounter,
                         skipped_outputs: Optional[List[stitch_utils.DCModelOutput]] = None
                         ) -> List[Optional[str]]:
  """Windows -> FASTQ records without per-window Python objects: `run_model_on_examples`, the merge with the windows
  that bypassed the model, the sort, and per read `stitch_utils.stitch_to_fastq` (quick_inference.py:341-415, :686 and
  :721-760), with the byte work on the device.

  `feature_dicts`: the windows to score (the `for_model` list of `split_skipped_windows`).  `skipped_outputs`: the
  DCModelOutputs `split_skipped_windows` produced for overflow / high-quality windows (`process_skipped_window`); they
  are interleaved with the model's outputs exactly as the reference does -- concatenate, sort by (molecule_name,
  window_pos), group by name (quick_inference.py:686,721-736).  Returns one FASTQ record (or None when a filter drops
  the read) per read, in sorted-name order; `outcome_counter` is updated like the reference's.
  """
  from deepconsensus_b200 import stitch_gpu
  L = int(model_params.max_length)
  names, positions, bases, quals = [], [], [], []

  def collect(data, out):
    bases.append(out["bases"])
    quals.append(out["quals"])
    names.extend(_as_str(x) for x in data["name"])
    positions.extend(int(x) for x in data["window_pos"])

  _pipelined(model, batch_examples(feature_dicts, model_params, options), collect)
  widths = [L] * len(names)
  for o in skipped_outputs or []:                 # an overflow window (CCS smart windows) keeps its own width
    seq, qual = o.sequence.encode("latin-1"), o.quality_string.encode("latin-1")
    if len(seq) != len(qual):
      raise ValueError("skipped window %s@%s: sequence and quality differ in length" % (o.molecule_name, o.window_pos))
    bases.append(np.frombuffer(seq, np.uint8))
    quals.append(np.frombuffer(qual, np.uint8))
    widths.append(len(seq))
    names.append(_as_str(o.molecule_name))
    positions.append(int(o.window_pos))
  if not names:
    return []
  order = sorted(range(len(names)), key=lambda i: (names[i], positions[i]))     # quick_inference.py:721-728
  widths = np.asarray(widths, np.int64)
  window_off = np.concatenate([[0], np.cumsum(widths[order])])
  at = _ranges(np.concatenate([[0], np.cumsum(widths)])[order], widths[order])
  all_b = np.concatenate([b.reshape(-1) for b in bases])[at]
  all_q = np.concatenate([q.reshape(-1) for q in quals])[at]
  return stitch_gpu.stitch_batch_to_fastq(model, all_b, all_q, [names[i] for i in order], [positions[i] for i in order], L,
                                          options.min_quality, options.min_length, outcome_counter, window_off=window_off)


def inference_on_zmw_windows(feature_dicts_for_zmws: Iterable[Iterable[Dict[str, Any]]], model: engine_lib.B200Model,
                             model_params: params_lib.Params, options: InferenceOptions,
                             outcome_counter: stitch_utils.OutcomeCounter) -> List[Optional[str]]:
  """The model-facing part of `inference_on_n_zmws` + the stitching of `run()` for a batch of ZMWs
  (quick_inference.py:657-686,721-760) with every per-window / per-read byte and arithmetic step on the device:

    skip decision   avg_phred(ccs_base_quality_scores) > skip_windows_above     dcb_skip_mask
    model           run_model_on_examples on the windows that are not skipped    dcb_submit / dcb_wait
    skipped windows process_skipped_window: adopt CCS bases / calibrated quals    dcb_fill_skipped_ragged
    stitch          sort by (name, window_pos), stitch_to_fastq per read          dcb_stitch_fastq_ragged

  Returns one FASTQ record (or None) per read in sorted-name order -- identical to the reference flow built from
  `split_skipped_windows`, `run_model_on_examples`, `sorted(...)` and `stitch_utils.stitch_to_fastq`.
  """
  from deepconsensus_b200 import stitch_gpu
  L = int(model_params.max_length)
  windows = [w for one_zmw in feature_dicts_for_zmws for w in one_zmw]
  n = len(windows)
  if n == 0:
    return []
  names = [_as_str(w["name"]) for w in windows]
  positions = [int(w["window_pos"]) for w in windows]
  skip = np.array([bool(w.get("overflow", False)) for w in windows])
  widths = np.array([len(w["ccs_base_quality_scores"]) if o else L for w, o in zip(windows, skip)], np.int64)
  fit = np.nonzero(~skip)[0]                                  # overflow windows are skipped before the quality decision
  if options.skip_windows_above and len(fit):
    bq = np.stack([np.asarray(windows[i]["ccs_base_quality_scores"]) for i in fit]).astype(np.int16)
    mask, _ = model.skip_mask(bq, options.skip_windows_above)
    for i in np.nonzero(mask == 2)[0]:                       # within 1e-7 of the threshold: the reference's expression
      mask[i] = utils.avg_phred(windows[fit[i]]["ccs_base_quality_scores"]) > options.skip_windows_above
    skip[fit] |= mask.astype(bool)
  order = sorted(range(n), key=lambda i: (names[i], positions[i]))          # quick_inference.py:721-728
  dest = np.empty(n, np.int64)
  dest[order] = np.arange(n)
  window_off, all_b, all_q = _window_layout(widths, dest)
  scored = np.nonzero(~skip)[0]
  cursor = [0]

  def collect(data, out):
    k = out["bases"].shape[0]
    _place(all_b, all_q, window_off, dest[scored[cursor[0]:cursor[0] + k]], out, L)
    cursor[0] += k

  _pipelined(model, batch_examples([windows[i] for i in scored], model_params, options), collect)
  skipped = np.nonzero(skip)[0]
  if len(skipped):
    ccs_row = params_lib.get_indices(options.max_passes, options.use_ccs_bq)[4][0]
    ccs_ids = np.concatenate([np.asarray(windows[i]["subreads"])[ccs_row, :, 0] for i in skipped]).astype(np.uint8)
    bq = np.concatenate([np.asarray(windows[i]["ccs_base_quality_scores"]) for i in skipped]).astype(np.int16)
    model.fill_skipped_ragged(ccs_ids, bq, np.concatenate([[0], np.cumsum(widths[skipped])]), window_off[dest[skipped]],
                              all_b, all_q, calibration=options.ccs_calibration_values)
  return stitch_gpu.stitch_batch_to_fastq(model, all_b, all_q, [names[i] for i in order], [positions[i] for i in order],
                                          L, options.min_quality, options.min_length, outcome_counter, window_off=window_off)


def inference_on_packed_zmws(zmws: List[Dict[str, Any]], model: engine_lib.B200Model, model_params: params_lib.Params,
                             options: InferenceOptions, outcome_counter: stitch_utils.OutcomeCounter
                             ) -> Tuple[bytes, np.ndarray, np.ndarray, List[str]]:
  """`inference_on_zmw_windows` without any per-window Python object: `zmws` are the per-ZMW array bundles of
  `preprocess.BamFeatureStream.next_zmw(want_rows=False, want_packed=True)` (packed rows, window_pos, ccs_bq, overflow,
  name).  Skip decision, model (dcb_forward_packed), skipped-window fill, sort and stitch as there.

  Returns (fastq bytes, rec_off, passed, names): read z (sorted-name order) has the record
  fastq[rec_off[z]:rec_off[z + 1]] when passed[z].
  """
  from deepconsensus_b200 import stitch_gpu
  L, P = int(model_params.max_length), int(model_params.max_passes)
  zmws = [z for z in zmws if len(z["window_pos"])]
  if not zmws:
    return b"", np.zeros(1, np.int64), np.zeros(0, bool), []
  packed = np.concatenate([z["packed"] for z in zmws])
  pos = np.concatenate([z["window_pos"] for z in zmws]).astype(np.int64)
  bq = np.concatenate([z["ccs_bq"] for z in zmws])
  over = np.concatenate([z["overflow"] for z in zmws]).astype(bool)
  widths = np.where(over, np.concatenate([z["widths"] for z in zmws]), L).astype(np.int64)
  skip = over.copy()
  counts = np.array([len(z["window_pos"]) for z in zmws])
  names_z = [z["name"] for z in zmws]
  n = len(pos)
  fit = np.nonzero(~over)[0]                                  # overflow windows are skipped before the quality decision
  if options.skip_windows_above and len(fit):
    mask, _ = model.skip_mask(bq[fit], options.skip_windows_above)
    for i in np.nonzero(mask == 2)[0]:
      mask[i] = utils.avg_phred(bq[fit[i]].astype(np.int64)) > options.skip_windows_above
    skip[fit] |= mask.astype(bool)
  # sort by (name, window_pos): ZMW order by name, windows inside a ZMW by position (quick_inference.py:721-728)
  zorder = sorted(range(len(zmws)), key=lambda k: names_z[k])
  starts = np.concatenate([[0], np.cumsum(counts)])
  order = np.concatenate([starts[k] + np.argsort(pos[starts[k]:starts[k + 1]], kind="stable") for k in zorder])
  dest = np.empty(n, np.int64)
  dest[order] = np.arange(n)
  window_off, all_b, all_q = _window_layout(widths, dest)
  scored = np.nonzero(~skip)[0]
  for b0 in range(0, len(scored), options.batch_size):          # batch_examples (quick_inference.py:304-338)
    idx = scored[b0:b0 + options.batch_size]
    _place(all_b, all_q, window_off, dest[idx], model.forward_packed(packed[idx]), L)
  skipped = np.nonzero(skip)[0]
  if len(skipped):
    # CCS ids / qualities of the skipped windows back to back: the CCS plane of the packed rows and ccs_bq for windows
    # that fit, the wide arrays of next_zmw for overflow windows (which come in window order)
    start = np.arange(n, dtype=np.int64) * L
    start[over] = n * L + np.concatenate([[0], np.cumsum(widths[over])])[:-1]
    at = _ranges(start[skipped], widths[skipped])
    ccs_ids = np.concatenate([packed[:, 3 * P * L:3 * P * L + L].reshape(-1)] + [z["wide_ccs_ids"] for z in zmws])[at]
    ccs_bq = np.concatenate([bq.reshape(-1)] + [z["wide_ccs_bq"] for z in zmws])[at]
    model.fill_skipped_ragged(ccs_ids, ccs_bq, np.concatenate([[0], np.cumsum(widths[skipped])]),
                              window_off[dest[skipped]], all_b, all_q, calibration=options.ccs_calibration_values)
  names_sorted = [names_z[k] for k in zorder for _ in range(counts[k])]
  fastq, rec_off, passed = stitch_gpu.stitch_batch_to_fastq_bytes(model, all_b, all_q, names_sorted, pos[order].tolist(), L,
                                                                  options.min_quality, options.min_length, outcome_counter,
                                                                  window_off=window_off)
  return fastq, rec_off, passed, [names_z[k] for k in zorder]


# Windows of their own width (CCS smart windows: an overflow window keeps all W columns): the post-model stage holds
# every window's bytes back to back in sorted order and addresses them through int64 offsets.
def _window_layout(widths: np.ndarray, dest: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
  """(window_off [n + 1], bases, quals) for windows whose sorted position is dest[i]."""
  sorted_widths = np.empty(len(widths), np.int64)
  sorted_widths[dest] = widths
  window_off = np.concatenate([[0], np.cumsum(sorted_widths)])
  return window_off, np.empty(int(window_off[-1]), np.uint8), np.empty(int(window_off[-1]), np.uint8)


def _place(all_b: np.ndarray, all_q: np.ndarray, window_off: np.ndarray, rows: np.ndarray, out: Dict[str, Any], L: int):
  """The model's [k, L] outputs into sorted windows `rows`."""
  if window_off[-1] == L * (len(window_off) - 1):             # every window L wide: whole rows
    all_b.reshape(-1, L)[rows], all_q.reshape(-1, L)[rows] = out["bases"], out["quals"]
  else:
    at = window_off[rows][:, None] + np.arange(L)
    all_b[at], all_q[at] = out["bases"], out["quals"]


def _ranges(start: np.ndarray, widths: np.ndarray) -> np.ndarray:
  """Indices start[j] .. start[j] + widths[j] - 1 for every j, back to back."""
  off = np.concatenate([[0], np.cumsum(widths)])
  return np.repeat(np.asarray(start, np.int64) - off[:-1], widths) + np.arange(off[-1])


def _as_str(x) -> str:
  return x.decode() if isinstance(x, (bytes, np.bytes_)) else str(x)


def load_weights_npz(path: str) -> weights_lib.Weights:
  """Variables exported as an .npz keyed by the checkpoint variable names (SURVEY.md Appendix B)."""
  with np.load(path) as z:
    return {k: z[k] for k in z.files}


def load_weights(checkpoint_path: str) -> weights_lib.Weights:
  """What `--checkpoint` may point at (quick_inference.py:515-529): a TF2 checkpoint prefix (".../checkpoint-50"), its
  `.index` file, a directory holding a `checkpoint` state file -- read without TensorFlow by `tf_checkpoint` -- or an
  .npz export of the same variables."""
  if checkpoint_path.endswith(".npz"):
    return load_weights_npz(checkpoint_path)
  from deepconsensus_b200 import tf_checkpoint
  return tf_checkpoint.load_variables(tf_checkpoint.resolve_prefix(checkpoint_path))


def read_params_from_json(checkpoint_path: str) -> params_lib.Params:
  """params.json next to the checkpoint (model_utils.read_params_from_json, model_utils.py:434-465)."""
  return params_lib.read_params_from_json(checkpoint_path)


def initialize_model(checkpoint_path: str, params: params_lib.Params, options: InferenceOptions,
                     weights: Optional[weights_lib.Weights] = None, device: int = 0, precision: str = "bf16"
                     ) -> Tuple[engine_lib.B200Model, params_lib.Params]:
  """Builds the engine for `params` and loads variables (quick_inference.py:485-532).

  `checkpoint_path`: a TF2 checkpoint (prefix / directory / .index) or an .npz export; `weights` overrides it.
  Like the reference's `assert_existing_objects_matched()`, a variable the model needs but the checkpoint lacks (or
  holds with another shape) raises; extra keys (optimizer slots) are ignored as with `expect_partial()`.
  """
  params_lib.modify_params(params, max_length=options.max_length, is_training=False)
  if weights is None:
    weights = load_weights(checkpoint_path)
  model = engine_lib.B200Model(params, weights, max_batch=options.batch_size, device=device,
                               max_base_quality=options.max_base_quality,
                               calibration=options.dc_calibration_values, precision=precision)
  return model, params

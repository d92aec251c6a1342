"""`deepconsensus run` on the dcb200 engine (mirror of `quick_inference.run`, quick_inference.py:800-960): subreads-to-CCS
BAM + CCS BAM in, polished reads (FASTQ or unaligned BAM) out.

  python -m deepconsensus_b200.run --subreads_to_ccs S.bam --ccs_bam C.bam --checkpoint model_dir/checkpoint-50 \\
         --output out.fastq [--batch_zmws 100 --batch_size 1024 --min_quality 20 --skip_windows_above 45
         --use_ccs_smart_windows ...]

Stages (all but the driver loop in native code): feature construction from BAM (csrc/bam_prep.cpp), skip decision,
model, skipped-window fill, sort, stitch + filters + FASTQ bytes (CUDA, `inference.inference_on_zmw_windows`), output
writer (FASTQ text or BGZF/BAM, csrc/bam_prep.cpp).  `--checkpoint` is a TF2 checkpoint (read without TensorFlow), a
directory, or an .npz; params.json is read from next to it.  `--random_weights SEED` replaces the variables by seeded
ones (the reference's bundled test checkpoints ship without their data shard).
"""
from __future__ import annotations

import argparse
import itertools
import json
import os
import time
from typing import Any, Dict, List, Optional

from deepconsensus_b200 import calibration as calibration_lib
from deepconsensus_b200 import inference
from deepconsensus_b200 import params as params_lib
from deepconsensus_b200 import preprocess
from deepconsensus_b200 import stitch_utils
from deepconsensus_b200 import weights as weights_lib


def run(subreads_to_ccs: str, ccs_bam: str, checkpoint: str, output: str, batch_zmws: int = 100, batch_size: int = 1024,
        min_quality: int = 20, min_length: int = 0, skip_windows_above: int = 45, ins_trim: int = 5,
        max_base_quality: int = 93, dc_calibration: Optional[str] = None, ccs_calibration: str = "skip",
        limit: int = 0, random_weights: Optional[int] = None, precision: str = "bf16", device: int = 0, cpus: int = 0,
        use_ccs_smart_windows: bool = False) -> stitch_utils.OutcomeCounter:
  """One inference run; returns the OutcomeCounter (quick_inference.run's return value).

  use_ccs_smart_windows: window widths come from the `wl` tag of every CCS record (quick_inference.py:113-120); windows
  wider than max_length bypass the model with the CCS call."""
  params = params_lib.read_params_from_json(checkpoint)
  if dc_calibration is None:
    dc_calibration = params.get("dc_calibration", "skip")                      # quick_inference.py:817-831
  options = inference.InferenceOptions(
      max_length=int(params.max_length), example_height=params_lib.get_total_rows(params.max_passes, params.use_ccs_bq),
      max_passes=int(params.max_passes), min_quality=min_quality, min_length=min_length, batch_size=batch_size,
      use_ccs_bq=bool(params.use_ccs_bq), cpus=0, skip_windows_above=skip_windows_above, use_saved_model=False,
      max_base_quality=max_base_quality, dc_calibration_values=calibration_lib.parse_calibration_string(dc_calibration),
      ccs_calibration_values=calibration_lib.parse_calibration_string(ccs_calibration))
  weights = None
  if random_weights is not None:
    params_lib.modify_params(params, max_length=options.max_length)
    weights = weights_lib.init_weights(params, seed=random_weights)
  model, params = inference.initialize_model(checkpoint, params, options, weights=weights, device=device, precision=precision)
  counter = stitch_utils.OutcomeCounter()
  stream = preprocess.BamFeatureStream(subreads_to_ccs, ccs_bam, options.max_passes, options.max_length,
                                       options.use_ccs_bq, ins_trim, threads=cpus,
                                       use_ccs_smart_windows=use_ccs_smart_windows)
  as_bam = output.endswith(".bam")
  writer: Any = preprocess.BamWriter(output, stream.ccs_header) if as_bam else open(output, "wb")
  stats = dict(zmws=0, windows=0, seconds_features=0.0, seconds_model_and_stitch=0.0)
  try:
    done = False
    while not done:
      t0 = time.time()
      batch = []                      # per-ZMW array bundles: packed rows + metadata, no per-window objects
      while len(batch) < batch_zmws:
        z = stream.next_zmw(want_rows=False, want_packed=True)
        if z is None or (limit and stats["zmws"] + len(batch) >= limit):
          done = True
          break
        batch.append(z)
      stats["seconds_features"] += time.time() - t0
      if not batch:
        break
      t0 = time.time()
      fastq, rec_off, passed, names = inference.inference_on_packed_zmws(batch, model, params, options, counter)
      stats["seconds_model_and_stitch"] += time.time() - t0
      stats["zmws"] += len(batch)
      stats["windows"] += sum(len(z["window_pos"]) for z in batch)
      tags = {z["name"]: z for z in batch}
      if as_bam:
        for k, name in enumerate(names):
          if passed[k]:
            t = tags[name]
            writer.write_fastq_record(fastq[int(rec_off[k]):int(rec_off[k + 1])].decode("latin-1"), t["ec"],
                                      t["np_num_passes"], t["rq"], t["rg"])
      elif passed.all():
        writer.write(fastq)           # every read passed: the device's byte buffer IS the FASTQ text of the batch
      else:
        for k in range(len(names)):
          if passed[k]:
            writer.write(fastq[int(rec_off[k]):int(rec_off[k + 1])])
  finally:
    writer.close()
    stream.close()
    model.close()
  with open(output + ".inference.json", "w") as f:                               # save_counters (quick_inference.py:790-797)
    json.dump(dict(counter.__dict__, **stats), f, indent=True)
  return counter


def main(argv: Optional[List[str]] = None) -> None:
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--subreads_to_ccs", required=True)
  ap.add_argument("--ccs_bam", required=True)
  ap.add_argument("--checkpoint", required=True)
  ap.add_argument("--output", required=True)
  ap.add_argument("--batch_zmws", type=int, default=100)
  ap.add_argument("--batch_size", type=int, default=1024)
  ap.add_argument("--min_quality", type=int, default=20)
  ap.add_argument("--min_length", type=int, default=0)
  ap.add_argument("--skip_windows_above", type=int, default=45)
  ap.add_argument("--ins_trim", type=int, default=5)
  ap.add_argument("--max_base_quality", type=int, default=93)
  ap.add_argument("--dc_calibration", default=None)
  ap.add_argument("--ccs_calibration", default="skip")
  ap.add_argument("--limit", type=int, default=0)
  ap.add_argument("--random_weights", type=int, default=None)
  ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
  ap.add_argument("--cpus", type=int, default=0, help="native feature-construction threads (0: on the calling thread)")
  ap.add_argument("--use_ccs_smart_windows", action="store_true",
                  help="window widths from the CCS records' wl tag instead of max_length columns")
  a = ap.parse_args(argv)
  c = run(**vars(a))
  print(json.dumps(c.__dict__))


if __name__ == "__main__":
  main()

"""Digest of the reference's own preprocessing output for its BAM fixtures.

deepconsensus/testdata/human_1m/tf_examples/inference/inference.tfrecord.gz holds the 1 593 examples the reference's
`deepconsensus preprocess` (v1.2.0, ins_trim=5: see tf_examples/summary/summary.inference.json) wrote from
testdata/human_1m/{subreads_to_ccs,ccs}.bam.  This script reduces every example to (name, window_pos, num_passes,
sha1 of the float32 rows, sha1 of the CCS base qualities) -> tests/golden/human_1m/inference_digest.json; ccs.bam and
7 of the 10 ZMWs of subreads_to_ccs.bam (scripts/make_bam_subset.py) sit next to it.  tests/test_bam_prep.py rebuilds
the windows of those ZMWs with csrc/bam_prep.cpp and requires their digest entries, window for window.  Run here (needs /root/reference); output is committed.
"""
import hashlib
import importlib.util
import json
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference/deepconsensus/testdata/human_1m/"
spec = importlib.util.spec_from_file_location("mg", os.path.join(REPO, "scripts", "make_golden.py"))
mg = importlib.util.module_from_spec(spec)
spec.loader.exec_module(mg)


def main():
  out = []
  for ex in mg.read_tfrecords(REF + "tf_examples/inference/inference.tfrecord.gz"):
    rows = np.frombuffer(ex["subreads/encoded"][0], "<f4").reshape(ex["subreads/shape"])[..., 0]
    bq = np.asarray(ex["ccs_base_quality_scores"], np.int64)
    out.append(dict(name=ex["name"][0].decode(), window_pos=int(ex["window_pos"][0]),
                    num_passes=int(ex["subreads/num_passes"][0]), shape=list(rows.shape),
                    rows_sha1=hashlib.sha1(np.ascontiguousarray(rows, "<f4").tobytes()).hexdigest(),
                    bq_sha1=hashlib.sha1(bq.astype("<i8").tobytes()).hexdigest()))
  with open(REF + "tf_examples/summary/summary.inference.json") as f:
    summary = json.load(f)
  path = os.path.join(REPO, "tests", "golden", "human_1m", "inference_digest.json")
  with open(path, "w") as f:
    json.dump(dict(source="deepconsensus/testdata/human_1m/tf_examples/inference/inference.tfrecord.gz",
                   summary={k: summary[k] for k in ("ins_trim", "max_passes", "max_length", "n_examples", "n_zmw_pass", "version")},
                   windows=out), f)
  print(len(out), "windows ->", path)


if __name__ == "__main__":
  main()

"""Batch stitching on the device (`dcb_stitch_fastq`): windows of many reads -> FASTQ records.

`stitch_utils.stitch_to_fastq` (mirror of postprocess/stitch_utils.py:131-189) handles one read at a time from
per-window strings.  Here a whole batch of reads goes through at once, straight from the engine's per-window byte
arrays, and everything per-read happens in CUDA kernels (csrc/kernels.cu stitch_kernel, csrc/post_kernels.cu):
get_full_sequence + remove_gaps (stitch_utils.py:51-98), the missing-window check, the only-gaps / quality / length
filters (same order, same counters) and the FASTQ byte assembly.  The host only turns outcome codes into
`OutcomeCounter` increments and slices records out of one byte buffer.

The quality filter is `round(avg_phred, 5) >= min_quality` in float64 (stitch_utils.py:101-109).  The device forms the
mean error probability from an exact integer histogram, NumPy sums per-base terms pairwise; the two can differ in the
last bits, so reads within 1e-7 of the threshold come back flagged DCB_READ_BORDERLINE and are re-decided here with the
reference's own NumPy expression.  The result is identical, read for read, to stitch_utils.stitch_to_fastq.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np

from deepconsensus_b200 import engine as engine_lib
from deepconsensus_b200 import stitch_utils, utils


def group_reads(molecule_names: Sequence[str]) -> np.ndarray:
  """zmw_start for windows already grouped by read: index of the first window of every run of equal names, + end."""
  n = len(molecule_names)
  starts = [0] if n else []
  for i in range(1, n):
    if molecule_names[i] != molecule_names[i - 1]:
      starts.append(i)
  return np.asarray(starts + [n], dtype=np.int32)


def stitch_batch_to_fastq_bytes(model, bases, quals, molecule_names: Sequence[str], window_pos: Sequence[int],
                                max_length: int, min_quality: int, min_length: int,
                                outcome_counter: stitch_utils.OutcomeCounter,
                                n_windows: Optional[int] = None, on_device: bool = False,
                                window_off: Optional[np.ndarray] = None) -> Tuple[bytes, np.ndarray, np.ndarray]:
  """(fastq bytes, rec_off, passed): read z's record is fastq[rec_off[z]:rec_off[z + 1]] when passed[z].

  window_off (int64 [n_windows + 1]): the ragged form for windows of their own width (CCS smart windows): `bases` /
  `quals` are flat host arrays and window w is bytes [window_off[w], window_off[w + 1]) (dcb_stitch_fastq_ragged)."""
  zs = group_reads(molecule_names)
  nz = len(zs) - 1
  names = [molecule_names[int(zs[z])] for z in range(nz)]
  fastq, rec_off, outcome, _ = model.stitch_fastq(bases, quals, zs, window_pos, names, min_quality, min_length,
                                                  n_windows=n_windows, on_device=on_device, length=max_length,
                                                  window_off=window_off)
  passed = np.zeros(nz, bool)
  for z in range(nz):
    code = int(outcome[z])
    if code & engine_lib.DCB_READ_BORDERLINE:
      # quality within 1e-7 of the threshold: decide with the reference's expression (its record was written)
      code &= 0x7F
      rec = fastq[int(rec_off[z]):int(rec_off[z + 1])] if code == engine_lib.DCB_READ_OK else None
      if rec is not None:
        qual = rec.split(b"\n")[3]
      elif window_off is not None:            # too short, ragged host arrays: remove_gaps in NumPy
        a, b = int(window_off[zs[z]]), int(window_off[zs[z + 1]])
        seg_b, seg_q = np.asarray(bases).reshape(-1)[a:b], np.asarray(quals).reshape(-1)[a:b]
        qual = seg_q[seg_b != ord(" ")].tobytes()
      else:                                   # too short: the record was not written; recompute from the windows
        qual = _read_quality_bytes(model, bases, quals, zs, z, max_length, n_windows, on_device)
      ok = round(utils.avg_phred(np.frombuffer(qual, np.uint8).astype(np.int64) - 33), 5) >= min_quality
      if not ok:
        code = engine_lib.DCB_READ_LOW_QUALITY
    if code == engine_lib.DCB_READ_OK:
      outcome_counter.success += 1
      passed[z] = True
    elif code == engine_lib.DCB_READ_EMPTY:
      outcome_counter.empty_sequence += 1
    elif code == engine_lib.DCB_READ_ONLY_GAPS:
      outcome_counter.only_gaps += 1
    elif code == engine_lib.DCB_READ_LOW_QUALITY:
      outcome_counter.failed_quality_filter += 1
    else:
      outcome_counter.failed_length_filter += 1
  return fastq, rec_off, passed


def _read_quality_bytes(model, bases, quals, zs, z, max_length, n_windows, on_device) -> bytes:
  seq, qual, lens = model.stitch(bases, quals, zs, n_windows=n_windows, on_device=on_device, length=max_length)
  o = int(zs[z]) * max_length
  return qual[o:o + int(lens[z])].tobytes()


def stitch_batch_to_fastq(model, bases, quals, molecule_names: Sequence[str], window_pos: Sequence[int],
                          max_length: int, min_quality: int, min_length: int,
                          outcome_counter: stitch_utils.OutcomeCounter,
                          n_windows: Optional[int] = None, on_device: bool = False,
                          window_off: Optional[np.ndarray] = None) -> List[Optional[str]]:
  """One FASTQ record (or None) per read, for windows grouped by read and sorted by window position.

  `bases` / `quals`: uint8 [n_windows, max_length] arrays as `B200Model.forward` returns them, or device addresses
  of the same (`on_device=True`, e.g. the DCB_OUT_ON_DEVICE outputs of `forward_raw`); with `window_off`, flat host
  arrays of windows of their own width (see stitch_batch_to_fastq_bytes).
  """
  fastq, rec_off, passed = stitch_batch_to_fastq_bytes(model, bases, quals, molecule_names, window_pos, max_length,
                                                       min_quality, min_length, outcome_counter, n_windows, on_device,
                                                       window_off)
  return [fastq[int(rec_off[z]):int(rec_off[z + 1])].decode("latin-1") if passed[z] else None
          for z in range(len(passed))]

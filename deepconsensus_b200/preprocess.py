"""Feature construction from BAM without pysam / htslib (mirror of the inference half of
`deepconsensus/preprocess/pre_lib.py` and of `quick_inference.stream_bam` / `preprocess`).

The work is done by host C++ behind the C ABI (csrc/bam_prep.cpp, `dcb_prep_*`): BGZF / BAM decoding, SubreadGrouper,
trim_insertions, expand_clip_indent, construct_ccs_read, space_out_subreads, DcExample.iter_examples and
extract_features.  This module hands the results out in the reference's own shapes:

  stream_zmw_windows(...)   per ZMW a list of feature dicts with the keys of DcExample.to_features_dict
                            (pre_lib.py:746-762) -- what quick_inference.preprocess returns (quick_inference.py:535-564)
  stream_zmw_packed(...)    the same windows as packed rows (include/dcb200.h "packed input rows") + per-window metadata,
                            with no float32 rows and no per-window Python objects in between
  BamWriter                 the unaligned-BAM output of `deepconsensus run --output *.bam` (quick_inference.py:742-760)

Needs no GPU.
"""
from __future__ import annotations

import ctypes
from typing import Any, Dict, Iterator, List, Optional, Tuple

import numpy as np

from deepconsensus_b200 import engine as engine_lib
from deepconsensus_b200 import params as params_lib


class DcbZmwInfo(ctypes.Structure):
  _fields_ = [("n_windows", ctypes.c_int32), ("n_subreads", ctypes.c_int32), ("name", ctypes.c_char_p),
              ("has_ec", ctypes.c_int32), ("has_np", ctypes.c_int32), ("has_rq", ctypes.c_int32),
              ("ec", ctypes.c_float), ("rq", ctypes.c_float), ("np_num_passes", ctypes.c_int32),
              ("rg", ctypes.c_char_p), ("ccs_length", ctypes.c_int32), ("spaced_width", ctypes.c_int32)]


class PrepError(RuntimeError):
  pass


def _lib():
  lib = engine_lib.load_library()
  if not getattr(lib, "_prep_bound", False):
    vp, i32 = ctypes.c_void_p, ctypes.c_int32
    lib.dcb_prep_open.argtypes = [ctypes.c_char_p, ctypes.c_char_p, i32, i32, i32, i32, ctypes.POINTER(vp)]
    lib.dcb_prep_set_threads.argtypes = [vp, i32]
    lib.dcb_prep_set_smart_windows.argtypes = [vp, i32]
    lib.dcb_prep_get_window_widths.argtypes = [vp, vp]
    lib.dcb_prep_get_overflow_windows.argtypes = [vp, vp, vp, vp]
    lib.dcb_prep_next_zmw.argtypes = [vp, ctypes.POINTER(DcbZmwInfo)]
    lib.dcb_prep_get_windows.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.dcb_prep_ccs_header.argtypes = [vp]
    lib.dcb_prep_ccs_header.restype = ctypes.c_char_p
    lib.dcb_prep_close.argtypes = [vp]
    lib.dcb_prep_close.restype = None
    lib.dcb_prep_last_error.restype = ctypes.c_char_p
    lib.dcb_bamw_open.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(vp)]
    lib.dcb_bamw_write.argtypes = [vp, ctypes.c_char_p, vp, vp, i32, i32, ctypes.c_float, i32, ctypes.c_float, ctypes.c_char_p]
    lib.dcb_bamw_close.argtypes = [vp]
    lib._prep_bound = True
  return lib


class BamFeatureStream:
  """Iterates the ZMWs of a subreads-to-CCS BAM + CCS BAM pair (create_proc_feeder + subreads_to_dc_example +
  iter_examples, pre_lib.py:1279-1384,625-697)."""

  def __init__(self, subreads_to_ccs: str, ccs_bam: str, max_passes: int, max_length: int, use_ccs_bq: bool = False,
               ins_trim: int = 5, threads: int = 0, use_ccs_smart_windows: bool = False):
    """threads > 0: ZMWs are processed by that many native worker threads (plus one BAM-decoding thread) while the
    caller consumes them; the order of the ZMWs is the file's either way (`--cpus` of `deepconsensus run`).
    use_ccs_smart_windows: window widths come from the CCS records' `wl` tags (`--use_ccs_smart_windows`); windows
    wider than max_length are overflow windows, handed out in full by `next_zmw`."""
    self._lib = _lib()
    self._h = ctypes.c_void_p()
    self.max_passes, self.max_length, self.use_ccs_bq = int(max_passes), int(max_length), bool(use_ccs_bq)
    self.total_rows = params_lib.get_total_rows(self.max_passes, self.use_ccs_bq)
    rc = self._lib.dcb_prep_open(subreads_to_ccs.encode(), ccs_bam.encode(), self.max_passes, self.max_length,
                                 int(self.use_ccs_bq), int(ins_trim), ctypes.byref(self._h))
    if rc:
      raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))
    if threads > 0 and self._lib.dcb_prep_set_threads(self._h, int(threads)):
      raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))
    if use_ccs_smart_windows and self._lib.dcb_prep_set_smart_windows(self._h, 1):
      raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))
    self._stride = ((3 * self.max_passes + 1 + int(self.use_ccs_bq)) * self.max_length + 15) // 16 * 16 + 16   # PackedLayout

  @property
  def ccs_header(self) -> str:
    return self._lib.dcb_prep_ccs_header(self._h).decode("latin-1")

  @property
  def packed_window_bytes(self) -> int:
    return self._stride

  def close(self) -> None:
    if self._h and self._h.value:
      self._lib.dcb_prep_close(self._h)
      self._h = ctypes.c_void_p()

  def __del__(self):
    try:
      self.close()
    except Exception:
      pass

  def next_zmw(self, want_rows: bool = True, want_packed: bool = False) -> Optional[Dict[str, Any]]:
    """The next ZMW's windows as arrays: dict(name, n_subreads, ec, np_num_passes, rq, rg, window_pos [n], overflow
    [n], num_passes [n], widths [n] (spaced width W of every window), ccs_bq int16 [n, L], rows float32 [n, R, L] and / or
    packed uint8 [n, stride]); None at EOF.  Overflow windows (W > L, smart windows only) hold their first L columns in
    those arrays and come in full, ragged in window order, as wide_ccs_ids uint8 [S], wide_ccs_bq int16 [S] and, with
    want_rows, wide_rows float32 [S * R] (window after window, each [R, W]; S = sum of their widths)."""
    info = DcbZmwInfo()
    rc = self._lib.dcb_prep_next_zmw(self._h, ctypes.byref(info))
    if rc < 0:
      raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))
    if rc == 0:
      return None
    n, L, R = int(info.n_windows), self.max_length, self.total_rows
    out: Dict[str, Any] = dict(name=info.name.decode("utf-8", "replace"), n_subreads=int(info.n_subreads),
                               ec=float(info.ec) if info.has_ec else None,
                               np_num_passes=int(info.np_num_passes) if info.has_np else None,
                               rq=float(info.rq) if info.has_rq else None,
                               rg=info.rg.decode("utf-8", "replace") if info.rg else None,
                               window_pos=np.zeros(n, np.int32), overflow=np.zeros(n, np.uint8),
                               num_passes=np.zeros(n, np.int32), ccs_bq=np.zeros((n, L), np.int16))
    if want_rows:
      out["rows"] = np.empty((n, R, L), np.float32)
    if want_packed:
      out["packed"] = np.empty((n, self._stride), np.uint8)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = self._lib.dcb_prep_get_windows(self._h, vp(out["rows"]) if want_rows else None,
                                        vp(out["packed"]) if want_packed else None, vp(out["window_pos"]),
                                        vp(out["overflow"]), vp(out["ccs_bq"]), vp(out["num_passes"]))
    if rc:
      raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))
    out["widths"] = np.zeros(n, np.int32)
    self._lib.dcb_prep_get_window_widths(self._h, vp(out["widths"]))
    wide = int(out["widths"][out["overflow"] != 0].sum())
    out["wide_ccs_ids"], out["wide_ccs_bq"] = np.zeros(wide, np.uint8), np.zeros(wide, np.int16)
    if want_rows:
      out["wide_rows"] = np.zeros(wide * R, np.float32)
    if wide:
      rc = self._lib.dcb_prep_get_overflow_windows(self._h, vp(out["wide_rows"]) if want_rows else None,
                                                   vp(out["wide_ccs_ids"]), vp(out["wide_ccs_bq"]))
      if rc:
        raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))
    return out

  def __iter__(self):
    while True:
      z = self.next_zmw()
      if z is None:
        return
      yield z


def stream_zmw_windows(subreads_to_ccs: str, ccs_bam: str, max_passes: int, max_length: int, use_ccs_bq: bool = False,
                       ins_trim: int = 5, limit: int = 0, use_ccs_smart_windows: bool = False
                       ) -> Iterator[List[Dict[str, Any]]]:
  """Per ZMW, the feature dicts `quick_inference.preprocess` returns (keys of DcExample.to_features_dict).  An overflow
  window (smart windows only) has subreads [R, W, 1] and W CCS base qualities, as the reference leaves it unpadded."""
  stream = BamFeatureStream(subreads_to_ccs, ccs_bam, max_passes, max_length, use_ccs_bq, ins_trim,
                            use_ccs_smart_windows=use_ccs_smart_windows)
  try:
    done = 0
    for z in stream:
      rows, bq = list(z["rows"]), list(z["ccs_bq"])
      off = 0
      for i in np.nonzero(z["overflow"])[0]:
        w = int(z["widths"][i])
        rows[i] = z["wide_rows"][off * stream.total_rows:(off + w) * stream.total_rows].reshape(stream.total_rows, w)
        bq[i] = z["wide_ccs_bq"][off:off + w]
        off += w
      yield [dict(subreads=rows[i][..., None], **{"subreads/num_passes": int(z["num_passes"][i])},
                  name=z["name"], window_pos=int(z["window_pos"][i]),
                  ccs_base_quality_scores=bq[i].astype(np.int64), overflow=bool(z["overflow"][i]),
                  ec=z["ec"], np_num_passes=z["np_num_passes"], rq=z["rq"], rg=z["rg"])
             for i in range(len(z["window_pos"]))]
      done += 1
      if limit and done >= limit:
        return
  finally:
    stream.close()


class BamWriter:
  """Unaligned BAM output (quick_inference.py:742-760,892-897): one record per polished read, header of the CCS BAM."""

  def __init__(self, path: str, header_text: str = ""):
    self._lib = _lib()
    self._h = ctypes.c_void_p()
    if self._lib.dcb_bamw_open(path.encode(), header_text.encode("latin-1"), ctypes.byref(self._h)):
      raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))

  def write_fastq_record(self, fastq_string: str, ec: Optional[float], np_num_passes: Optional[int], rq: Optional[float],
                         rg: Optional[str]) -> None:
    name, seq, _, qual = fastq_string.splitlines()
    s, q = seq.encode("latin-1"), qual.encode("latin-1")
    rc = self._lib.dcb_bamw_write(self._h, name[1:].encode(), s, q, len(s), int(ec is not None), float(ec or 0.0),
                                  int(np_num_passes or 0), float(rq or 0.0), rg.encode() if rg is not None else None)
    if rc:
      raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))

  def close(self) -> None:
    if self._h and self._h.value:
      rc = self._lib.dcb_bamw_close(self._h)
      self._h = ctypes.c_void_p()
      if rc:
        raise PrepError(self._lib.dcb_prep_last_error().decode("utf-8", "replace"))

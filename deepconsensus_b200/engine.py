"""ctypes binding of the dcb200 C-ABI (include/dcb200.h) and the model object built on it.

`B200Model` stands where the reference's `tf.keras.Model` stands in
`quick_inference.run_model_on_examples` (quick_inference.py:341-415):

  * `model.predict(rows)` -> object with `.numpy()` giving softmax output [B, L, 5]
    (the contract quick_inference.py:368-370 relies on), and
  * `model.forward(rows)` -> base / quality characters straight from the device epilogue
    (what quick_inference.py:377-414 computes on the host).

There is no CPU fallback: if the CUDA library is missing or no sm_100 GPU is present,
construction raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Any, Dict, Optional, Tuple

import numpy as np

from deepconsensus_b200 import calibration as calibration_lib
from deepconsensus_b200 import params as params_lib
from deepconsensus_b200 import weights as weights_lib

# DCB200_LIB: developer override to load an experiment build of the same library (never a different implementation)
_LIB_PATH = os.environ.get("DCB200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc",
                                                         "libdcb200.so")
_lib = None

DCB_ROWS_ON_DEVICE = 1
DCB_OUT_ON_DEVICE = 2
DCB_STRICT_FP32 = 4
DCB_FAST_BF16 = 8
DCB_PRECISION_BF16 = 0
DCB_PRECISION_FP32 = 1
# per-read outcome codes of dcb_stitch_fastq (the OutcomeCounter field the reference would bump)
DCB_READ_OK, DCB_READ_EMPTY, DCB_READ_ONLY_GAPS, DCB_READ_LOW_QUALITY, DCB_READ_TOO_SHORT = 0, 1, 2, 3, 4
DCB_READ_BORDERLINE = 0x80


class DcbError(RuntimeError):
  def __init__(self, code: int, message: str):
    super().__init__("dcb200 error %d: %s" % (code, message))
    self.code = code


class DcbConfig(ctypes.Structure):
  _fields_ = [
      ("struct_size", ctypes.c_int32), ("device", ctypes.c_int32),
      ("max_passes", ctypes.c_int32), ("max_length", ctypes.c_int32),
      ("use_ccs_bq", ctypes.c_int32),
      ("hidden_size", ctypes.c_int32), ("num_heads", ctypes.c_int32),
      ("num_hidden_layers", ctypes.c_int32), ("filter_size", ctypes.c_int32),
      ("attn_win_size", ctypes.c_int32), ("rezero", ctypes.c_int32),
      ("add_pos_encoding", ctypes.c_int32), ("condense_transformer_input", ctypes.c_int32),
      ("per_base_hidden_size", ctypes.c_int32), ("pw_hidden_size", ctypes.c_int32),
      ("ip_hidden_size", ctypes.c_int32), ("strand_hidden_size", ctypes.c_int32),
      ("ccs_bq_hidden_size", ctypes.c_int32), ("sn_hidden_size", ctypes.c_int32),
      ("pw_max", ctypes.c_int32), ("ip_max", ctypes.c_int32), ("sn_max", ctypes.c_int32),
      ("ccs_bq_max", ctypes.c_int32), ("strand_max", ctypes.c_int32),
      ("max_base_quality", ctypes.c_int32), ("calibration_enabled", ctypes.c_int32),
      ("calibration_threshold", ctypes.c_double), ("calibration_w", ctypes.c_double),
      ("calibration_b", ctypes.c_double),
      ("max_batch", ctypes.c_int32), ("chunk_tiles", ctypes.c_int32),
      ("precision", ctypes.c_int32),
      ("reserved", ctypes.c_int32 * 5),
  ]


class DcbTensor(ctypes.Structure):
  _fields_ = [("name", ctypes.c_char_p), ("data", ctypes.POINTER(ctypes.c_float)),
              ("ndim", ctypes.c_int32), ("shape", ctypes.c_int64 * 4)]


# Every symbol include/dcb200.h declares; tests check the built library exports all of them.
ABI_SYMBOLS = (
    "dcb_create", "dcb_load_weights", "dcb_forward", "dcb_submit", "dcb_wait", "dcb_stitch", "dcb_last_forward_ms",
    "dcb_packed_window_bytes", "dcb_pack_rows", "dcb_forward_packed", "dcb_submit_packed",
    "dcb_stitch_fastq", "dcb_skip_mask", "dcb_fill_skipped",
    "dcb_stitch_fastq_ragged", "dcb_fill_skipped_ragged",
    "dcb_prep_open", "dcb_prep_set_threads", "dcb_prep_set_smart_windows", "dcb_prep_next_zmw", "dcb_prep_get_windows",
    "dcb_prep_get_window_widths", "dcb_prep_get_overflow_windows", "dcb_prep_ccs_header", "dcb_prep_close",
    "dcb_prep_last_error", "dcb_bamw_open", "dcb_bamw_write", "dcb_bamw_close",
    "dcb_last_forward_launches", "dcb_set_profile", "dcb_get_profile", "dcb_get_profile_kernels", "dcb_alloc_host",
    "dcb_free_host", "dcb_alloc_device", "dcb_free_device", "dcb_memcpy_h2d", "dcb_memcpy_d2h",
    "dcb_synchronize", "dcb_last_error", "dcb_version", "dcb_destroy",
)
# include/dcb200_debug.h: developer / test hooks, not part of the drop-in boundary
DEBUG_SYMBOLS = ("dcb_set_debug", "dcb_debug_residual", "dcb_debug_trace")


def library_path() -> str:
  return _LIB_PATH


def load_library() -> ctypes.CDLL:
  """Loads libdcb200.so (built in-tree by `__graft_entry__.build()` / csrc/build.sh)."""
  global _lib
  if _lib is None:
    _lib = _load(_LIB_PATH)
  return _lib


_dev_lib = None


def load_dev_library() -> ctypes.CDLL:
  """libdcb200_dev.so: the same sources built with -DDCB_DEV_SWITCHES, where DCB_* environment variables select the
  measured alternative kernel paths (tests and scripts only; pass as B200Model(..., library=...))."""
  global _dev_lib
  if _dev_lib is None:
    _dev_lib = _load(os.path.join(os.path.dirname(_LIB_PATH), "libdcb200_dev.so"))
  return _dev_lib


def _load(path: str) -> ctypes.CDLL:
  if not os.path.exists(path):
    raise FileNotFoundError(
        "%s not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; "
        "g.build()'); the dcb200 engine has no CPU fallback" % path)
  lib = ctypes.CDLL(path)
  vp, i32, u32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_uint32
  lib.dcb_create.argtypes = [ctypes.POINTER(DcbConfig), ctypes.POINTER(vp)]
  lib.dcb_load_weights.argtypes = [vp, ctypes.POINTER(DcbTensor), i32]
  lib.dcb_forward.argtypes = [vp, vp, i32, u32, vp, vp, vp, vp]
  lib.dcb_submit.argtypes = [vp, vp, i32, u32, vp, vp, vp, vp, ctypes.POINTER(ctypes.c_int64)]
  lib.dcb_wait.argtypes = [vp, ctypes.c_int64]
  lib.dcb_packed_window_bytes.argtypes = [ctypes.POINTER(DcbConfig)]
  lib.dcb_packed_window_bytes.restype = ctypes.c_size_t
  lib.dcb_pack_rows.argtypes = [ctypes.POINTER(DcbConfig), vp, i32, vp]
  lib.dcb_forward_packed.argtypes = [vp, vp, i32, u32, vp, vp, vp, vp]
  lib.dcb_submit_packed.argtypes = [vp, vp, i32, u32, vp, vp, vp, vp, ctypes.POINTER(ctypes.c_int64)]
  lib.dcb_stitch.argtypes = [vp, vp, vp, i32, i32, ctypes.POINTER(i32), i32, u32, vp, vp, vp]
  f64 = ctypes.c_double
  lib.dcb_stitch_fastq.argtypes = [vp, vp, vp, i32, i32, vp, i32, vp, vp, vp, f64, i32, u32, vp, ctypes.c_int64, vp, vp, vp]
  lib.dcb_skip_mask.argtypes = [vp, vp, i32, i32, f64, vp, vp]
  lib.dcb_fill_skipped.argtypes = [vp, vp, vp, vp, i32, i32, i32, f64, f64, f64, u32, vp, vp]
  lib.dcb_stitch_fastq_ragged.argtypes = [vp, vp, vp, i32, vp, i32, vp, i32, vp, vp, vp, f64, i32, u32, vp, ctypes.c_int64,
                                          vp, vp, vp]
  lib.dcb_fill_skipped_ragged.argtypes = [vp, vp, vp, vp, vp, i32, i32, f64, f64, f64, u32, vp, vp]
  lib.dcb_last_forward_ms.argtypes = [vp, ctypes.POINTER(ctypes.c_float)]
  lib.dcb_last_forward_launches.argtypes = [vp, ctypes.POINTER(i32)]
  lib.dcb_set_debug.argtypes = [vp, i32]
  lib.dcb_set_profile.argtypes = [vp, i32]
  lib.dcb_get_profile.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(i32),
                                  ctypes.POINTER(ctypes.c_int64)]
  lib.dcb_get_profile_kernels.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(i32),
                                          ctypes.POINTER(i32)]
  lib.dcb_debug_residual.argtypes = [vp, i32, vp, ctypes.c_int64]
  lib.dcb_alloc_host.argtypes = [ctypes.c_size_t, ctypes.POINTER(vp)]
  lib.dcb_free_host.argtypes = [vp]
  lib.dcb_alloc_device.argtypes = [vp, ctypes.c_size_t, ctypes.POINTER(vp)]
  lib.dcb_free_device.argtypes = [vp, vp]
  lib.dcb_memcpy_h2d.argtypes = [vp, vp, vp, ctypes.c_size_t]
  lib.dcb_memcpy_d2h.argtypes = [vp, vp, vp, ctypes.c_size_t]
  lib.dcb_synchronize.argtypes = [vp]
  lib.dcb_last_error.argtypes = [vp]
  lib.dcb_last_error.restype = ctypes.c_char_p
  lib.dcb_version.restype = ctypes.c_char_p
  lib.dcb_destroy.argtypes = [vp]
  lib.dcb_destroy.restype = None
  return lib


def make_config(params: params_lib.Params, max_batch: int, device: int = 0,
                max_base_quality: int = 93,
                calibration: Optional[calibration_lib.QualityCalibrationValues] = None,
                chunk_tiles: int = 0, precision: str = "bf16") -> DcbConfig:
  """params (params.json surface) + InferenceOptions fields -> dcb_config."""
  if precision not in ("bf16", "fp32"):
    raise ValueError("precision must be 'bf16' (tensor cores) or 'fp32' (strict, the reference's arithmetic)")
  c = DcbConfig()
  c.struct_size = ctypes.sizeof(DcbConfig)
  c.device = device
  c.max_passes, c.max_length = int(params.max_passes), int(params.max_length)
  c.use_ccs_bq = int(bool(params.use_ccs_bq))
  c.hidden_size, c.num_heads = int(params.hidden_size), int(params.num_heads)
  c.num_hidden_layers, c.filter_size = int(params.num_hidden_layers), int(params.filter_size)
  c.attn_win_size = int(params.attn_win_size or 0)
  c.rezero = int(bool(params.rezero))
  c.add_pos_encoding = int(bool(params.add_pos_encoding))
  c.condense_transformer_input = int(bool(params.condense_transformer_input))
  for f in ("per_base", "pw", "ip", "strand", "ccs_bq", "sn"):
    setattr(c, f + "_hidden_size", int(params[f + "_hidden_size"]))
  c.pw_max, c.ip_max, c.sn_max = int(params.PW_MAX), int(params.IP_MAX), int(params.SN_MAX)
  c.ccs_bq_max, c.strand_max = int(params.CCS_BQ_MAX), int(params.STRAND_MAX)
  c.max_base_quality = int(max_base_quality)
  if calibration is not None and calibration.enabled:
    c.calibration_enabled = 1
    c.calibration_threshold = float(calibration.threshold)
    c.calibration_w, c.calibration_b = float(calibration.w), float(calibration.b)
  c.max_batch = int(max_batch)
  c.chunk_tiles = int(chunk_tiles)
  c.precision = DCB_PRECISION_FP32 if precision == "fp32" else DCB_PRECISION_BF16
  for need in ("use_bases", "use_pw", "use_ip", "use_strand", "use_ccs", "use_sn"):
    if not params.get(need, True):
      raise DcbError(-1, "params.%s=False is not supported by the dcb200 engine" % need)
  return c


class _Prediction:
  """Stand-in for the EagerTensor `model.predict` returns (quick_inference.py:368-370)."""

  def __init__(self, array: np.ndarray):
    self._array = array

  def numpy(self) -> np.ndarray:
    return self._array


class B200Model:
  """The encoder-only learned-values transformer on one B200, behind the C-ABI."""

  def __init__(self, params: params_lib.Params, weights: weights_lib.Weights, max_batch: int = 1024,
               device: int = 0, max_base_quality: int = 93,
               calibration: Optional[calibration_lib.QualityCalibrationValues] = None,
               chunk_tiles: int = 0, precision: str = "bf16", library: Optional[ctypes.CDLL] = None):
    """precision: "bf16" = tensor-core path (default); "fp32" = strict path, the reference's float32 arithmetic
    (identical bases wherever the float32 top-2 logit margin exceeds 1e-3; ~25x slower).  Either can be overridden
    per call with forward(..., strict=True/False)."""
    self._lib = library if library is not None else load_library()
    self._handle = ctypes.c_void_p()
    self.params = params
    self.max_batch = max_batch
    self.max_length = int(params.max_length)
    self.total_rows = params_lib.get_total_rows(params.max_passes, params.use_ccs_bq)
    cfg = make_config(params, max_batch, device, max_base_quality, calibration, chunk_tiles, precision)
    rc = self._lib.dcb_create(ctypes.byref(cfg), ctypes.byref(self._handle))
    if rc:
      msg = self._lib.dcb_last_error(None).decode()
      self._handle = ctypes.c_void_p()
      raise DcbError(rc, msg)
    self.load_weights(weights)

  # -- lifecycle ---------------------------------------------------------------------------
  def close(self) -> None:
    if getattr(self, "_handle", None) and self._handle.value:
      self._lib.dcb_destroy(self._handle)
      self._handle = ctypes.c_void_p()
      for st in getattr(self, "_stage", {}).values():
        for addr in st["addrs"]:
          free_pinned(addr)
      self._stage = {}

  def __del__(self):
    try:
      self.close()
    except Exception:  # interpreter shutdown
      pass

  def _check(self, rc: int, tolerate: Tuple[int, ...] = ()) -> int:
    if rc and rc not in tolerate:
      raise DcbError(rc, self._lib.dcb_last_error(self._handle).decode())
    return rc

  def load_weights(self, weights: weights_lib.Weights) -> None:
    weights_lib.check_weights(self.params, weights)
    keep, tensors = [], (DcbTensor * len(weights))()
    for i, (name, arr) in enumerate(weights.items()):
      shape = np.shape(arr)                      # 0-d for the ReZero alphas
      a = np.ascontiguousarray(np.asarray(arr, dtype=np.float32)).reshape(-1)
      keep.append(a)
      tensors[i].name = name.encode()
      tensors[i].data = a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
      tensors[i].ndim = len(shape)
      for d, s in enumerate(shape):
        tensors[i].shape[d] = s
    self._check(self._lib.dcb_load_weights(self._handle, tensors, len(weights)))

  # -- the hot path ------------------------------------------------------------------------
  def _rows3(self, rows: np.ndarray) -> np.ndarray:
    rows = np.asarray(rows)
    if rows.ndim == 4:
      if rows.shape[-1] != 1:
        raise ValueError("rows must be [B, R, L, 1]")
      rows = rows[..., 0]
    if rows.ndim != 3 or rows.shape[1] != self.total_rows or rows.shape[2] != self.max_length:
      raise ValueError("rows must be [B, %d, %d(, 1)], got %s" %
                       (self.total_rows, self.max_length, rows.shape))
    return np.ascontiguousarray(rows, dtype=np.float32)

  @staticmethod
  def _precision_flag(strict: Optional[bool]) -> int:
    return 0 if strict is None else (DCB_STRICT_FP32 if strict else DCB_FAST_BF16)

  def forward(self, rows: np.ndarray, want_probs: bool = False, want_logits: bool = False,
              strict_input: bool = True, strict: Optional[bool] = None) -> Dict[str, np.ndarray]:
    """rows float32 [B, R, L(,1)] -> dict(bases u8 [B,L], quals u8 [B,L], [probs], [logits]).

    Batches larger than `max_batch` are split, like `batch_examples` does with
    `options.batch_size` (quick_inference.py:304-338).
    """
    rows = self._rows3(rows)
    B, L = rows.shape[0], self.max_length
    out = dict(bases=np.empty((B, L), np.uint8), quals=np.empty((B, L), np.uint8))
    if want_probs:
      out["probs"] = np.empty((B, L, 5), np.float32)
    if want_logits:
      out["logits"] = np.empty((B, L, 5), np.float32)
    ms, launches = 0.0, 0
    for b0 in range(0, B, self.max_batch):
      b1 = min(B, b0 + self.max_batch)
      ptr = lambda k: out[k][b0:b1].ctypes.data_as(ctypes.c_void_p) if k in out else None
      rc = self._lib.dcb_forward(self._handle, rows[b0:b1].ctypes.data_as(ctypes.c_void_p), b1 - b0,
                                 self._precision_flag(strict), ptr("bases"), ptr("quals"), ptr("probs"), ptr("logits"))
      self._check(rc, tolerate=() if strict_input else (-5,))
      ms += self.last_forward_ms()
      launches += self.last_forward_launches()
    self.last_ms, self.last_launches = ms, launches
    return out

  # -- packed input rows (include/dcb200.h "packed input rows"; SURVEY.md section 8(f)1) -------------------------
  @property
  def packed_window_bytes(self) -> int:
    return packed_window_bytes(self.params)

  def pack_rows(self, rows: np.ndarray, out: Optional[np.ndarray] = None, strict_input: bool = True) -> np.ndarray:
    return pack_rows(self.params, rows, out, strict_input)

  def forward_packed(self, packed: np.ndarray, want_probs: bool = False, want_logits: bool = False,
                     strict_input: bool = True, strict: Optional[bool] = None) -> Dict[str, np.ndarray]:
    """forward() on packed rows uint8 [B, packed_window_bytes]: bit-identical to forward() on the float32 rows they
    were packed from."""
    packed = np.ascontiguousarray(packed, dtype=np.uint8)
    if packed.ndim != 2 or packed.shape[1] != self.packed_window_bytes:
      raise ValueError("packed rows must be uint8 [B, %d]" % self.packed_window_bytes)
    B, L = packed.shape[0], self.max_length
    out = dict(bases=np.empty((B, L), np.uint8), quals=np.empty((B, L), np.uint8))
    if want_probs:
      out["probs"] = np.empty((B, L, 5), np.float32)
    if want_logits:
      out["logits"] = np.empty((B, L, 5), np.float32)
    ms, launches = 0.0, 0
    for b0 in range(0, B, self.max_batch):
      b1 = min(B, b0 + self.max_batch)
      ptr = lambda k: out[k][b0:b1].ctypes.data_as(ctypes.c_void_p) if k in out else None
      rc = self._lib.dcb_forward_packed(self._handle, packed[b0:b1].ctypes.data_as(ctypes.c_void_p), b1 - b0,
                                        self._precision_flag(strict), ptr("bases"), ptr("quals"), ptr("probs"),
                                        ptr("logits"))
      self._check(rc, tolerate=() if strict_input else (-5,))
      ms += self.last_forward_ms()
      launches += self.last_forward_launches()
    self.last_ms, self.last_launches = ms, launches
    return out

  def submit_packed_raw(self, packed_ptr: int, batch: int, flags: int, bases_ptr: int, quals_ptr: int) -> int:
    """dcb_submit_packed on caller-managed pointers; returns the ticket for wait_raw()."""
    ticket = ctypes.c_int64(-1)
    self._check(self._lib.dcb_submit_packed(self._handle, ctypes.c_void_p(packed_ptr), batch, flags,
                                            ctypes.c_void_p(bases_ptr), ctypes.c_void_p(quals_ptr), None, None,
                                            ctypes.byref(ticket)))
    return int(ticket.value)

  # -- the hot path, pipelined over a stream of batches ----------------------------------------
  # dcb_submit / dcb_wait: the host->device copy of batch i+1 overlaps the kernels of batch i.  Page-locked staging
  # (two sets, allocated on first use) is owned here so that callers can stack their windows straight into it.
  def staging_rows(self, slot: int) -> np.ndarray:
    """Pinned float32 [max_batch, R, L] buffer of pipeline slot 0/1 (fill [:batch], then submit(slot=...))."""
    st = self._staging(slot)
    return st["rows"]

  def _staging(self, slot: int) -> Dict[str, Any]:
    if not hasattr(self, "_stage"):
      self._stage = {}
    if slot not in self._stage:
      mb, R, L = self.max_batch, self.total_rows, self.max_length
      def pinned(shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        addr, raw = alloc_pinned(max(n, 1))
        return addr, raw[:n].view(dtype).reshape(shape)
      st = {"addrs": []}
      for key, shape, dt in (("rows", (mb, R, L), np.float32), ("bases", (mb, L), np.uint8),
                             ("quals", (mb, L), np.uint8)):
        addr, st[key] = pinned(shape, dt)
        st["addrs"].append(addr)
      self._stage[slot] = st
    return self._stage[slot]

  def _staging_opt(self, slot: int, key: str) -> np.ndarray:
    st = self._staging(slot)
    if key not in st:
      n = self.max_batch * self.max_length * 5 * 4
      addr, raw = alloc_pinned(n)
      st[key] = raw.view(np.float32).reshape(self.max_batch, self.max_length, 5)
      st["addrs"].append(addr)
    return st[key]

  def submit(self, rows: Optional[np.ndarray] = None, batch: Optional[int] = None, slot: Optional[int] = None,
             want_probs: bool = False, want_logits: bool = False, strict: Optional[bool] = None) -> Dict[str, Any]:
    """Enqueue one batch (<= max_batch windows) and return a handle for wait().  Either pass `rows` (copied into the
    slot's pinned staging) or fill staging_rows(slot)[:batch] yourself and pass `batch`.  At most two handles may be
    outstanding and they must be waited for in submission order."""
    busy = self.__dict__.setdefault("_slot_busy", {0: False, 1: False})
    if slot is None:
      slot = 1 - getattr(self, "_last_slot", 1)
      if busy[slot] and not busy[1 - slot]:
        slot = 1 - slot
    if busy[slot]:   # its pinned staging may still be read by the copy engine: refuse before touching it
      raise DcbError(-4, "two submissions in flight: wait() for the oldest first")
    self._last_slot = slot
    st = self._staging(slot)
    if rows is not None:
      rows = self._rows3(rows)
      batch = rows.shape[0]
      if batch > self.max_batch:
        raise ValueError("submit(): batch %d > max_batch %d" % (batch, self.max_batch))
      st["rows"][:batch] = rows
    elif batch is None:
      raise ValueError("submit(): rows or batch required")
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    probs = self._staging_opt(slot, "probs") if want_probs else None
    logits = self._staging_opt(slot, "logits") if want_logits else None
    ticket = ctypes.c_int64(-1)
    self._check(self._lib.dcb_submit(self._handle, vp(st["rows"]), batch, self._precision_flag(strict),
                                     vp(st["bases"]), vp(st["quals"]),
                                     vp(probs) if want_probs else None, vp(logits) if want_logits else None,
                                     ctypes.byref(ticket)))
    busy[slot] = True
    return dict(ticket=int(ticket.value), slot=slot, batch=batch, probs=want_probs, logits=want_logits)

  def wait(self, handle: Dict[str, Any], strict_input: bool = True) -> Dict[str, np.ndarray]:
    """Block until the submission's results are on the host; returns the same dict as forward()."""
    rc = self._lib.dcb_wait(self._handle, handle["ticket"])
    if rc != -4:   # anything but "not in flight" retires the slot
      self._slot_busy[handle["slot"]] = False
    self._check(rc, tolerate=() if strict_input else (-5,))
    st, b = self._stage[handle["slot"]], handle["batch"]
    out = dict(bases=st["bases"][:b].copy(), quals=st["quals"][:b].copy())
    if handle["probs"]:
      out["probs"] = st["probs"][:b].copy()
    if handle["logits"]:
      out["logits"] = st["logits"][:b].copy()
    self.last_ms, self.last_launches = self.last_forward_ms(), self.last_forward_launches()
    return out

  def drain(self, *handles) -> None:
    """Retire outstanding submissions whose results are no longer wanted (error paths): waits for each handle and
    swallows its status, so the engine's and this object's pipeline slots are free again."""
    for h in handles:
      if h is None:
        continue
      try:
        self.wait(h, strict_input=False)
      except DcbError:
        pass

  def forward_batches(self, batches, want_probs: bool = False, want_logits: bool = False,
                      strict_input: bool = True, strict: Optional[bool] = None):
    """Pipelined forward over an iterable of row batches; yields one output dict per batch, in order."""
    pending = None
    try:
      for rows in batches:
        h = self.submit(rows, want_probs=want_probs, want_logits=want_logits, strict=strict)
        prev, pending = pending, h
        if prev is not None:
          yield self.wait(prev, strict_input)
      if pending is not None:
        h, pending = pending, None
        yield self.wait(h, strict_input)
    finally:
      self.drain(pending)

  # -- stitch: per-read window concatenation + gap compaction on the device -------------------------
  def stitch(self, bases, quals, zmw_start: np.ndarray, n_windows: Optional[int] = None,
             on_device: bool = False, length: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """dcb_stitch: bases/quals are uint8 [n_windows, L] arrays (or device addresses when `on_device`); read z is the
    windows [zmw_start[z], zmw_start[z+1]).  Returns (seq, qual, lengths): read z's compacted characters are
    seq[zmw_start[z] * L : zmw_start[z] * L + lengths[z]] (same for qual)."""
    zs = np.ascontiguousarray(zmw_start, dtype=np.int32)
    nz = int(zs.shape[0]) - 1
    L = int(length) if length is not None else self.max_length   # characters per window
    if on_device:
      if n_windows is None:
        raise ValueError("stitch(on_device=True) needs n_windows")
      b_ptr, q_ptr = ctypes.c_void_p(int(bases)), ctypes.c_void_p(int(quals))
      flags = DCB_ROWS_ON_DEVICE
    else:
      bases = np.ascontiguousarray(bases, dtype=np.uint8)
      quals = np.ascontiguousarray(quals, dtype=np.uint8)
      n_windows = int(bases.shape[0])
      b_ptr, q_ptr = bases.ctypes.data_as(ctypes.c_void_p), quals.ctypes.data_as(ctypes.c_void_p)
      flags = 0
    seq = np.empty(n_windows * L, np.uint8)
    qual = np.empty(n_windows * L, np.uint8)
    lens = np.zeros(max(nz, 0), np.int32)
    self._check(self._lib.dcb_stitch(self._handle, b_ptr, q_ptr, n_windows, L,
                                     zs.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), nz, flags,
                                     seq.ctypes.data_as(ctypes.c_void_p), qual.ctypes.data_as(ctypes.c_void_p),
                                     lens.ctypes.data_as(ctypes.c_void_p)))
    return seq, qual, lens

  def stitch_fastq(self, bases, quals, zmw_start: np.ndarray, window_pos, names, min_quality: float, min_length: int,
                   n_windows: Optional[int] = None, on_device: bool = False, length: Optional[int] = None,
                   window_off: Optional[np.ndarray] = None):
    """dcb_stitch_fastq: stitch_utils.stitch_to_fastq for a batch of reads on the device.  Returns (fastq bytes,
    rec_off int64 [n_zmw + 1], outcome int32 [n_zmw], avg_q float64 [n_zmw]); read z's record is
    fastq[rec_off[z]:rec_off[z + 1]] (empty unless outcome[z] & 0x7f == DCB_READ_OK).
    window_off (int64 [n_windows + 1], host arrays only): windows of their own width, dcb_stitch_fastq_ragged -- bases /
    quals are flat and window w is bytes [window_off[w], window_off[w + 1])."""
    zs = np.ascontiguousarray(zmw_start, dtype=np.int32)
    nz = int(zs.shape[0]) - 1
    L = int(length) if length is not None else self.max_length
    if on_device:
      if n_windows is None:
        raise ValueError("stitch_fastq(on_device=True) needs n_windows")
      b_ptr, q_ptr, flags = ctypes.c_void_p(int(bases)), ctypes.c_void_p(int(quals)), DCB_ROWS_ON_DEVICE
    else:
      bases = np.ascontiguousarray(bases, dtype=np.uint8)
      quals = np.ascontiguousarray(quals, dtype=np.uint8)
      n_windows = int(bases.shape[0])
      b_ptr, q_ptr, flags = bases.ctypes.data_as(ctypes.c_void_p), quals.ctypes.data_as(ctypes.c_void_p), 0
    if window_off is not None:
      window_off = np.ascontiguousarray(window_off, dtype=np.int64)
      n_windows = int(window_off.shape[0]) - 1
      if on_device or int(window_off[-1]) > min(bases.size, quals.size):
        raise ValueError("stitch_fastq: window_off needs host arrays that hold window_off[-1] bytes")
    pos = np.ascontiguousarray(window_pos, dtype=np.int32)
    if pos.shape[0] != n_windows:
      raise ValueError("window_pos must have one entry per window")
    enc = [n.encode("latin-1") if isinstance(n, str) else bytes(n) for n in names]
    if len(enc) != nz:
      raise ValueError("names must have one entry per read")
    name_off = np.zeros(nz + 1, np.int32)
    if nz:
      name_off[1:] = np.cumsum([len(x) for x in enc])
    blob = np.frombuffer(b"".join(enc) or b"\0", np.uint8)
    cap = int(name_off[-1]) + 2 * (n_windows * L if window_off is None else int(window_off[-1])) + 6 * nz + 16
    fastq = np.empty(cap, np.uint8)
    rec_off = np.zeros(nz + 1, np.int64)
    outcome = np.zeros(max(nz, 0), np.int32)
    avg_q = np.zeros(max(nz, 0), np.float64)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    if window_off is None:
      self._check(self._lib.dcb_stitch_fastq(self._handle, b_ptr, q_ptr, n_windows, L, vp(zs), nz, vp(pos), vp(blob),
                                             vp(name_off), float(min_quality), int(min_length), flags, vp(fastq), cap,
                                             vp(rec_off), vp(outcome), vp(avg_q)))
    else:
      self._check(self._lib.dcb_stitch_fastq_ragged(self._handle, b_ptr, q_ptr, n_windows, vp(window_off), L, vp(zs), nz,
                                                    vp(pos), vp(blob), vp(name_off), float(min_quality),
                                                    int(min_length), flags, vp(fastq), cap, vp(rec_off), vp(outcome),
                                                    vp(avg_q)))
    return fastq[:int(rec_off[-1])].tobytes(), rec_off, outcome, avg_q

  def skip_mask(self, ccs_base_quality_scores: np.ndarray, skip_windows_above: float) -> Tuple[np.ndarray, np.ndarray]:
    """dcb_skip_mask: per window avg_phred(ccs_base_quality_scores) > skip_windows_above on the device
    (quick_inference.py:663-672).  Returns (mask uint8 [n] with 2 = within 1e-7 of the threshold, avg float64 [n])."""
    bq = np.ascontiguousarray(ccs_base_quality_scores, dtype=np.int16)
    if bq.ndim != 2:
      raise ValueError("ccs_base_quality_scores must be [n_windows, L]")
    n, L = bq.shape
    mask, avg = np.zeros(n, np.uint8), np.zeros(n, np.float64)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    self._check(self._lib.dcb_skip_mask(self._handle, vp(bq), n, L, float(skip_windows_above), vp(mask), vp(avg)))
    return mask, avg

  def fill_skipped(self, ccs_ids: np.ndarray, ccs_base_quality_scores: np.ndarray, dst_window: np.ndarray,
                   bases, quals, calibration: Optional[calibration_lib.QualityCalibrationValues] = None,
                   on_device: bool = False) -> None:
    """dcb_fill_skipped: process_skipped_window (quick_inference.py:567-594) for k windows on the device; window j
    lands in row dst_window[j] of `bases` / `quals` (uint8 [*, L] arrays, or device addresses with on_device)."""
    ids = np.ascontiguousarray(ccs_ids, dtype=np.uint8)
    bq = np.ascontiguousarray(ccs_base_quality_scores, dtype=np.int16)
    dst = np.ascontiguousarray(dst_window, dtype=np.int32)
    k, L = ids.shape
    if bq.shape != (k, L) or dst.shape != (k,):
      raise ValueError("fill_skipped: ccs_ids / ccs_base_quality_scores [k, L] and dst_window [k] expected")
    cal = calibration
    en = int(bool(cal is not None and cal.enabled))
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    if on_device:
      b_ptr, q_ptr, flags = ctypes.c_void_p(int(bases)), ctypes.c_void_p(int(quals)), DCB_OUT_ON_DEVICE
    else:
      if not (bases.flags.c_contiguous and quals.flags.c_contiguous and bases.dtype == np.uint8 and quals.dtype == np.uint8):
        raise ValueError("fill_skipped: bases / quals must be C-contiguous uint8 arrays")
      if k and int(dst.max()) >= bases.shape[0]:
        raise ValueError("fill_skipped: destination window outside the output arrays")
      b_ptr, q_ptr, flags = vp(bases), vp(quals), 0
    self._check(self._lib.dcb_fill_skipped(self._handle, vp(ids), vp(bq), vp(dst), k, L, en,
                                           float(cal.threshold) if en else 0.0, float(cal.w) if en else 1.0,
                                           float(cal.b) if en else 0.0, flags, b_ptr, q_ptr))

  def fill_skipped_ragged(self, ccs_ids: np.ndarray, ccs_base_quality_scores: np.ndarray, src_off: np.ndarray,
                          dst_off: np.ndarray, bases: np.ndarray, quals: np.ndarray,
                          calibration: Optional[calibration_lib.QualityCalibrationValues] = None) -> None:
    """dcb_fill_skipped_ragged: `fill_skipped` for windows of their own width.  Window j is entries
    [src_off[j], src_off[j + 1]) of ccs_ids / ccs_base_quality_scores (flat) and lands at byte dst_off[j] of the flat
    host uint8 arrays bases / quals."""
    ids = np.ascontiguousarray(ccs_ids, dtype=np.uint8).reshape(-1)
    bq = np.ascontiguousarray(ccs_base_quality_scores, dtype=np.int16).reshape(-1)
    src = np.ascontiguousarray(src_off, dtype=np.int64)
    dst = np.ascontiguousarray(dst_off, dtype=np.int64)
    k = int(src.shape[0]) - 1
    if dst.shape != (k,) or int(src[-1]) > min(ids.shape[0], bq.shape[0]):
      raise ValueError("fill_skipped_ragged: src_off [k + 1] within ccs_ids / ccs_base_quality_scores and dst_off [k] expected")
    if not (bases.flags.c_contiguous and quals.flags.c_contiguous and bases.dtype == np.uint8 and quals.dtype == np.uint8):
      raise ValueError("fill_skipped_ragged: bases / quals must be C-contiguous uint8 arrays")
    if k and int((dst + np.diff(src)).max()) > min(bases.size, quals.size):
      raise ValueError("fill_skipped_ragged: destination outside the output arrays")
    cal = calibration
    en = int(bool(cal is not None and cal.enabled))
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    self._check(self._lib.dcb_fill_skipped_ragged(self._handle, vp(ids), vp(bq), vp(src), vp(dst), k, en,
                                                  float(cal.threshold) if en else 0.0, float(cal.w) if en else 1.0,
                                                  float(cal.b) if en else 0.0, 0, vp(bases), vp(quals)))

  def stitch_raw(self, bases_ptr: int, quals_ptr: int, n_windows: int, zmw_start: np.ndarray, flags: int,
                 seq_ptr: int, qual_ptr: int, len_ptr: int, length: Optional[int] = None) -> None:
    """dcb_stitch on caller-managed pointers (host or device per `flags`)."""
    zs = np.ascontiguousarray(zmw_start, dtype=np.int32)
    self._check(self._lib.dcb_stitch(self._handle, ctypes.c_void_p(bases_ptr), ctypes.c_void_p(quals_ptr), n_windows,
                                     int(length) if length is not None else self.max_length,
                                     zs.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), int(zs.shape[0]) - 1, flags,
                                     ctypes.c_void_p(seq_ptr), ctypes.c_void_p(qual_ptr), ctypes.c_void_p(len_ptr)))

  def predict(self, rows: np.ndarray) -> _Prediction:
    """Softmax output [B, L, 5], shaped like `EncoderOnlyTransformer.predict` (networks.py:357-365)."""
    return _Prediction(self.forward(rows, want_probs=True)["probs"])

  # -- introspection -----------------------------------------------------------------------
  def last_forward_ms(self) -> float:
    v = ctypes.c_float()
    self._check(self._lib.dcb_last_forward_ms(self._handle, ctypes.byref(v)))
    return float(v.value)

  def last_forward_launches(self) -> int:
    v = ctypes.c_int32()
    self._check(self._lib.dcb_last_forward_launches(self._handle, ctypes.byref(v)))
    return int(v.value)

  def set_profile(self, enabled: bool = True) -> None:
    self._check(self._lib.dcb_set_profile(self._handle, int(enabled)))

  def get_profile(self) -> Dict[str, float]:
    ms, n, tok = ctypes.c_float(), ctypes.c_int32(), ctypes.c_int64()
    self._check(self._lib.dcb_get_profile(self._handle, ctypes.byref(ms), ctypes.byref(n),
                                          ctypes.byref(tok)))
    ms6, n6, fused = (ctypes.c_float * 6)(), (ctypes.c_int32 * 6)(), ctypes.c_int32()
    self._check(self._lib.dcb_get_profile_kernels(self._handle, ms6, n6, ctypes.byref(fused)))
    names = ("embed", "row_gemm", "qkv_gemm", "attention", "ffn", "head")
    return dict(ffn_ms_total=float(ms.value), ffn_launches=int(n.value), ffn_tokens=int(tok.value),
                fused_oproj=int(fused.value),   # 0: separate out-proj, 1: fused into the FFN kernel, 2: whole stack in one kernel
                kernels={k: dict(ms=float(ms6[i]), launches=int(n6[i])) for i, k in enumerate(names)})

  def set_debug(self, enabled: bool = True) -> None:
    self._check(self._lib.dcb_set_debug(self._handle, int(enabled)))

  def debug_residual(self, stage: int, tokens: int) -> np.ndarray:
    out = np.empty((tokens, 280), np.float32)
    self._check(self._lib.dcb_debug_residual(self._handle, stage, out.ctypes.data_as(ctypes.c_void_p),
                                             out.size))
    return out

  # -- raw device / pinned buffers (bench, multi-GPU driver) ----------------------------------
  def alloc_device(self, nbytes: int) -> int:
    p = ctypes.c_void_p()
    self._check(self._lib.dcb_alloc_device(self._handle, nbytes, ctypes.byref(p)))
    return p.value

  def free_device(self, ptr: int) -> None:
    self._check(self._lib.dcb_free_device(self._handle, ctypes.c_void_p(ptr)))

  def memcpy_h2d(self, dst: int, src: np.ndarray) -> None:
    src = np.ascontiguousarray(src)
    self._check(self._lib.dcb_memcpy_h2d(self._handle, ctypes.c_void_p(dst),
                                         src.ctypes.data_as(ctypes.c_void_p), src.nbytes))

  def memcpy_d2h(self, dst: np.ndarray, src: int) -> None:
    self._check(self._lib.dcb_memcpy_d2h(self._handle, dst.ctypes.data_as(ctypes.c_void_p),
                                         ctypes.c_void_p(src), dst.nbytes))

  def submit_raw(self, rows_ptr: int, batch: int, flags: int, bases_ptr: int, quals_ptr: int,
                 probs_ptr: int = 0, logits_ptr: int = 0) -> int:
    """dcb_submit on caller-managed pointers; returns the ticket for wait_raw()."""
    ticket = ctypes.c_int64(-1)
    self._check(self._lib.dcb_submit(self._handle, ctypes.c_void_p(rows_ptr), batch, flags,
                                     ctypes.c_void_p(bases_ptr), ctypes.c_void_p(quals_ptr),
                                     ctypes.c_void_p(probs_ptr) if probs_ptr else None,
                                     ctypes.c_void_p(logits_ptr) if logits_ptr else None, ctypes.byref(ticket)))
    return int(ticket.value)

  def wait_raw(self, ticket: int) -> None:
    self._check(self._lib.dcb_wait(self._handle, ticket))

  def forward_raw(self, rows_ptr: int, batch: int, flags: int, bases_ptr: int, quals_ptr: int,
                  probs_ptr: int = 0, logits_ptr: int = 0) -> None:
    """dcb_forward on caller-managed pointers (host or device per `flags`)."""
    self._check(self._lib.dcb_forward(self._handle, ctypes.c_void_p(rows_ptr), batch, flags,
                                      ctypes.c_void_p(bases_ptr), ctypes.c_void_p(quals_ptr),
                                      ctypes.c_void_p(probs_ptr) if probs_ptr else None,
                                      ctypes.c_void_p(logits_ptr) if logits_ptr else None))

  def synchronize(self) -> None:
    self._check(self._lib.dcb_synchronize(self._handle))


def packed_window_bytes(params: params_lib.Params) -> int:
  """Bytes per window of the packed row format (include/dcb200.h "packed input rows")."""
  cfg = make_config(params, max_batch=1)
  return int(load_library().dcb_packed_window_bytes(ctypes.byref(cfg)))


def pack_rows(params: params_lib.Params, rows: np.ndarray, out: Optional[np.ndarray] = None,
              strict_input: bool = True) -> np.ndarray:
  """float32 rows [B, R, L(,1)] -> packed uint8 [B, packed_window_bytes] (dcb_pack_rows; host code, needs no GPU).
  Raises DcbError(-5) when a base / strand / ccs / ccs_bq value lies outside its vocabulary (TensorFlow's gather would
  raise) or an SN row is not constant, unless `strict_input` is False (values are clamped either way)."""
  rows = np.asarray(rows)
  if rows.ndim == 4:
    rows = rows[..., 0]
  R = params_lib.get_total_rows(params.max_passes, params.use_ccs_bq)
  if rows.ndim != 3 or rows.shape[1] != R or rows.shape[2] != int(params.max_length):
    raise ValueError("rows must be [B, %d, %d(, 1)], got %s" % (R, int(params.max_length), rows.shape))
  rows = np.ascontiguousarray(rows, dtype=np.float32)
  lib, cfg = load_library(), make_config(params, max_batch=1)
  stride = int(lib.dcb_packed_window_bytes(ctypes.byref(cfg)))
  B = rows.shape[0]
  if out is None:
    out = np.empty((B, stride), np.uint8)
  if out.shape != (B, stride) or out.dtype != np.uint8 or not out.flags.c_contiguous:
    raise ValueError("pack_rows(out=...): need C-contiguous uint8 [%d, %d]" % (B, stride))
  rc = lib.dcb_pack_rows(ctypes.byref(cfg), rows.ctypes.data_as(ctypes.c_void_p), B, out.ctypes.data_as(ctypes.c_void_p))
  if rc and not (rc == -5 and not strict_input):
    raise DcbError(rc, lib.dcb_last_error(None).decode())
  return out


def unpack_rows(params: params_lib.Params, packed: np.ndarray) -> np.ndarray:
  """The float32 rows [B, R, L] a packed batch stands for (NumPy mirror of csrc/common.h packed_value; tests and
  debugging -- the engine never needs it)."""
  P, L, bq = int(params.max_passes), int(params.max_length), int(bool(params.use_ccs_bq))
  R = 4 * P + 5 + bq
  packed = np.asarray(packed, np.uint8)
  B = packed.shape[0]
  sn_off = ((3 * P + 1 + bq) * L + 15) & ~15
  planes = packed[:, :(3 * P + 1 + bq) * L].reshape(B, 3 * P + 1 + bq, L)
  rows = np.zeros((B, R, L), np.float32)
  rows[:, :P] = planes[:, :P] & 7
  rows[:, P:3 * P] = planes[:, P:3 * P]
  rows[:, 3 * P:4 * P] = (planes[:, :P] >> 3) & 3
  rows[:, 4 * P] = planes[:, 3 * P]
  if bq:
    rows[:, 4 * P + 1] = planes[:, 3 * P + 1].astype(np.float32) - 1
  sn = np.ascontiguousarray(packed[:, sn_off:sn_off + 16]).view(np.float32)
  rows[:, R - 4:] = sn[:, :, None]
  return rows


def alloc_pinned(nbytes: int) -> Tuple[int, np.ndarray]:
  """Pinned host buffer as (address, uint8 ndarray view). Free with free_pinned(address)."""
  lib = load_library()
  p = ctypes.c_void_p()
  rc = lib.dcb_alloc_host(nbytes, ctypes.byref(p))
  if rc:
    raise DcbError(rc, "cudaMallocHost failed")
  arr = np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctypes.c_uint8)), shape=(nbytes,))
  return p.value, arr


def free_pinned(addr: int) -> None:
  load_library().dcb_free_host(ctypes.c_void_p(addr))

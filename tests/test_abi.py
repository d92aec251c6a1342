"""The C-ABI library: loads without a GPU, exports every symbol include/dcb200.h declares, and the
product path fails loudly (no CPU fallback) when no GPU is present."""
import ctypes
import os
import re

import pytest

from deepconsensus_b200 import engine, params as params_lib, weights as weights_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols(header="dcb200.h"):
  text = open(os.path.join(ROOT, "include", header)).read()
  text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
  return sorted(set(re.findall(r"\b(dcb_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
  assert _declared_symbols() == sorted(engine.ABI_SYMBOLS)
  assert _declared_symbols("dcb200_debug.h") == sorted(engine.DEBUG_SYMBOLS)


def test_library_exports_every_declared_symbol():
  if not os.path.exists(engine.library_path()):
    import __graft_entry__
    __graft_entry__.build()
  for path in (engine.library_path(), os.path.join(os.path.dirname(engine.library_path()), "libdcb200_dev.so")):
    lib = ctypes.CDLL(path)
    for sym in _declared_symbols() + _declared_symbols("dcb200_debug.h"):
      assert hasattr(lib, sym), (path, sym)
  assert b"sm_100a" in engine.load_library().dcb_version()


def test_config_struct_matches_header_field_order():
  text = open(os.path.join(ROOT, "include", "dcb200.h")).read()
  body = text[text.index("typedef struct dcb_config {") + len("typedef struct dcb_config {"):text.index("} dcb_config;")]
  body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
  names = []
  for decl in body.split(";"):
    decl = decl.strip()
    m = re.match(r"(int32_t|double)\s+(.*)", decl, flags=re.S)
    if m:
      names += [n.strip().split("[")[0] for n in m.group(2).split(",")]
  assert names == [f[0] for f in engine.DcbConfig._fields_]


def test_kernel_path_switches_exist_only_in_the_developer_build():
  """The DCB_* kernel-path switches exist only in the developer build; retired ones exist in neither."""
  prod = open(engine.library_path(), "rb").read()
  dev = open(os.path.join(os.path.dirname(engine.library_path()), "libdcb200_dev.so"), "rb").read()
  for name in (b"DCB_STACK", b"DCB_FUSE_QA", b"DCB_FUSE_HEAD", b"DCB_ALIGN", b"DCB_CHUNK_TILES"):
    assert name not in prod, name
    assert name in dev, name
  for name in (b"DCB_QKV2", b"DCB_FFN_PAIR", b"DCB_FFN_CLUSTER"):   # retired switches: neither build reads them
    assert name not in prod and name not in dev, name


def test_no_cpu_fallback_without_gpu():
  import torch
  if torch.cuda.is_available():
    pytest.skip("GPU present")
  p = params_lib.synthetic_params(20, 100)
  with pytest.raises(engine.DcbError, match="no CUDA device|CPU fallback"):
    engine.B200Model(p, weights_lib.init_weights(p), max_batch=2)


def test_product_code_never_imports_oracle():
  pkg = os.path.join(ROOT, "deepconsensus_b200")
  for dirpath, _, files in os.walk(pkg):
    for f in files:
      if f.endswith((".py", ".cu", ".cuh", ".h", ".sh")):
        src = open(os.path.join(dirpath, f)).read()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(dirpath, f)

"""The C-ABI library loads on a CPU-only box and exports every entry point that
include/tfr_b200.h declares (no compute calls here)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
  text = open(os.path.join(ROOT, 'include', 'tfr_b200.h')).read()
  text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
  return sorted(set(re.findall(r'\b(tfr_[a-z0-9_]+)\s*\(', text)))


def test_build_and_exports():
  import __graft_entry__ as g
  lib_path = g.build()
  lib = ctypes.CDLL(lib_path)
  declared = _declared_symbols()
  assert len(declared) >= 14, declared
  for name in declared:
    assert hasattr(lib, name), 'missing symbol ' + name


def test_binding_matches_header():
  import __graft_entry__ as g
  g.build()
  from ranking_b200 import _C
  assert sorted(_C.EXPORTED_SYMBOLS) == _declared_symbols()
  assert _C.lib.tfr_version() >= 1
  assert isinstance(_C.last_error(), str)


def test_argument_validation_without_gpu():
  """Argument errors are reported before any CUDA call."""
  import __graft_entry__ as g
  g.build()
  from ranking_b200 import _C
  rc = _C.lib.tfr_approx_loss_fwd_bwd(None, None, None, 0, None, 1, 4, 1.0, 0,
                                      1.0, 0, None, None, None, None)
  assert rc == 1 and 'NULL' in _C.last_error()
  cfg = _C.MlpCfg()
  cfg.n_dense = 0
  assert _C.lib.tfr_mlp_param_count(ctypes.byref(cfg)) == 0
  cfg.n_dense = 4
  for i, d in enumerate([136, 256, 128, 64, 1]):
    cfg.dims[i] = d
  assert _C.lib.tfr_mlp_param_count(ctypes.byref(cfg)) == (
      136 * 256 + 256 + 256 * 128 + 128 + 128 * 64 + 64 + 64 + 1)


def test_product_has_no_oracle_import():
  """The product package must never route through the oracle."""
  pkg = os.path.join(ROOT, 'ranking_b200')
  for dirpath, _, files in os.walk(pkg):
    for f in files:
      if f.endswith('.py'):
        src = open(os.path.join(dirpath, f)).read()
        assert not re.search(r'^\s*(from|import)\s+oracle\b', src, flags=re.M), f


def test_native_code_reads_no_environment():
  """Which kernel runs follows from shapes and arguments only: an environment variable
  must not switch a library call to another code path."""
  csrc = os.path.join(ROOT, 'ranking_b200', 'csrc')
  sources = sorted(f for f in os.listdir(csrc) if f.endswith(('.cu', '.cuh', '.h')))
  assert any(f.endswith('.cu') for f in sources), sources
  for f in sources:
    src = open(os.path.join(csrc, f)).read()
    assert not re.search(r'getenv\s*\(', src), f

"""CPU-side checks of the C-ABI boundary: the library loads, exports every symbol the header
declares, and refuses to compute without a GPU (no silent CPU fallback)."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from omnidirectional_collaborative_filtering_b200 import _lib


def test_library_exports_every_declared_symbol():
    lib = _lib.lib()
    names = _lib.header_symbols()
    assert len(names) >= 30
    for name in names:
        assert hasattr(lib, name), "include/ocf.h declares %s but libocf_b200.so does not export it" % name
    assert set(names) == set(_lib._SIGNATURES), "ctypes signatures out of sync with include/ocf.h"
    assert lib.ocf_version() == 101


def test_exports_are_plain_c():
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.SO_PATH], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert set(_lib.header_symbols()) <= exported


def test_kernels_are_sm100a():
    out = subprocess.run(["cuobjdump", "-lelf", _lib.SO_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_argument_validation_needs_no_gpu():
    lib = _lib.lib()
    out = C.c_void_p()
    rowptr = np.array([0, 2, 1], dtype=np.int64)           # not monotone
    col = np.zeros(2, dtype=np.int32); val = np.zeros(2, dtype=np.float32)
    st = lib.ocf_store_create(2, 4, _lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(val), C.byref(out))
    assert st == -1 and b"monotone" in lib.ocf_last_error()
    cfg = _lib.ModelConfig()
    cfg.n_cols = 10; cfg.n_cols_total = 10; cfg.n_layers = 0
    st = lib.ocf_model_create(C.byref(cfg), C.byref(out))
    assert st == -1 and b"n_layers" in lib.ocf_last_error()


@pytest.mark.skipif(_lib.lib().ocf_device_count() > 0, reason="only meaningful without a GPU")
def test_no_cpu_fallback():
    from omnidirectional_collaborative_filtering_b200.store import RatingStore
    from omnidirectional_collaborative_filtering_b200.synthetic import Csr
    s = RatingStore(Csr(1, 3, np.array([0, 1], dtype=np.int64), np.array([1], dtype=np.int32),
                        np.array([2.0], dtype=np.float32)))
    with pytest.raises(_lib.OcfError):
        s.handle


def test_header_is_plain_c_and_links(tmp_path):
    """include/ocf.h compiles as C99 (no C++ in the signatures) and a C program linked against the
    library can call it: here the host-only ingest of a rating file, start to finish."""
    import json
    import os
    src = tmp_path / "use.c"
    src.write_text(r'''
#include <stdio.h>
#include "ocf.h"
int main(int argc, char** argv) {
  ocf_vocab* v = 0; ocf_ratings* r = 0; int64_t info[4];
  if (ocf_version() != OCF_VERSION) return 2;
  if (ocf_vocab_load_json(argv[1], &v)) { printf("%s\n", ocf_last_error()); return 3; }
  if (ocf_ratings_load_json(argv[2], v, 0, &r)) { printf("%s\n", ocf_last_error()); return 4; }
  if (ocf_ratings_info(r, info)) return 5;
  printf("%lld rows %lld ratings\n", (long long)info[0], (long long)info[2]);
  ocf_ratings_destroy(r); ocf_vocab_destroy(v);
  return ocf_ratings_load_json("/nonexistent.json", 0, 0, &r) == OCF_ERR_INVALID ? 0 : 6;
}
''')
    root = os.path.dirname(_lib.HEADER_PATH)
    exe = str(tmp_path / "use")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", root, str(src), "-o", exe, _lib.SO_PATH,
                    "-Wl,-rpath," + os.path.dirname(_lib.SO_PATH)], check=True)
    (tmp_path / "v.json").write_text(json.dumps([10, 20, 30]))
    (tmp_path / "t.json").write_text(json.dumps({"a": [[10, 1.0], [30.0, 2.5]], "b": [[20, 4]]}))
    out = subprocess.run([exe, str(tmp_path / "v.json"), str(tmp_path / "t.json")], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip() == "2 rows 3 ratings", (out.returncode, out.stdout, out.stderr)


def test_product_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under the package imports it, and importing the whole package
    leaves `oracle` out of sys.modules (a product path routed through the oracle would void every parity claim)."""
    import os
    import sys
    pkg = os.path.dirname(_lib.HERE + "/")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                with open(os.path.join(root, f), errors="replace") as fh:
                    text = fh.read()
                assert "import oracle" not in text and "from oracle" not in text, f
    code = ("import sys; sys.path.insert(0, %r); "
            "import omnidirectional_collaborative_filtering_b200 as p; "
            "from omnidirectional_collaborative_filtering_b200 import data_reader, model, train, dist, ingest, splitter, store, synthetic, optimizers; "
            "assert not [m for m in sys.modules if m == 'oracle' or m.startswith('oracle.')]" % os.path.dirname(pkg))
    subprocess.run([sys.executable, "-c", code], check=True)

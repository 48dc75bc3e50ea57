"""CPU tests: the C-ABI library loads, exports every symbol include/lbic.h declares, and refuses to run
without an sm_100 GPU (no CPU fallback)."""
import os
import re
import subprocess
import sys

import pytest
import torch

import lbic_b200
from lbic_b200 import _lib
from conftest import ROOT


def _declared():
    src = open(os.path.join(ROOT, "include", "lbic.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lbic_[a-z_0-9]+)\s*\(", src)))


def test_exports_every_declared_symbol():
    L = _lib.lib()
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), f"liblbic_b200.so does not export {n}"
        assert n in _lib.PROTOTYPES, f"python binding lacks a prototype for {n}"
    assert sorted(_lib.PROTOTYPES) == names


def test_option_constants_match_the_header_without_reusing_removed_numbers():
    """Every LBIC_OPT_* of include/lbic.h has the same value in the python binding and a name in set_option(); the
    numbers of removed options (13, 21, 24) are not given to new ones."""
    src = open(os.path.join(ROOT, "include", "lbic.h")).read()
    opts = {k: int(v) for k, v in re.findall(r"#define\s+(LBIC_OPT_[A-Z0-9_]+)\s+(\d+)", src)}
    assert len(opts) >= 18 and len(set(opts.values())) == len(opts), "duplicate option numbers"
    assert not {13, 21, 24} & set(opts.values()), "numbers of removed options are not reused"
    for k, v in opts.items():
        assert getattr(_lib, k, None) == v, f"{k}: header says {v}, _lib.py says {getattr(_lib, k, None)}"


def test_blackwell_instructions_in_sass():
    """The shipped kernels are tcgen05/TMA code, not a legacy mma.sync path."""
    import shutil
    from lbic_b200 import build
    # the cuobjdump of the toolkit that built the library, when it is not on PATH
    tool = shutil.which("cuobjdump") or os.path.join(os.path.dirname(build.NVCC), "cuobjdump")
    sass = subprocess.run([tool, "-sass", _lib.SO_PATH], capture_output=True, text=True, check=True).stdout
    assert "UTCHMMA" in sass and "UTMALDG" in sass and "LDTM" in sass
    assert "HMMA.16816" not in sass


_NO_GPU_CHECK = """
import ctypes
import sys
sys.path.insert(0, %r)
import pytest
import torch
import lbic_b200
from lbic_b200 import _lib
assert not torch.cuda.is_available()
L = _lib.lib()
cfg = _lib.LbicConfig(8, (ctypes.c_int * 4)(3, 1, 1, 1), 768, 96)
h = ctypes.c_void_p()
rc = L.lbic_create(ctypes.byref(cfg), 0, ctypes.byref(h))
assert rc == -5 and b"no CPU fallback" in L.lbic_last_error()
m = lbic_b200.BlockBasedImgCompLossyNetv9(lbic_b200.load_config("B8_lowrate"))
with pytest.raises(RuntimeError):
    m.update(force=True)
with pytest.raises(RuntimeError):
    m.to("cpu")
"""


def test_fails_loudly_without_gpu():
    # in a child process that sees no GPU, so that this also runs on a machine that has one
    out = subprocess.run([sys.executable, "-c", _NO_GPU_CHECK % ROOT], capture_output=True, text=True, timeout=600, cwd=ROOT,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-3000:]


def test_config_loader_reads_reference_json(tmp_path):
    import json
    p = tmp_path / "c.json"
    p.write_text(json.dumps({"block_size": 8, "KS": [3, 1, 1, 1], "N": 768, "M": 96, "net_version": "v9",
                             "mode": "eval_model", "lambda_": [117.045], "seed": 1337}))
    c = lbic_b200.load_config(str(p))
    assert (c.block_size, c.N, c.M, c.KS) == (8, 768, 96, [3, 1, 1, 1]) and c.lambda_ == [117.045]
    with pytest.raises(KeyError):
        lbic_b200.load_config({"block_size": 8})
    with pytest.raises(ValueError):
        lbic_b200.load_config({"block_size": 8, "KS": [5, 1, 1, 1], "N": 768, "M": 96})
    m = lbic_b200.BlockBasedImgCompLossyNetv9(c)
    assert len(m.expected_keys()) == 14 * 3 + 6 * 6
    with pytest.raises(RuntimeError):
        m.load_state_dict({"prtr_forward1.weight": torch.zeros(1)})

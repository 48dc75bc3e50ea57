"""The drop-in boundary exercised FROM THE REFERENCE SIDE (VERDICT r1 item 6).

needs_reference tests import the UNMODIFIED reference agent (agents/blkbsdimgcomp_agent.py) through oracle/ref_shim,
build its own config / checkpoint / PNG folder, and run eval_model (AGENT:560-641):
  * with the stock model on the CPU, against the committed golden log line (the golden generator and this test share
    their code, so the fixture cannot drift from what the reference prints);
  * with the INTEGRATION.md patch applied (`backend: "b200"`): the python block is taken FROM INTEGRATION.md and executed
    inside a subclass of the reference agent.  Without a GPU the B200 model must refuse loudly (no CPU fallback); with
    a GPU (and the reference tree present) eval_model runs through liblbic_b200 and its log line is diffed against
    the stock one.
The GPU box has no reference tree: there tests/test_gpu_parity.py::test_eval_model_matches_reference_log_line compares
the B200 path with the committed golden."""
import json
import os
import re
import sys
import tempfile

import pytest
import torch

from conftest import GOLDEN, ROOT
from oracle.ref_shim import load_reference

sys.path.insert(0, GOLDEN)
pytestmark = pytest.mark.needs_reference

GOLD = os.path.join(GOLDEN, "eval_model_B8_lowrate_208x176.json")


def integration_patch_source():
    """The python block of INTEGRATION.md that a maintainer adds to the agent's __init__."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    m = re.search(r"```python\n# agents/blkbsdimgcomp_agent.py, in __init__ after self.model0 is built.*?\n(.*?)```", text, re.S)
    assert m, "INTEGRATION.md lost its agent patch"
    return m.group(1)


@pytest.fixture(scope="module")
def ref_agent():
    if not load_reference.available():
        pytest.skip("reference tree not present (LBIC_REFERENCE_ROOT)")
    return load_reference.load_agent()


def test_stock_eval_model_reproduces_golden_log_line(ref_agent):
    import make_golden_eval_model as G
    gold = json.load(open(GOLD))
    with tempfile.TemporaryDirectory() as tmp:
        G.prepare_inputs(tmp)
        recs, lines = G.run_eval_model(ref_agent.BlockBasedImgCompLossyAgent, G.reference_config(tmp))
    assert len(recs) == 1
    r, g = recs[0], gold["record"]
    assert r["bytes"] == g["bytes"] and r["bpp"] == g["bpp"] and r["psnr"] == g["psnr"]
    assert (r["enc_dec_mad"], r["enc_dec_max"], r["enc_dec_min"]) == (0.0, 0.0, 0.0)       # AGENT:601-602
    strip = lambda ln: re.sub(r"Enc/DecTime:[\d.]+/[\d.]+ ", "", ln)                       # wall-clock seconds differ
    assert strip([ln for ln in lines if ln.startswith("Image")][0]) == strip(gold["log_line"])


def test_integration_patch_routes_eval_model_into_liblbic(ref_agent):
    import make_golden_eval_model as G
    patch = integration_patch_source()
    Stock = ref_agent.BlockBasedImgCompLossyAgent

    class PatchedAgent(Stock):
        def __init__(self, config):
            super().__init__(config)
            exec(patch, {}, {"self": self})          # the INTEGRATION.md lines, verbatim

    with tempfile.TemporaryDirectory() as tmp:
        G.prepare_inputs(tmp)
        cfg = G.reference_config(tmp, backend="b200")
        if not torch.cuda.is_available():
            # the reference agent now builds the B200 model, which refuses to exist without an sm_100 GPU
            with pytest.raises(RuntimeError, match="no CPU path|no CUDA device|no CPU fallback"):
                PatchedAgent(cfg)
            # and without the config key nothing changes
            agent = PatchedAgent(G.reference_config(tmp))
            assert type(agent.model0).__module__.startswith("graphs.models")
            return
        cfg["cuda"] = True
        recs, lines = G.run_eval_model(PatchedAgent, cfg)
        gold = json.load(open(GOLD))["record"]
        r = recs[0]
        assert abs(r["bytes"] - gold["bytes"]) <= max(8, gold["bytes"] // 1000)          # bpp within 0.1 %
        assert abs(r["psnr"] - gold["psnr"]) <= 0.01
        assert (r["enc_dec_mad"], r["enc_dec_max"], r["enc_dec_min"]) == (0.0, 0.0, 0.0)

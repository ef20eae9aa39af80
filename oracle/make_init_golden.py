"""ORACLE tooling — the state-dict layout and initial values of the REAL reference's Basic2DNet under torch.manual_seed(1) for the
configurations of oracle/interface_configs.py: per entry name, shape, dtype and the SHA-256 of its bytes, plus the named_parameters()
order, to tests/golden/init_state.json. Needs a checkout of the reference (DL4VC_REFERENCE), CPU only, seconds.
TEST INFRASTRUCTURE ONLY.     python oracle/make_init_golden.py"""
from __future__ import annotations

import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim      # noqa: E402
from oracle.interface_configs import CONFIGS      # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "init_state.json")
SEED = 1


def describe(model):
    state = [[k, list(v.shape), str(v.dtype).replace("torch.", ""), hashlib.sha256(v.detach().cpu().contiguous().numpy().tobytes()).hexdigest()]
             for k, v in model.state_dict().items()]
    return {"state": state, "parameters": [n for n, _ in model.named_parameters()]}


def main():
    import torch

    if not ref_shim.reference_available():
        sys.exit(f"no reference checkout at {ref_shim.REFERENCE_ROOT} (set DL4VC_REFERENCE): the golden is recorded from the reference only")
    out = {"source": f"reference dl4vc/model.py ({ref_shim.REFERENCE_ROOT})", "torch": torch.__version__, "seed": SEED, "configs": {}}
    for name in sorted(CONFIGS):
        torch.manual_seed(SEED)
        out["configs"][name] = describe(ref_shim.build_reference_model(CONFIGS[name])[0])
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", OUT)


if __name__ == "__main__":
    main()

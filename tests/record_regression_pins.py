"""Write tests/golden/regression_pins.json: what one implementation gives for the host-side parity checks of
tests/test_host_cpu.py (seeded default init, checkpoints loaded the tools' way, public signatures, host helpers,
model_locked / get_params).  The tests compare with these values only when the reference is not importable.

    python tests/record_regression_pins.py <tree>      # default: controlnet-pytorch_b200/dropin

The tree is put first on sys.path and its `models.*` / `scheduler.*` modules are imported.  The committed file was
recorded from the drop-ins (controlnet-pytorch_b200/dropin) of commit 70d0cc0, because no copy of the reference was at
hand: it is a regression pin of the drop-ins, not reference data.  "_source" and "_torch" in the file say which tree and
which torch version it came from (the default initialisers' bytes depend on the torch version).
"""
import importlib
import json
import os
import sys
import tempfile

import torch

import helpers as H

if __name__ == "__main__":
    src = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else os.path.join(H.ROOT, "controlnet-pytorch_b200", "dropin"))
    sys.path.insert(0, src)
    get = importlib.import_module
    dropin = hasattr(get("models.controlnet"), "__cnb200_real__")
    rel = os.path.relpath(src, H.ROOT)
    pins = {"_source": rel if not rel.startswith("..") else os.path.basename(src),
            "_kind": "drop-in regression pins, not reference data" if dropin else "reference data",
            "_torch": torch.__version__, "init": H.init_digests(get)}
    with tempfile.TemporaryDirectory() as d:
        pins["tool_checkpoints"] = H.write_tool_checkpoints(get, d)[1]
    pins["public_surface"] = H.public_surface(get, reexports=dropin)
    pins["host_helpers"] = H.host_helper_digests(get)
    pins["locked_params"] = {str(locked): H.locked_params(get, locked) for locked in (True, False)}
    with open(H.PINS, "w") as f:
        json.dump(pins, f, indent=1)
        f.write("\n")
    print("wrote", H.PINS, "from", pins["_source"])

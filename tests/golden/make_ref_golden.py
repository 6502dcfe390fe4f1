"""Writes tests/golden/ref_golden.json: what the reference's own code (oracle/_ref, built from the original engine's sources by
`make -C oracle`) returns on the cases of tests/ref_golden.py, and the struct layouts of tests/test_struct_layout_ref.py.

Where a reference library is built its value is recorded and the port (oracle / product) must return the same; where it is not,
the value is only recorded with --from-port, from the port, which the live tests require to equal the reference bit for bit.
The file notes which source each section came from."""
import json
import os
import pathlib
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

import oracle_lib as orc  # noqa: E402
import ref_golden as rg  # noqa: E402
import test_struct_layout_ref as sl  # noqa: E402

from_port = "--from-port" in sys.argv
out = {"source": {}}
for kind, case, libname in rg.cases():
    have = os.path.exists(os.path.join(orc.ORACLE_DIR, "_ref", libname))
    if not have and not from_port:
        sys.exit(f"oracle/_ref/{libname} is not built: build it with `make -C oracle REF=<engine sources>` or pass --from-port")
    mine = rg.port(kind, case)
    if have:
        assert rg.reference(kind, case) == mine, (kind, case)
    out["source"][kind] = f"oracle/_ref/{libname}" if have else "port (equal to the reference wherever the live test ran)"
    out.setdefault(kind, {})[rg.key(*case) if isinstance(case, tuple) else str(case)] = mine

with tempfile.TemporaryDirectory() as td:
    mine = sl.probe(pathlib.Path(td))
    if sl.REF:
        assert sl.probe(pathlib.Path(td), reference=True) == mine
    elif not from_port:
        sys.exit("VQ_REFERENCE is not set: point it at the engine sources or pass --from-port")
out["struct_layout"] = mine
out["source"]["struct_layout"] = ("Shaders/LightingConstantBufferData.h" if sl.REF
                                  else "include/vq_shader_data.h (equal to the reference header wherever the live test ran)")
json.dump(out, open(rg.PATH, "w"), indent=0, sort_keys=True)
print(f"wrote {rg.PATH}: {sum(len(v) for k, v in out.items() if k != 'source')} values")

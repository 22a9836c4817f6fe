"""Writes tests/golden/reference_abi.json: the C ABI of the reference's Sources/MFAFFI/include/mfa_ffi.h as
tests/test_abi_cpu.py sees it (normalised mfa_* prototypes, and what its enum / struct probe prints), so that
include/mfa_ffi.h is checked against the reference without a reference checkout at test time.

The committed file was written from include/mfa_ffi.h at a commit where both header tests passed against the
reference header itself; rerun this on the reference header to refresh it:

    python tests/golden/make_reference_abi.py <reference checkout>/Sources/MFAFFI/include/mfa_ffi.h
"""
import importlib.util
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "reference_abi.json")


def main(header):
    spec = importlib.util.spec_from_file_location("test_abi_cpu", os.path.join(HERE, "..", "test_abi_cpu.py"))
    t = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(t)
    with open(header) as f:
        protos = t._prototypes(f.read())
    with tempfile.TemporaryDirectory() as tmp:
        probe = t.probe_output(header, tmp)
    rows = ",\n".join(f"  {json.dumps(n)}: {json.dumps([r, list(a)])}" for n, (r, a) in sorted(protos.items()))
    with open(OUT, "w") as f:
        f.write('{\n "header": "Sources/MFAFFI/include/mfa_ffi.h",\n "prototypes": {\n' + rows + "\n },\n"
                f' "probe": {json.dumps(probe)}\n}}\n')
    print("wrote", OUT, len(protos), "prototypes")


if __name__ == "__main__":
    main(sys.argv[1])

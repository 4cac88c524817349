"""Generates tests/golden/fmi_golden.json from the REFERENCE ITSELF (oracle/_ref/libseal_ref.so = unmodified
seal/cpp_modules/fm_index.cpp + vendored sdsl-lite, built by `make -C oracle ref`):

    python tests/golden/make_fmi_golden.py

For every text of tests/test_host_logic.py::sdsl_writer_texts, the reference's FMIndex::save writes an .fmi file;
the fixture keeps its length and SHA-256, which the product's writer must reproduce byte for byte.
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle.fm_oracle import RefFM  # noqa: E402
from test_host_logic import sdsl_writer_texts  # noqa: E402


def main():
    files = {}
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ref.fmi")
        for name, text in sdsl_writer_texts().items():
            RefFM(np.asarray(text, dtype=np.uint64)).save(path)
            with open(path, "rb") as f:
                data = f.read()
            files[name] = {"bytes": len(data), "sha256": hashlib.sha256(data).hexdigest()}
    out = os.path.join(HERE, "fmi_golden.json")
    with open(out, "w") as f:
        json.dump({"written_by": "seal/cpp_modules/fm_index.cpp FMIndex::save (sdsl store_to_file)", "files": files}, f,
                  indent=1)
        f.write("\n")
    print("wrote", out, len(files), "files")


if __name__ == "__main__":
    main()

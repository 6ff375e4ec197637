#!/usr/bin/env python
"""Writes tests/golden/reference.json and tests/golden/reference_{zstd,zlib}.npz: what the UNMODIFIED
reference returns for the cases the tests compare against (digests of transcripts, verdicts, chunk
sizes and headers, exported symbols) and the zstd frames / zlib and zstd chunks it writes.

Needs the reference build in oracle/_ref (`make -C oracle ref REF=<reference checkout>`) and the
reference's blosc/blosc.h:

    python scripts/record_reference_golden.py <reference checkout>
"""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import datagen  # noqa: E402
import test_abi  # noqa: E402
import test_decoder_edges  # noqa: E402
import test_fast_parse  # noqa: E402
import test_hostile_input  # noqa: E402
import test_oracle_vs_ref  # noqa: E402
import test_zlib_decode  # noqa: E402
import test_zstd_decode  # noqa: E402


def load(path, names):
    lib = C.CDLL(path)
    for f in names:
        getattr(lib, f).restype = C.c_int
    return lib


def main():
    ref_path = os.path.join(ROOT, "oracle", "_ref", "libblosc_ref.so")
    ref = load(ref_path, ("blosc_compress_ctx", "blosc_decompress_ctx", "blosc_getitem", "LZ4_compress_fast",
                          "LZ4_decompress_safe", "blosclz_compress", "blosclz_decompress"))
    orc = load(os.path.join(ROOT, "oracle", "liboracle.so"), ("orc_compress_ctx", "orc_decompress_ctx", "orc_getitem",
                                                               "orc_lz4_compress_fast", "orc_lz4_decompress_safe"))
    for name, mod in (("zstd", test_zstd_decode), ("zlib", test_zlib_decode)):
        np.savez_compressed(os.path.join(datagen.GOLDEN, f"reference_{name}.npz"), **mod.reference_golden(ref, orc))
    datagen.golden_arrays.cache_clear()

    out = {"transcripts": {}}
    for part in (test_oracle_vs_ref.reference_golden(ref, orc), test_hostile_input.reference_golden(ref, orc),
                 test_fast_parse.reference_golden(ref, orc), test_decoder_edges.reference_golden(ref, orc),
                 test_zstd_decode.reference_verdicts(ref, orc),
                 test_abi.reference_golden(ref_path, os.path.join(sys.argv[1], "blosc", "blosc.h"))):
        out["transcripts"].update(part.pop("transcripts", {}))
        out.update(part)
    with open(os.path.join(datagen.GOLDEN, "reference.json"), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()

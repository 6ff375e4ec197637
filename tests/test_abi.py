"""The C-ABI shared library loads (no GPU needed for that) and exports every symbol that
include/blosc_b200.h declares; the 25 public symbols of the reference's libblosc.so.1
(SURVEY.md section 8b) that belong to the hot path and its front end are all there."""
import ctypes as C
import os
import re

from datagen import golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_exports_match_header(pkg):
    hdr = open(os.path.join(ROOT, "include", "blosc_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(blosc_[a-z0-9_]+)\s*\(", hdr))
    assert {"blosc_compress_ctx", "blosc_decompress_ctx", "blosc_getitem"} <= names
    lib = C.CDLL(pkg.LIB_PATH)
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing


def _dynamic_symbols(path):
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    return {l.split()[-1] for l in out.splitlines() if len(l.split()) >= 3 and l.split()[-2] in ("T", "t", "W")}


def test_reference_public_symbols_present(pkg):
    """Every public blosc_* symbol of the reference is exported here.  The list SURVEY.md section 8b recorded is checked
    against the reference's own header (BLOSC_EXPORT declarations) and against `nm -D` of the reference build, both
    stored in tests/golden/reference.json."""
    ref_syms = """blosc_init blosc_destroy blosc_compress blosc_compress_ctx blosc_decompress blosc_decompress_ctx
    blosc_getitem blosc_get_nthreads blosc_set_nthreads blosc_get_compressor blosc_set_compressor
    blosc_compcode_to_compname blosc_compname_to_compcode blosc_list_compressors blosc_get_version_string
    blosc_get_complib_info blosc_free_resources blosc_cbuffer_sizes blosc_cbuffer_validate blosc_cbuffer_metainfo
    blosc_cbuffer_versions blosc_cbuffer_complib blosc_get_blocksize blosc_set_blocksize blosc_set_splitmode""".split()
    assert len(ref_syms) == 25
    # the public API is what blosc.h marks BLOSC_EXPORT (everything else is hidden by -fvisibility=hidden,
    # blosc/CMakeLists.txt:6-8): the recorded list must be exactly that
    public = set(golden()["abi"]["header_exports"])
    assert public == set(ref_syms), (sorted(public - set(ref_syms)), sorted(set(ref_syms) - public))
    # ... and each of them is a symbol the reference build really defines (it is built without the visibility flag,
    # so it exports some internals on top: those are not part of the contract)
    defined = set(golden()["abi"]["defined"])
    assert set(ref_syms) <= defined, sorted(set(ref_syms) - defined)
    ours = _dynamic_symbols(pkg.LIB_PATH)
    missing = [s for s in ref_syms if s not in ours]
    assert not missing, missing


def test_host_only_entry_points(pkg):
    """Header readers and name tables run without a device."""
    import numpy as np
    lib = pkg.lib
    chunk = np.frombuffer(bytes.fromhex("02012104" "00001000" "00000800" "90220000"), np.uint8).copy()
    nb, cb, bs = C.c_size_t(), C.c_size_t(), C.c_size_t()
    lib.blosc_cbuffer_sizes(chunk.ctypes.data_as(C.c_void_p), C.byref(nb), C.byref(cb), C.byref(bs))
    assert (nb.value, cb.value, bs.value) == (1 << 20, 8848, 524288)
    lib.blosc_compname_to_compcode.argtypes = [C.c_char_p]
    assert lib.blosc_compname_to_compcode(b"lz4") == 1 and lib.blosc_compname_to_compcode(b"blosclz") == 0
    assert lib.blosc_compname_to_compcode(b"zstd") == -1
    lib.blosc_cbuffer_complib.restype = C.c_char_p
    assert lib.blosc_cbuffer_complib(chunk.ctypes.data_as(C.c_void_p)) == b"LZ4"
    lib.blosc_list_compressors.restype = C.c_char_p
    assert lib.blosc_list_compressors() == b"blosclz,lz4,lz4hc"
    assert lib.blosc_compname_to_compcode(b"lz4hc") == 2


def test_product_does_not_touch_the_oracle():
    """The product path must never import, link or execute anything under oracle/ or tests/."""
    bad = []
    for dirpath, _, files in os.walk(os.path.join(ROOT, "c-blosc_b200")):
        for f in files:
            if f.endswith((".c", ".cu", ".cuh", ".h", ".py")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                for line in txt.splitlines():
                    if re.search(r"#\s*include.*(oracle|simt_emu)|import.*oracle|liboracle|libblosc_ref|orc_[a-z]", line):
                        bad.append((f, line.strip()))
    assert not bad, bad


def reference_golden(ref_path, header_path):
    hdr = re.sub(r"/\*.*?\*/", "", open(header_path).read(), flags=re.S)
    public = sorted(set(re.findall(r"BLOSC_EXPORT[^;(]*?\b(blosc_[a-z0-9_]+)\s*\(", hdr)))
    defined = sorted(s for s in _dynamic_symbols(ref_path) if s.startswith("blosc_"))
    return {"abi": {"header_exports": public, "defined": defined}}

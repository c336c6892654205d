"""The drop-in boundary: libpumitally.so must load without a GPU, export every
symbol include/pumitally_c.h declares, and export the Itanium-mangled members
of pumitally::PumiTally exactly as the reference header declares them
(reference: src/pumitally/PumiTally.h:34-107)."""
import ctypes
import json
import os
import re
import subprocess

import pytest

from helpers import ROOT
from pumiumtally_b200 import build as pbuild
from pumiumtally_b200 import tally

REF_MANGLED = [
    "_ZN9pumitally9PumiTallyC1ERKNSt7__cxx1112basic_stringIcSt11char_traitsIcESaIcEEEiRiRPPc",
    "_ZN9pumitally9PumiTallyC2ERKNSt7__cxx1112basic_stringIcSt11char_traitsIcESaIcEEEiRiRPPc",
    "_ZN9pumitally9PumiTallyD1Ev",
    "_ZN9pumitally9PumiTallyD2Ev",
    "_ZNK9pumitally9PumiTally19CopyInitialPositionEPdi",
    "_ZNK9pumitally9PumiTally18MoveToNextLocationEPdS1_PaS1_i",
    "_ZNK9pumitally9PumiTally17WriteTallyResultsEv",
]


@pytest.fixture(scope="module")
def lib_path():
    return pbuild.build_library()


def _exported(lib_path):
    out = subprocess.check_output(["nm", "-D", "--defined-only", lib_path], text=True)
    return {line.split()[-1] for line in out.splitlines() if line.strip()}


def test_c_abi_symbols_declared_and_exported(lib_path):
    hdr = open(os.path.join(ROOT, "include", "pumitally_c.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(pumitally_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    exported = _exported(lib_path)
    missing = declared - exported
    assert not missing, f"declared in pumitally_c.h but not exported: {sorted(missing)}"
    # the Python binding table must cover the header too
    assert declared == set(tally.C_API), declared ^ set(tally.C_API)


def test_library_loads_without_gpu(lib_path):
    L = tally.load_library()
    assert b"sm_100a" in L.pumitally_version()


def test_cxx_class_abi_matches_reference(lib_path):
    exported = _exported(lib_path)
    for sym in REF_MANGLED:
        assert sym in exported, sym


def test_facade_header_is_layout_compatible(tmp_path, lib_path):
    """A TU compiled against our header needs exactly the reference's symbols and
    sees sizeof(PumiTally) == sizeof(void*)."""
    src = tmp_path / "use.cpp"
    src.write_text(
        '#include "pumitally/PumiTally.h"\n'
        "static_assert(sizeof(pumitally::PumiTally) == sizeof(void*), \"pimpl only\");\n"
        "int run(int argc, char** argv, double* a, double* b, signed char* f, double* w) {\n"
        "  pumitally::PumiTally t(\"box:1,1,1\", 5, argc, argv);\n"
        "  t.CopyInitialPosition(a, 15); t.MoveToNextLocation(a, b, f, w, 15); t.WriteTallyResults();\n"
        "  return 0; }\n")
    obj = tmp_path / "use.o"
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-c", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(obj)])
    und = subprocess.check_output(["nm", "-u", str(obj)], text=True)
    needed = {l.split()[-1] for l in und.splitlines() if "pumitally" in l}
    assert needed == {s for s in REF_MANGLED if "C2" not in s and "D2" not in s}, needed
    # the same TU compiled against the reference header needs exactly these symbols
    with open(os.path.join(ROOT, "tests", "golden", "reference_facade_symbols.json")) as f:
        assert needed == set(json.load(f)["undefined"])


def test_no_gpu_means_loud_failure(lib_path):
    """There is no CPU fallback: without a device the constructor fails."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        tally.PumiTally("box:1,1,1", 5)

"""Record tests/golden/reference.npz: the reference's answers for the inputs of the tests that pin this project to it.

Needs a checkout of the reference (intel/neural-speed): its code is compiled into oracle/_ref by oracle/Makefile, and its
converter's common.py and core/ne.h are read from it.  Runs those tests with oracle/golden.py recording: every answer comes
from the reference itself and is still compared, so the fixture is written only when the tests pass against the live reference.

    python tests/golden/make_golden_reference.py <neural-speed checkout>
"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import golden  # noqa: E402

TESTS = [
    "tests/test_oracle_vs_ref.py",
    "tests/test_lowbit_cpu.py::test_planes_and_integers_against_the_reference_kernels",
    "tests/test_lowbit_cpu.py::test_f4_codebooks_against_the_reference_kernels",
    "tests/test_abi_cpu.py::test_oracle_blob_layout_against_reference_kernels",
    "tests/test_moe_cpu.py::test_restatement_matches_the_reference_engine",
    "tests/test_ne_abi_cpu.py::test_layout_matches_the_reference_header",
    "tests/test_ne_loader_cpu.py::test_parse_ne_llama_file_with_btla_blobs",
]


def main():
    src = os.path.abspath(sys.argv[1])
    assert os.path.isdir(os.path.join(src, "neural_speed")), f"{src} is not a neural-speed checkout"
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "-s", f"REF={src}", "liboracle.so", "_ref/libref_ggml.so",
                    "_ref/libref_btla.so", "_ref/libref_ne.so"], check=True)
    golden.start_recording(src)
    rc = pytest.main(["-q", "-p", "no:cacheprovider", "--rootdir", ROOT] + [os.path.join(ROOT, t) for t in TESTS])
    assert rc == 0, "the tests fail against the live reference: nothing written"
    print("wrote", golden.save_recording(), "answers to", golden.PATH)


if __name__ == "__main__":
    main()

"""Regenerate rise_sdf_b200/csrc/mcubes_table.cuh from the face-walk generator in oracle/mcubes.py.

    python scripts/gen_mcubes_table.py

The header is committed so that the library build never imports the oracle package;
tests/test_oracle_mcubes.py checks that the committed file equals this script's output.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import mcubes  # noqa: E402

if __name__ == "__main__":
    with open(mcubes.HEADER, "w") as f:
        f.write(mcubes.header_text())
    print("wrote", mcubes.HEADER)

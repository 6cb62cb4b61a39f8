#!/usr/bin/env python3
"""Store the reports of nvCOMP's own benchmark and example programs in reference_harness.json.

Needs a GPU and the programs built into oracle/_ref/ (NVCOMP_REFERENCE_DIR=<nvCOMP tree> during build(), or
oracle/build_reference_harness.sh <nvCOMP tree>).  Runs every program with the arguments and data files
tests/test_reference_harness_gpu.py uses and keeps the deterministic part of each report (exit status, byte counts,
validation lines); the tests replay the same workloads against it.
Run from the repo root: python tests/golden/make_reference_reports.py
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from test_reference_harness_gpu import GOLDEN, RUNS, parse_report, run_program, write_data_files  # noqa: E402


def main():
    files = write_data_files(tempfile.mkdtemp())
    reports = {}
    for key in RUNS:
        rc, out, _ = run_program(key, files)
        reports[key] = parse_report(rc, out)
        print(key, reports[key], flush=True)
    json.dump(reports, open(GOLDEN, "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()

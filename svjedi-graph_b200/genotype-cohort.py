#!/usr/bin/env python3
"""Cohort genotyping (not in the reference): one SV catalogue, many samples' GAF files, one multi-sample VCF whose
column s is what filter-alignments.py + predict-genotype.py write for sample s alone (svjg/cli.py: cohort_main)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from svjg import cli  # noqa: E402

if __name__ == "__main__":
    cli.leave(cli.cohort_main())

"""Generate tests/golden/live_twins.npz: the stored values behind the reference-free twins of four live reference comparisons.

    python oracle/make_twin_golden.py

Four tests compare novic_b200 with the unmodified reference live and need its source tree, which this repository does not include:
tests/test_stats.py::test_stats_match_reference_generation_task, tests/test_targets.py::test_random_vocabularies_match_the_reference_embedder,
tests/test_cache.py::test_header_struct_and_offsets_match_the_reference and tests/test_abi_and_host.py::test_drop_in_through_the_reference_loader.
Each runs on fixed, seeded inputs and asserts that novic_b200's values equal the reference's.  This script stores novic_b200's values
on those inputs, computed by the same functions the twins call (stats_values, random_vocabulary_values, header_values,
state_dict_values).  The code involved (novic_b200/stats.py, targets.py, cache.py, the decoder's state dict and get_num_params) passed
those live comparisons and computes the same values since, so the stored values are the ones the reference gave.  When one of
those modules changes on purpose, run the live tests against a reference tree (NOVIC_REFERENCE_ROOT) first and only then
regenerate this file.
TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import test_abi_and_host, test_cache, test_stats, test_targets  # noqa: E402
from tests.golden_util import TWINS_PATH  # noqa: E402


def main():
    out = {}
    for use_classes in (False, True):
        out.update({f"stats__{int(use_classes)}__{k}": v for k, v in test_stats.stats_values(use_classes).items()})
    out.update({f"rand__{k}": v for k, v in test_targets.random_vocabulary_values().items()})
    out.update({f"cache__{k}": v for k, v in test_cache.header_values().items()})
    out.update({f"sd__{k}": v for k, v in test_abi_and_host.state_dict_values().items()})
    np.savez_compressed(TWINS_PATH, **out)
    print(f"{len(out)} arrays, {os.path.getsize(TWINS_PATH)} bytes -> {TWINS_PATH}")


if __name__ == "__main__":
    main()

"""CPU-side checks of the drop-in boundary: the library builds for sm_100a, loads, exports every
symbol include/plaid_b200.h declares, and fails loudly (no fallback) without a device."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def npb():
    import next_plaid_b200 as m
    m.build_library()
    return m


def test_header_symbols_all_exported(npb):
    hdr = open(os.path.join(ROOT, "include", "plaid_b200.h")).read()
    declared = set(re.findall(r"PB_API\s+[\w\s\*]+?\b(pb_\w+)\s*\(", hdr))
    assert declared, "no PB_API declarations parsed"
    L = npb.load_library()
    missing = [s for s in sorted(declared) if not hasattr(L, s)]
    assert not missing, missing
    assert declared == set(npb.EXPORTS), declared ^ set(npb.EXPORTS)


def test_library_targets_sm100a_only(npb):
    import subprocess
    from importlib import import_module
    cuobjdump = import_module("next_plaid_b200.build").cuda_tool("cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", npb.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert not re.search(r"sm_(?!100a)\d+", out), out


def test_default_params_match_reference(npb):
    # search.rs:58-69
    import ctypes as C
    from importlib import import_module
    idx = import_module("next_plaid_b200.index")
    p = idx._Params()
    npb.load_library().pb_search_params_default(C.byref(p))
    assert (p.batch_size, p.n_full_scores, p.top_k, p.n_ivf_probe, p.centroid_batch_size) == \
        (2000, 4096, 10, 8, 100000)
    assert p.has_centroid_score_threshold == 1 and abs(p.centroid_score_threshold - 0.4) < 1e-7
    d = npb.SearchParameters()
    assert (d.batch_size, d.n_full_scores, d.top_k, d.n_ivf_probe) == (2000, 4096, 10, 8)


def test_no_cpu_fallback_without_device(npb):
    if npb.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(npb.PlaidError) as e:
        npb.MmapIndex.from_arrays(np.zeros((4, 32), np.float32), np.zeros(16, np.float32),
                                  np.zeros(2, np.int64), np.zeros((2, 16), np.uint8),
                                  np.array([2], np.int64), np.zeros(1, np.int64),
                                  np.array([1, 0, 0, 0], np.int32), 4)
    assert e.value.status == 2 and "no CPU fallback" in str(e.value)
    with pytest.raises(npb.PlaidError):
        npb.maxsim_scores(np.zeros((2, 32), np.float32), [np.zeros((3, 32), np.float32)])


def test_argument_validation_precedes_device_use(npb):
    # nbits must divide 8 (codec.rs:161-166) -> PB_ERR_INVALID even without a GPU
    with pytest.raises(npb.PlaidError) as e:
        npb.MmapIndex.from_arrays(np.zeros((4, 32), np.float32), np.zeros(8, np.float32),
                                  np.zeros(2, np.int64), np.zeros((2, 12), np.uint8),
                                  np.array([2], np.int64), np.zeros(1, np.int64),
                                  np.array([1, 0, 0, 0], np.int32), 3)
    assert e.value.status == 1 and "divisor of 8" in str(e.value)


def test_load_reports_missing_directory(npb, tmp_path):
    with pytest.raises(npb.PlaidError) as e:
        npb.MmapIndex.load(str(tmp_path / "nope"))
    assert e.value.status == 3


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "next-plaid_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dp, f)).read()
                # comments may cite the oracle's pinned order; code may not import, include or dlopen it
                assert not re.search(r"^\s*(import|from)\s+oracle", txt, re.M), f
                assert "libplaid_oracle" not in txt and not re.search(r"#include\s+.*oracle", txt), f


def test_build_sizing_rules_match_the_reference_formulas(npb=None):
    # kmeans.rs:273-312 and index.rs:195-212 are pure arithmetic: no device needed
    import next_plaid_b200 as m
    from oracle import oracle
    for D, avg in ((10_000, 64.0), (1_000_000, 300.0), (123, 17.5), (1, 5.0)):
        n_docs = min(int(1.0 + 16.0 * np.sqrt(120.0 * D)), D)
        s = m.kmeans_sizing(D, avg, 10 ** 12, int(D * avg))
        assert s["kmeans_sample_docs"] == n_docs
        assert s["num_partitions"] == oracle.num_partitions_heuristic(D, [avg] * 4)
        assert s["codec_sample_docs"] == max(min(int(16.0 * np.sqrt(120.0 * D)), D), 1)
        assert s["heldout_tokens"] == int(min(0.05 * int(D * avg), 50000.0))
    assert m.kmeans_sizing(10_000, 64.0, 100, 640_000)["num_partitions"] == 100      # capped at the sampled tokens

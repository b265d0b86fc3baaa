"""Pins the oracle and the host-side mirrors against the reference's OWN code: tests/golden/reference_blocks.npz holds what
the reference's classes returned on the seeded inputs of oracle/make_golden.py (`python oracle/make_golden.py
--reference-blocks`, run where the reference tree is present); here the same inputs go through this project's classes."""
import os

import numpy as np
import pytest

from oracle import make_golden as mg

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_blocks.npz")


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLD)


def test_oracle_clustering_equals_reference_class(ref):
    from oracle.clustering import OracleClustering

    got = mg.clustering_trace(OracleClustering, lambda clu, s, e: clu(s, e)[1])
    n = len(mg.CLASS_CONFIGS) * mg.CLASS_CHUNKS
    for key in ("cluster_out", "cluster_centers", "cluster_active"):
        assert len(got[key]) == len(ref[key]) == n, key
        differ = np.flatnonzero((got[key] != ref[key]).reshape(n, -1).any(axis=1))
        assert differ.size == 0, (f"{key}: first difference in config {differ[0] // mg.CLASS_CHUNKS}, "
                                  f"chunk {differ[0] % mg.CLASS_CHUNKS}")


def test_post_path_blocks_equal_reference(ref):
    """Binarize and DelayedAggregation (host-side 'next' rows) against the reference implementations"""
    from diart_b200 import blocks

    got = mg.aggregation_outputs(blocks.DelayedAggregation, blocks.Binarize)
    assert sorted(got) == sorted(k for k in ref.files if k.startswith("agg_")) and len(got) == 32
    for key, value in got.items():
        if key.endswith("_data"):
            np.testing.assert_allclose(value, ref[key], rtol=1e-12, err_msg=key)
        elif key.endswith("_window"):
            assert np.abs(value - ref[key]).max() < 1e-12, key
        else:
            assert value == ref[key], key
    n_buf = {"0.5": 1, "2": 4, "5": 10}
    for key in got:
        if key.startswith("agg_hamming_loose_") and key.endswith("_num_windows"):
            assert got[key] == n_buf[key.split("_")[3]]


def test_formatter_equals_reference(ref):
    from diart_b200.features import TemporalFeatureFormatter

    got = mg.formatter_outputs(TemporalFeatureFormatter)
    assert got["formatter_cast"].dtype == ref["formatter_cast"].dtype
    assert np.array_equal(got["formatter_cast"], ref["formatter_cast"])
    assert np.array_equal(got["formatter_restored_window"], ref["formatter_restored_window"])


def test_preprocessing_blocks_equal_reference(ref):
    """Resample and AdjustVolume (optional pre-processing next to the path) against the reference implementations"""
    from diart_b200 import blocks

    got = mg.preprocessing_outputs(blocks.AdjustVolume, blocks.Resample)
    assert sorted(got) == sorted(k for k in ref.files if k.startswith(("volume_", "resample_"))) and len(got) == 13
    assert got["resample_up_shape"].tolist() == [16000, 1]
    assert np.array_equal(got["resample_up_window"], ref["resample_up_window"])
    for key, value in got.items():
        if key.endswith("_shape"):
            assert np.array_equal(value, ref[key]), key
        elif key.startswith("volume_"):
            np.testing.assert_allclose(value, ref[key], rtol=1e-6, err_msg=key)
        elif key.endswith("_sample"):
            np.testing.assert_allclose(value, ref[key], rtol=1e-6, atol=1e-7, err_msg=key)

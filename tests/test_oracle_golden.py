"""Pins the oracle (oracle/snn_oracle.c) against the LIVE reference: every fixture under
tests/golden/ was produced by running the original package itself (gen_golden.py).  CPU only."""
import numpy as np
import pytest

import cases
import helpers

SMALL = [c for c in cases.CASES if c not in ("dc2015_c2", "dc2015_metric_t40")]


@pytest.mark.parametrize("name", SMALL)
def test_oracle_matches_reference(name):
    fx, state, counts = helpers.run_case_oracle(name)
    helpers.assert_close_to_golden(fx, state, counts)


@pytest.mark.parametrize("name", ["c1_lif_postpre", "lif_postpre_batch", "lif_wdep", "lif_clamps", "dc2015_onespike", "dc2015v2"])
def test_oracle_dense_equals_sparse(name):
    """The costed dense restatement (zeros multiplied like the reference does) and the
    zero-skipping fast mode are bit-identical."""
    _, s_sparse, c_sparse = helpers.run_case_oracle(name, dense=0)
    _, s_dense, c_dense = helpers.run_case_oracle(name, dense=1)
    helpers.assert_bit_identical(s_sparse, s_dense, name)
    helpers.assert_bit_identical(c_sparse, c_dense, name)


@pytest.mark.parametrize("name", ["dc2015_c2", "dc2015_metric_t40"])
def test_oracle_matches_reference_baseline_configs(name):
    """BASELINE.json config 2 (n=400, B=32, T=250) and the metric configuration (n=1600, B=128;
    the live reference needs ~2 s per step there, so the fixture stops at T=40)."""
    fx, state, counts = helpers.run_case_oracle(name)
    helpers.assert_close_to_golden(fx, state, counts)

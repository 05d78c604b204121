"""Retrieval-metric restatements of the oracle against the reference's own numpy code (utils/mAP.py, utils/nDCG.py) and
its one known-answer test (utils/nDCG.py:154-181).

tests/golden/retrieval_metrics.json holds the values the comparison with the reference looks at (_metric_values): they
were recorded from the oracle, are compared with it everywhere, and are themselves compared with the original project's
code by the live test whenever $HH_REFERENCE_ROOT names a checkout of it."""
import importlib
import json
import os
import sys

import numpy as np
import pytest

from oracle import hh_oracle as O
from oracle import ref_import

from oracle.golden_cases import KNOWN_K, KNOWN_NDCG, KNOWN_REL, KNOWN_SIM, synth_retrieval  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "retrieval_metrics.json")


def _metric_values(calculate_mAP, calculate_nDCG):
    """{"N_M_seed": [mAP, nDCG, mAP of the transposed problem]} of three synthetic retrieval problems, float64."""
    out = {}
    for N, M, seed in [(5, 7, 0), (40, 300, 1), (16, 2000, 2)]:
        sim, rel = synth_retrieval(N, M, seed)
        out["%d_%d_%d" % (N, M, seed)] = [float(calculate_mAP(sim, rel)), float(calculate_nDCG(sim, rel)),
                                          float(calculate_mAP(sim.T.copy(), rel.T.copy()))]
    return out


def _oracle_values():
    return _metric_values(lambda s, r: O.calculate_mAP(s, r)[0], lambda s, r: O.calculate_nDCG(s, r)[0])


def test_known_answer():
    assert (O.calculate_k_counts(KNOWN_REL) == KNOWN_K).all()
    assert O.calculate_nDCG(KNOWN_SIM, KNOWN_REL, KNOWN_K)[0] == KNOWN_NDCG


def test_against_stored_reference_values():
    with open(GOLDEN) as f:
        assert _oracle_values() == json.load(f)


@pytest.mark.skipif(not ref_import.reference_available(), reason="needs a checkout of the original project (HH_REFERENCE_ROOT)")
def test_against_live_reference():
    if ref_import.REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, ref_import.REFERENCE_ROOT)
    ref_map = importlib.import_module("utils.mAP")
    ref_ndcg = importlib.import_module("utils.nDCG")
    want = _metric_values(ref_map.calculate_mAP, ref_ndcg.calculate_nDCG)
    assert _oracle_values() == want
    with open(GOLDEN) as f:
        assert json.load(f) == want

"""The oracle (oracle/hh_oracle.py) against the reference's outputs.

* everywhere: against the committed fixtures in tests/golden/ (made by oracle/make_golden.py from the
  unmodified reference);
* where $HH_REFERENCE_ROOT names a checkout of the original project: against the live reference as well.
"""
import os

import pytest
import torch

from oracle import golden_cases as gc
from oracle import ref_import

TOL = 1e-5   # fp32 CPU vs fp32 CPU, different op order (masked dense attention vs rearrange/cat)


def _compare(ref, mine, name):
    for k, v in ref.items():
        if isinstance(v, torch.Tensor) and not v.dtype.is_floating_point:
            assert torch.equal(mine[k], v), (name, k)           # indices / masks: exact
        elif isinstance(v, torch.Tensor):
            assert mine[k].shape == v.shape, (name, k)
            err = (mine[k] - v).abs().max().item()
            assert err <= TOL * max(1.0, v.abs().max().item()), (name, k, err)
        else:
            for kk in v:
                assert abs(v[kk] - mine[k][kk]) < 1e-4, (name, k, kk)


@pytest.mark.parametrize("name", sorted(gc.CASES))
def test_oracle_matches_golden_fixture(name):
    path = os.path.join(gc.GOLDEN_DIR, name + ".pt")
    ref = torch.load(path)
    _compare(ref, gc.run_oracle(gc.CASES[name]), name)


@pytest.mark.skipif(not ref_import.reference_available(), reason="needs a checkout of the original project (HH_REFERENCE_ROOT)")
@pytest.mark.parametrize("name", ["enc_tiny", "enc_l14", "enc_l14_t16", "dec_tiny_traj", "dec_tiny_notraj", "dec_train_dropout", "boxes", "score", "losses"])
def test_fixture_is_what_the_live_reference_says(name):
    from oracle import make_golden
    live = make_golden.run_reference(gc.CASES[name])
    ref = torch.load(os.path.join(gc.GOLDEN_DIR, name + ".pt"))
    for k, v in ref.items():
        if isinstance(v, torch.Tensor) and not v.dtype.is_floating_point:
            assert torch.equal(live[k], v), (name, k)
        elif isinstance(v, torch.Tensor):
            assert torch.allclose(live[k], v, atol=1e-6, rtol=1e-6), (name, k)


def test_group_mask_semantics():
    """CLS sees all, patches see CLS + own group (model/LaviLa.py:255-270)."""
    from oracle import hh_oracle as O
    m = O._group_mask(T=3, n=4, mode="time")
    assert m[0].all() and m[:, 0].all()
    # token (f=1,p=2) -> index 1+1*4+2 = 7 ; same p across frames: 3, 7, 11
    assert m[7].nonzero().flatten().tolist() == [0, 3, 7, 11]
    s = O._group_mask(T=3, n=4, mode="space")
    assert s[7].nonzero().flatten().tolist() == [0, 5, 6, 7, 8]


def test_grouped_and_masked_attention_statements_agree():
    """The oracle's O(N(n+T)) grouped attention equals its masked dense second statement."""
    from oracle import hh_oracle as O
    g = torch.Generator().manual_seed(3)
    for (B, T, n, H) in [(2, 3, 5, 2), (1, 4, 16, 3), (1, 1, 7, 1)]:
        D = H * 64
        z = torch.randn(B, 1 + T * n, D, generator=g)
        wq = torch.randn(3 * D, D, generator=g) / D ** 0.5
        bq = torch.randn(3 * D, generator=g) * 0.1
        wp = torch.randn(D, D, generator=g) / D ** 0.5
        bp = torch.randn(D, generator=g) * 0.1
        for mode in ("time", "space"):
            a = O.var_attention(z, wq, bq, wp, bp, H, T, n, mode)
            b = O.var_attention_masked(z, wq, bq, wp, bp, H, T, n, mode)
            assert torch.allclose(a, b, atol=2e-5), (B, T, n, H, mode, (a - b).abs().max())

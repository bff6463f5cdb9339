"""CPU: pin the data-layer restatements (oracle/data_oracle.py, oracle/stft_oracle.stft_transform, and the closed-form
prior the product's synthetic batches use) against outputs of the reference's own functions (fixtures written by
tests/make_golden.py) and against scipy's beta-binomial."""
import os

import numpy as np
import torch

from conftest import GOLDEN
from oracle import data_oracle as D
from flowtron_b200 import synth
from oracle import stft_oracle as S


def _load(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def test_closed_form_prior_equals_scipy_loop():
    for P, M, s in [(7, 13, 1.0), (40, 200, 1.0), (23, 61, 0.5), (1, 5, 1.0)]:
        a = synth.beta_binomial_prior(P, M, s)
        b = D.beta_binomial_prior_distribution(P, M, s).numpy()
        assert a.shape == b.shape == (M, P)
        assert np.abs(a - b).max() <= 1e-12 + 1e-9 * np.abs(b).max()


def test_data_oracle_matches_reference_data_py():
    gold = _load("data_collate.npz")
    p_ref = torch.from_numpy(gold["prior_11_29"])
    assert torch.equal(p_ref, D.beta_binomial_prior_distribution(11, 29, 1.0))
    batch = [tuple(torch.from_numpy(gold[f"in_{k}_{i}"]) for k in ("mel", "speaker", "text", "prior")) for i in range(4)]
    ref = [torch.from_numpy(gold[f"collate_{i}"]) for i in range(7)]
    mine = D.collate(batch, 1, use_attn_prior=True)
    assert len(mine) == len(ref)
    for a, b in zip(ref, mine):
        assert a.shape == b.shape and torch.equal(a.float(), b.float())


def test_stft_transform_oracle_matches_reference():
    gold = _load("stft_transform.npz")
    m_ref, p_ref = torch.from_numpy(gold["magnitude"]), torch.from_numpy(gold["phase"])
    m, p = S.stft_transform(torch.from_numpy(gold["y"]))
    assert torch.allclose(m, m_ref, atol=1e-6) and torch.allclose(p, p_ref, atol=1e-6)


def test_forced_alignment_branch_matches_reference_ar_step_infer():
    """AR_Step.infer / AR_Back_Step.infer with `attns` given (flowtron.py:585-588, 797): oracle vs the reference modules.
    (Flowtron.infer itself cannot be driven with attns in the reference: `reversed(attns)[i]` at :924 raises.)"""
    from oracle import flowtron_oracle as O
    gold = _load("ar_step_forced_attns.npz")
    cfg = dict(synth.DEFAULT_MODEL_CONFIG, n_flows=2, use_gate_layer=False)
    params = synth.synth_params(cfg, int(gold["seed"]))
    residual, enc, attns = (torch.from_numpy(gold[k]) for k in ("residual", "enc", "attns"))
    r0, r1 = torch.from_numpy(gold["flow0"]), torch.from_numpy(gold["flow1"])
    with torch.no_grad():
        o0, _ = O.ar_step_infer(params, O.flow_prefix(0), residual, enc, attns=attns)
        o1, _ = O.ar_back_step_infer(params, "flows.1", residual, enc, attns=attns)
    assert (r0 - o0).abs().max().item() <= 1e-5 * r0.abs().max().item()
    assert (r1 - o1).abs().max().item() <= 1e-5 * r1.abs().max().item()

"""CPU restatement of the reference's data-layer pieces that sit next to the hot path (TEST INFRASTRUCTURE):
beta_binomial_prior_distribution (data.py:31-41) and DataCollate.__call__ (data.py:197-246).  Pinned against the
reference's own outputs (tests/golden/data_collate.npz, written by tests/make_golden.py) in tests/test_oracle_data.py."""
from __future__ import annotations

import numpy as np
import torch


def beta_binomial_prior_distribution(phoneme_count, mel_count, scaling_factor=1.0):
    """data.py:31-41, literally: one scipy.stats.betabinom pmf per mel frame.  float64 [mel_count, phoneme_count]."""
    from scipy.stats import betabinom
    P, M = phoneme_count, mel_count
    x = np.arange(0, P)
    rows = []
    for i in range(1, M + 1):
        a, b = scaling_factor * i, scaling_factor * (M + 1 - i)
        rows.append(betabinom(P - 1, a, b).pmf(x))
    return torch.tensor(np.array(rows))


def collate(batch, n_frames_per_step=1, use_attn_prior=False):
    """data.py:197-246.  batch: list of (mel [n_mel,F], speaker_id tensor/int, text 1-D long, attn_prior [F,P] or None)."""
    input_lengths, ids = torch.sort(torch.LongTensor([len(x[2]) for x in batch]), dim=0, descending=True)
    max_input_len = int(input_lengths[0])
    text_padded = torch.zeros(len(batch), max_input_len, dtype=torch.long)
    for i in range(len(ids)):
        t = batch[ids[i]][2]
        text_padded[i, :t.size(0)] = t
    n_mel = batch[0][0].size(0)
    max_target_len = max(x[0].size(1) for x in batch)
    if max_target_len % n_frames_per_step != 0:
        max_target_len += n_frames_per_step - max_target_len % n_frames_per_step
    mel_padded = torch.zeros(len(batch), n_mel, max_target_len)
    gate_padded = torch.zeros(len(batch), max_target_len)
    output_lengths = torch.zeros(len(batch), dtype=torch.long)
    prior_padded = torch.zeros(len(batch), max_target_len, max_input_len) if use_attn_prior else None
    speaker_ids = torch.zeros(len(batch), dtype=torch.long)
    for i in range(len(ids)):
        mel = batch[ids[i]][0]
        mel_padded[i, :, :mel.size(1)] = mel
        gate_padded[i, mel.size(1) - 1:] = 1
        output_lengths[i] = mel.size(1)
        speaker_ids[i] = int(batch[ids[i]][1])
        if use_attn_prior:
            p = batch[ids[i]][3]
            prior_padded[i, :p.size(0), :p.size(1)] = p
    return mel_padded, speaker_ids, text_padded, input_lengths, output_lengths, gate_padded, prior_padded

"""CPU fp32 restatement of the Flowtron AR-flow hot path (TEST INFRASTRUCTURE).

Functional style: every function takes ``p``, a flat ``{state_dict key: tensor}``
dict in the reference's checkpoint layout (SURVEY.md §8a row 15), so the same
weights drive the reference, this oracle and the CUDA path.  Everything is
ordinary differentiable torch, so ``torch.autograd`` of these functions is the
gradient oracle as well.  They compute in the dtype of their inputs: given float64
tensors they are a float64 reference (tests/test_gpu_flow_step.py).

Each function cites the reference lines it restates (paths relative to
/root/reference).  Pinned against reference-generated fixtures by
``tests/test_oracle_golden.py``.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor
Params = Dict[str, Tensor]


# --------------------------------------------------------------------------- masks
def get_mask_from_lengths(lengths: Tensor, max_len: Optional[int] = None) -> Tensor:
    """flowtron.py:39-50 — ``arange(max_len) < lengths[:, None]`` (bool [B, max_len])."""
    if max_len is None:
        max_len = int(lengths.max().item())
    ids = torch.arange(0, max_len, device=lengths.device, dtype=lengths.dtype)
    return ids < lengths.unsqueeze(1)


# --------------------------------------------------------------------------- LSTM
def lstm_layer_explicit(x: Tensor, w_ih: Tensor, w_hh: Tensor, b_ih: Tensor, b_hh: Tensor,
                        h0: Optional[Tensor] = None, c0: Optional[Tensor] = None,
                        return_state: bool = False):
    """One ``nn.LSTM`` layer, zero initial state, gate order i,f,g,o (flowtron.py:654-655).

    x: [T, B, I] -> h: [T, B, H].  Python loop over T: this is the specification.
    """
    T, B, _ = x.shape
    H = w_hh.shape[1]
    h = x.new_zeros(B, H) if h0 is None else h0
    c = x.new_zeros(B, H) if c0 is None else c0
    xp = x @ w_ih.t() + (b_ih + b_hh)
    outs = []
    for t in range(T):
        a = xp[t] + h @ w_hh.t()
        i, f, g, o = a.split(H, dim=1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
        h = torch.sigmoid(o) * torch.tanh(c)
        outs.append(h)
    out = torch.stack(outs, 0)
    if return_state:
        return out, (h, c)
    return out


def lstm_layer_fast(x: Tensor, w_ih: Tensor, w_hh: Tensor, b_ih: Tensor, b_hh: Tensor) -> Tensor:
    """Same layer through ATen's fused CPU LSTM (what the reference's nn.LSTM calls).
    Used for the timed CPU baseline; ``test_oracle_golden`` checks it equals the explicit loop."""
    B = x.shape[1]
    H = w_hh.shape[1]
    hx = (x.new_zeros(1, B, H), x.new_zeros(1, B, H))
    out, _, _ = torch._VF.lstm(x, hx, [w_ih, w_hh, b_ih, b_hh], True, 1, 0.0, False, False, False)
    return out


def _lstm(x, p, prefix, layer, fast):
    fn = lstm_layer_fast if fast else lstm_layer_explicit
    return fn(x, p[f"{prefix}.weight_ih_l{layer}"], p[f"{prefix}.weight_hh_l{layer}"],
              p[f"{prefix}.bias_ih_l{layer}"], p[f"{prefix}.bias_hh_l{layer}"])


def _zero_after_len(h: Tensor, out_lens: Optional[Tensor]) -> Tensor:
    """pack_padded/pad_packed semantics (flowtron.py:689-694): outputs are 0 at t >= len.
    The LSTM is causal and its final state is unused, so packing == full run + zeroing
    (SURVEY.md §8a row 3)."""
    if out_lens is None:
        return h
    T = h.shape[0]
    m = (torch.arange(T, device=h.device)[:, None] < out_lens[None, :]).to(h.dtype)
    return h * m[:, :, None]


# --------------------------------------------------------------------------- attention
def attention_forward(p: Params, pre: str, queries: Tensor, text: Tensor, mask: Optional[Tensor],
                      attn_prior: Optional[Tensor], temperature: float = 1.0,
                      attn: Optional[Tensor] = None):
    """flowtron.py:559-592 (+ compute_attention_posterior :544-557).

    queries [T,B,H], text [L,B,E], mask [B,L,1] bool (True = pad).
    Returns ctx [B,A,T], attn [B,T,L], attn_logprob [B,T,L] (or None if attn was given).
    """
    Wq = p[f"{pre}.query.linear_layer.weight"]
    Wk = p[f"{pre}.key.linear_layer.weight"]
    Wv = p[f"{pre}.value.linear_layer.weight"]
    wv = p[f"{pre}.v.linear_layer.weight"]
    values = (text @ Wv.t()).transpose(0, 1)                     # [B,L,A]
    if attn is None:
        keys = (text @ Wk.t()).transpose(0, 1)                   # [B,L,A]
        q = (queries @ Wq.t()).transpose(0, 1)                   # [B,T,A]
        e = torch.tanh(q[:, :, None] + keys[:, None]) @ wv.t()   # [B,T,L,1]   :572
        e = e[..., 0] / temperature                              # :573
        if mask is not None:
            e = e.masked_fill(mask.transpose(1, 2), -float("inf"))   # :574-576
        a = torch.softmax(e, dim=2)                              # :577
        if attn_prior is not None:
            lp = torch.log(a + 1e-20) + torch.log(attn_prior.to(a.dtype) + 1e-20)  # :546-548
            attn_logprob = lp.clone()                            # :550 (before masking)
            if mask is not None:
                lp = lp.masked_fill(mask.transpose(1, 2), -float("inf"))
            a = torch.softmax(lp, dim=2)                         # :556
        else:
            attn_logprob = torch.log(a + 1e-8)                   # :583
    else:
        a = attn
        attn_logprob = None
    ctx = torch.bmm(a, values).transpose(1, 2)                   # :590-591
    return ctx, a, attn_logprob


# --------------------------------------------------------------------------- flows
def _dense_conv(p: Params, pre: str, h: Tensor) -> Tensor:
    """DenseLayer (flowtron.py:453-464) then the 1x1 conv (:651, :768): [T,B,H] -> [T,B,2M]."""
    y = torch.tanh(h @ p[f"{pre}.dense_layer.layers.0.linear_layer.weight"].t()
                   + p[f"{pre}.dense_layer.layers.0.linear_layer.bias"])
    y = torch.tanh(y @ p[f"{pre}.dense_layer.layers.1.linear_layer.weight"].t()
                   + p[f"{pre}.dense_layer.layers.1.linear_layer.bias"])
    return y @ p[f"{pre}.conv.weight"][:, :, 0].t() + p[f"{pre}.conv.bias"]


def ar_step_forward(p: Params, pre: str, mel: Tensor, text: Tensor, mask: Optional[Tensor],
                    out_lens: Optional[Tensor], attn_prior: Optional[Tensor] = None,
                    temperature: float = 1.0, fast: bool = False):
    """AR_Step.forward, flowtron.py:725-773 (SURVEY.md Appendix A.1).

    mel [T,B,M], text [L,B,E], mask [B,L,1].  Returns
    (mel_out [T,B,M], log_s [T,B,M], gates [T,B,1]|None, attn [B,T,L], attn_logprob [B,T,L]).
    """
    M = mel.shape[2]
    mel0 = torch.cat([torch.zeros_like(mel[:1]), mel[:-1]], 0)              # :726-729
    hA = _zero_after_len(_lstm(mel0, p, f"{pre}.attention_lstm", 0, fast), out_lens)   # :737-740
    ctx, attn, attn_logprob = attention_forward(
        p, f"{pre}.attention_layer", hA, text, mask, attn_prior, temperature)           # :748-750
    ctx = ctx.permute(2, 0, 1)                                              # :752
    d = torch.cat((hA, ctx), -1)                                            # :753
    gates = None
    if f"{pre}.gate_layer.linear_layer.weight" in p:                        # :756-758
        gates = d @ p[f"{pre}.gate_layer.linear_layer.weight"].t() + p[f"{pre}.gate_layer.linear_layer.bias"]
    h = _zero_after_len(_lstm(d, p, f"{pre}.lstm", 0, fast), out_lens)      # :762-765 (2 layers)
    h = _zero_after_len(_lstm(h, p, f"{pre}.lstm", 1, fast), out_lens)
    o = _dense_conv(p, pre, h)                                              # :767-768
    log_s, b = o[:, :, :M], o[:, :, M:]                                     # :770-771
    mel_out = torch.exp(log_s) * mel + b                                    # :772
    return mel_out, log_s, gates, attn, attn_logprob


def back_step_index(out_lens: Tensor, T: int) -> Tensor:
    """AR_Back_Step's flip+roll as a gather index (flowtron.py:606-613, SURVEY.md §8a row 5):
    src(q) = len-1-q for q < len, else T-1-q+len.  Returns idx [T,B] (an involution per column)."""
    q = torch.arange(T, device=out_lens.device)[:, None]
    ln = out_lens[None, :]
    return torch.where(q < ln, ln - 1 - q, T - 1 - q + ln)


def ar_back_step_forward(p: Params, pre: str, mel: Tensor, text: Tensor, mask: Optional[Tensor],
                         out_lens: Tensor, attn_prior: Optional[Tensor] = None,
                         temperature: float = 1.0, fast: bool = False):
    """AR_Back_Step.forward, flowtron.py:605-627: time-reverse each utterance (valid frames stay
    left-aligned), run the child step, un-reverse ``mel`` only."""
    T, B, M = mel.shape
    idx = back_step_index(out_lens, T)                                      # [T,B]
    mel_r = torch.gather(mel, 0, idx[:, :, None].expand(T, B, M))
    prior_r = None
    if attn_prior is not None:
        L = attn_prior.shape[2]
        prior_r = torch.gather(attn_prior, 1, idx.t()[:, :, None].expand(B, T, L))
    mel_o, log_s, gates, attn, lp = ar_step_forward(
        p, f"{pre}.ar_step", mel_r, text, mask, out_lens, prior_r, temperature, fast)
    mel_o = torch.gather(mel_o, 0, idx[:, :, None].expand(T, B, M))        # same map is its own inverse
    return mel_o, log_s, gates, attn, lp


def ar_step_infer(p: Params, pre: str, residual: Tensor, text: Tensor, temperature: float = 1.0,
                  gate_threshold: float = 0.5, attn_prior: Optional[Tensor] = None,
                  attns: Optional[Tensor] = None, per_sample_stop: bool = False):
    """AR_Step.infer, flowtron.py:775-828 (Appendix A.3).  residual [T,B,M] -> (out [T',B,M], [attn]).

    The reference breaks when the (single) sample's gate fires; the frame that trips the gate IS
    emitted.  ``per_sample_stop`` is the B>1 extension (SURVEY.md §3.2): every row behaves like
    its own B=1 run; rows that already stopped emit zeros, the loop ends when all rows stopped.
    """
    T, B, M = residual.shape
    H = p[f"{pre}.attention_lstm.weight_hh_l0"].shape[1]
    z = lambda: residual.new_zeros(B, H)
    hA, cA, h0, c0, h1, c1 = z(), z(), z(), z(), z(), z()
    out_prev = residual.new_zeros(B, M)
    has_gate = f"{pre}.gate_layer.linear_layer.weight" in p
    alive = torch.ones(B, dtype=torch.bool)
    outs, attn_list = [], []

    def cell(x, h, c, lp, layer):
        a = (x @ p[f"{lp}.weight_ih_l{layer}"].t() + p[f"{lp}.bias_ih_l{layer}"]
             + h @ p[f"{lp}.weight_hh_l{layer}"].t() + p[f"{lp}.bias_hh_l{layer}"])
        i, f, g, o = a.split(H, dim=1)
        c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
        return torch.sigmoid(o) * torch.tanh(c), c

    for i in range(T):
        hA, cA = cell(out_prev, hA, cA, f"{pre}.attention_lstm", 0)         # :789-791
        prior_i = None if attn_prior is None else attn_prior[:, i][:, None]    # :798 (B=1: [None])
        attn_i = None if attns is None else attns[i][None, None]            # :797
        ctx, a, _ = attention_forward(p, f"{pre}.attention_layer", hA[None], text, None,
                                      prior_i, temperature, attn=attn_i)    # :800-803 (no mask in infer)
        attn_list.append(a)
        d = torch.cat((hA, ctx[:, :, 0]), -1)                               # :809-811
        h0, c0 = cell(d, h0, c0, f"{pre}.lstm", 0)                          # :812-815
        h1, c1 = cell(h0, h1, c1, f"{pre}.lstm", 1)
        o = _dense_conv(p, pre, h1[None])[0]                                # :816-817
        log_s, b = o[:, :M], o[:, M:]                                       # :819-820
        out_prev = (residual[i] - b) / torch.exp(log_s)                     # :821
        if per_sample_stop:
            outs.append(out_prev * alive[:, None].to(out_prev.dtype))
        else:
            outs.append(out_prev)
        if has_gate:                                                        # :823-826
            g = torch.sigmoid(d @ p[f"{pre}.gate_layer.linear_layer.weight"].t()
                              + p[f"{pre}.gate_layer.linear_layer.bias"])[:, 0]
            if per_sample_stop:
                alive = alive & ~(g > gate_threshold)
                if not bool(alive.any()):
                    break
            elif bool((g > gate_threshold).all()) and B == 1:
                break
    return torch.stack(outs, 0), attn_list


def ar_back_step_infer(p, pre, residual, text, temperature=1.0, gate_threshold=0.5, attn_prior=None,
                       per_sample_stop=False, attns=None):
    """AR_Back_Step.infer, flowtron.py:629-642: flip in time, run, flip back (no roll); `attns` is passed through
    unflipped (:634-635), i.e. consumed in the back step's own time order."""
    if attn_prior is not None:
        attn_prior = torch.flip(attn_prior, (1,))
    out, attns = ar_step_infer(p, f"{pre}.ar_step", torch.flip(residual, (0,)), text, temperature,
                               gate_threshold, attn_prior, attns=attns, per_sample_stop=per_sample_stop)
    return torch.flip(out, (0,)), attns


# --------------------------------------------------------------------------- encoder
def _masked_instance_norm(x: Tensor, mask: Optional[Tensor], w: Tensor, b: Tensor, eps: float = 1e-5):
    """flowtron.py:53-92 with use_input_stats=True (track_running_stats=False)."""
    if mask is None:
        return F.instance_norm(x, None, None, w, b, True, 0.1, eps)
    lengths = mask.sum((-1,))
    mean = (x * mask).sum((-1,)) / lengths
    var = (((x - mean[..., None]) * mask) ** 2).sum((-1,)) / lengths
    out = (x - mean[..., None]) / torch.sqrt(var[..., None] + eps)
    return out * w[None, :, None] + b[None, :, None]


def encoder_forward(p: Params, x: Tensor, in_lens: Optional[Tensor], infer: bool = False) -> Tensor:
    """Encoder.forward / .infer in eval mode (no dropout), flowtron.py:492-525.
    x [B,C,L] -> [B,L,C].  ``in_lens`` sorted descending as DataCollate provides."""
    B = x.shape[0]
    mask = None
    if not infer and B > 1:
        mask = get_mask_from_lengths(in_lens, x.shape[2]).unsqueeze(1)
    for i in range(3):
        if mask is not None:
            x = x.masked_fill(~mask, 0.0)
        x = F.conv1d(x, p[f"encoder.convolutions.{i}.0.conv.weight"],
                     p[f"encoder.convolutions.{i}.0.conv.bias"], padding=2)
        # Encoder.infer iterates the Sequential(ConvNorm, norm) blocks, so the (unmasked) instance
        # norm is applied there too (flowtron.py:517-518); forward with B == 1 also has mask=None.
        x = F.relu(_masked_instance_norm(x, mask.to(x.dtype) if mask is not None else None,
                                         p[f"encoder.convolutions.{i}.1.weight"],
                                         p[f"encoder.convolutions.{i}.1.bias"]))
    x = x.transpose(1, 2)                        # [B,L,C]
    Hh = p["encoder.lstm.weight_hh_l0"].shape[1]
    L = x.shape[1]
    outs = []
    for b in range(B):                           # packed BiLSTM: each row runs over its own length
        n = L if (infer or in_lens is None) else int(in_lens[b])
        xb = x[b, :n][:, None]                   # [n,1,C]
        fwd = lstm_layer_explicit(xb, p["encoder.lstm.weight_ih_l0"], p["encoder.lstm.weight_hh_l0"],
                                  p["encoder.lstm.bias_ih_l0"], p["encoder.lstm.bias_hh_l0"])
        bwd = lstm_layer_explicit(torch.flip(xb, (0,)), p["encoder.lstm.weight_ih_l0_reverse"],
                                  p["encoder.lstm.weight_hh_l0_reverse"],
                                  p["encoder.lstm.bias_ih_l0_reverse"], p["encoder.lstm.bias_hh_l0_reverse"])
        o = torch.cat([fwd, torch.flip(bwd, (0,))], -1)[:, 0]              # [n,2Hh]
        outs.append(F.pad(o, (0, 0, 0, L - n)))
    out = torch.stack(outs, 0)
    if not infer and in_lens is not None:
        out = out[:, : int(in_lens.max())]
    return out


# --------------------------------------------------------------------------- model
def n_flows_of(p: Params) -> int:
    return 1 + max(int(k.split(".")[1]) for k in p if k.startswith("flows."))


def flow_prefix(i: int) -> str:
    return f"flows.{i}"


def flowtron_forward(p: Params, mel: Tensor, speaker_ids: Tensor, text: Tensor, in_lens: Tensor,
                     out_lens: Tensor, attn_prior: Optional[Tensor] = None, fast: bool = False,
                     encoder_outputs: Optional[Tensor] = None):
    """Flowtron.forward, flowtron.py:870-899 (n_components=0 branch, eval-mode encoder)."""
    if encoder_outputs is None:
        spk = F.embedding(speaker_ids, p["speaker_embedding.weight"])
        t = F.embedding(text, p["embedding.weight"]).transpose(1, 2)
        t = encoder_forward(p, t, in_lens).transpose(0, 1)                   # [L,B,512]
        encoder_outputs = torch.cat([t, spk.expand(t.size(0), -1, -1)], 2)   # :886-887
    mel = mel.permute(2, 0, 1)
    mask = ~get_mask_from_lengths(in_lens, encoder_outputs.shape[0])[..., None]   # :891
    log_s_list, attns, lps, gate = [], [], [], None
    for i in range(n_flows_of(p)):
        fn = ar_step_forward if i % 2 == 0 else ar_back_step_forward
        mel, log_s, gate, a, lp = fn(p, flow_prefix(i), mel, encoder_outputs, mask, out_lens,
                                     attn_prior, fast=fast)
        log_s_list.append(log_s)
        attns.append(a)
        lps.append(lp)
    return mel, log_s_list, gate, attns, lps, None, None, None


def flowtron_infer(p: Params, residual: Tensor, speaker_ids: Tensor, text: Tensor,
                   temperature: float = 1.0, gate_threshold: float = 0.5,
                   per_sample_stop: bool = False, attns=None):
    """Flowtron.infer, flowtron.py:901-930.  `attns`: per-flow forced alignments [T,L] indexed by flow (the reference's
    `reversed(attns)[i]` at :924 is not subscriptable; the evident intent -- flow k gets attns[k] -- is restated)."""
    spk = F.embedding(speaker_ids, p["speaker_embedding.weight"])
    t = F.embedding(text, p["embedding.weight"]).transpose(1, 2)
    t = encoder_forward(p, t, None, infer=True).transpose(0, 1)
    enc = torch.cat([t, spk.expand(t.size(0), -1, -1)], 2)
    residual = residual.permute(2, 0, 1)
    attn_all = []
    for i in reversed(range(n_flows_of(p))):
        forced = None if attns is None else attns[i]
        if i % 2 == 0:
            residual, a = ar_step_infer(p, flow_prefix(i), residual, enc, temperature, gate_threshold,
                                        attns=forced, per_sample_stop=per_sample_stop)
        else:
            residual, a = ar_back_step_infer(p, flow_prefix(i), residual, enc, temperature,
                                             gate_threshold, per_sample_stop=per_sample_stop, attns=forced)
        attn_all.append(a)
    return residual.permute(1, 2, 0), attn_all


def flowtron_loss(model_output, gate_target: Tensor, in_lens: Tensor, out_lens: Tensor,
                  sigma: float = 1.0, gate_loss: bool = True):
    """FlowtronLoss.forward default branch (no GMM, no CTC), flowtron.py:200-243 (Appendix A.5)."""
    z, log_s_list, gate_pred = model_output[0], model_output[1], model_output[2]
    mask = get_mask_from_lengths(out_lens, z.shape[0]).transpose(0, 1)[..., None].to(z.dtype)
    n = mask.sum()
    log_s_total = sum(torch.sum(ls * mask) for ls in log_s_list)
    zm = z * mask
    nll = (torch.sum(zm * zm) / (2 * sigma * sigma) - log_s_total) / (n * z.size(2))
    gl = torch.zeros(1)
    if gate_loss and gate_pred is not None:
        gp = (gate_pred * mask)[..., 0].permute(1, 0)
        gl = F.binary_cross_entropy_with_logits(gp, gate_target.to(gp.dtype), reduction="none")
        gl = (gl.permute(1, 0) * mask[:, :, 0]).sum() / n
    return nll, gl


def attention_ctc_loss(attn_logprob: Tensor, in_lens: Tensor, out_lens: Tensor, blank_logprob: float = -1.0) -> Tensor:
    """AttentionCTCLoss.forward, flowtron.py:162-182: attn_logprob [B,T,L] (natural time) -> scalar."""
    padded = F.pad(attn_logprob[:, None], (1, 0, 0, 0, 0, 0, 0, 0), value=blank_logprob)     # blank column in front, :166-168
    ctc = torch.nn.CTCLoss(zero_infinity=True)
    total = 0.0
    for b in range(attn_logprob.shape[0]):
        K, Tq = int(in_lens[b]), int(out_lens[b])
        cur = padded[b].permute(1, 0, 2)[:Tq, :, :K + 1]                                    # :172-175
        cur = torch.log_softmax(cur[None], dim=3)[0]
        total = total + ctc(cur, torch.arange(1, K + 1)[None], input_lengths=torch.tensor([Tq]),
                            target_lengths=torch.tensor([K]))
    return total / attn_logprob.shape[0]


def flowtron_ctc_loss(model_output, in_lens: Tensor, out_lens: Tensor, blank_logprob: float = -1.0) -> Tensor:
    """The use_ctc_loss branch of FlowtronLoss.forward, flowtron.py:245-274: back-step flows are un-rolled and
    un-flipped to natural time first (index map instead of the reference's in-place roll/flip/restore)."""
    lps = model_output[4]
    T = lps[0].shape[1]
    total = 0.0
    for i, lp in enumerate(lps):
        if i % 2 != 0:
            idx = back_step_index(out_lens, T)                        # [T, B]: natural t -> flow-time row
            lp = torch.stack([lp[b][idx[:, b]] for b in range(lp.shape[0])])
        total = total + attention_ctc_loss(lp, in_lens, out_lens, blank_logprob)
    return total / float(len(lps))


# --------------------------------------------------------------------------- attention prior
def beta_binomial_prior(phoneme_count: int, mel_count: int, scaling: float = 1.0) -> np.ndarray:
    """data.py:31-41 restated literally with scipy.stats.betabinom (the closed-form version used by the
    data helpers is checked against this in tests/test_oracle_golden.py)."""
    from scipy.stats import betabinom
    x = np.arange(0, phoneme_count)
    rows = []
    for i in range(1, mel_count + 1):
        a, b = scaling * i, scaling * (mel_count + 1 - i)
        rows.append(betabinom(phoneme_count - 1, a, b).pmf(x))
    return np.array(rows)

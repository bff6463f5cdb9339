"""GPU: one flow step (ft_ar_step_fwd and both backward schedules) against the float64 oracle, at the shapes where
ar_step.cu changes kernel schedule, with the gradient of every output injected on its own.

A flow module is called directly (``model.flows[i](mel, text, mask, out_lens, attn_prior)``), so no batch splitting gets in
the way: B up to 64 reaches the kernels as one launch.  The reference is ``oracle.ar_step_forward`` /
``oracle.ar_back_step_forward`` in float64 on the GPU with the explicit LSTM loop, fed the same parameters cast up.

Schedules chosen by shape in ar_step.cu with default settings (each case below sits on one of these boundaries):
  B <= 32, T <= 100   attention LSTM with the folded input projection, one launch per layer; BPTT as one cluster launch
  B <= 32, T > 100    layer pipeline in 100-step chunks; from T >= 200 the BPTT runs in chunks with the dc carry hand-over
  B <= 32, T >= 320   attention LSTM in 256-step chunks with attention / gate / layer-0 projection on a second stream; the
                      one-call backward (ft_ar_step_bwd) overlaps the attention backward with the chunked attention-LSTM BPTT
  32 < B <= 64        separate projection GEMM, 128-CTA forward, no pipeline, no overlap, ring-of-groups BPTT kernel

Bars: forward outputs within 1e-3 of the tensor's max |value| on valid positions; gradients per tensor relative L2 <= 5e-3 and
cosine >= 0.99995.  Padded query rows (t >= out_len) are outside the contract: nothing is injected or compared there.
"""
import pytest
import torch

from conftest import record_parity
from flowtron_b200 import synth
from oracle import flowtron_oracle as O

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-3
REL_L2_TOL = 5e-3
COS_TOL = 0.99995
DEV = "cuda"

OUTPUTS = ("mel_out", "log_s", "gates", "attn", "attn_logprob")

# in_lens / out_lens: explicit lists, or None for seeded ragged lengths (row 0 full length, the others in [1, max]).
CASES = [
    # smallest everything: one step, one key.  Its one gate logit (0.016) is the cancelling sum of terms of size ~1, so the
    # fp16 rounding of the value projection's operands (~5e-4 absolute in the logit) is 3 % of the tensor's max |value|: the
    # reference takes the same fp16-rounded attention operands (fp16_attention_operands)
    dict(id="b1_t1_l1_step", B=1, T=1, L=1, back=False, gate=True, prior=False, out_lens=[1], in_lens=[1],
         fp16_attention_operands=True),
    # last one-launch T; a one-frame utterance and a one-key row (softmax over a single key)
    dict(id="b3_t100_l37_back", B=3, T=100, L=37, back=True, gate=True, prior=True, out_lens=[100, 1, 63], in_lens=[37, 19, 1]),
    # forward layer pipeline with a 1-step tail chunk; exactly one attention key block (AT_LB = 128)
    dict(id="b5_t101_l128_step", B=5, T=101, L=128, back=False, gate=False, prior=True),
    # BPTT pipeline with exactly two chunks; one key past a key block
    dict(id="b8_t200_l129_back", B=8, T=200, L=129, back=True, gate=True, prior=False),
    # attention overlap at its threshold (one 256-step chunk + a 64-step chunk); widest batch of the folded projection
    dict(id="b32_t320_l24_step", B=32, T=320, L=24, back=False, gate=True, prior=True),
    # overlap with a 77-step tail chunk; the largest L the attention backward takes
    dict(id="b2_t333_l256_back", B=2, T=333, L=256, back=True, gate=False, prior=True),
    # smallest wide batch (Bbox 40): projection GEMM, 128-CTA forward, lstm_bwd_kernel
    dict(id="b33_t150_l50_step", B=33, T=150, L=50, back=False, gate=True, prior=True),
    # widest batch
    dict(id="b64_t130_l24_back", B=64, T=130, L=24, back=True, gate=True, prior=False),
    # temperature != 1, and keys scaled so that a large share of |q + k| is beyond the +-40 clamp of e^{2x} (and the score's
    # 2^60 clamp): tanh is saturated there, so the clamps must not change a thing.  With keys of size ~50, the fp16 rounding
    # of the key projection's operands moves the unsaturated scores by ~1e-2 (1.5e-3 on attn, 1.8e-2 relative L2 on d_text
    # against the exact reference, reproduced by the float64 reference on fp16-rounded operands): the reference takes the
    # same fp16-rounded attention operands, so what is measured here is the clamping, not the operand precision
    dict(id="b6_t70_l20_temp_bigkeys", B=6, T=70, L=20, back=False, gate=True, prior=True, temperature=1.3,
         key_scale=50.0, query_scale=8.0, fp16_attention_operands=True),
]
CASE_BY_ID = {c["id"]: c for c in CASES}


# --------------------------------------------------------------------------------------------------------- set-up
def _lengths(case, g):
    B, T, L = case["B"], case["T"], case["L"]
    out_lens = case.get("out_lens")
    if out_lens is None:
        out_lens = torch.randint(1, T + 1, (B,), generator=g)
        out_lens[0] = T
    in_lens = case.get("in_lens")
    if in_lens is None:
        in_lens = torch.randint(1, L + 1, (B,), generator=g)
        in_lens[0] = L
    return torch.as_tensor(out_lens, dtype=torch.long), torch.as_tensor(in_lens, dtype=torch.long)


def _setup(case, seed=1234):
    """The flow module under test (fp32, CUDA) and its inputs."""
    from flowtron_b200 import _lib
    from flowtron_b200.flowtron import Flowtron
    _lib.set_lstm_half_sm(False)                 # process-wide switch that Flowtron.forward sets; calling a flow skips that
    cfg = dict(synth.DEFAULT_MODEL_CONFIG, n_flows=2 if case["back"] else 1, use_gate_layer=case["gate"])
    params = synth.synth_params(cfg, seed)
    i = 1 if case["back"] else 0
    pre = f"flows.{i}.ar_step" if case["back"] else f"flows.{i}"
    params[f"{pre}.attention_layer.key.linear_layer.weight"] *= case.get("key_scale", 1.0)
    params[f"{pre}.attention_layer.query.linear_layer.weight"] *= case.get("query_scale", 1.0)
    model = Flowtron(**cfg)
    model.load_state_dict(params, strict=True)
    flow = model.flows[i].to(DEV)
    step = flow.ar_step if case["back"] else flow
    assert hasattr(step, "gate_layer") == case["gate"]
    step.attention_layer.temperature = case.get("temperature", 1.0)

    B, T, L = case["B"], case["T"], case["L"]
    M, E = cfg["n_mel_channels"], cfg["n_text_dim"] + cfg["n_speaker_dim"]
    g = torch.Generator().manual_seed(seed + B * 1000 + T)
    out_lens, in_lens = _lengths(case, g)
    mel = torch.randn(T, B, M, generator=g)              # padded frames hold data too: they must not leak into valid ones
    text = torch.randn(L, B, E, generator=g)
    prior = None
    if case["prior"]:
        prior = torch.zeros(B, T, L)
        for b in range(B):
            pb = synth.beta_binomial_prior(int(in_lens[b]), int(out_lens[b]))
            prior[b, : int(out_lens[b]), : int(in_lens[b])] = torch.from_numpy(pb).float()
    dev = DEV
    inp = dict(mel=mel.to(dev), text=text.to(dev), out_lens=out_lens.to(dev), in_lens=in_lens.to(dev),
               mask=~(torch.arange(L)[None, :] < in_lens[:, None])[..., None].to(dev),
               prior=None if prior is None else prior.to(dev))
    tmask = torch.arange(T, device=dev)[:, None] < inp["out_lens"][None, :]                     # [T, B] valid frames
    kmask = torch.arange(L, device=dev)[None, :] < inp["in_lens"][:, None]                      # [B, L] valid keys
    inp["tmask"], inp["kmask"] = tmask, kmask
    inp["btl"] = tmask.t()[:, :, None] & kmask[:, None, :]                                      # [B, T, L] valid (row, key)
    return flow, step, inp


ATTENTION_PROJECTIONS = ("attention_layer.query.linear_layer.weight", "attention_layer.key.linear_layer.weight",
                         "attention_layer.value.linear_layer.weight")


def _ref_inputs(case, step, inp):
    """float64 leaves of the reference: parameters keyed like AR_Step.named_parameters(), mel and text (inp["mel64"],
    inp["text64"]).  With fp16_attention_operands, text and the query / key / value weights are first rounded to fp16,
    the operands of the kernel's projection GEMMs."""
    r16 = case.get("fp16_attention_operands", False)
    P = {}
    for n, p in step.named_parameters():
        t = p.detach()
        if r16 and n in ATTENTION_PROJECTIONS:
            t = t.half()
        P[n] = t.double().requires_grad_(True)
    inp["mel64"] = inp["mel"].double().requires_grad_(True)
    inp["text64"] = (inp["text"].half() if r16 else inp["text"]).double().requires_grad_(True)
    return P


def _ref_forward(P, inp, back, temperature, out_lens=None):
    """float64 oracle of the flow; P is keyed like AR_Step.named_parameters()."""
    mel = inp["mel64"]
    text = inp["text64"]
    prior = None if inp["prior"] is None else inp["prior"].double()
    out_lens = inp["out_lens"] if out_lens is None else out_lens
    if back:
        p = {f"f.ar_step.{n}": t for n, t in P.items()}
        return O.ar_back_step_forward(p, "f", mel, text, inp["mask"], out_lens, prior, temperature)
    p = {f"f.{n}": t for n, t in P.items()}
    return O.ar_step_forward(p, "f", mel, text, inp["mask"], out_lens, prior, temperature)


def _injections(case, inp, seed=99):
    """Six sets of output gradients: N(0,1) into exactly one output (valid positions only), then all five at once at mixed
    magnitudes (d_gates ~1e3 x d_mel_out, like the gate BCE gradient 1/n next to the NLL gradient 1/(n*80)), which exercises
    the per-flow power-of-two loss scale."""
    B, T, L, M = case["B"], case["T"], case["L"], inp["mel"].shape[2]
    g = torch.Generator().manual_seed(seed + T)
    tm = inp["tmask"][..., None].float()
    btl = inp["btl"].float()
    shapes = dict(mel_out=((T, B, M), tm), log_s=((T, B, M), tm), gates=((T, B, 1), tm), attn=((B, T, L), btl),
                  attn_logprob=((B, T, L), btl))
    names = [n for n in OUTPUTS if n != "gates" or case["gate"]]
    rnd = {n: torch.randn(*shapes[n][0], generator=g).to(DEV) * shapes[n][1] for n in names}
    out = []
    for n in names:
        out.append((n, {m: (rnd[m] if m == n else torch.zeros_like(rnd[m])) for m in names}))
    mags = dict(mel_out=1e-3, log_s=1e-3, gates=1.0, attn=1e-2, attn_logprob=1e-2)
    out.append(("mixed", {m: rnd[m] * mags[m] for m in names}))
    return out


def _as_dict(outs, gate):
    mel_out, log_s, gates, attn, lp = outs
    d = dict(mel_out=mel_out, log_s=log_s, attn=attn, attn_logprob=lp)
    if gate:
        d["gates"] = gates
    return d


def _run_kernel(flow, step, inp, grads, fused):
    """Fresh forward (the kernel releases its saved activations after one backward), then backward with `grads`."""
    step._fuse_bwd = fused
    for p in flow.parameters():
        p.grad = None
    mel = inp["mel"].clone().requires_grad_(True)
    text = inp["text"].clone().requires_grad_(True)
    outs = _as_dict(flow(mel, text, inp["mask"], inp["out_lens"], inp["prior"]), hasattr(step, "gate_layer"))
    names = list(outs)
    torch.autograd.backward([outs[n] for n in names], [grads[n] for n in names])
    torch.cuda.synchronize()
    got = {"d_mel": mel.grad, "d_text": text.grad}
    got.update({n: p.grad for n, p in step.named_parameters()})
    return {n: o.detach() for n, o in outs.items()}, got


def _ref_grads(ref_outs, inp, P, grads):
    names = list(ref_outs)
    leaves = [inp["mel64"], inp["text64"]] + list(P.values())
    gs = torch.autograd.grad([ref_outs[n] for n in names], leaves, [grads[n].double() for n in names],
                             retain_graph=True, allow_unused=True)
    keys = ["d_mel", "d_text"] + list(P)
    return {k: (torch.zeros_like(l) if g is None else g) for k, g, l in zip(keys, gs, leaves)}


# --------------------------------------------------------------------------------------------------------- metrics
def _fwd_errors(got, ref, inp):
    """max |got - ref| / max |ref| per output on valid positions (valid keys for the [B,T,L] outputs; attn_logprob's padded
    keys of valid rows hold defined constants and are checked on their own)."""
    btl = inp["btl"]
    frames = inp["tmask"][..., None]                                       # [T, B, 1]
    pad_keys = inp["tmask"].t()[:, :, None] & ~btl                         # valid rows, padded keys

    def err(a, b, m, floor=1e-30):
        a, b = a.double()[m.expand_as(a)], b.detach()[m.expand_as(b)]
        return float((a - b).abs().max() / b.abs().max().clamp_min(floor)) if b.numel() else 0.0

    # log-probabilities are measured on a scale of at least 1 nat: with a single valid key, log(1 + 1e-8) is 1e-8 in float64
    # and exactly 0 in float32, which is no error at all
    errs = {n: err(got[n], r, frames if n in ("mel_out", "log_s", "gates") else btl, 1.0 if n == "attn_logprob" else 1e-30)
            for n, r in ref.items()}
    if bool(pad_keys.any()):
        errs["attn_logprob_padkeys"] = err(got["attn_logprob"], ref["attn_logprob"], pad_keys, 1.0)
    return errs


def _grad_errors(got, ref):
    """Per tensor: relative L2 and cosine against the float64 gradient.  Tensors whose reference gradient is (near) zero --
    e.g. the dense layers when only `attn` receives a gradient -- are measured against 1e-4 of the largest gradient norm."""
    floor = 1e-4 * max(float(r.norm()) for r in ref.values())
    rows = {}
    for k, r in ref.items():
        g = got[k]
        assert g is not None, f"no gradient for {k}"
        g, r = g.double().reshape(-1), r.reshape(-1)
        rn = float(r.norm())
        rel = float((g - r).norm()) / max(rn, floor) if max(rn, floor) > 0 else float(g.norm())
        cos = float((g @ r) / (g.norm() * r.norm() + 1e-300)) if rn > floor else 1.0
        rows[k] = (rel, cos)
    return rows


def _fails(fwd, grads, fwd_tol=FWD_TOL, rel_tol=REL_L2_TOL, cos_tol=COS_TOL):
    bad = {k: v for k, v in fwd.items() if not v <= fwd_tol}
    bad.update({k: v for k, v in grads.items() if not (v[0] <= rel_tol and v[1] >= cos_tol)})
    return bad


# --------------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_flow_step_matches_float64_reference_per_output_gradient(case):
    from flowtron_b200 import _lib
    flow, step, inp = _setup(case)
    back, gate, temperature = case["back"], case["gate"], case.get("temperature", 1.0)
    B, T, L = case["B"], case["T"], case["L"]
    P = _ref_inputs(case, step, inp)
    ref = _as_dict(_ref_forward(P, inp, back, temperature), gate)

    if "key_scale" in case:        # the case must do what it claims: a good share of |q + k| beyond the clamp
        with torch.no_grad():
            hA = O._zero_after_len(O._lstm(torch.cat([torch.zeros_like(inp["mel64"][:1]), inp["mel64"][:-1]]),
                                           {f"f.{n}": t for n, t in P.items()}, "f.attention_lstm", 0, False), inp["out_lens"])
            q = hA @ P["attention_layer.query.linear_layer.weight"].t()                     # [T, B, A]
            k = inp["text64"] @ P["attention_layer.key.linear_layer.weight"].t()            # [L, B, A]
            s = (q.permute(1, 0, 2)[:, :, None] + k.permute(1, 0, 2)[:, None]).abs()        # [B, T, L, A]
            share = float((s > 40).double()[inp["btl"]].mean())
        record_parity(f"flow_step_{case['id']}_clamp_share", {"share_abs_q_plus_k_over_40": share})
        assert share >= 0.2, share

    failures = {}
    for inj_i, (inj, grads) in enumerate(_injections(case, inp)):
        rg = _ref_grads(ref, inp, P, grads)
        for sched, fused in (("two_call", False), ("one_call", True)):
            outs, got = _run_kernel(flow, step, inp, grads, fused)
            assert _lib.device_status() == 0
            fwd = {}
            if inj_i == 0:
                # ---- forward: bar, finiteness everywhere, attention rows, the text gradient on padded keys
                for n, o in outs.items():
                    assert bool(torch.isfinite(o).all()), f"{sched}: non-finite {n}"
                fwd = _fwd_errors(outs, ref, inp)
                rows = inp["tmask"].t()                                                   # [B, T]
                row_sum_err = float((outs["attn"].double().sum(2)[rows] - 1).abs().max())
                assert row_sum_err <= 1e-5, (sched, row_sum_err)
                pad_keys = rows[:, :, None] & ~inp["kmask"][:, None, :]
                if bool(pad_keys.any()):
                    assert float(outs["attn"][pad_keys].abs().max()) == 0.0, f"{sched}: attention on padded keys"
            for k, g in got.items():
                assert g is not None and bool(torch.isfinite(g).all()), f"{sched}/{inj}: non-finite or missing {k}"
            pad_text = ~inp["kmask"].t()                                                  # [L, B]
            if bool(pad_text.any()):
                assert float(got["d_text"][pad_text].abs().max()) == 0.0, f"{sched}/{inj}: d_text nonzero on padded keys"
            gerr = _grad_errors(got, rg)
            worst = max(gerr, key=lambda k: gerr[k][0])
            rec = {"rel_l2_worst": gerr[worst][0], "cos_worst": min(v[1] for v in gerr.values()), "worst_tensor": worst,
                   "d_mel_rel_l2": gerr["d_mel"][0], "d_text_rel_l2": gerr["d_text"][0]}
            if fwd:
                rec["fwd_worst"] = max(fwd.values())
                rec.update({f"fwd_{k}": v for k, v in fwd.items()})
            record_parity(f"flow_step_{case['id']}_{sched}_{inj}", rec)
            bad = _fails(fwd, gerr)
            if bad:
                failures[f"{sched}/{inj}"] = bad
            del outs, got
        del rg
    assert not failures, failures


# Each entry: (case, deliberate change to the reference).  The changed reference must miss the bar against the true one;
# then a kernel that passes is not off by a mask (out_len), a scale (temperature) or a time map (back-step flag).
SELF_CHECKS = [("b8_t200_l129_back", "out_len"), ("b8_t200_l129_back", "back_flag"), ("b5_t101_l128_step", "out_len"),
               ("b5_t101_l128_step", "temperature"), ("b6_t70_l20_temp_bigkeys", "temperature"),
               ("b3_t100_l37_back", "back_flag")]


@pytest.mark.parametrize("case_id,change", SELF_CHECKS, ids=[f"{c}-{m}" for c, m in SELF_CHECKS])
def test_bar_rejects_a_semantically_changed_reference(case_id, change):
    case = CASE_BY_ID[case_id]
    flow, step, inp = _setup(case)
    back, gate, temperature = case["back"], case["gate"], case.get("temperature", 1.0)
    P = _ref_inputs(case, step, inp)
    ref = _as_dict(_ref_forward(P, inp, back, temperature), gate)
    out_lens = None
    if change == "out_len":                  # a row that is not the longest, one frame short
        ol = inp["out_lens"].clone()
        b = int(torch.argmin(torch.where(ol > 1, ol, ol.max() + 1)))
        ol[b] -= 1
        out_lens = ol
    elif change == "temperature":
        temperature = temperature * 1.05
    elif change == "back_flag":
        back = not back
    alt = _as_dict(_ref_forward(P, inp, back, temperature, out_lens), gate)
    _, grads = _injections(case, inp)[-1]
    rg = _ref_grads(ref, inp, P, grads)
    ag = _ref_grads(alt, inp, P, grads)
    fwd = _fwd_errors({k: v.detach() for k, v in alt.items()}, ref, inp)
    gerr = _grad_errors(ag, rg)
    bad = _fails(fwd, gerr)
    record_parity(f"flow_step_selfcheck_{case_id}_{change}", {"fwd_worst": max(fwd.values()),
                                                               "rel_l2_worst": max(v[0] for v in gerr.values()),
                                                               "n_failing": len(bad)})
    assert bad, f"the bar does not tell the reference from one with a changed {change}"

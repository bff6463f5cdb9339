#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) on CPU fp32.

Run in the build container only (the GPU box has no /root/reference):
    python tests/make_golden.py
Weights come from flowtron_b200.synth.synth_params(cfg, seed), so fixtures carry outputs only.
Reference entry points exercised: Flowtron.forward (flowtron.py:870-899), FlowtronLoss.forward
(:200-243), autograd of both, Flowtron.infer (:901-930), TacotronSTFT.mel_spectrogram
(audio_processing.py:117-134), RAdam.step (radam.py:44-122) after clip_grad_norm_ (train.py:326).
"""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shims  # noqa: E402
from flowtron_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
N_GRAD_SAMPLES = 32


def grad_sample_index(name: str, numel: int) -> np.ndarray:
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    return torch.randint(0, numel, (N_GRAD_SAMPLES,), generator=g).numpy()


def train_case(tag, n_flows, B, T, L, out_lens, with_prior, seed, in_lens=None, logmel_stats=False, store_attn=True,
               ctc_weight=0.0):
    cfg = dict(synth.DEFAULT_MODEL_CONFIG, n_flows=n_flows)
    params = synth.synth_params(cfg, seed)
    F, model = ref_shims.reference_model(cfg, params)
    batch = synth.synth_batch(B, T, L, cfg, seed, out_lens=out_lens, in_lens=in_lens, with_prior=with_prior,
                              logmel_stats=logmel_stats)
    crit = F.FlowtronLoss(sigma=1.0, gm_loss=False, gate_loss=True, use_ctc_loss=ctc_weight > 0, ctc_loss_weight=ctc_weight)
    for p in model.parameters():
        p.requires_grad_(True)
    # Encoder dropout (flowtron.py:502) is random in train mode, and in eval mode F.dropout returns
    # its input so the in-place masked_fill_ at :501 breaks autograd.  Shim for the gradient fixture:
    # dropout := identity copy (== eval-mode values, differentiable).
    F.F.dropout = lambda x, p=0.5, training=True, inplace=False: x.clone()
    out = model(batch["mel"], batch["speaker_ids"], batch["text"], batch["in_lens"], batch["out_lens"],
                batch["attn_prior"])
    z, log_s_list, gate, attns, lps = out[:5]
    nll, gl, ctc = crit(out, batch["gate_target"], batch["in_lens"], batch["out_lens"])
    (nll + gl + ctc * ctc_weight).sum().backward()        # train.py:301-304
    rec = dict(ctc_weight=np.float32(ctc_weight), loss_ctc=ctc.detach().numpy(),cfg_n_flows=n_flows, B=B, T=T, L=L, seed=seed, with_prior=int(with_prior), logmel_stats=int(logmel_stats),
               out_lens=batch["out_lens"].numpy(), in_lens=batch["in_lens"].numpy(),
               z=z.detach().numpy(), gate=gate.detach().numpy(),
               nll=nll.detach().numpy(), gate_loss=gl.detach().numpy())
    for i in range(n_flows):
        rec[f"log_s_{i}"] = log_s_list[i].detach().numpy()
        if store_attn:
            rec[f"attn_{i}"] = attns[i].detach().numpy()
            rec[f"attn_logprob_{i}"] = lps[i].detach().numpy()
        else:                                   # BASELINE-size cases: keep the fixture to a few MB (one utterance's attention)
            rec[f"attn_{i}_b0"] = attns[i][0].detach().numpy()
    for name, p in model.named_parameters():
        gflat = p.grad.detach().reshape(-1)
        rec[f"gnorm::{name}"] = np.float64(gflat.double().norm().item())
        rec[f"gsamp::{name}"] = gflat[grad_sample_index(name, gflat.numel())].numpy()
    np.savez_compressed(os.path.join(OUT, f"train_{tag}.npz"), **rec)
    print(f"train_{tag}: nll={float(nll):.6f} gate={float(gl):.6f}")


def infer_case(tag, n_flows, B, T, L, seed, gate_bias, sigma=0.5, use_gate=True):
    cfg = dict(synth.DEFAULT_MODEL_CONFIG, n_flows=n_flows, use_gate_layer=use_gate)
    params = synth.synth_params(cfg, seed)
    if use_gate:
        key = [k for k in params if k.endswith("gate_layer.linear_layer.bias")][0]
        params[key] = torch.full_like(params[key], gate_bias)
    F, model = ref_shims.reference_model(cfg, params)
    g = torch.Generator().manual_seed(seed)
    residual = torch.randn(B, 80, T, generator=g) * sigma
    text = torch.randint(0, cfg["n_text"], (B, L), generator=g)
    spk = torch.zeros(B, dtype=torch.long)
    with torch.no_grad():
        mel, attn = model.infer(residual, spk, text, temperature=1.0, gate_threshold=0.5)
    rec = dict(cfg_n_flows=n_flows, B=B, T=T, L=L, seed=seed, gate_bias=gate_bias, sigma=sigma,
               use_gate=int(use_gate), residual=residual.numpy(), text=text.numpy(), mel=mel.numpy())
    np.savez_compressed(os.path.join(OUT, f"infer_{tag}.npz"), **rec)
    print(f"infer_{tag}: frames out {mel.shape[-1]} of {T}")


def mel_case():
    AP = ref_shims.import_audio_processing()
    stft = AP.TacotronSTFT(1024, 256, 1024, 80, 22050, 0.0, 8000.0)
    g = torch.Generator().manual_seed(7)
    rec = {"mel_basis": stft.mel_basis.numpy()}
    # (1) first second of the only real audio in the reference tree; (2) noise; (3) short ragged lengths
    from scipy.io.wavfile import read
    sr, wav = read(os.path.join(ref_shims.REF, "tacotron2", "demo.wav"))
    wav = torch.from_numpy(np.asarray(wav)).float()
    if wav.abs().max() > 1.0:
        wav = wav / 32768.0
    sigs = {"demo": wav[:22050][None], "noise": (torch.rand(2, 8192, generator=g) * 1.9 - 0.95),
            "short": (torch.rand(1, 1300, generator=g) * 1.9 - 0.95),
            "quiet": (torch.rand(1, 4096, generator=g) * 2e-4 - 1e-4)}
    for k, y in sigs.items():
        rec[f"y_{k}"] = y.numpy()
        rec[f"mel_{k}"] = stft.mel_spectrogram(y).numpy()
    np.savez_compressed(os.path.join(OUT, "mel.npz"), **rec)
    print("mel: ", {k: tuple(rec[f'mel_{k}'].shape) for k in sigs})


def radam_case():
    """Trajectory of the UNMODIFIED reference optimizer (radam.py:25-122) preceded by train.py:326's clip, CPU fp32."""
    import warnings
    sys.path.insert(0, "/root/reference")
    from radam import RAdam
    g = torch.Generator().manual_seed(77)
    shapes = [(7, 5), (33,), (1,)]
    ps = [torch.nn.Parameter(torch.randn(*s, generator=g)) for s in shapes]
    opt = RAdam(ps, lr=1e-3, weight_decay=1e-6)
    rec = {"n_steps": np.int64(9), "max_norm": np.float32(1.0)}
    for i, p in enumerate(ps):
        rec[f"p0_{i}"] = p.detach().numpy().copy()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for s in range(9):                       # steps 1-5 take the N_sma < 5 branch, 6+ the adaptive one
            for i, p in enumerate(ps):
                p.grad = torch.randn(*shapes[i], generator=g) * (3.0 if s % 2 else 0.05)
                rec[f"g{s}_{i}"] = p.grad.numpy().copy()
            total = torch.nn.utils.clip_grad_norm_(ps, 1.0)
            rec[f"norm{s}"] = total.numpy().copy()
            opt.step()
            for i, p in enumerate(ps):
                rec[f"p{s + 1}_{i}"] = p.detach().numpy().copy()
    for i, p in enumerate(ps):
        rec[f"m_{i}"] = opt.state[p]["exp_avg"].numpy().copy()
        rec[f"v_{i}"] = opt.state[p]["exp_avg_sq"].numpy().copy()
    np.savez_compressed(os.path.join(OUT, "radam.npz"), **rec)
    print("radam: 9 steps recorded")


def host_layer_cases():
    """Reference outputs the CPU restatements of the data layer, the STFT and the forced-alignment infer branch are pinned
    against (tests/test_oracle_data.py, tests/test_abi_and_host.py), with the inputs that produced them."""
    import types
    cwd = os.getcwd()
    os.chdir(ref_shims.REF)                                 # text/__init__ opens data/cmudict_dictionary relative to the cwd
    try:
        ref_shims.import_audio_processing()                 # librosa stub before data.py imports audio_processing
        for name in ("unidecode", "inflect"):                # text-cleaning dependencies (absent here, unused by the collate)
            if name not in sys.modules:
                m = types.ModuleType(name)
                m.unidecode = lambda s: s
                m.engine = lambda: None
                sys.modules[name] = m
        sys.path.insert(0, ref_shims.REF)
        import data as RD
    finally:
        os.chdir(cwd)
    rec = {"prior_11_29": RD.beta_binomial_prior_distribution(11, 29, 1.0).numpy()}
    g = torch.Generator().manual_seed(0)
    batch = []
    for i, (F_, P_) in enumerate([(29, 11), (40, 17), (5, 17), (33, 3)]):
        item = (torch.randn(80, F_, generator=g), torch.LongTensor([F_ % 3]), torch.randint(1, 100, (P_,), generator=g),
                RD.beta_binomial_prior_distribution(P_, F_, 1.0))
        batch.append(item)
        for k, t in zip(("mel", "speaker", "text", "prior"), item):
            rec[f"in_{k}_{i}"] = t.numpy()
    for i, t in enumerate(RD.DataCollate(1, use_attn_prior=True)(batch)):
        rec[f"collate_{i}"] = t.numpy()
    np.savez_compressed(os.path.join(OUT, "data_collate.npz"), **rec)

    AP = ref_shims.import_audio_processing()
    g = torch.Generator().manual_seed(3)
    y = torch.rand(2, 3000, generator=g) * 1.9 - 0.95
    m, p = AP.STFT(1024, 256, 1024).transform(y)
    np.savez_compressed(os.path.join(OUT, "stft_transform.npz"), y=y.numpy(), magnitude=m.numpy(), phase=p.numpy())

    # AR_Step.infer / AR_Back_Step.infer with `attns` given (flowtron.py:585-588, 797)
    cfg = dict(synth.DEFAULT_MODEL_CONFIG, n_flows=2, use_gate_layer=False)
    F, model = ref_shims.reference_model(cfg, synth.synth_params(cfg, 17))
    g = torch.Generator().manual_seed(2)
    T, L = 10, 6
    residual = torch.randn(T, 1, 80, generator=g) * 0.5
    enc = torch.randn(L, 1, 640, generator=g)
    attns = torch.softmax(torch.randn(T, L, generator=g), -1)
    with torch.no_grad():
        r0, _ = model.flows[0].infer(residual, enc, attns)
        r1, _ = model.flows[1].infer(residual, enc, attns)
    np.savez_compressed(os.path.join(OUT, "ar_step_forced_attns.npz"), seed=np.int64(17), residual=residual.numpy(),
                        enc=enc.numpy(), attns=attns.numpy(), flow0=r0.numpy(), flow1=r1.numpy())

    # the reference's state_dict layout for the default config: key order and shapes
    cfg = dict(synth.DEFAULT_MODEL_CONFIG)
    F, model = ref_shims.reference_model(cfg, synth.synth_params(cfg, 5))
    sd = model.state_dict()
    rec = {"keys": np.array(list(sd.keys()))}
    rec.update({f"shape::{k}": np.array(v.shape, dtype=np.int64) for k, v in sd.items()})
    np.savez_compressed(os.path.join(OUT, "state_dict_layout.npz"), **rec)
    print("host layer: data_collate, stft_transform, ar_step_forced_attns, state_dict_layout")


def big_cases():
    """BASELINE-shape fixtures (VERDICT r1 #1): a T=1000 training step (cfg 2 shapes at the largest B the CPU reference
    finishes in minutes) and cfg-4 inference requests (T=400 default, T=1000), all 2-flow."""
    train_case("t1000", n_flows=2, B=4, T=1000, L=150, out_lens=[1000, 873, 640, 512], in_lens=[150, 134, 98, 79],
               with_prior=True, seed=2024, logmel_stats=True, store_attn=False)
    infer_case("b1_t400", n_flows=2, B=1, T=400, L=100, seed=11, gate_bias=-10.0)
    infer_case("b1_t1000", n_flows=2, B=1, T=1000, L=100, seed=12, gate_bias=-10.0)
    infer_case("b4nogate_t400", n_flows=2, B=4, T=400, L=100, seed=13, gate_bias=0.0, use_gate=False)


def main():
    assert ref_shims.available(), "needs /root/reference"
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    train_case("cfg1", n_flows=1, B=2, T=128, L=32, out_lens=[128, 100], with_prior=False, seed=1234)
    train_case("f2prior", n_flows=2, B=3, T=96, L=24, out_lens=[96, 61, 80], with_prior=True, seed=4321)
    train_case("f2ragged", n_flows=2, B=5, T=64, L=20, out_lens=[64, 1, 33, 64, 17], with_prior=False, seed=99)
    train_case("f2ctc", n_flows=2, B=3, T=80, L=20, out_lens=[80, 47, 66], with_prior=True, seed=777, ctc_weight=1.0)
    infer_case("b1", n_flows=2, B=1, T=48, L=20, seed=5, gate_bias=-10.0)
    infer_case("b1gate", n_flows=2, B=1, T=48, L=20, seed=6, gate_bias=0.25)
    infer_case("b4nogate", n_flows=2, B=4, T=32, L=16, seed=8, gate_bias=0.0, use_gate=False)
    mel_case()
    radam_case()
    host_layer_cases()
    big_cases()


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "radam":     # regenerate only the optimizer fixture
        radam_case()
    elif len(sys.argv) > 1 and sys.argv[1] == "host":    # only the data-layer / STFT / forced-alignment / layout fixtures
        host_layer_cases()
    elif len(sys.argv) > 1 and sys.argv[1] == "ctc":     # only the CTC-loss fixture
        torch.manual_seed(0)
        torch.set_num_threads(8)
        train_case("f2ctc", n_flows=2, B=3, T=80, L=20, out_lens=[80, 47, 66], with_prior=True, seed=777, ctc_weight=1.0)
    elif len(sys.argv) > 1 and sys.argv[1] == "big":     # only the BASELINE-shape fixtures (minutes of CPU time)
        torch.manual_seed(0)
        torch.set_num_threads(8)
        big_cases()
    else:
        main()

"""CPU: the C-ABI library loads and exports every symbol include/flowtron_b200.h declares; the host-side module
mirror keeps the reference's state_dict layout; product code never imports oracle/ and fails loudly on CPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from flowtron_b200 import synth


def test_library_exports_every_declared_symbol():
    from flowtron_b200 import _lib, build
    path = build.build()
    L = ctypes.CDLL(path)
    hdr = open(os.path.join(ROOT, "include", "flowtron_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(ft_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 15
    missing = [n for n in sorted(names) if not hasattr(L, n)]
    assert not missing, missing
    assert _lib.lib().ft_version() >= 100


def test_state_dict_layout_matches_reference_spec():
    from flowtron_b200.flowtron import Flowtron
    for n_flows in (1, 2, 3):
        cfg = dict(synth.DEFAULT_MODEL_CONFIG, n_flows=n_flows)
        m = Flowtron(**cfg)
        spec = synth.param_shapes(cfg)
        sd = m.state_dict()
        assert set(sd.keys()) == set(spec.keys())
        for k, v in sd.items():
            assert tuple(v.shape) == tuple(spec[k]), k
        m.load_state_dict(synth.synth_params(cfg, 3), strict=True)


def test_state_dict_loads_into_reference_and_back():
    """Against the reference model's state_dict layout for the default config (key order and shapes, written by
    tests/make_golden.py): a reference checkpoint loads strictly into ours, and ours has exactly its keys and shapes."""
    from flowtron_b200.flowtron import Flowtron
    gold = np.load(os.path.join(GOLDEN, "state_dict_layout.npz"), allow_pickle=False)
    ref_keys = [str(k) for k in gold["keys"]]
    ref_sd = {k: torch.zeros(tuple(int(d) for d in gold[f"shape::{k}"])) for k in ref_keys}
    cfg = dict(synth.DEFAULT_MODEL_CONFIG)
    ours = Flowtron(**cfg)
    ours.load_state_dict(synth.synth_params(cfg, 5), strict=True)
    ours.load_state_dict(ref_sd, strict=True)
    sd = ours.state_dict()
    assert list(sd.keys()) == ref_keys
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(ref_sd[k].shape), k


def test_product_path_fails_loudly_on_cpu():
    from flowtron_b200._lib import FlowtronB200Error
    from flowtron_b200.flowtron import Flowtron
    cfg = dict(synth.DEFAULT_MODEL_CONFIG, n_flows=1)
    m = Flowtron(**cfg).eval()
    b = synth.synth_batch(2, 8, 6, cfg, 1)
    with pytest.raises(FlowtronB200Error):
        m(b["mel"], b["speaker_ids"], b["text"], b["in_lens"], b["out_lens"])


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "flowtron_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


def test_encoder_matches_oracle_restatement():
    """The torch Encoder kept on the host side equals the oracle's explicit restatement (eval mode)."""
    from flowtron_b200.flowtron import Flowtron
    from oracle import flowtron_oracle as O
    cfg = dict(synth.DEFAULT_MODEL_CONFIG, n_flows=1)
    p = synth.synth_params(cfg, 9)
    m = Flowtron(**cfg)
    m.load_state_dict(p, strict=True)
    m.eval()
    b = synth.synth_batch(3, 8, 11, cfg, 2)
    with torch.no_grad():
        x = m.embedding(b["text"]).transpose(1, 2)
        ours = m.encoder(x, b["in_lens"])
        ref = O.encoder_forward(p, torch.nn.functional.embedding(b["text"], p["embedding.weight"]).transpose(1, 2), b["in_lens"])
        assert (ours - ref).abs().max().item() < 1e-5
        ours_i = m.encoder.infer(x[:1])
        ref_i = O.encoder_forward(p, x[:1], None, infer=True)
        assert (ours_i - ref_i).abs().max().item() < 1e-5


def test_default_switches_are_the_validated_configuration(monkeypatch):
    """The GPU validation of record (profiles/r2_*) ran with: encoder overlap ON, two-stream BiLSTM OFF, fused optimizer
    ON (capturable), layer pipeline ON (forward and BPTT), CUDA-graph step ON in bench.py.  Anything else is opt-in through the
    environment (DESIGN.md 4.9)."""
    import flowtron_b200.flowtron as F
    if "FT_ENC_OVERLAP" not in os.environ:                 # class attribute, read at import
        assert F.Flowtron.overlap_encoder is True
    monkeypatch.delenv("FT_ENC_STREAMS", raising=False)
    assert F.Encoder().two_streams is False
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'os.environ.get("FT_FUSED_OPT", "1")' in src
    csrc = open(os.path.join(ROOT, "flowtron_b200", "csrc", "ar_step.cu")).read()
    assert 'getenv("FT_PIPE_FWD"); v = (!e || atoi(e) != 0) ? 1 : 0' in csrc
    assert 'getenv("FT_PIPE_BWD"); v = (!e || atoi(e) != 0) ? 1 : 0' in csrc
    assert 'os.environ.get("FT_GRAPH", "1")' in src


def test_encoder_abi_host_side():
    """ft_encoder_*_bytes are pure host functions: sizes grow with the batch, an unsupported descriptor gives 0 and an error
    string (no GPU needed)."""
    from ctypes import byref
    from flowtron_b200 import _lib
    L = _lib.lib()
    small, big = _lib.encoder_desc(2, 16, True, 0.0), _lib.encoder_desc(32, 160, True, 0.5)
    for fn in (L.ft_encoder_saved_bytes, L.ft_encoder_fwd_scratch_bytes, L.ft_encoder_bwd_scratch_bytes):
        a, b = fn(byref(small)), fn(byref(big))
        assert 0 < a < b
    bad = _lib.encoder_desc(2, 16, True, 0.0)
    bad.C = 256
    assert L.ft_encoder_saved_bytes(byref(bad)) == 0
    assert b"512" in L.ft_last_error()
    # the weight / gradient structs have one pointer per reference parameter of Encoder (flowtron.py:473-490)
    assert sum(k for _, k in _lib.ENC_PARAM_FIELDS) == 20

"""Import the UNMODIFIED reference modules on CPU: from the reference tree (``FLOWTRON_REFERENCE``; used by
tests/make_golden.py to generate the fixtures the tests compare against), or from their byte-compiled staging in
oracle/_ref/ (oracle/build_ref.py), which ONLY bench.py's reference arm / cpu_baseline leg may use (no test and not
smoke() reads the reference).  Shims (SURVEY.md §8c / Appendix B):
  1. flowtron.get_mask_from_lengths hard-codes torch.cuda.LongTensor (flowtron.py:48) -> arange version;
  2. AR_Step.infer allocates torch.cuda.FloatTensor (flowtron.py:785) -> alias to torch.FloatTensor;
  3. audio_processing imports librosa (absent here) -> stub providing filters.mel / util.pad_center /
     util.tiny / util.normalize from oracle.stft_oracle (the restated published algorithm).
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("FLOWTRON_REFERENCE", "/root/reference")
if not os.path.isfile(os.path.join(REF, "flowtron.py")):
    # GPU box: the byte-compiled reference modules staged by oracle/build_ref.py (bench.py's reference arm only)
    REF = os.path.join(_HERE, "_ref")


def available() -> bool:
    """The reference tree itself (build container): fixtures may only be generated from this."""
    return os.path.isfile(os.path.join(REF, "flowtron.py"))


def runnable() -> bool:
    """The reference modules can be imported: the tree, or its byte-compiled staging in oracle/_ref/."""
    return available() or os.path.isfile(os.path.join(REF, "flowtron.pyc"))


def import_flowtron():
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import flowtron as F  # noqa: the reference module

    def _mask(lengths):
        max_len = int(torch.max(lengths).item())
        ids = torch.arange(0, max_len, device=lengths.device, dtype=torch.long)
        return (ids < lengths.unsqueeze(1)).bool()

    F.get_mask_from_lengths = _mask
    F.get_gate_mask_from_lengths = _mask
    # the reference is only ever RUN ON THE CPU here (fixtures, CPU baseline): AR_Step.infer allocates its first frame as
    # torch.cuda.FloatTensor (flowtron.py:785), which on a GPU box would land on cuda:0 while the model sits on the host
    torch.cuda.FloatTensor = torch.FloatTensor
    return F


def import_audio_processing():
    from . import stft_oracle as so
    if "librosa" not in sys.modules:
        lib = types.ModuleType("librosa")
        filt = types.ModuleType("librosa.filters")
        util = types.ModuleType("librosa.util")
        filt.mel = lambda sr, n_fft, n_mels=128, fmin=0.0, fmax=None: so.slaney_mel_basis(sr, n_fft, n_mels, fmin, fmax)
        util.pad_center = lambda data, size: so.pad_center(np.asarray(data), size)
        util.tiny = lambda x: np.finfo(np.asarray(x).dtype if np.issubdtype(np.asarray(x).dtype, np.floating) else np.float32).tiny
        util.normalize = lambda S, norm=np.inf, **kw: S / max(np.max(np.abs(S)), 1e-30) if norm is not None else S
        lib.filters, lib.util = filt, util
        sys.modules["librosa"] = lib
        sys.modules["librosa.filters"] = filt
        sys.modules["librosa.util"] = util
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import audio_processing as AP  # noqa
    return AP


def reference_model(cfg: dict, params: dict):
    """Build reference Flowtron(**cfg) and load ``params`` strictly."""
    F = import_flowtron()
    model = F.Flowtron(**cfg)
    missing, unexpected = model.load_state_dict(params, strict=True), None
    model.eval()
    return F, model

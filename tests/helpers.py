"""Shared test helpers (seeded inputs, RNG replay, fixtures)."""
from __future__ import annotations

import contextlib
import io
from pathlib import Path

import numpy as np
import torch

GOLDEN = Path(__file__).resolve().parent / "golden"

CTOR = dict(rnn_dims=512, fc_dims=512, bits=9, pad=2, upsample_factors=(5, 5, 11), feat_dims=80,
            compute_dims=128, res_out_dims=128, res_blocks=10, hop_length=275, sample_rate=22050)


def make_model(seed=0, mode="MOL", device="cpu"):
    """OUR WaveRNN, random-init under torch.manual_seed(seed) -- bit-identical to the reference's
    init under the same seed (checked against tests/golden/weights_*.npz)."""
    from wavernn_b200 import WaveRNN
    torch.manual_seed(seed)
    with contextlib.redirect_stdout(io.StringIO()):
        m = WaveRNN(mode=mode, **CTOR)
    m.gen_verbose = False
    return m.to(device)


def make_mel(T, seed=0):
    torch.manual_seed(seed)
    return torch.rand(1, 80, T)


def replay_uniforms(seed, S, B):
    """The draws the reference's generate() makes from torch's CPU generator (MOL):
    manual_seed -> two GRUCell constructions (fatchord_version.py:178-179) -> per step
    (1,B,10) then (1,B) uniform_(1e-5, 1-1e-5) (utils/distribution.py:106,118)."""
    torch.manual_seed(seed)
    torch.nn.GRUCell(512, 512)
    torch.nn.GRUCell(544, 512)
    return torch.empty(S, 11 * B).uniform_(1e-5, 1.0 - 1e-5).numpy()


def replay_expo(seed, S, B, n_classes):
    """RAW head: one exponential_() of shape (B, n_classes) per step (Categorical.sample ->
    torch.multinomial(n=1))."""
    torch.manual_seed(seed)
    torch.nn.GRUCell(512, 512)
    torch.nn.GRUCell(544, 512)
    e = torch.empty(S, B, n_classes)
    for t in range(S):
        e[t].exponential_()
    return e.numpy()


def state_numpy(model):
    return {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}


def weight_fingerprint(sd) -> dict:
    out = {}
    for k, v in sd.items():
        a = np.asarray(v, dtype=np.float64).ravel()
        out[k] = np.array([a.sum(), np.abs(a).sum(), a[0], a[-1]])
    return out


def sample_index(n, k, seed):
    """Sorted indices of a fixed, seeded sample of k out of n entries (the stored sample of a fixture too large to keep
    whole)."""
    return np.sort(np.random.default_rng(seed).choice(n, size=min(n, k), replace=False))


def first_exceed(diff, thr):
    """First step (axis -1) at which any row exceeds thr, or None."""
    bad = (np.abs(diff) > thr)
    while bad.ndim > 1:
        bad = bad.any(axis=0)
    return int(np.argmax(bad)) if bad.any() else None


def load_golden(name):
    return np.load(GOLDEN / name, allow_pickle=False)


def tacotron_mels():
    """The 16 Tacotron mels of BASELINE configs[3] (tests/golden/make_tacotron_mels.py), de-quantised: list of
    (80, T) float32 in [0, 1]."""
    g = load_golden("tacotron_mels.npz")
    return [g[f"mel_{i:02d}"].astype(np.float32) / np.float32(65535.0) for i in range(16)]


def mol_component_picks(logits, U):
    """Mixture component chosen per (step, fold) (utils/distribution.py:106-108): argmax(logit - log(-log u)) with the
    replayed draws U[S, 11*B].  logits (S, B, 30)."""
    S, B = logits.shape[:2]
    u = U[:S, :10 * B].reshape(S, B, 10).astype(np.float32)
    return np.argmax(logits[:, :, :10] - np.log(-np.log(u)), axis=-1)


def pretrained_state_dict():
    """state_dict of the reference's shipped LJSpeech checkpoint (fixture copy under tests/golden/pretrained)."""
    import zipfile
    with zipfile.ZipFile(GOLDEN / "pretrained" / "ljspeech.wavernn.mol.800k.zip") as z:
        blob = z.read("latest_weights.pyt")
    return torch.load(io.BytesIO(blob), map_location="cpu")

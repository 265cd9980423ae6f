"""Fixtures of the reference pins in tests/test_oracle_vs_reference.py and the reference-surface test in
tests/test_dropin_api.py, taken from the UNMODIFIED reference (needs a checkout of it, named by WAVERNN_REFERENCE):

    WAVERNN_REFERENCE=<checkout> python tests/golden/make_golden_pins.py [surface] [pretrained] [forward]

  pins_pretrained.npz  -- the reference's generate() with its shipped LJSpeech checkpoint (torch.rand mel T=30, seed 0;
                          target=2750 overlap=275, sampler seed 1234): raw (3, 3300) samples
  pins_forward.npz     -- the reference's training forward (`WaveRNN.forward`, what train_wavernn.py calls) on
                          random-init weights (seed 0), MOL and RAW heads, eval then train mode, then the gradient of
                          square().mean() of a third call.  Full outputs and gradients are too large to store
                          (RAW: 20 MB per output), so each is kept as a summary vector: sample seed, float64 sum and
                          sum of |x| of the whole tensor, then a fixed sample of its entries (helpers.sample_index);
                          the gradients' summaries are concatenated in named_parameters() order.  The state_dict after
                          the calls is kept whole for buffers and as helpers.weight_fingerprint for parameters
  reference_surface.json -- parameter names of the reference WaveRNN's public methods
"""
import json
import sys
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

from oracle import ref_shim  # noqa: E402
import helpers  # noqa: E402

SURFACE = ("__init__", "forward", "generate", "get_gru_cell", "pad_tensor", "fold_with_overlap", "xfade_and_unfold",
           "get_step", "log", "load", "save", "num_params", "gen_display")
N_SAMPLE = 2048          # sampled entries per output tensor
N_SAMPLE_GRAD = 64       # sampled entries per gradient tensor


def summarise(t: torch.Tensor, k: int, seed: int) -> np.ndarray:
    a = t.detach().double().numpy().ravel()
    return np.concatenate([[seed, a.sum(), np.abs(a).sum()], a[helpers.sample_index(a.size, k, seed)]])


def forward_pins(mode: str, out: dict):
    """The same calls, inputs and order as test_training_forward_equals_reference_forward."""
    ref_model = ref_shim.build_reference_model(seed=0, mode=mode)
    ours0 = helpers.make_model(0, mode)                    # the test takes its weights from here: must be the reference's
    for k, v in ref_model.state_dict().items():
        assert torch.equal(v, ours0.state_dict()[k]), k
    torch.manual_seed(5)
    mels = torch.rand(3, 80, 12 + 4)
    x = torch.rand(3, 12 * 275) * 2 - 1
    for train in (False, True):
        ref_model.train(train)
        out[f"{mode}.out_{'train' if train else 'eval'}"] = summarise(ref_model(x, mels), N_SAMPLE, 1 + train)
    out[f"{mode}.step"] = np.int64(ref_model.get_step())
    sd = ref_model.state_dict()
    params = [k for k, _ in ref_model.named_parameters()]
    buffers = [k for k in sd if k not in params]
    out[f"{mode}.param_keys"] = np.array(params)
    out[f"{mode}.param_fp"] = np.stack([helpers.weight_fingerprint({k: sd[k].numpy()})[k] for k in params])
    out[f"{mode}.buffer_keys"] = np.array(buffers)
    out[f"{mode}.buffers"] = np.concatenate([sd[k].double().numpy().ravel() for k in buffers])
    ref_model.zero_grad()
    ref_model(x, mels).square().mean().backward()
    out[f"{mode}.grad"] = np.concatenate([summarise(p.grad, N_SAMPLE_GRAD, 100 + i)
                                          for i, (_, p) in enumerate(ref_model.named_parameters())])


def main():
    only = sys.argv[1:] or ["surface", "pretrained", "forward"]
    ref = ref_shim.load_reference()
    import inspect
    surface = {name: list(inspect.signature(getattr(ref.WaveRNN, name)).parameters) for name in SURFACE}
    if "surface" in only:
        (HERE / "reference_surface.json").write_text(json.dumps(surface, indent=1) + "\n")
    if "pretrained" in only:
        pretrained_pins()
    if "forward" in only:
        out = {}
        for mode in ("MOL", "RAW"):
            forward_pins(mode, out)
        np.savez_compressed(HERE / "pins_forward.npz", **out)


def pretrained_pins():
    model = ref_shim.build_reference_model(seed=0, mode="MOL", pretrained=True)
    model.eval()
    ours = helpers.make_model(0, "MOL")                    # the test's weights: ours loading the committed checkpoint copy
    ours.load_state_dict(helpers.pretrained_state_dict(), strict=False)
    for k, v in model.state_dict().items():
        assert torch.equal(v, ours.state_dict()[k]), k
    r = ref_shim.ref_generate(model, helpers.make_mel(30, 0), True, 2750, 275, seed=1234)
    np.savez_compressed(HERE / "pins_pretrained.npz", T=30, mel_seed=0, target=2750, overlap=275, seed=1234, raw=r["raw"])


if __name__ == "__main__":
    main()

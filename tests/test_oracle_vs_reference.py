"""Pins of the oracle, the CPU timing port and the training forward against the UNMODIFIED reference, through what
the reference computed on the same seeded inputs (fixtures tests/golden/pins_*.npz and mol_batched.npz, generators
tests/golden/make_golden_pins.py and make_golden.py)."""
import numpy as np
import pytest
import torch

import helpers
from oracle import torch_port
from oracle import wavernn_oracle as O


def test_oracle_tracks_reference_with_pretrained_weights():
    """Trained weights make the sampler chaotic (SURVEY 7.2): agreement is a PREFIX property.  After the prefix the two
    runs are different draws of the same process, and one loud burst in either moves the std of 3 x 3300 samples by
    more than 20 % (it does on some hosts), so the level of the whole run is compared through the median |sample|."""
    g = helpers.load_golden("pins_pretrained.npz")
    model = helpers.make_model(0, "MOL")
    model.load_state_dict(helpers.pretrained_state_dict(), strict=False)
    model.eval()
    sd = helpers.state_numpy(model)
    mel = helpers.make_mel(int(g["T"]), int(g["mel_seed"]))
    U = helpers.replay_uniforms(1234, 3300, 3)
    wav, pre = O.generate(O.hot_weights(sd), sd, mel[0].numpy(), batched=True, target=2750, overlap=275,
                          uniforms=U, return_pre=True)
    ref_raw = g["raw"]
    d = np.abs(pre - ref_raw)
    assert d[:, :1000].max() < 1e-4
    level, ref_level = np.median(np.abs(pre)), np.median(np.abs(ref_raw))
    assert abs(level - ref_level) < 0.2 * ref_level


def test_torch_port_reproduces_reference_samples():
    """Same torch operators in the same order as the reference's loop: bit-identical on one host (bench.py's CPU arm
    relies on it).  The fixture comes from another host, whose CPU kernels sum in another order (last bits), and
    random-init weights keep that from growing."""
    g = helpers.load_golden("mol_batched.npz")
    model = helpers.make_model(0, "MOL")                   # bit-identical to the reference's init (test_oracle_golden.py)
    model.eval()
    mel = helpers.make_mel(30, 0)
    with torch.no_grad():
        mp = model.pad_tensor(mel.transpose(1, 2), pad=2, side="both").transpose(1, 2)
        m_up, aux = model.upsample(mp)
        mf, af = model.fold_with_overlap(m_up, 2750, 275), model.fold_with_overlap(aux, 2750, 275)
    torch.manual_seed(1234)
    out, _ = torch_port.generate_segments_torch({k: v.detach() for k, v in model.state_dict().items()}, mf, af)
    np.testing.assert_allclose(out, g["raw"], rtol=0, atol=1e-6)


def test_dropin_class_loads_pretrained_checkpoint():
    ours = helpers.make_model(0, "MOL")
    missing = ours.load_state_dict(helpers.pretrained_state_dict(), strict=False)
    assert not missing.missing_keys and not missing.unexpected_keys
    assert ours.get_step() == 797232


GRAD_SAMPLE = 64          # entries sampled per gradient (make_golden_pins.py: N_SAMPLE_GRAD)


def _assert_close_to_pin(pin, t, rtol, atol, what):
    """pin = the reference tensor's summary (make_golden_pins.py): sample seed, sum, sum of |x|, sampled entries.
    Elementwise |t - ref| <= atol + rtol*|ref| on the sampled entries; on the whole tensor the bound the same
    elementwise condition implies for the sum and the sum of |x|: sum(atol + rtol*|ref|)."""
    seed, ref_sum, ref_abssum, val = int(pin[0]), pin[1], pin[2], pin[3:]
    a = t.detach().double().numpy().ravel()
    np.testing.assert_allclose(a[helpers.sample_index(a.size, val.size, seed)], val, rtol=rtol, atol=atol, err_msg=what)
    bound = atol * a.size + rtol * ref_abssum
    assert abs(a.sum() - ref_sum) <= bound, what
    assert abs(np.abs(a).sum() - ref_abssum) <= bound, what


@pytest.mark.parametrize("mode", ["MOL", "RAW"])
def test_training_forward_equals_reference_forward(mode):
    """SURVEY 8f-4: `WaveRNN.forward(x, mels)` (reference :131-167, what train_wavernn.py:91-155 calls) on identical
    weights and inputs -- eval mode and train mode (BatchNorm batch statistics, running-stat updates, `step` counter)."""
    g = helpers.load_golden("pins_forward.npz")
    ref_init = helpers.make_model(0, mode)                 # the reference's init under seed 0 (make_golden_pins.py checks)
    ours = helpers.make_model(1, mode)                     # different init: everything must come from the state_dict
    ours.load_state_dict(ref_init.state_dict())
    torch.manual_seed(5)
    mels = torch.rand(3, 80, 12 + 4)                       # (B, 80, T + 2*pad)
    x = torch.rand(3, 12 * 275) * 2 - 1                    # (B, T*hop)
    for train in (False, True):
        ours.train(train)
        b = ours(x, mels)
        assert b.shape == (3, 12 * 275, 30 if mode == "MOL" else 512)
        _assert_close_to_pin(g[f"{mode}.out_{'train' if train else 'eval'}"], b, 0, 1e-6, f"train={train}")
    assert ours.get_step() == int(g[f"{mode}.step"])
    sb = ours.state_dict()
    params = [k for k, _ in ours.named_parameters()]
    buffers = [k for k in sb if k not in params]
    assert params == list(g[f"{mode}.param_keys"]) and buffers == list(g[f"{mode}.buffer_keys"])
    np.testing.assert_allclose(np.stack([helpers.weight_fingerprint({k: sb[k].numpy()})[k] for k in params]),
                               g[f"{mode}.param_fp"], rtol=0, atol=1e-6)
    # BatchNorm running statistics moved identically
    np.testing.assert_allclose(np.concatenate([sb[k].double().numpy().ravel() for k in buffers]), g[f"{mode}.buffers"],
                               rtol=0, atol=1e-6)
    # gradients of the training loss flow through the same parameters
    ours.zero_grad()
    ours(x, mels).square().mean().backward()
    pins, pos = g[f"{mode}.grad"], 0
    for k, p in ours.named_parameters():
        n = 3 + min(p.numel(), GRAD_SAMPLE)
        _assert_close_to_pin(pins[pos:pos + n], p.grad, 1e-4, 1e-7, k)
        pos += n
    assert pos == pins.size

"""Host-side mirror of the reference interface: WaveRNN surface, hparams singleton, fold /
xfade helpers, sliced conditioning, failure modes.  CPU only."""
import inspect
import io
import contextlib

import numpy as np
import pytest
import torch

import helpers
from oracle import wavernn_oracle as O


def test_ctor_state_dict_layout():
    m = helpers.make_model(0, "MOL")
    sd = m.state_dict()
    assert len(sd) == 148
    for k, shape in {"I.weight": (512, 113), "rnn1.weight_ih_l0": (1536, 512), "rnn2.weight_ih_l0": (1536, 544),
                     "fc1.weight": (512, 544), "fc2.weight": (512, 544), "fc3.weight": (30, 512),
                     "upsample.up_layers.5.weight": (1, 1, 1, 23), "step": (1,)}.items():
        assert tuple(sd[k].shape) == shape, k
    assert helpers.make_model(0, "RAW").state_dict()["fc3.weight"].shape == (512, 512)
    with pytest.raises(RuntimeError):
        helpers.make_model(0, "nope")
    assert m.training is True
    sig = list(inspect.signature(m.generate).parameters)
    assert sig == ["mels", "save_path", "batched", "target", "overlap", "mu_law"]


def test_generate_without_cuda_fails_loudly():
    m = helpers.make_model(0, "MOL")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.generate(helpers.make_mel(30), None, True, 2750, 275, False)


def test_fold_and_xfade_helpers_match_oracle():
    m = helpers.make_model(0, "MOL")
    x = torch.arange(1000 * 3, dtype=torch.float32).reshape(1, 1000, 3)
    np.testing.assert_array_equal(m.fold_with_overlap(x, 300, 30).numpy(), O.fold_with_overlap(x[0].numpy(), 300, 30))
    np.testing.assert_array_equal(m.fold_with_overlap(x[:, :1020], 300, 30).numpy(),
                                  O.fold_with_overlap(x[0, :1020].numpy(), 300, 30))
    y = np.random.RandomState(0).randn(5, 360)
    np.testing.assert_allclose(m.xfade_and_unfold(y.copy(), 300, 30), O.xfade_and_unfold(y, 300, 30), atol=1e-15)


def test_sliced_conditioning_equals_full_upsample():
    """Per-rank / chunked conditioning (halo slices) == one UpsampleNetwork call (:186).  Up to the last bits: torch's
    CPU convolution sums in an order that depends on the input length and the thread count."""
    m = helpers.make_model(0, "MOL").eval()
    mel = helpers.make_mel(61)
    mp = torch.nn.functional.pad(mel, (2, 2))
    with torch.no_grad():
        full_m, full_a = m.upsample(mp)
        m.gen_upsample_chunk = 16
        cm, ca = m.conditioning(mp, 0, 61)
        sm, sa = m.conditioning(mp, 20, 45)
    np.testing.assert_allclose(cm.numpy(), full_m[0].numpy(), atol=5e-6)
    np.testing.assert_allclose(ca.numpy(), full_a[0].numpy(), rtol=0, atol=2e-6)
    np.testing.assert_allclose(sm.numpy(), full_m[0, 20 * 275:45 * 275].numpy(), atol=5e-6)
    np.testing.assert_allclose(sa.numpy(), full_a[0, 20 * 275:45 * 275].numpy(), rtol=0, atol=2e-6)
    sd = helpers.state_numpy(m)
    om, oa = O.upsample_network(sd, mp[0].numpy(), pad=2)
    np.testing.assert_allclose(full_m[0].numpy(), om, atol=5e-6)
    np.testing.assert_allclose(full_a[0].numpy(), oa, atol=5e-6)


def test_forward_training_path_runs():
    m = helpers.make_model(0, "MOL")
    x = torch.rand(2, 275 * 3) * 2 - 1
    mel = torch.rand(2, 80, 3 + 4)
    out = m(x, mel)
    assert out.shape == (2, 825, 30) and m.get_step() == 1


def test_hparams_singleton_contract(tmp_path):
    from wavernn_b200.hp import _HParams, DEFAULT_HPARAMS_FILE
    hp = _HParams()
    with pytest.raises(AttributeError, match="not configured"):
        hp.sample_rate
    hp.configure(DEFAULT_HPARAMS_FILE)
    assert hp.sample_rate == 22050 and hp.voc_target == 11000 and hp.voc_overlap == 550 and hp.voc_mode == "MOL"
    with pytest.raises(RuntimeError, match="Cannot reconfigure"):
        hp.configure(DEFAULT_HPARAMS_FILE)
    with pytest.raises(FileNotFoundError):
        _HParams().configure(tmp_path / "nope.py")
    bad = tmp_path / "x.txt"; bad.write_text("a=1")
    with pytest.raises(ValueError):
        _HParams().configure(bad)


def test_save_load_roundtrip_and_wav(tmp_path):
    from wavernn_b200.dsp import save_wav, decode_mu_law
    m = helpers.make_model(0, "MOL")
    p = tmp_path / "w.pyt"
    m.save(p)
    m2 = helpers.make_model(1, "MOL")
    m2.load(p)
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k
    save_wav(np.linspace(-1, 1, 100), tmp_path / "a.wav", 22050)
    from scipy.io import wavfile
    sr, data = wavfile.read(tmp_path / "a.wav")
    assert sr == 22050 and data.dtype == np.float32 and len(data) == 100
    g = helpers.load_golden("functions.npz")
    np.testing.assert_allclose(decode_mu_law(g["mulaw_in"], 512, False), g["mulaw_out"], rtol=1e-15)


def test_public_surface_matches_reference_class():
    """Parameter names of the reference WaveRNN's methods (fixture tests/golden/reference_surface.json,
    generator tests/golden/make_golden_pins.py)."""
    import json
    import wavernn_b200 as W
    ref = json.loads((helpers.GOLDEN / "reference_surface.json").read_text())
    for name in ("forward", "generate", "get_gru_cell", "pad_tensor", "fold_with_overlap", "xfade_and_unfold",
                 "get_step", "log", "load", "save", "num_params", "gen_display"):
        assert ref[name] == list(inspect.signature(getattr(W.WaveRNN, name)).parameters), name
    assert ref["__init__"] == list(inspect.signature(W.WaveRNN.__init__).parameters)


def test_upsample_taps_reproduce_the_interpolation_cascade():
    """The 5-tap-per-phase table the kernel uses for in-kernel conditioning == UpsampleNetwork's stretch+conv cascade
    (reference fatchord_version.py:73-88), for freshly initialised and for perturbed (as-if-trained) conv weights."""
    m = helpers.make_model(0, "MOL").eval()
    for perturb in (False, True):
        if perturb:
            with torch.no_grad():
                for layer in m.upsample.up_layers:
                    if hasattr(layer, "weight"):
                        layer.weight.mul_(0.9).add_(0.01 * torch.randn_like(layer.weight))
        taps = m.upsample_taps(torch.device("cpu")).numpy().astype(np.float64)
        assert taps.shape == (275, 5) and (np.abs(taps) > 0).sum(1).max() <= 4
        T = 37
        mp = torch.nn.functional.pad(helpers.make_mel(T, 2), (2, 2))
        with torch.no_grad():
            full_m, full_a = m.upsample(mp)
            aux_fr = m.upsample.resnet(mp)[0].T.numpy()
        xp = mp[0].T.numpy().astype(np.float64)
        n = np.arange(T * 275)
        rec = sum(taps[n % 275, d][:, None] * xp[n // 275 + d] for d in range(5))
        np.testing.assert_allclose(rec, full_m[0].numpy(), atol=2e-6)
        np.testing.assert_array_equal(np.repeat(aux_fr, 275, 0), full_a[0].numpy())


@pytest.mark.parametrize("mode", ["MOL", "RAW"])
def test_native_generator_replay_equals_torch_operators(mode):
    """cabi.torch_rng_uniform / wrnn_mt19937_uniform: the native replay of torch's CPU generator gives the same
    draws as the reference's own sequence (two nn.GRUCell ctors, then uniform_ / exponential_) and leaves the
    generator in the same state."""
    import torch
    from wavernn_b200 import cabi
    from wavernn_b200.sharding import fold_geometry
    if not cabi.is_built():
        pytest.skip("library not built")
    assert cabi.torch_rng_replay_ok()
    model = helpers.make_model(0, mode, "cpu")
    geo = fold_geometry(30 * 275, 2750, 275)
    got = {}
    for native in (True, False):
        model.gen_native_rng = native
        torch.manual_seed(4321)
        torch.rand(77)                                   # start mid-block
        u, e = model._reference_draws(geo, 300 if mode == "MOL" else 5)
        got[native] = (u if u is not None else e, torch.rand(9))
    assert torch.equal(got[True][0], got[False][0]) and torch.equal(got[True][1], got[False][1])


def _epilogue_kernel_emulation(samples, stride, overlap, tabs, n_classes, wave_len, tail_len):
    """numpy restatement of csrc/wrnn_epilogue.cu (same table lookups, same order of float64 operations)."""
    B, S = samples.shape
    y = samples.astype(np.float64)
    if tabs["mu"] is not None:
        lbl = np.clip(np.rint((samples + np.float32(1)) * np.float32(0.5 * (n_classes - 1))).astype(np.int64), 0, n_classes - 1)
        y = tabs["mu"].numpy()[lbl]
    if overlap:
        y[:, :overlap] = y[:, :overlap] * tabs["fade_in"].numpy()
        y[:, S - overlap:] = y[:, S - overlap:] * tabs["fade_out"].numpy()
    n = np.arange(wave_len)
    i_hi = np.minimum(n // stride, B - 1)
    k_hi = n - i_hi * stride
    v = np.zeros(wave_len)
    lo = (i_hi >= 1) & (k_hi + stride < S)
    v[lo] = v[lo] + y[i_hi[lo] - 1, k_hi[lo] + stride]
    hi = k_hi < S
    v[hi] = v[hi] + y[i_hi[hi], k_hi[hi]]
    v[wave_len - tail_len:] = v[wave_len - tail_len:] * tabs["tail"].numpy()
    return v


@pytest.mark.parametrize("mode,batched,mu_law", [("MOL", True, False), ("MOL", False, False), ("RAW", True, True)])
def test_device_epilogue_tables_and_algorithm_equal_host_epilogue(mode, batched, mu_law):
    """The float64 tables handed to wrnn_epilogue + the kernel's gather formulation (each output sample = at most two
    fold samples, folds ascending) reproduce the reference's in-place cross-fade / overlap-add bit for bit.  (The CUDA
    kernel itself is checked against the host epilogue in tests/test_gpu_parity.py.)"""
    from wavernn_b200.sharding import fold_geometry, unbatched_geometry
    model = helpers.make_model(0, mode, "cpu")
    T, hop = 33, 275
    geo = fold_geometry(T * hop, 2750, 275) if batched else unbatched_geometry(T * hop)
    rs = np.random.RandomState(3)
    if mode == "RAW":
        samples = (np.float32(2) * rs.randint(0, 512, size=(geo.n_seg, geo.seg_len)).astype(np.float32) / np.float32(511) - np.float32(1))
    else:
        samples = rs.uniform(-1, 1, size=(geo.n_seg, geo.seg_len)).astype(np.float32)
    wave_len = (T - 1) * hop
    tabs = model._epilogue_tables(geo, batched, mu_law, torch.device("cpu"))
    got = _epilogue_kernel_emulation(samples, geo.seg_stride, geo.overlap if batched else 0, tabs, model.n_classes, wave_len, 20 * hop)
    want = model._epilogue(samples.astype(np.float64), geo, batched, wave_len, mu_law)
    assert np.array_equal(got, want)


def test_rank_local_draws_are_the_columns_of_the_full_draw_matrix():
    """Sharded jobs: every rank advances torch's generator over the WHOLE (steps, 11*B) matrix of the reference's draws
    but converts and keeps only its own folds' columns (wrnn_mt19937_uniform_cols)."""
    import torch
    from wavernn_b200 import cabi
    from wavernn_b200.sharding import fold_geometry, shard_folds
    if not cabi.is_built():
        pytest.skip("library not built")
    model = helpers.make_model(0, "MOL", "cpu")
    geo = fold_geometry(60 * 275, 2750, 275)            # 6 folds (the last one zero-padded)
    assert geo.n_seg == 6
    torch.manual_seed(77)
    full, _ = model._reference_draws(geo, 123)
    after = torch.rand(4)
    B = geo.n_seg
    for world in (2, 3, 8):                             # 8 ranks: some own no fold at all
        for rank in range(world):
            sh = shard_folds(geo, rank, world, 275)
            torch.manual_seed(77)
            loc, _ = model._reference_draws(geo, 123, shard=sh)
            f0, n = sh.seg_first, sh.n_seg
            want = torch.cat([full[:, 10 * f0:10 * (f0 + n)], full[:, 10 * B + f0:10 * B + f0 + n]], 1)
            assert loc.shape == (123, 11 * n) and torch.equal(loc, want), (world, rank)
            assert torch.equal(torch.rand(4), after)                     # generator left where the full draw leaves it


def test_kernel_conditioning_is_refused_for_geometries_the_tap_table_does_not_encode():
    """The reference accepts any voc_pad / voc_upsample_factors (fatchord_version.py:64-89).  The 5-tap frame-rate
    path is exact only for pad == 2 and an interpolation response that fits 5 frames; anything else must take the
    materialised torch conditioning (which equals the reference's upsample by construction)."""
    import contextlib, io
    from wavernn_b200 import WaveRNN
    base = dict(helpers.CTOR)

    def build(**over):
        with contextlib.redirect_stdout(io.StringIO()):
            return WaveRNN(mode="MOL", **{**base, **over})
    assert build()._kernel_conditioning_ok()
    assert not build(pad=1)._kernel_conditioning_ok()
    assert not build(pad=3)._kernel_conditioning_ok()
    wide = build(upsample_factors=(1, 5, 55))              # first factor 1: the response spans more than 5 frames
    assert wide.upsample.total_scale == 275 and not wide._kernel_conditioning_ok()
    # the fallback path is the reference layout for every one of them
    for m in (build(pad=1), build(pad=3), wide):
        m.eval()
        T = 9
        mp = torch.nn.functional.pad(helpers.make_mel(T, 1), (m.pad, m.pad))
        with torch.no_grad():
            want_m, want_a = m.upsample(mp)
            got_m, got_a = m.conditioning(mp, 0, T)
        np.testing.assert_allclose(got_m.numpy(), want_m[0].numpy(), atol=1e-6)
        np.testing.assert_allclose(got_a.numpy(), want_a[0].numpy(), atol=1e-6)


def test_raw_reference_draws_keep_only_the_local_folds_and_are_bounded():
    """RAW parity draws (one exponential_() of shape (B, 512) per step): a rank keeps its own folds' rows of the same
    stream, and an over-large request fails with a pointer to gen_rng='philox' instead of exhausting host memory."""
    from wavernn_b200.sharding import fold_geometry, shard_folds
    m = helpers.make_model(0, "RAW")
    m.gen_native_rng = False
    geo = fold_geometry(22 * 275, 550, 55)
    torch.manual_seed(3)
    _, full = m._reference_draws(geo, 40)
    assert full.shape == (40, geo.n_seg, 512)
    np.testing.assert_array_equal(full.numpy(), helpers.replay_expo(3, 40, geo.n_seg, 512))
    sh = shard_folds(geo, 1, 2, 275)
    torch.manual_seed(3)
    _, part = m._reference_draws(geo, 40, shard=sh)
    np.testing.assert_array_equal(part.numpy(), full[:, sh.seg_first:sh.seg_first + sh.n_seg].numpy())
    m.gen_max_draw_bytes = 1 << 20
    with pytest.raises(RuntimeError, match="philox"):
        m._reference_draws(geo, 660)


def test_streamed_draw_chunks_cover_the_steps_and_start_short(monkeypatch):
    """Streamed reference draws (vocoder.py::_streamed_draws): the chunk boundaries cover [0, steps] without gaps, no chunk
    exceeds `gen_draw_chunk` steps, and the first one (replayed before the launch, i.e. on the critical path) stays near
    128 k draws however many folds the job has; under serialised launches (CUDA_LAUNCH_BLOCKING=1, WRNN_STREAM_DRAWS=0)
    streaming is off -- the kernel would wait for rows an upload stream cannot deliver."""
    from wavernn_b200 import WaveRNN
    for steps, chunk, folds in ((12100, 1024, 19), (12100, 1024, 152), (3000, 1024, 4096), (2050, 1024, 1), (12100, 64, 19)):
        b = WaveRNN._draw_chunk_bounds(steps, chunk, folds)
        sizes = np.diff(b)
        assert b[0] == 0 and b[-1] == steps and (sizes > 0).all() and sizes.max() <= chunk
        assert sizes[0] * 11 * folds <= max(1 << 17, 8 * 11 * folds) or sizes[0] == 8
        assert all(sizes[i + 1] <= 2 * sizes[i] for i in range(len(sizes) - 2))       # doubling, never a jump
    model = helpers.make_model(0, "MOL")
    ok = lambda: model._can_stream_draws(12100, None, None)
    base = ok()                                         # False here when the library is not built; the guards below only ever turn it off
    monkeypatch.setenv("WRNN_STREAM_DRAWS", "0")
    assert ok() is False
    monkeypatch.delenv("WRNN_STREAM_DRAWS")
    monkeypatch.setenv("CUDA_LAUNCH_BLOCKING", "1")
    assert ok() is False
    monkeypatch.delenv("CUDA_LAUNCH_BLOCKING")
    assert ok() == base

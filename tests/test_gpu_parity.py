"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle
on the same seeded inputs, against the committed golden fixtures, and -- at BASELINE.json's
full batch -- through size-independent properties.

Tolerances (north_star: "decoded event-token ids matching the reference within fp32 logit
tolerance (mel frames within 1e-4 rel)"):
  mel frames   |mel - mel64| <= 1e-4 * mel64 + 1e-6 * max_bin(mel64[frame])   in the linear mel
               domain, i.e. 1e-4 relative plus the fp32 noise floor of the frame (leakage bins
               100+ dB below the partials carry the FFT's own fp32 rounding noise);
  logits       |l - l64| <= LOGIT_TOL * max|l64| with LOGIT_TOL = 5e-4, and never worse than
               4x what the fp32 *oracle* itself deviates from the fp64 oracle on that input;
  tokens       identical to the fp64 oracle's greedy tokens wherever its top-2 logit margin
               exceeds 2x the measured logit error (SURVEY 7.2-1).
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import mt3_oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
LOGIT_TOL = 5e-4
DEV = "cuda:0"


def _mel_close(lm_gpu: np.ndarray, lm64: np.ndarray):
    mel, mel64 = np.exp(lm_gpu.astype(np.float64)), np.exp(lm64)
    tol = 1e-4 * mel64 + 1e-6 * mel64.max(axis=-1, keepdims=True)
    err = np.abs(mel - mel64)
    worst = float((err / tol).max())
    assert worst <= 1.0, f"mel frames outside tolerance: worst err/tol = {worst:.3f}"
    return worst


@pytest.fixture(scope="module")
def spec_cfg():
    from mt3_b200 import spectrograms
    return spectrograms.SpectrogramConfig()


# ------------------------------------------------------------------------------------------------
# K1 log-mel
# ------------------------------------------------------------------------------------------------
def test_logmel_vs_oracle_and_golden(spec_cfg):
    from mt3_b200 import spectrograms
    audio = np.stack([O.sine_mix(32768, seed=1234 + i) for i in range(6)] +
                     [O.sine_mix(32768, seed=7)])
    lm = spectrograms.compute_spectrogram(torch.from_numpy(audio).to(DEV), spec_cfg).cpu().numpy()
    assert lm.shape == (7, 256, 512) and lm.dtype == np.float32
    lm64 = O.compute_spectrogram(audio.astype(np.float64), np.float64)
    _mel_close(lm, lm64)
    g = np.load(os.path.join(GOLD, "logmel_sine_seed7.npz"))
    _mel_close(lm[6][g["rows"]], g["logmel"])


def test_logmel_edge_cases(spec_cfg):
    from mt3_b200 import spectrograms
    rng = np.random.default_rng(3)
    # all-zero audio: safe_log's replace branch -> exactly log(1e-5)
    z = spectrograms.compute_spectrogram(torch.zeros(32768, device=DEV), spec_cfg).cpu().numpy()
    assert z.shape == (256, 512)
    np.testing.assert_allclose(z, np.log(np.float32(1e-5)), rtol=1e-6)
    # full-scale white noise
    noise = rng.uniform(-1, 1, 32768).astype(np.float32)
    ln = spectrograms.compute_spectrogram(torch.from_numpy(noise).to(DEV), spec_cfg).cpu().numpy()
    _mel_close(ln, O.compute_spectrogram(noise.astype(np.float64), np.float64))
    # ragged length (not a multiple of hop) against the committed fixture
    g = np.load(os.path.join(GOLD, "logmel_noise_5000.npz"))
    lr = spectrograms.compute_spectrogram(torch.from_numpy(g["audio"]).to(DEV), spec_cfg).cpu().numpy()
    assert lr.shape == (40, 512)
    _mel_close(lr, g["logmel"])
    # 1 sample, and empty input (tf.signal.frame gives 1 frame / 0 frames)
    one = spectrograms.compute_spectrogram(torch.full((1,), 0.5, device=DEV), spec_cfg).cpu().numpy()
    assert one.shape == (1, 512)
    _mel_close(one, O.compute_spectrogram(np.full((1,), 0.5), np.float64))
    empty = spectrograms.compute_spectrogram(torch.zeros((3, 0), device=DEV), spec_cfg)
    assert tuple(empty.shape) == (3, 0, 512)
    # short last segment: rows past n_valid are the feature converter's 0.0 padding (models.py:96)
    a = torch.from_numpy(np.stack([O.sine_mix(32768, 1), O.sine_mix(32768, 2)])).to(DEV)
    a[1, 229 * 128:] = 0
    nv = torch.tensor([256, 229], dtype=torch.int32, device=DEV)
    lv = spectrograms.compute_spectrogram(a, spec_cfg, n_valid_frames=nv).cpu().numpy()
    assert (lv[1, 229:] == 0).all() and (lv[0] != 0).any()
    short = O.compute_spectrogram(a[1, :229 * 128].cpu().numpy().astype(np.float64), np.float64)
    _mel_close(lv[1, :229], short)
    # strided rows
    big = torch.zeros((4, 40000), device=DEV)
    big[:, :32768] = a[0]
    ls = spectrograms.compute_spectrogram(big[:, :32768], spec_cfg).cpu().numpy()
    np.testing.assert_array_equal(ls[2], lv[0])


def test_logmel_shift_property_full_batch(spec_cfg):
    """Size-independent property at the full B=64: a frame's output depends only on its own 2048
    samples, so shifting a segment by k hops shifts the frames bit-exactly."""
    from mt3_b200 import spectrograms
    audio = np.stack([O.sine_mix(32768 + 5 * 128, seed=100 + i) for i in range(64)])
    a = torch.from_numpy(audio).to(DEV)
    base = spectrograms.compute_spectrogram(a[:, :32768], spec_cfg)
    shifted = spectrograms.compute_spectrogram(a[:, 5 * 128:], spec_cfg)
    # frames whose 2048-sample window lies inside both views
    n_ok = 256 - 16 - 5
    assert torch.equal(base[:, 5:5 + n_ok], shifted[:, :n_ok])


# ------------------------------------------------------------------------------------------------
# Encoder / decoder
# ------------------------------------------------------------------------------------------------
MODEL_MODES = [("simt", "f32"), ("tf32x3", "f32"), ("tf32x3", "f16"), ("tf32x3", "p24")]   # the last one is what bench.py times


def _mode_ids(mode):
    from mt3_b200 import _lib
    gm = {"simt": _lib.GEMM_FP32_SIMT, "tf32x3": _lib.GEMM_TF32X3, "tf32": _lib.GEMM_TF32}[mode[0]]
    kv = {"f32": _lib.KV_F32, "f16": _lib.KV_F16, "p24": _lib.KV_P24}[mode[1]]
    return gm, kv


def _mt3_cfg(**kw):
    from mt3_b200 import network
    d = dict(vocab_size=1536, emb_dim=512, num_heads=6, num_encoder_layers=8, num_decoder_layers=8, head_dim=64, mlp_dim=1024,
             mlp_activations=('gelu', 'linear'))
    d.update(kw)
    return network.T5Config(**d)


@pytest.fixture(scope="module", params=MODEL_MODES, ids=lambda m: f"{m[0]}-kv{m[1]}")
def mt3_model(request):
    """The full mt3 model at B = 64, T = 256, L = 1024 in every arithmetic configuration the library ships:
    exact-fp32 SIMT GEMMs (parity anchor), tcgen05 3xTF32 GEMMs + tcgen05 attention with fp32 K/V, and the same with
    fp16 K/V rows, or 24-bit rows -- the configuration bench.py times."""
    from mt3_b200 import network
    gm, kv = _mode_ids(request.param)
    ocfg = O.T5Config()
    params = O.init_params(ocfg, seed=0, norm_scale_jitter=0.05)
    model = network.Transformer(_mt3_cfg(), params, device=DEV, max_batch=64, max_input_length=256, max_decode_length=1024,
                                gemm_mode=gm, kv_format=kv)
    model.mode = request.param
    yield model, ocfg, params
    del model
    torch.cuda.empty_cache()


def _inputs(b, t=256, seed=0):
    audio = np.stack([O.sine_mix(t * 128, seed=1234 + seed + i) for i in range(b)])
    return O.compute_spectrogram(audio, np.float32)


def test_encoder_parity(mt3_model):
    model, ocfg, params = mt3_model
    x = _inputs(2)
    enc = model.encode(torch.from_numpy(x).to(DEV)).cpu().numpy()
    enc64 = O.encode(params, ocfg, x, np.float64)
    enc32 = O.encode(params, ocfg, x, np.float32)
    scale = np.abs(enc64).max()
    e_gpu, e_f32 = np.abs(enc - enc64).max() / scale, np.abs(enc32 - enc64).max() / scale
    print(f"encoder: gpu vs fp64 {e_gpu:.3e}   fp32-oracle vs fp64 {e_f32:.3e}")
    assert e_gpu <= max(LOGIT_TOL, 4 * e_f32)
    if model.mode[0] == "simt":
        assert e_gpu <= 4 * e_f32 + 1e-5, "CUDA encoder is much less accurate than the reference's fp32 arithmetic"


def test_decoder_teacher_forced_logits_and_tokens(mt3_model):
    model, ocfg, params = mt3_model
    x = _inputs(2, seed=10)
    enc64 = O.encode(params, ocfg, x, np.float64)
    steps = 12
    toks64, logits64 = O.greedy_decode(params, ocfg, enc64, steps, np.float64, stop_at_eos=False, return_logits=True)
    dec_in = np.concatenate([np.zeros((2, 1), np.int64), toks64[:, :steps - 1]], axis=1)
    _, logits32 = O.greedy_decode(params, ocfg, enc64.astype(np.float32), steps, np.float32, stop_at_eos=False,
                                  return_logits=True, forced_tokens=dec_in)
    enc_gpu = model.encode(torch.from_numpy(x).to(DEV))
    lg = model.teacher_forced_logits(enc_gpu, torch.from_numpy(dec_in).to(DEV).to(torch.int32)).cpu().numpy()
    scale = np.abs(logits64).max()
    e_gpu, e_f32 = np.abs(lg - logits64).max() / scale, np.abs(logits32 - logits64).max() / scale
    print(f"logits: gpu vs fp64 {e_gpu:.3e}   fp32-oracle vs fp64 {e_f32:.3e}")
    assert e_gpu <= max(LOGIT_TOL, 4 * e_f32)
    # free-running greedy tokens where the margin allows
    out = model.generate(torch.from_numpy(x).to(DEV), num_steps=steps, stop_at_eos=False, use_graph=False).cpu().numpy()
    srt = np.sort(logits64, axis=-1)
    margin = srt[..., -1] - srt[..., -2]
    safe = np.cumprod(margin > 2 * e_gpu * scale, axis=1).astype(bool)     # only up to the first risky step
    np.testing.assert_array_equal(out[:, :steps][safe], toks64[:, :steps][safe])
    assert (out[:, steps:] == 0).all()


@pytest.fixture(scope="module")
def long_decode_oracle():
    """float64 teacher-forced logits over 1024 positions (one numpy pass, layers.py:246-314 in its full-sequence form)
    at the positions the long-cache tests probe, plus the float32 oracle's own deviation there."""
    ocfg = O.T5Config()
    params = O.init_params(ocfg, seed=0, norm_scale_jitter=0.05)
    x = _inputs(2, seed=40)
    enc64 = O.encode(params, ocfg, x, np.float64)
    rng = np.random.default_rng(12)
    toks = rng.integers(3, 1500, size=(2, 1024))
    toks[:, 0] = 0
    probe = np.array(LONG_PROBE)
    l64 = O.decode_teacher_forced(params, ocfg, enc64, toks, np.float64)[:, probe]
    l32 = O.decode_teacher_forced(params, ocfg, enc64.astype(np.float32), toks, np.float32)[:, probe]
    return x, enc64, toks, l64, float(np.abs(l32 - l64).max() / np.abs(l64).max())


LONG_PROBE = [0, 1, 31, 32, 63, 64, 65, 191, 192, 257, 383, 511, 512, 767, 1022, 1023]


def test_decoder_long_cache_teacher_forced(mt3_model, long_decode_oracle):
    """The regime bench.py times: KV-cache lengths up to 1024 (32 fp32 / 16 fp16 K tiles and as many V tiles through the
    6-stage ring of dec_attention_bulk_kernel, 1024 scores in shared memory, the fused append at every position) against
    the float64 oracle at cache positions 63, 257, 511, 1023 and at the tile boundaries around them."""
    model, ocfg, params = mt3_model
    x, enc64, toks, l64, e_f32 = long_decode_oracle
    enc_gpu = model.encode(torch.from_numpy(x).to(DEV))
    model.init_cache(enc_gpu)
    t = torch.from_numpy(toks).to(DEV).to(torch.int32)
    got = {}
    for i in range(1024):
        lg = model.decode(enc_gpu, None, t[:, i:i + 1])
        if i in LONG_PROBE:
            got[i] = lg[:, 0].cpu().numpy()
    scale = np.abs(l64).max()
    errs = np.array([np.abs(got[p] - l64[:, j]).max() / scale for j, p in enumerate(LONG_PROBE)])
    print(f"long-cache logits [{model.mode}]: gpu vs fp64 per probe " + " ".join(f"{p}:{e:.1e}" for p, e in zip(LONG_PROBE, errs)) +
          f"   fp32-oracle vs fp64 {e_f32:.1e}")
    assert errs.max() <= LOGIT_TOL, (model.mode, errs)
    if model.mode[1] in ("f32", "p24"):   # fp32 / 24-bit K/V rows: as accurate as the reference's own float32 arithmetic
        assert errs.max() <= max(4 * e_f32, 2e-5), (model.mode, errs, e_f32)
    # the argmax agrees with the oracle wherever the oracle's top-2 margin exceeds twice the measured error
    srt = np.sort(l64, axis=-1)
    for j, p in enumerate(LONG_PROBE):
        safe = (srt[:, j, -1] - srt[:, j, -2]) > 2 * errs[j] * scale
        np.testing.assert_array_equal(got[p].argmax(-1)[safe], l64[:, j].argmax(-1)[safe])


def test_encoder_full_batch_vs_oracle(mt3_model):
    """B = 64, T = 256: the M = 16384-row tcgen05 GEMMs and the persistent attention kernel's multi-item loop (768 work items
    on 148 CTAs) against the float64 oracle on sequences 0, 17 and 63 (segments are independent, so the oracle only
    needs those three)."""
    model, ocfg, params = mt3_model
    x = _inputs(64, seed=900)
    enc = model.encode(torch.from_numpy(x).to(DEV)).cpu().numpy()
    pick = [0, 17, 63]
    enc64 = O.encode(params, ocfg, x[pick], np.float64)
    enc32 = O.encode(params, ocfg, x[pick], np.float32)
    scale = np.abs(enc64).max()
    e_gpu, e_f32 = np.abs(enc[pick] - enc64).max() / scale, np.abs(enc32 - enc64).max() / scale
    print(f"encoder B=64 [{model.mode}]: gpu vs fp64 {e_gpu:.3e}   fp32-oracle vs fp64 {e_f32:.3e}")
    assert e_gpu <= max(LOGIT_TOL, 4 * e_f32)
    if model.mode[0] == "simt":
        assert e_gpu <= 4 * e_f32 + 1e-5
    # and the decoder on top of it: 4 teacher-forced steps at B = 64 (M = 64-row decode GEMMs, 384 attention CTAs)
    toks = np.random.default_rng(5).integers(3, 1500, size=(64, 4))
    toks[:, 0] = 0
    lg = model.teacher_forced_logits(torch.from_numpy(enc).to(DEV), torch.from_numpy(toks).to(DEV).to(torch.int32)).cpu().numpy()
    l64 = O.decode_teacher_forced(params, ocfg, enc64, toks[pick], np.float64)
    e_l = np.abs(lg[pick] - l64).max() / np.abs(l64).max()
    print(f"logits B=64 [{model.mode}]: gpu vs fp64 {e_l:.3e}")
    assert e_l <= LOGIT_TOL


@pytest.mark.parametrize("attn", ["tc", "simt"])
def test_encoder_parity_t512_ismir2021(attn, monkeypatch):
    """ismir2021's input length (gin/ismir2021.gin:4): T = 512 keys do not fit one pass of the tcgen05 attention kernel (512 + 64
    TMEM columns), so it runs two key parts of 256 and merges them (softmax is associative over key blocks); against the
    float64 oracle, and against the exact-fp32 SIMT attention kernel on the same GEMMs."""
    from mt3_b200 import _lib, network
    monkeypatch.setenv("MT3_TC_ATTENTION", "1" if attn == "tc" else "0")
    ocfg = O.T5Config(vocab_size=1664, num_encoder_layers=3, num_decoder_layers=1)
    params = O.init_params(ocfg, seed=3, norm_scale_jitter=0.05)
    cfg = _mt3_cfg(vocab_size=1664, num_encoder_layers=3, num_decoder_layers=1)
    m = network.Transformer(cfg, params, device=DEV, max_batch=3, max_input_length=512, max_decode_length=8, gemm_mode=_lib.GEMM_TF32X3)
    x = _inputs(3, t=512, seed=60)
    enc = m.encode(torch.from_numpy(x).to(DEV)).cpu().numpy()
    enc64 = O.encode(params, ocfg, x, np.float64)
    scale = np.abs(enc64).max()
    e = np.abs(enc - enc64).max() / scale
    print(f"encoder T=512 [{attn}]: gpu vs fp64 {e:.3e}")
    assert e <= 2e-5


def test_model_tiny_golden_fixture():
    """Committed oracle fixture (mt3 layer sizes, 1+1 layers, T=32)."""
    from mt3_b200 import network
    g = np.load(os.path.join(GOLD, "model_tiny.npz"))
    ocfg = O.T5Config(vocab_size=1536, num_encoder_layers=1, num_decoder_layers=1)
    params = O.init_params(ocfg, seed=int(g["weight_seed"]), norm_scale_jitter=float(g["jitter"]))
    cfg = network.T5Config(vocab_size=1536, emb_dim=512, num_heads=6, num_encoder_layers=1, num_decoder_layers=1,
                           head_dim=64, mlp_dim=1024, mlp_activations=('gelu', 'linear'))
    m = network.Transformer(cfg, params, device=DEV, max_batch=2, max_input_length=32, max_decode_length=16)
    x = torch.from_numpy(g["x"]).to(DEV)
    enc = m.encode(x)
    np.testing.assert_allclose(enc.cpu().numpy()[:, ::8, ::16], g["encoded"], rtol=1e-3, atol=2e-4)
    dec_in = np.concatenate([np.zeros((2, 1), np.int64), g["tokens"][:, :5]], axis=1)
    lg = m.teacher_forced_logits(enc, torch.from_numpy(dec_in).to(DEV).to(torch.int32)).cpu().numpy()
    assert np.abs(lg[:, :, ::16] - g["logits"]).max() <= LOGIT_TOL * np.abs(g["logits"]).max()
    toks = m.generate(x, num_steps=6, stop_at_eos=False, use_graph=True).cpu().numpy()
    np.testing.assert_array_equal(toks[:, :6], g["tokens"])


def _eos_params(ocfg, seed, boost):
    """Random weights never emit EOS at a useful rate; scaling the EOS column of logits_dense
    makes EOS win whenever its projection is positive, so sequences end at scattered steps."""
    p = O.init_params(ocfg, seed=seed)
    w = p["decoder/logits_dense/kernel"].copy()
    w[:, O.EOS_ID] *= boost
    p["decoder/logits_dense/kernel"] = w
    return p


@pytest.mark.parametrize("pdl", ["0", "1"])
def test_generate_eos_semantics_and_graph_equivalence(pdl, monkeypatch):
    """pdl=1: the decode-step kernels are chained with programmatic dependent launch (weights / cross
    K/V are prefetched before griddepcontrol.wait); results must be bit-identical to pdl=0."""
    from mt3_b200 import network
    monkeypatch.setenv("MT3_PDL", pdl)
    ocfg = O.T5Config(vocab_size=1536, num_encoder_layers=2, num_decoder_layers=2)
    params = _eos_params(ocfg, seed=9, boost=6.0)
    cfg = network.T5Config(vocab_size=1536, emb_dim=512, num_heads=6, num_encoder_layers=2, num_decoder_layers=2,
                           head_dim=64, mlp_dim=1024, mlp_activations=('gelu', 'linear'))
    L = 48
    m = network.Transformer(cfg, params, device=DEV, max_batch=4, max_input_length=64, max_decode_length=L)
    x = _inputs(4, t=64, seed=50)
    enc64 = O.encode(params, ocfg, x, np.float64)
    ref = O.greedy_decode(params, ocfg, enc64, L, np.float64, stop_at_eos=True)
    has_eos = (ref == O.EOS_ID).any(axis=1)
    assert has_eos.any(), "test weights did not produce any EOS; raise the boost"
    xg = torch.from_numpy(x).to(DEV)
    t_plain = m.generate(xg, stop_at_eos=True, use_graph=False).cpu().numpy()
    steps_plain = m.last_steps_run
    t_graph = m.generate(xg, stop_at_eos=True, use_graph=True).cpu().numpy()
    t_full = m.generate(xg, stop_at_eos=False, use_graph=True).cpu().numpy()
    np.testing.assert_array_equal(t_plain, t_graph)
    np.testing.assert_array_equal(t_plain, t_full)          # finished sequences keep emitting PAD
    if has_eos.all():
        assert steps_plain < L                               # the loop really stopped early
    # zeros after the first EOS, identical prefix to the oracle where margins are safe
    for b in range(4):
        row = t_plain[b]
        if (row == 1).any():
            first = int(np.argmax(row == 1))
            assert (row[first + 1:] == 0).all()
    _, logits64 = O.greedy_decode(params, ocfg, enc64, L, np.float64, stop_at_eos=False, return_logits=True)
    srt = np.sort(logits64, axis=-1)
    safe = np.cumprod((srt[..., -1] - srt[..., -2]) > 1e-3 * np.abs(logits64).max(), axis=1).astype(bool)
    ref_full = O.greedy_decode(params, ocfg, enc64, L, np.float64, stop_at_eos=False)
    alive = np.cumsum(ref_full == 1, axis=1) - (ref_full == 1) == 0   # up to and including first EOS
    sel = safe & alive
    np.testing.assert_array_equal(t_plain[sel], ref_full[sel])
    # vocabulary decode kernel == oracle (vocabularies.py:241-271)
    from mt3_b200 import vocabularies
    vocab = vocabularies.GenericTokenVocabulary(1388, extra_ids=100)
    dec = vocab.decode_tf(torch.from_numpy(t_plain).to(DEV)).cpu().numpy()
    np.testing.assert_array_equal(dec, O.vocab_decode(t_plain, 1388))


@pytest.mark.parametrize("seed,boost", [(9, 4.0), (11, 2.5)])
def test_generate_beam1_matches_t5x_beam_search_restatement(seed, boost):
    """MT3_GEN_BEAM1: T5X decoding.beam_search at num_decodes=1 (the reference's decode_fn, models.py:127) on the device,
    against oracle/beam_search.py driven by the float64 oracle's step logits.  EOS-boosted weights make EOS compete at
    scattered steps, so some sequences end where greedy ends, some earlier (a runner-up EOS with a better normalised
    score) and some later (a first-ranked EOS that loses to a later finish)."""
    from mt3_b200 import network
    from oracle import beam_search as BS
    ocfg = O.T5Config(vocab_size=1536, num_encoder_layers=2, num_decoder_layers=2)
    params = _eos_params(ocfg, seed=seed, boost=boost)       # chosen so that one of the 8 sequences ends elsewhere than greedy's
    cfg = _mt3_cfg(num_encoder_layers=2, num_decoder_layers=2)
    L, Bn = 48, 8
    m = network.Transformer(cfg, params, device=DEV, max_batch=Bn, max_input_length=64, max_decode_length=L)
    x = _inputs(Bn, t=64, seed=50)
    enc64 = O.encode(params, ocfg, x, np.float64)
    p64 = O._cast(params, np.float64)
    state = O.init_decode_state(ocfg, Bn, L, np.float64)
    margins = []

    def logits_fn(prefixes, step):          # K = 1: the live prefix only ever grows, so the oracle's KV cache can be reused
        assert prefixes.shape[1] == 1 and state.position_index == step
        cur = prefixes[:, 0, step - 1] if step > 0 else np.zeros((Bn,), np.int64)
        lg = O.decode_step(p64, ocfg, enc64, cur, state)
        margins.append(lg)
        return lg[:, None, :]

    want, score = BS.beam_search(logits_fn, Bn, L, eos_id=O.EOS_ID, num_decodes=1)
    xg = torch.from_numpy(x).to(DEV)
    got = m.generate(xg, stop_at_eos=False, use_graph=True, decode='beam1').cpu().numpy()
    got_stop = m.generate(xg, stop_at_eos=True, use_graph=False, decode='beam1').cpu().numpy()
    greedy = m.generate(xg, stop_at_eos=True, use_graph=True).cpu().numpy()
    np.testing.assert_array_equal(got, got_stop)                 # graph replay == plain launches, early stop changes nothing
    n_diff = int((got != greedy).any(axis=1).sum())
    print(f"beam1: {n_diff} of {Bn} sequences differ from greedy; lengths beam1 {[(int(np.argmax(r == 1)) if (r == 1).any() else -1) for r in got]}"
          f" greedy {[(int(np.argmax(r == 1)) if (r == 1).any() else -1) for r in greedy]}")
    np.testing.assert_array_equal(got, want)
    assert n_diff > 0, "the crafted weights should make beam-1 and greedy disagree somewhere"


@pytest.mark.parametrize("kv", ["f32", "f16", "p24"])
@pytest.mark.parametrize("gm,pdl,cluster", [("tf32x3", "0", "1"), ("tf32x3", "1", "1"), ("tf32x3", "6", "1"), ("simt", "1", "1"),
                                            ("simt", "2", "0")])
def test_decode_variants(gm, pdl, cluster, kv, monkeypatch):
    """The remaining scheduling switches, under the tensor-core encoder (tf32x3) and the exact-fp32 one (simt).
    MT3_PDL only changes when kernels start (default 2: attention launches): tokens AND logits are bit-identical to the
    default path.  MT3_DEC_CLUSTER=0 (global-scratch split-K) changes the K partition, i.e. the fp32 summation order:
    logits agree to 2e-5 of their scale."""
    from mt3_b200 import _lib, network
    ocfg = O.T5Config(vocab_size=1536, num_encoder_layers=1, num_decoder_layers=2)
    params = O.init_params(ocfg, seed=21)
    cfg = _mt3_cfg(num_encoder_layers=1, num_decoder_layers=2)
    x = torch.from_numpy(_inputs(32, t=64, seed=300)).to(DEV)
    gmode, kvf = _mode_ids((gm, kv))

    def run():
        m = network.Transformer(cfg, params, device=DEV, max_batch=32, max_input_length=64, max_decode_length=40, gemm_mode=gmode,
                                kv_format=kvf)
        toks = m.generate(x, stop_at_eos=False, use_graph=True).cpu().numpy()
        enc = m.encode(x)
        lg = m.teacher_forced_logits(enc, torch.from_numpy(toks[:, :4].astype(np.int32)).to(DEV)).cpu().numpy()
        return toks, lg

    for k in ("MT3_PDL", "MT3_DEC_CLUSTER"):
        monkeypatch.delenv(k, raising=False)
    base_t, base_l = run()
    monkeypatch.setenv("MT3_PDL", pdl)
    monkeypatch.setenv("MT3_DEC_CLUSTER", cluster)
    t, l = run()
    if cluster == "1":
        np.testing.assert_array_equal(t, base_t)
        np.testing.assert_array_equal(l, base_l)
    else:
        np.testing.assert_allclose(l, base_l, rtol=0, atol=2e-5 * np.abs(base_l).max())


@pytest.mark.parametrize("kv", ["f32", "f16", "p24"])
def test_kv_l2_prefetch_is_value_neutral(kv, monkeypatch):
    """MT3_PF_ATTN (default 16): the decode-step attention kernels pull the K/V tiles that follow their shared-memory ring
    into L2 while they wait under the preceding GEMM.  Only cache state changes: tokens of a graph-replayed greedy run over
    300 cache positions (5 / 10 tiles per stream, ragged last tile, cache capacity not a multiple of the tile; T = 256 so
    that the cross K/V has tiles beyond the ring too) and step-by-step logits are bit-identical with the prefetch off,
    shorter than the stream (3 tiles) and longer than it (64), in every K/V row format."""
    from mt3_b200 import network
    ocfg = O.T5Config(vocab_size=1536, num_encoder_layers=1, num_decoder_layers=3)
    params = O.init_params(ocfg, seed=21)
    cfg = _mt3_cfg(num_encoder_layers=1, num_decoder_layers=3)
    x = torch.from_numpy(_inputs(8, seed=700)).to(DEV)
    gmode, kvf = _mode_ids(("tf32x3", kv))
    forced = torch.from_numpy(np.random.default_rng(5).integers(3, 1500, size=(8, 70)).astype(np.int32)).to(DEV)

    def run():
        m = network.Transformer(cfg, params, device=DEV, max_batch=8, max_input_length=256, max_decode_length=300, gemm_mode=gmode,
                                kv_format=kvf)
        toks = m.generate(x, stop_at_eos=False, use_graph=True).cpu().numpy()
        lg = m.teacher_forced_logits(m.encode(x), forced).cpu().numpy()
        return toks, lg

    monkeypatch.setenv("MT3_PF_ATTN", "0")
    base_t, base_l = run()
    for n in (None, "3", "64"):
        if n is None:
            monkeypatch.delenv("MT3_PF_ATTN")
        else:
            monkeypatch.setenv("MT3_PF_ATTN", n)
        t, l = run()
        np.testing.assert_array_equal(t, base_t)
        np.testing.assert_array_equal(l, base_l)


def test_kv_cache_formats_vs_fp32():
    """fp16 rows (MT3_KV_F16) and 24-bit rows (MT3_KV_P24) against fp32 rows, everything else equal: the logits move by
    the rounding of the stored rows only (measured ~1e-4 of the logit scale for fp16 with these weights, ~5e-6 for
    p24), and all three stay inside the oracle bar."""
    from mt3_b200 import _lib, network
    ocfg = O.T5Config(vocab_size=1536, num_encoder_layers=1, num_decoder_layers=3)
    params = O.init_params(ocfg, seed=33, norm_scale_jitter=0.05)
    cfg = _mt3_cfg(num_encoder_layers=1, num_decoder_layers=3)
    x_np = _inputs(5, t=64, seed=500)
    x = torch.from_numpy(x_np).to(DEV)
    forced = np.random.default_rng(3).integers(3, 1500, size=(5, 70)).astype(np.int32)   # crosses the 64-key tile of the fp16 / p24 kernels

    def run(kv):
        m = network.Transformer(cfg, params, device=DEV, max_batch=8, max_input_length=64, max_decode_length=72, kv_format=kv)
        return m.teacher_forced_logits(m.encode(x), torch.from_numpy(forced).to(DEV)).cpu().numpy()

    l32, l16, l24 = run(_lib.KV_F32), run(_lib.KV_F16), run(_lib.KV_P24)
    ref = O.decode_teacher_forced(params, ocfg, O.encode(params, ocfg, x_np, np.float64), forced, np.float64)
    scale = np.abs(ref).max()
    d16, d24 = np.abs(l16 - l32).max() / scale, np.abs(l24 - l32).max() / scale
    print(f"kv f16 vs f32: {d16:.2e};  p24 vs f32: {d24:.2e};  vs oracle: f32 {np.abs(l32 - ref).max() / scale:.2e}"
          f"  f16 {np.abs(l16 - ref).max() / scale:.2e}  p24 {np.abs(l24 - ref).max() / scale:.2e}")
    assert 0 < d16 <= 4e-4
    assert 0 < d24 <= 2e-5
    assert np.abs(l32 - ref).max() <= 2e-5 * scale
    assert np.abs(l24 - ref).max() <= 3e-5 * scale
    assert np.abs(l16 - ref).max() <= LOGIT_TOL * scale


def test_kv_cache_formats_sharp_attention():
    """How the storage formats behave when the attention is SHARP.  The oracle's random-init weights give diffuse
    attention (scores of order 1), where every format is far inside the bar; a trained checkpoint need not.  Scaling the
    decoder's query kernels by 8 sharpens every softmax, and any perturbation of a stored row is then amplified through
    the following layers -- float32 arithmetic itself moves from 7e-7 to 6e-6 of the logit scale in the float64 oracle.
    Restated on the CPU (tests/kv_format_study.py: float64 decoder, rows rounded in numpy): fp16 rows 3e-3, p24 rows 1e-4,
    growing 4-6x with every further doubling of the scale; measured here on the B200: f32 1.5e-6, p24 3.4e-5, f16 1.2e-3.
    The bar (5e-4) is asserted for fp32 and p24 rows; fp16 rows are reported and must be the worst of the three --
    that is the reason MT3_KV_P24 exists and what DESIGN.md section 4 tells a user with a sharp checkpoint to select."""
    from mt3_b200 import _lib, network
    ocfg = O.T5Config(vocab_size=1536, num_encoder_layers=1, num_decoder_layers=3)
    params = O.init_params(ocfg, seed=33, norm_scale_jitter=0.05)
    for k in list(params):
        if k.startswith("decoder") and k.endswith("query/kernel"):
            params[k] = params[k] * np.float32(8.0)
    cfg = _mt3_cfg(num_encoder_layers=1, num_decoder_layers=3)
    x_np = _inputs(5, t=64, seed=500)
    x = torch.from_numpy(x_np).to(DEV)
    forced = np.random.default_rng(3).integers(3, 1500, size=(5, 70)).astype(np.int32)
    ref = O.decode_teacher_forced(params, ocfg, O.encode(params, ocfg, x_np, np.float64), forced, np.float64)
    scale = np.abs(ref).max()
    err = {}
    for name, kv in (("f32", _lib.KV_F32), ("p24", _lib.KV_P24), ("f16", _lib.KV_F16)):
        m = network.Transformer(cfg, params, device=DEV, max_batch=8, max_input_length=64, max_decode_length=72, kv_format=kv)
        lg = m.teacher_forced_logits(m.encode(x), torch.from_numpy(forced).to(DEV)).cpu().numpy()
        err[name] = np.abs(lg - ref).max() / scale
        del m
    print("sharp attention (decoder query kernels x8), max logit error / scale: " + "  ".join(f"{k} {v:.2e}" for k, v in err.items()))
    assert err["f32"] <= 1e-4
    assert err["p24"] <= LOGIT_TOL
    assert err["f16"] > err["p24"] > 0


def test_decode_fused_out_q_matches_unfused(monkeypatch):
    """The default step folds the self-attention out-projection into the cross-attention query projection
    (precomposed [Wo.Wq ; Wq] block, q scaled inside the attention kernel).  Same math as the two-launch
    path up to fp32 rounding of the precomposed product: logits agree to 2e-5 of their scale, and both sit
    within the standard tolerance of the fp64 oracle."""
    from mt3_b200 import network
    ocfg = O.T5Config(vocab_size=1536, num_encoder_layers=1, num_decoder_layers=3)
    params = O.init_params(ocfg, seed=33, norm_scale_jitter=0.05)
    cfg = network.T5Config(vocab_size=1536, emb_dim=512, num_heads=6, num_encoder_layers=1, num_decoder_layers=3,
                           head_dim=64, mlp_dim=1024, mlp_activations=('gelu', 'linear'))
    x_np = _inputs(5, t=64, seed=500)
    x = torch.from_numpy(x_np).to(DEV)
    forced = np.random.default_rng(3).integers(3, 1500, size=(5, 6)).astype(np.int32)

    def run():
        m = network.Transformer(cfg, params, device=DEV, max_batch=8, max_input_length=64, max_decode_length=16)
        enc = m.encode(x)
        return m.teacher_forced_logits(enc, torch.from_numpy(forced).to(DEV)).cpu().numpy()

    monkeypatch.setenv("MT3_DEC_FUSE", "0")
    unfused = run()
    monkeypatch.setenv("MT3_DEC_FUSE", "1")
    fused = run()
    scale = np.abs(unfused).max()
    assert np.abs(fused - unfused).max() <= 2e-5 * scale
    assert np.abs(fused - unfused).max() > 0          # the fused path really ran (different rounding)
    enc64 = O.encode(params, ocfg, x_np, np.float64)
    ref = O.decode_teacher_forced(params, ocfg, enc64, forced, np.float64)
    assert np.abs(fused - ref).max() <= 5e-4 * np.abs(ref).max()


def test_dot_product_attention_op_reference_kat():
    """layers_test.py:375-387, literally (np.random.seed(0); b, q, h, d, k = 2, 3, 4, 5, 6; full additive bias), plus the
    broadcast bias shapes the reference uses (mask-derived [b, 1, q, k]; relative-position [1, h, q, k]) and no bias."""
    from mt3_b200 import layers
    b, q, h, d, k = 2, 3, 4, 5, 6
    np.random.seed(0)
    query = np.random.randn(b, q, h, d)
    key = np.random.randn(b, k, h, d)
    value = np.random.randn(b, k, h, d)
    bias = np.random.randn(b, h, q, k)
    dev = lambda a: torch.from_numpy(a.astype(np.float32)).to(DEV)

    def expected(bias_):
        logits = np.einsum('bqhd,bkhd->bhqk', query, key) + (0.0 if bias_ is None else bias_)
        w = np.exp(logits - logits.max(-1, keepdims=True))
        w /= w.sum(-1, keepdims=True)
        return np.einsum('bhqk,bkhd->bqhd', w, value)

    for bias_ in (bias, None, bias[:, :1], bias[:1]):
        got = layers.dot_product_attention(dev(query), dev(key), dev(value), bias=None if bias_ is None else dev(bias_)).cpu().numpy()
        np.testing.assert_allclose(got, expected(bias_), atol=2e-6)
    # a larger shape with head_dim 64 against the oracle's restatement, mask bias of -1e10 included (layers.py:297-322)
    rng = np.random.default_rng(1)
    Q, K_, V_ = (rng.standard_normal((3, 40, 6, 64)) * 0.3 for _ in range(3))
    mask = np.tril(np.ones((40, 40)))[None, None]
    mb = np.where(mask > 0, 0.0, -1e10)
    got = layers.dot_product_attention(dev(Q), dev(K_), dev(V_), bias=dev(mb)).cpu().numpy()
    np.testing.assert_allclose(got, O.dot_product_attention(Q, K_, V_, mb), atol=5e-6)
    with pytest.raises(AssertionError):
        layers.dot_product_attention(dev(query), dev(key[:, :, :2]), dev(value))


def test_vocab_decode_kernel_random():
    from mt3_b200 import vocabularies
    # vocabularies_test.py:47-83, literally (GenericTokenVocabulary(32, extra_ids=4))
    v32 = vocabularies.GenericTokenVocabulary(32, extra_ids=4)
    for ids_, want in (([4, 5, 6], [1, 2, 3]), ([0, 2, 3, 4, 34, 35], [-2, -2, 0, 1, 31, -2]),
                       ([0, 2, 3, 4, 1, 0, 1, 0], [-2, -2, 0, 1, -1, -1, -1, -1])):
        got_ = v32.decode_tf(torch.tensor(ids_, dtype=torch.int32, device=DEV)).cpu().numpy()
        np.testing.assert_array_equal(got_, want)
    rng = np.random.default_rng(0)
    ids = rng.integers(0, 1536, size=(64, 1024)).astype(np.int32)
    ids[rng.random(ids.shape) < 0.002] = 1
    ids[5] = 7            # no EOS at all
    vocab = vocabularies.GenericTokenVocabulary(1388, extra_ids=100)
    got = vocab.decode_tf(torch.from_numpy(ids).to(DEV)).cpu().numpy()
    np.testing.assert_array_equal(got, O.vocab_decode(ids, 1388))


def test_batch_invariance_full_batch(mt3_model):
    """Size-independent property at the full B=64: segments are independent (data-parallel unit),
    so a segment's tokens do not depend on which batch it was decoded in."""
    model, _, _ = mt3_model
    x = torch.from_numpy(_inputs(64, seed=200)).to(DEV)
    steps = 24
    full = model.generate(x, num_steps=steps, stop_at_eos=False, use_graph=True)
    sub = model.generate(x[8:16].contiguous(), num_steps=steps, stop_at_eos=False, use_graph=True)
    assert torch.equal(full[8:16], sub)
    enc_full = model.encode(x)
    enc_sub = model.encode(x[40:44].contiguous())
    assert torch.equal(enc_full[40:44], enc_sub)


def test_error_paths(mt3_model):
    from mt3_b200 import _lib
    model, _, _ = mt3_model
    with pytest.raises(TypeError):
        model.encode(torch.zeros(1, 256, 512))                       # CPU tensor
    with pytest.raises(ValueError):
        model.encode(torch.zeros(1, 256, 100, device=DEV))           # wrong depth
    with pytest.raises(_lib.Mt3Error):
        model.encode(torch.zeros(65, 256, 512, device=DEV))          # batch > max_batch
    with pytest.raises(_lib.Mt3Error):
        model.generate(torch.zeros(1, 256, 512, device=DEV), num_steps=2000)
    enc = model.encode(torch.zeros(1, 256, 512, device=DEV))
    model.init_cache(enc)
    with pytest.raises(ValueError):
        model.decode(enc, None, torch.zeros(1, 2, dtype=torch.int32, device=DEV))   # layers.py:266-270
    with pytest.raises(ValueError):
        model.decode(enc, None, torch.zeros(1, 1, device=DEV))                      # layers.py:528-529


def test_inference_model_api_end_to_end():
    from mt3_b200 import inference
    im = inference.InferenceModel('synthetic:0', 'mt3', device=DEV, batch_size=8)
    assert (im.inputs_length, im.outputs_length, im.batch_size) == (256, 1024, 8)
    assert im.sequence_length == {'inputs': 256, 'targets': 1024}
    assert im.input_shapes['encoder_input_tokens'] == (8, 256)
    assert im.model.config.vocab_size == 1536
    audio = np.concatenate([O.sine_mix(32768, 1), O.sine_mix(32768, 2), O.sine_mix(20000, 3)])   # 2.6 segments
    ds = im.preprocess(im.audio_to_dataset(audio))
    assert len(ds) == 3 and ds[2]['inputs'].shape[0] == (len(audio) + 128 - len(audio) % 128) // 128 - 512
    # predict_tokens on a hand-made batch == oracle pipeline semantics (decoded ids)
    spec = O.compute_spectrogram(np.stack([audio[:32768], audio[32768:65536]]), np.float32)
    toks = im.model.generate(torch.from_numpy(spec).to(DEV), num_steps=8, stop_at_eos=False).cpu().numpy()
    dec = im.vocabulary.decode_tf(toks)
    np.testing.assert_array_equal(dec, O.vocab_decode(toks, 1388))
    with pytest.raises(ValueError):
        inference.InferenceModel('synthetic', 'bogus')
    # __call__: audio -> segments -> GPU -> tokens -> stitched NoteSequence (notebook :283-308); the stitch of the
    # GPU's tokens must equal the stitch of the same tokens done segment by segment on the host
    from mt3_b200 import note_decoding
    im.outputs_length = 1024
    preds = im.predict_segments(audio)
    # segment starts 0 / 2.048 / 4.096 s, rounded DOWN to the 10 ms token grid (notebook :349-351)
    assert len(preds) == 3 and [round(p['start_time'], 3) for p in preds] == [0.0, 2.04, 4.09]
    ns = im(audio)
    assert isinstance(ns, note_decoding.NoteSequence)
    ref_ns = note_decoding.event_predictions_to_ns(preds, im.codec, im.encoding_spec)['est_ns']
    assert [(n.pitch, n.start_time, n.end_time, n.program) for n in ns.notes] == \
           [(n.pitch, n.start_time, n.end_time, n.program) for n in ref_ns.notes]
    ism = inference.InferenceModel('synthetic:1', 'ismir2021', device=DEV, batch_size=1)
    assert ism.inputs_length == 512 and ism.model.config.vocab_size == 1664
    clip = O.sine_mix(32000, 5)                                   # BASELINE config 1: single 2 s clip
    frames, times = ism._audio_to_frames(clip)
    assert frames.shape == (251, 128)
    seg = np.zeros((1, 512 * 128), np.float32)
    seg[0, :251 * 128] = frames.reshape(-1)
    out = ism.transcribe_segments(seg, n_valid_frames=np.array([251], np.int32), num_steps=6, stop_at_eos=False)
    assert out.shape == (1, 1024) and out.dtype == np.int32
    # against the oracle's encoder/decoder on the spectrogram the GPU frontend produced (the frontend
    # has its own parity test; feeding the oracle its own float64 log-mel would let the frontend's
    # permitted 1e-4 mel error in near-silent bins, amplified by 16 layers, flip near-tie tokens)
    ocfg = O.T5Config(vocab_size=1664)
    from mt3_b200 import spectrograms, weights
    params = weights.synthetic_params(ism.model.config, 1)
    spec_gpu = spectrograms.compute_spectrogram(torch.from_numpy(seg).to(DEV), ism.spectrogram_config,
                                                n_valid_frames=torch.tensor([251], dtype=torch.int32, device=DEV))
    spec = spec_gpu.cpu().numpy()
    assert spec.shape == (1, 512, 512) and (spec[0, 251:] == 0).all()
    _mel_close(spec[0, :251], O.compute_spectrogram(frames.reshape(-1).astype(np.float64), np.float64))
    enc64 = O.encode(params, ocfg, spec, np.float64)
    ref, lg = O.greedy_decode(params, ocfg, enc64, 6, np.float64, stop_at_eos=False, return_logits=True)
    srt = np.sort(lg, -1)
    safe = np.cumprod((srt[..., -1] - srt[..., -2]) > 1e-3 * np.abs(lg).max(), axis=1).astype(bool)
    np.testing.assert_array_equal(out[:, :6][safe], O.vocab_decode(ref[:, :6], 1514)[safe])


def test_baseline_config4_ten_minute_stream_logmel(spec_cfg):
    """BASELINE configs[3]: log-mel of a 10 min / 16 kHz stream (9.6 M samples -> 75 001 frames -> 293 segments, the
    last one short).  Segment-wise GPU frames == one-shot GPU frames (segments are independent, spectral_ops.py:35-48
    frames never cross a segment), and sampled segments == the float64 oracle."""
    from mt3_b200 import spectrograms
    n = 10 * 60 * 16000
    rng = np.random.default_rng(11)
    t = np.arange(n, dtype=np.float64) / 16000.0
    audio = (0.3 * np.sin(2 * np.pi * (220.0 + 40.0 * np.sin(0.05 * t)) * t) + 0.05 * rng.standard_normal(n)).astype(np.float32)
    padded = np.pad(audio, [0, 128 - n % 128])
    frames = padded.reshape(-1, 128)
    assert frames.shape[0] == 75001
    S = -(-frames.shape[0] // 256)
    assert S == 293
    segs = np.zeros((S, 256 * 128), np.float32)
    flat = frames.reshape(-1)
    segs.reshape(-1)[:flat.size] = flat
    n_valid = np.full((S,), 256, np.int32)
    n_valid[-1] = frames.shape[0] - 292 * 256
    lm = spectrograms.compute_spectrogram(torch.from_numpy(segs).to(DEV), spec_cfg,
                                          n_valid_frames=torch.from_numpy(n_valid).to(DEV)).cpu().numpy()
    assert lm.shape == (293, 256, 512)
    assert (lm[-1, n_valid[-1]:] == 0).all()                     # feature-converter zero rows
    for i in (0, 146, 291):
        _mel_close(lm[i], O.compute_spectrogram(segs[i].astype(np.float64), np.float64))
    last = O.compute_spectrogram(segs[-1, :n_valid[-1] * 128].astype(np.float64), np.float64)
    _mel_close(lm[-1, :n_valid[-1]], last)
    # batch composition does not matter: a segment alone == the same segment inside the 293-segment launch
    solo = spectrograms.compute_spectrogram(torch.from_numpy(segs[146]).to(DEV), spec_cfg).cpu().numpy()
    np.testing.assert_array_equal(solo, lm[146])


@pytest.mark.parametrize("fft", [512, 1024, 4096])
def test_logmel_other_fft_sizes(fft):
    """BASELINE configs[3] sweeps FFT sizes 1024 / 2048 / 4096 at hop 128 and 512 mel bins.  Only 2048 exists in the
    reference (spectrograms.py:27-28); the other sizes go through the generic power-of-two kernel and are checked
    against the same restated pipeline (spectral_ops.py:29-88) in float64."""
    from mt3_b200 import spectral_ops
    bins, hop = (512 if fft >= 1024 else 128), 128
    audio = np.stack([O.sine_mix(8 * 1024 + 77, 900 + i) for i in range(3)]).astype(np.float32)
    audio[2] = np.random.default_rng(9).uniform(-1, 1, audio.shape[1]).astype(np.float32)
    got = spectral_ops.compute_logmel(torch.from_numpy(audio).to(DEV), lo_hz=20.0, hi_hz=7600.0, bins=bins, fft_size=fft,
                                      overlap=1.0 - hop / fft).cpu().numpy()
    want = O.compute_logmel(audio.astype(np.float64), bins=bins, lo_hz=20.0, hi_hz=7600.0, fft_size=fft, hop=hop, dtype=np.float64)
    assert got.shape == want.shape == (3, -(-audio.shape[1] // hop), bins)
    _mel_close(got, want)
    z = spectral_ops.compute_logmel(torch.zeros(1000, device=DEV), lo_hz=20.0, hi_hz=7600.0, bins=bins, fft_size=fft,
                                    overlap=1.0 - hop / fft).cpu().numpy()
    np.testing.assert_allclose(z, np.log(np.float32(1e-5)), rtol=1e-6)
    # frames depend only on their own window: a long stream cut at a frame boundary gives the same frames (bit-exact) as the
    # whole stream wherever the window does not cross the cut -- exercises every frame slot of a CTA and many CTAs
    long = np.concatenate([O.sine_mix(40 * 1024, 950), np.random.default_rng(2).uniform(-0.5, 0.5, 3000).astype(np.float32)])
    whole = spectral_ops.compute_logmel(torch.from_numpy(long).to(DEV), lo_hz=20.0, hi_hz=7600.0, bins=bins, fft_size=fft,
                                        overlap=1.0 - hop / fft)
    cut = 100 * hop
    tail = spectral_ops.compute_logmel(torch.from_numpy(long[cut:]).to(DEV), lo_hz=20.0, hi_hz=7600.0, bins=bins, fft_size=fft,
                                       overlap=1.0 - hop / fft)
    assert torch.equal(whole[100:], tail)
    _mel_close(whole.cpu().numpy(), O.compute_logmel(long.astype(np.float64), bins=bins, lo_hz=20.0, hi_hz=7600.0, fft_size=fft, hop=hop,
                                                      dtype=np.float64))


def test_baseline_config5_long_form_three_minutes():
    """BASELINE configs[4]: 3 min of audio -> 88 non-overlapping segments (87 full + one of 229 frames) -> tokens ->
    stitched NoteSequence, in two GPU batches of 64 + 24; batch composition must not change any token stream."""
    from mt3_b200 import inference, note_decoding
    im = inference.InferenceModel('synthetic:0', 'mt3', device=DEV, batch_size=64)
    n = 3 * 60 * 16000
    audio = np.concatenate([O.sine_mix(32768, 100 + i) for i in range(-(-n // 32768))])[:n]
    ds = im.preprocess(im.audio_to_dataset(audio))
    assert len(ds) == 88 and ds[-1]['inputs'].shape[0] == 229
    im.outputs_length = 1024
    preds = im.predict_segments(audio)
    assert len(preds) == 88
    assert round(preds[1]['start_time'], 3) == 2.04 and round(preds[87]['start_time'], 2) == round(int(87 * 2.048 * 100) / 100, 2)
    ns = note_decoding.event_predictions_to_ns(preds, im.codec, im.encoding_spec)['est_ns']
    assert isinstance(ns, note_decoding.NoteSequence)
    # the same segments one at a time (batch of 1) give the same decoded token streams
    hop = im.spectrogram_config.hop_width
    for i in (0, 63, 64, 87):
        flat = np.asarray(ds[i]['inputs'], np.float32).reshape(-1)
        seg = np.zeros((1, 256 * hop), np.float32)
        seg[0, :flat.size] = flat
        one = im.transcribe_segments(seg, n_valid_frames=np.array([flat.size // hop], np.int32))
        trimmed = one[0][:len(preds[i]['est_tokens'])]
        np.testing.assert_array_equal(trimmed, preds[i]['est_tokens'])


# ------------------------------------------------------------------------------------------------
# tcgen05 GEMM modes (encoder + cross-K/V on the tensor cores)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("attn", ["simt", "tc"])
@pytest.mark.parametrize("mode,tol", [("tf32x3", None), ("tf32", 3e-2)])
def test_tensor_core_encoder_parity(mode, tol, attn, monkeypatch):
    """MT3_GEMM_TF32X3 must meet the same fp32 bar as the exact-fp32 SIMT path; single-pass TF32
    is reported with its own (10-bit mantissa) tolerance and is not the default."""
    from mt3_b200 import _lib, network
    # attn = "simt": exact-fp32 attention between tcgen05 GEMMs (isolates the GEMM); "tc": tcgen05 attention too
    monkeypatch.setenv("MT3_TC_ATTENTION", "1" if attn == "tc" else "0")
    cfg = _mt3_cfg()
    ocfg = O.T5Config()
    params = O.init_params(ocfg, seed=0, norm_scale_jitter=0.05)
    gm = _lib.GEMM_TF32X3 if mode == "tf32x3" else _lib.GEMM_TF32
    model = network.Transformer(cfg, params, device=DEV, max_batch=4, max_input_length=256, max_decode_length=64, gemm_mode=gm)
    x = _inputs(3, seed=77)        # M = 768 rows: 6 row tiles
    enc = model.encode(torch.from_numpy(x).to(DEV)).cpu().numpy()
    enc64 = O.encode(params, ocfg, x, np.float64)
    enc32 = O.encode(params, ocfg, x, np.float32)
    scale = np.abs(enc64).max()
    e_gpu, e_f32 = np.abs(enc - enc64).max() / scale, np.abs(enc32 - enc64).max() / scale
    print(f"encoder[{mode},{attn}]: gpu vs fp64 {e_gpu:.3e}   fp32-oracle vs fp64 {e_f32:.3e}")
    if tol is None:
        assert e_gpu <= max(LOGIT_TOL, 4 * e_f32)
    else:
        assert e_gpu <= tol
    # decode on top of the tensor-core encoder / cross-K/V: teacher-forced logits
    steps = 6
    toks64, logits64 = O.greedy_decode(params, ocfg, enc64, steps, np.float64, stop_at_eos=False, return_logits=True)
    dec_in = np.concatenate([np.zeros((3, 1), np.int64), toks64[:, :steps - 1]], axis=1)
    enc_gpu = model.encode(torch.from_numpy(x).to(DEV))
    lg = model.teacher_forced_logits(enc_gpu, torch.from_numpy(dec_in).to(DEV).to(torch.int32)).cpu().numpy()
    e_l = np.abs(lg - logits64).max() / np.abs(logits64).max()
    print(f"logits[{mode}]: gpu vs fp64 {e_l:.3e}")
    assert e_l <= (LOGIT_TOL if tol is None else tol)


def test_bench_dump_outputs_are_the_timed_paths_tokens(tmp_path):
    """`bench.py --dump-outputs DIR` saves the token ids of its last timed step: bench's seeded 64-segment batch through
    the same pass via InferenceModel gives them again, bit for bit."""
    import subprocess
    import sys
    import bench
    from mt3_b200 import inference
    steps = 8
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--dec-steps", str(steps),
           "--no-alt-kv", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    got = np.load(tmp_path / "tokens.npy")
    assert got.dtype == np.float32 and got.shape == (bench.BATCH_PER_GPU, 1024)
    assert (got[:, steps:] == 0).all() and (got[:, :steps] > 0).any()
    im = inference.InferenceModel('synthetic:0', 'mt3', device=DEV, batch_size=bench.BATCH_PER_GPU)
    want = im.transcribe_segments(bench.synth_audio(bench.BATCH_PER_GPU, 1234), num_steps=steps, stop_at_eos=False,
                                  decoded=False)
    np.testing.assert_array_equal(got, want.astype(np.float32))

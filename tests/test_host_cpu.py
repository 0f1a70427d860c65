"""CPU-side tests (-m "not gpu"): golden vectors, host logic, and that the C-ABI library
loads and exports every symbol include/mt3_b200.h declares (no compute without a GPU)."""
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import mt3_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


# ---- golden: codec vectors produced by the reference's own event_codec.py --------------------
def test_codec_matches_reference_golden():
    from mt3_b200 import event_codec, vocabularies
    gold = json.load(open(os.path.join(GOLD, "event_codec.json")))
    for name in ("mt3", "ismir2021"):
        g = gold[name]
        codec = vocabularies.build_codec(vocabularies.VocabularyConfig(num_velocity_bins=g["num_velocity_bins"]))
        assert codec.num_classes == g["num_classes"]
        for t, (lo, hi) in g["ranges"].items():
            assert codec.event_type_range(t) == (lo, hi)
        for i, t, v in g["decode"]:
            ev = codec.decode_event_index(i)
            assert (ev.type, ev.value) == (t, v)
        for t, v, i in g["encode"]:
            assert codec.encode_event(event_codec.Event(t, v)) == i
        for i, flag in g["is_shift"]:
            assert codec.is_shift_event_index(i) == flag
        vocab = vocabularies.vocabulary_from_codec(codec)
        assert vocabularies.num_embeddings(vocab) == O.num_embeddings(g["num_classes"])
    # event_codec_test.py:26-40
    c = event_codec.Codec(100, 100, [event_codec.EventRange('pitch', 0, 127)])
    for t, v, i in gold["event_codec_test"]["encode"]:
        assert c.encode_event(event_codec.Event(t, v)) == i
    assert [i for _, _, i in gold["event_codec_test"]["encode"]] == [161, 5, 163]
    with pytest.raises(ValueError):
        c.encode_event(event_codec.Event('pitch', 128))
    with pytest.raises(ValueError):
        c.encode_event(event_codec.Event('nope', 0))
    with pytest.raises(ValueError):
        c.decode_event_index(10 ** 6)


def test_vocabulary_contract():
    # vocabularies_test.py:47-83
    from mt3_b200 import vocabularies as V
    vocab = V.GenericTokenVocabulary(10, extra_ids=4)
    assert vocab.vocab_size == 17 and vocab.eos_id == 1 and vocab.unk_id == 2
    assert vocab.encode([0, 1, 9]) == [3, 4, 12]
    with pytest.raises(ValueError):
        vocab.encode([10])
    assert vocab.decode([3, 4, 12, 1, 5]) == [0, 1, 9, -1]
    assert vocab.decode([0, 2, 13, 3]) == [-2, -2, -2, 0]
    ids = np.array([[3, 4, 1, 5, 6], [0, 2, 13, 16, 3]])
    np.testing.assert_array_equal(vocab.decode_tf(ids), O.vocab_decode(ids, 10))
    np.testing.assert_array_equal(vocab.decode_tf(torch.from_numpy(ids)).numpy(), O.vocab_decode(ids, 10))
    # velocity bins round trip (vocabularies_test.py:28-45)
    for nb in (1, 127):
        for vel in (0, 1, 64, 127):
            b = V.velocity_to_bin(vel, nb)
            assert 0 <= b <= nb
            if vel == 0:
                assert b == 0 and V.bin_to_velocity(b, nb) == 0
            else:
                assert V.velocity_to_bin(V.bin_to_velocity(b, nb), nb) == b


# ---- golden: oracle regression vectors ---------------------------------------------------------
def test_oracle_logmel_golden():
    g = np.load(os.path.join(GOLD, "logmel_sine_seed7.npz"))
    x = O.sine_mix(32768, seed=int(g["seed"]))
    lm64 = O.compute_spectrogram(x.astype(np.float64), np.float64)
    np.testing.assert_allclose(lm64[g["rows"]], g["logmel"], rtol=1e-12, atol=1e-12)
    lm32 = O.compute_spectrogram(x, np.float32)
    # fp32 vs fp64 oracle: the tolerance north_star states for mel frames (1e-4 rel) plus the
    # fp32 noise floor of the frame (leakage bins sit > 100 dB below the partials)
    mel64, mel32 = np.exp(lm64), np.exp(lm32.astype(np.float64))
    tol = 1e-4 * mel64 + 1e-6 * mel64.max(axis=-1, keepdims=True)
    assert (np.abs(mel32 - mel64) <= tol).all()
    n = np.load(os.path.join(GOLD, "logmel_noise_5000.npz"))
    ln = O.compute_spectrogram(n["audio"].astype(np.float64), np.float64)
    assert ln.shape == (40, 512)            # ceil(5000/128)
    np.testing.assert_allclose(ln, n["logmel"], rtol=1e-12, atol=1e-12)


def test_oracle_model_golden_and_fp32_budget():
    g = np.load(os.path.join(GOLD, "model_tiny.npz"))
    cfg = O.T5Config(vocab_size=1536, num_encoder_layers=1, num_decoder_layers=1)
    params = O.init_params(cfg, seed=int(g["weight_seed"]), norm_scale_jitter=float(g["jitter"]))
    enc = O.encode(params, cfg, g["x"], np.float64)
    np.testing.assert_allclose(enc[:, ::8, ::16], g["encoded"], rtol=1e-10, atol=1e-10)
    toks, logits = O.greedy_decode(params, cfg, enc, 6, np.float64, stop_at_eos=False, return_logits=True)
    np.testing.assert_array_equal(toks[:, :6], g["tokens"])
    np.testing.assert_allclose(logits[:, :, ::16], g["logits"], rtol=1e-9, atol=1e-9)
    # what "fp32 logit tolerance" means here: the fp32 oracle vs the fp64 oracle
    enc32 = O.encode(params, cfg, g["x"], np.float32)
    _, logits32 = O.greedy_decode(params, cfg, enc32, 6, np.float32, stop_at_eos=False, return_logits=True,
                                  forced_tokens=np.concatenate([np.zeros((2, 1), np.int64), toks[:, :5]], axis=1))
    assert np.abs(logits32 - logits).max() < 2e-4 * np.abs(logits).max()


def test_torch_cpu_port_matches_numpy_oracle():
    from oracle import torch_cpu as TC
    cfg = O.T5Config(vocab_size=256, emb_dim=64, num_heads=2, num_encoder_layers=2, num_decoder_layers=2,
                     head_dim=16, mlp_dim=96, input_depth=512)
    params = O.init_params(cfg, seed=2, norm_scale_jitter=0.1)
    audio = np.stack([O.sine_mix(4096, 3), O.sine_mix(4096, 4)])
    spec_np = O.compute_spectrogram(audio, np.float32)
    spec_t = TC.compute_logmel(torch.from_numpy(audio)).numpy()
    mel_np, mel_t = np.exp(spec_np.astype(np.float64)), np.exp(spec_t.astype(np.float64))
    assert (np.abs(mel_t - mel_np) <= 1e-4 * mel_np + 1e-6 * mel_np.max(-1, keepdims=True)).all()
    m = TC.TorchCpuModel(params, cfg)
    with torch.no_grad():
        enc_t = m.encode(torch.from_numpy(spec_np))
        enc_np = O.encode(params, cfg, spec_np, np.float64)
        np.testing.assert_allclose(enc_t.numpy(), enc_np, rtol=2e-4, atol=2e-4)
        toks_np, logits_np = O.greedy_decode(params, cfg, enc_np, 8, np.float64, stop_at_eos=False, return_logits=True)
        forced = torch.from_numpy(np.concatenate([np.zeros((2, 1), np.int64), toks_np[:, :7]], axis=1))
        for hoist in (True, False):
            toks_t, logits_t = m.greedy_decode(torch.from_numpy(enc_np.astype(np.float32)), 8, 16, hoist_cross_kv=hoist,
                                               return_logits=True, forced_tokens=forced)
            np.testing.assert_allclose(logits_t.numpy(), logits_np, rtol=5e-4, atol=5e-4)


# ---- host logic ------------------------------------------------------------------------------
def test_gin_lite_reads_package_configs():
    from mt3_b200 import gin_lite
    d = os.path.join(ROOT, "mt3_b200", "gin")
    for mt, (t, nvb) in {"mt3": (256, 1), "ismir2021": (512, 127)}.items():
        c = gin_lite.parse_config_files_and_bindings(
            [os.path.join(d, "model.gin"), os.path.join(d, mt + ".gin")],
            ['VOCAB_CONFIG=@vocabularies.VocabularyConfig()',
             'vocabularies.VocabularyConfig.num_velocity_bins=%NUM_VELOCITY_BINS'])
        p = c.params('network.T5Config')
        assert (p['emb_dim'], p['num_heads'], p['head_dim'], p['mlp_dim']) == (512, 6, 64, 1024)
        assert p['num_encoder_layers'] == p['num_decoder_layers'] == 8
        assert tuple(p['mlp_activations']) == ('gelu', 'linear') and p['logits_via_embedding'] is False
        assert c.macro('TASK_FEATURE_LENGTHS') == {'inputs': t, 'targets': 1024}
        assert c.binding('vocabularies.VocabularyConfig', 'num_velocity_bins') == nvb


def test_gin_lite_syntax():
    from mt3_b200 import gin_lite
    c = gin_lite.Config().parse_lines([
        "# comment", "import x", "A = 3  # trailing", "B = %A", "S = 'has # hash'",
        "mod.Cls:", "  p = (1,", "       2)", "  q = @other.fn()", "scope/mod.fn.r = {'k': %A}", "mod.fn2.s = @fn3",
    ])
    assert c.macro('A') == 3 and c.macro('B') == 3 and c.macro('S') == 'has # hash'
    assert c.params('mod.Cls')['p'] == (1, 2)
    assert isinstance(c.params('mod.Cls')['q'], gin_lite.Ref) and c.params('mod.Cls')['q'].call
    assert isinstance(c.binding('mod.fn', 'r')['k'], gin_lite.Macro)
    assert not c.binding('mod.fn2', 's').call
    with pytest.raises(ValueError):
        gin_lite.Config().parse_lines(["what is this"])


def test_weight_layout_matches_oracle_and_abi():
    import ctypes as C
    from mt3_b200 import _lib, network, weights
    cfg = network.T5Config(vocab_size=1536, emb_dim=512, num_heads=6, num_encoder_layers=8, num_decoder_layers=8,
                           head_dim=64, mlp_dim=1024, mlp_activations=('gelu', 'linear'))
    ocfg = O.T5Config()
    assert list(weights.param_shapes(cfg).items()) == list(O.param_shapes(ocfg).items())
    assert weights.num_params(cfg) == 45896704          # SURVEY.md 8a aggregate
    # synthetic generator == the oracle's (tests hand oracle params to the CUDA model)
    small = network.T5Config(vocab_size=128, emb_dim=32, num_heads=2, num_encoder_layers=1, num_decoder_layers=1,
                             head_dim=64, mlp_dim=48, mlp_activations=('gelu', 'linear'))
    osmall = O.T5Config(vocab_size=128, emb_dim=32, num_heads=2, num_encoder_layers=1, num_decoder_layers=1,
                        head_dim=64, mlp_dim=48)
    a, b = weights.synthetic_params(small, 3), O.init_params(osmall, 3)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    lib = _lib.load()
    mc = _lib.ModelConfig(1536, 512, 6, 64, 8, 8, 1024, 512, 8, 256, 1024, 0)
    assert lib.mt3_model_num_params(C.byref(mc)) == 45896704
    off = 0
    for name, shape in weights.param_shapes(cfg).items():
        n = C.c_int64(0)
        assert lib.mt3_model_param_offset(C.byref(mc), name.encode(), C.byref(n)) == off, name
        assert n.value == int(np.prod(shape))
        off += n.value
    assert lib.mt3_model_param_offset(C.byref(mc), b"no/such/param", None) == -1
    flat = weights.flatten(a, small)
    assert flat.dtype == np.float32 and flat.size == weights.num_params(small)
    with pytest.raises(KeyError):
        weights.flatten({}, small)


def test_weights_roundtrip(tmp_path):
    from mt3_b200 import network, weights
    small = network.T5Config(vocab_size=128, emb_dim=32, num_heads=1, num_encoder_layers=1, num_decoder_layers=1,
                             head_dim=64, mlp_dim=48, mlp_activations=('gelu', 'linear'))
    p = weights.synthetic_params(small, 1)
    f = str(tmp_path / "w.npz")
    weights.save(f, p)
    q = weights.load(f)
    assert p.keys() == q.keys() and all(np.array_equal(p[k], q[k]) for k in p)


def test_abi_library_exports_every_declared_symbol():
    import ctypes as C
    from mt3_b200 import _lib
    header = open(os.path.join(ROOT, "include", "mt3_b200.h")).read()
    declared = set(re.findall(r"\b(mt3_[a-z0-9_]+)\s*\(", header))
    declared -= {"mt3_last_error"} - {"mt3_last_error"}
    assert len(declared) >= 18
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/mt3_b200.h but not exported"
    assert set(_lib.EXPORTS) == declared
    assert lib.mt3_abi_version() == 2
    for name, val in (("MT3_KV_F32", _lib.KV_F32), ("MT3_KV_F16", _lib.KV_F16), ("MT3_KV_P24", _lib.KV_P24), ("MT3_GEN_BEAM1", _lib.GEN_BEAM1)):
        assert int(re.search(name + r"\s*=\s*(\d+)", header).group(1)) == val, name
    assert isinstance(lib.mt3_kernel_launch_count(), int)
    # argument validation happens before any CUDA call -> testable without a GPU
    assert lib.mt3_frontend_create(None, None, None) == -1
    assert b"null" in lib.mt3_last_error()
    cfg = _lib.FrontendConfig(16000, 128, 1000, 512, 1e-5)       # FFT sizes must be powers of two
    h = C.c_void_p()
    mel = np.zeros((501, 512), np.float32)
    assert lib.mt3_frontend_create(C.byref(cfg), mel.ctypes.data_as(C.c_void_p), C.byref(h)) == -3
    assert b"power of two" in lib.mt3_last_error() and b"2048" in lib.mt3_last_error()
    cfg = _lib.FrontendConfig(16000, 127, 2048, 512, 1e-5)       # odd hop
    assert lib.mt3_frontend_create(C.byref(cfg), mel.ctypes.data_as(C.c_void_p), C.byref(h)) == -1
    assert lib.mt3_workspace_bytes(None, 1, 1) == -1
    assert lib.mt3_encode(None, None, None, None) == -1


def test_spectrogram_host_helpers():
    from mt3_b200 import spectrograms
    cfg = spectrograms.SpectrogramConfig()
    assert cfg.frames_per_second == 125.0 and cfg.abbrev_str == '' and spectrograms.input_depth(cfg) == 512
    assert spectrograms.SpectrogramConfig(hop_width=64).abbrev_str == 'hw64'
    fr = spectrograms.split_audio(np.arange(300, dtype=np.float32), cfg)
    assert fr.shape == (3, 128) and fr[2, 44:].sum() == 0
    np.testing.assert_array_equal(spectrograms.flatten_frames(fr)[:300], np.arange(300))
    with pytest.raises(TypeError):
        spectrograms.compute_spectrogram(torch.zeros(1000), cfg)      # CPU tensor: no fallback


def test_no_cpu_fallback_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from mt3_b200 import inference
    with pytest.raises(RuntimeError):
        inference.InferenceModel('synthetic', 'mt3')
    with pytest.raises(ValueError):
        inference.InferenceModel('synthetic', 'nope')


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU port on the host cores) runs without a GPU and prints ONE JSON line with
    the contract's keys; under torchrun only rank 0 prints (the others exit 0 without work)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
           "--dec-steps", "3", "--ref-batch", "2", "--ref-budget-s", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "audio_seconds_per_second" and line["unit"] == "audio-s/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["n_gpus"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["e2e"]["value"] == line["value"]
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    other = subprocess.run(cmd[:2] + ["--impl", "reference", "--gpus", "2"], capture_output=True, text=True, timeout=120, cwd=root, env=env)
    assert other.returncode == 0 and other.stdout.strip() == ""
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"], ["--workload", "longform", "--dump-outputs", "d"]):
        rejected = subprocess.run(cmd[:2] + bad, capture_output=True, text=True, timeout=120, cwd=root)
        assert rejected.returncode == 2 and rejected.stdout == "" and bad[-2] in rejected.stderr, bad


@pytest.mark.parametrize("top_level_target", [False, True])
def test_t5x_checkpoint_reader_roundtrip(tmp_path, top_level_target):
    """checkpoints.load_t5x_checkpoint reads the T5X directory layout (msgpack state with inlined small arrays and
    PLACEHOLDER:// references to gzip zarr-v2 arrays, chunked) back to the Flax tree paths weights.flatten expects."""
    from mt3_b200 import checkpoints, network, weights
    cfg = network.T5Config(vocab_size=256, emb_dim=64, num_heads=2, num_encoder_layers=1, num_decoder_layers=1, head_dim=64,
                           mlp_dim=128, mlp_activations=('gelu', 'linear'))
    params = weights.synthetic_params(cfg, 5)
    d = tmp_path / "ckpt"
    checkpoints.save_t5x_checkpoint(str(d), params, step=123, inline_below=200, max_chunk=48, top_level_target=top_level_target)
    assert (d / "checkpoint").exists()
    zdir = d / "target.decoder.logits_dense.kernel"              # T5X names arrays 'target.<dotted path>' in both variants
    assert (zdir / ".zarray").exists() and (zdir / "0.0").exists() and (zdir / "1.5").exists()      # 64x256 in 48x48 chunks
    got = weights.load(str(d))
    assert set(got) == set(params)
    for k in params:
        assert got[k].dtype == np.float32 and np.array_equal(got[k], params[k]), k
    np.testing.assert_array_equal(weights.flatten(got, cfg), weights.flatten(params, cfg))
    np.testing.assert_array_equal(checkpoints.load_t5x_checkpoint(str(d / "checkpoint"))["encoder/encoder_norm/scale"],
                                  params["encoder/encoder_norm/scale"])
    # uncompressed, F-order, missing chunk -> fill value
    import json
    a = np.arange(12, dtype=np.float32).reshape(3, 4)
    z = tmp_path / "arr"
    z.mkdir()
    (z / ".zarray").write_text(json.dumps({"zarr_format": 2, "shape": [3, 4], "chunks": [2, 4], "dtype": "<f4", "order": "F",
                                           "compressor": None, "fill_value": 7.0, "filters": None}))
    (z / "0.0").write_bytes(np.asfortranarray(a[:2]).tobytes(order="F"))
    r = checkpoints.read_zarr_array(str(z))
    np.testing.assert_array_equal(r[:2], a[:2])
    assert (r[2] == 7.0).all()


def test_vocabulary_reference_tests_literal():
    """vocabularies_test.py:28-45 (velocity quantisation, every bin), :85-102 (encode range errors), :104-109 (dtypes)."""
    from mt3_b200 import vocabularies as V
    assert V.velocity_to_bin(0, num_velocity_bins=1) == 0 and V.velocity_to_bin(0, num_velocity_bins=127) == 0
    assert V.bin_to_velocity(0, num_velocity_bins=1) == 0 and V.bin_to_velocity(0, num_velocity_bins=127) == 0
    assert V.velocity_to_bin(V.bin_to_velocity(1, num_velocity_bins=1), num_velocity_bins=1) == 1
    for velocity_bin in range(1, 128):
        assert V.velocity_to_bin(V.bin_to_velocity(velocity_bin, num_velocity_bins=127), num_velocity_bins=127) == velocity_bin
    vocab = V.GenericTokenVocabulary(32)
    assert list(vocab.encode([0, 15, 31])) == [3, 18, 34]
    np.testing.assert_array_equal(vocab.encode_tf(np.array([0, 15, 31])), [3, 18, 34])
    for bad in ([-1, 15, 31], [0, 15, 32]):
        with pytest.raises(ValueError):
            vocab.encode(bad)
        with pytest.raises(ValueError):
            vocab.encode_tf(np.array(bad))
    assert vocab.encode_tf(np.array([0, 15, 31], np.int32)).dtype == np.int32
    assert vocab.encode_tf(np.array([0, 15, 31], np.int64)).dtype == np.int64


def test_program_granularities():
    """vocabularies.PROGRAM_GRANULARITIES (vocabularies.py:77-116): 'flat' drops program tokens, 'midi_class' maps a program to
    the first of its class of 8, 'full' is the identity; token and program maps are idempotent and agree with each other."""
    from mt3_b200 import event_codec, vocabularies as V
    codec = V.build_codec(V.VocabularyConfig(num_velocity_bins=1))
    E = event_codec.Event
    toks = np.array([codec.encode_event(e) for e in (E('shift', 10), E('program', 42), E('velocity', 1), E('pitch', 60),
                                                     E('program', 7), E('pitch', 62), E('tie', 0), E('drum', 38))])
    prog = lambda p: codec.encode_event(E('program', p))
    flat = V.PROGRAM_GRANULARITIES['flat'].tokens_map_fn(toks, codec)
    np.testing.assert_array_equal(flat, [t for t in toks if t not in (prog(42), prog(7))])
    cls = V.PROGRAM_GRANULARITIES['midi_class'].tokens_map_fn(toks, codec)
    np.testing.assert_array_equal(cls, [prog(40) if t == prog(42) else prog(0) if t == prog(7) else t for t in toks])
    np.testing.assert_array_equal(V.PROGRAM_GRANULARITIES['full'].tokens_map_fn(toks, codec), toks)
    for name, g in V.PROGRAM_GRANULARITIES.items():
        once = g.tokens_map_fn(toks, codec)
        np.testing.assert_array_equal(g.tokens_map_fn(once, codec), once)
        for p in (0, 7, 8, 42, 127):
            assert g.program_map_fn(g.program_map_fn(p)) == g.program_map_fn(p)
            mapped = g.tokens_map_fn(np.array([prog(p)]), codec)
            assert (len(mapped) == 0 and name == 'flat') or mapped[0] == prog(g.program_map_fn(p))


# ---- against what the reference's own files give (stored by tests/golden/make_golden.py) ----------------------------
def test_gin_lite_reads_the_references_own_gin_files():
    """The reference's gin files, unmodified, give the same model surface as the package's copies (gin/model.gin:47-59,
    gin/mt3.gin, gin/ismir2021.gin); gin_reference.json holds what gin_lite read from the reference's files."""
    from mt3_b200 import gin_lite
    gold = json.load(open(os.path.join(GOLD, "gin_reference.json")))
    bindings = ['VOCAB_CONFIG=@vocabularies.VocabularyConfig()', 'vocabularies.VocabularyConfig.num_velocity_bins=%NUM_VELOCITY_BINS']
    for mt in ("mt3", "ismir2021"):
        ours = gin_lite.parse_config_files_and_bindings([os.path.join(ROOT, "mt3_b200", "gin", f) for f in ("model.gin", mt + ".gin")], bindings)
        ref = gold[mt]
        po, pr = ours.params('network.T5Config'), ref["T5Config"]
        for k in ('emb_dim', 'num_heads', 'head_dim', 'mlp_dim', 'num_encoder_layers', 'num_decoder_layers', 'dropout_rate',
                  'logits_via_embedding'):
            assert po[k] == pr[k], k
        assert tuple(po['mlp_activations']) == tuple(pr['mlp_activations'])
        assert ours.macro('TASK_FEATURE_LENGTHS') == ref["TASK_FEATURE_LENGTHS"]
        assert ours.binding('vocabularies.VocabularyConfig', 'num_velocity_bins') == ref["num_velocity_bins"]


def test_event_codec_equals_the_references_module_on_random_events():
    """mt3/event_codec.py is the one reference module that imports with the standard library alone: mt3_b200.event_codec
    and the tables it produced (event_codec_tables.json) agree on every index of the mt3 and ismir2021 codecs, on the
    event type ranges and on the errors."""
    from mt3_b200 import event_codec as ours, vocabularies as V
    gold = json.load(open(os.path.join(GOLD, "event_codec_tables.json")))
    for nvb in (1, 127):
        co = V.build_codec(V.VocabularyConfig(num_velocity_bins=nvb))
        cr = gold[str(nvb)]
        assert co.num_classes == cr["num_classes"] == len(cr["events"])
        for i in range(co.num_classes):
            eo, er = co.decode_event_index(i), cr["events"][i]
            assert [eo.type, eo.value] == er
            assert co.encode_event(ours.Event(eo.type, eo.value)) == i
            assert co.is_shift_event_index(i) == bool(cr["is_shift"][i])
        for t in ('shift', 'pitch', 'velocity', 'tie', 'program', 'drum'):
            assert list(co.event_type_range(t)) == cr["ranges"][t]
        assert [['pitch', 128], ['nope', 0]] == cr["encode_raises"]
        for t, v in cr["encode_raises"]:
            with pytest.raises(ValueError):
                co.encode_event(ours.Event(t, v))
        assert cr["decode_raises"] == [co.num_classes]
        with pytest.raises(ValueError):
            co.decode_event_index(co.num_classes)

"""Generates the committed golden fixtures.

  python tests/golden/make_golden.py REFERENCE_MT3_DIR

REFERENCE_MT3_DIR is the `mt3/` package directory of a checkout of the original MT3 project; only
this script reads it, the tests read the fixtures.

  event_codec.json   produced by importing the reference's own mt3/event_codec.py (stdlib only:
                     the one reference module importable here) -- REFERENCE-DERIVED.
  event_codec_tables.json  the same module's full index tables of the mt3 and ismir2021 codecs
                     -- REFERENCE-DERIVED.
  gin_reference.json the model surface gin_lite reads from the reference's own gin files
                     -- REFERENCE-DERIVED.
  logmel_*.npz,      produced by oracle/mt3_oracle.py in float64 -- ORACLE-DERIVED regression
  model_tiny.npz     vectors (the frontend and full-model logits are "parity unpinned" by the
                     reference's own tests; see the oracle header).
"""
import importlib.util
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import mt3_oracle as O  # noqa: E402

REF = None    # the reference's mt3/ directory (command line)
GIN_BINDINGS = ['VOCAB_CONFIG=@vocabularies.VocabularyConfig()',
                'vocabularies.VocabularyConfig.num_velocity_bins=%NUM_VELOCITY_BINS']
GIN_T5_KEYS = ('emb_dim', 'num_heads', 'head_dim', 'mlp_dim', 'num_encoder_layers', 'num_decoder_layers', 'dropout_rate',
               'logits_via_embedding', 'mlp_activations')


def reference_event_codec():
    path = os.path.join(REF, "event_codec.py")
    spec = importlib.util.spec_from_file_location("ref_event_codec", path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules["ref_event_codec"] = mod
    spec.loader.exec_module(mod)
    return mod


def make_codec_golden():
    ec = reference_event_codec()
    out = {}
    for name, nvb in (("mt3", 1), ("ismir2021", 127)):
        ranges = [ec.EventRange('pitch', 0, 127), ec.EventRange('velocity', 0, nvb), ec.EventRange('tie', 0, 0),
                  ec.EventRange('program', 0, 127), ec.EventRange('drum', 0, 127)]
        codec = ec.Codec(max_shift_steps=1000, steps_per_second=100, event_ranges=ranges)
        rng = np.random.default_rng(0)
        idx = sorted(set([0, 1, 1000, 1001, 1128, 1129, codec.num_classes - 1] +
                         [int(i) for i in rng.integers(0, codec.num_classes, 64)]))
        dec = [[i, codec.decode_event_index(i).type, codec.decode_event_index(i).value] for i in idx]
        out[name] = {
            "num_velocity_bins": nvb,
            "num_classes": codec.num_classes,
            "ranges": {t: list(codec.event_type_range(t)) for t in ("shift", "pitch", "velocity", "tie", "program", "drum")},
            "decode": dec,
            "encode": [[t, v, codec.encode_event(ec.Event(t, v))] for _, t, v in dec],
            "is_shift": [[i, bool(codec.is_shift_event_index(i))] for i in (0, 999, 1000, 1001, 1387)],
        }
    # event_codec_test.py:26-40 (pitch 60 -> 161 with a 100-step shift range etc.)
    codec = ec.Codec(max_shift_steps=100, steps_per_second=100,
                     event_ranges=[ec.EventRange('pitch', 0, 127)])
    out["event_codec_test"] = {"encode": [[t, v, codec.encode_event(ec.Event(t, v))]
                                          for t, v in (("pitch", 60), ("shift", 5), ("pitch", 62))]}
    with open(os.path.join(HERE, "event_codec.json"), "w") as f:
        json.dump(out, f, indent=1)


def make_codec_tables_golden():
    """Every index of the mt3 (1 velocity bin) and ismir2021 (127 bins) codecs, as the reference module decodes it,
    and the inputs on which the reference raises ValueError."""
    ec = reference_event_codec()
    out = {}
    for nvb in (1, 127):
        ranges = [ec.EventRange('pitch', 0, 127), ec.EventRange('velocity', 0, nvb), ec.EventRange('tie', 0, 0),
                  ec.EventRange('program', 0, 127), ec.EventRange('drum', 0, 127)]
        codec = ec.Codec(max_shift_steps=1000, steps_per_second=100, event_ranges=ranges)
        events = [codec.decode_event_index(i) for i in range(codec.num_classes)]
        assert all(codec.encode_event(e) == i for i, e in enumerate(events))
        bad_events = [('pitch', 128), ('nope', 0)]
        for t, v in bad_events:
            try:
                codec.encode_event(ec.Event(t, v))
                raise AssertionError((t, v))
            except ValueError:
                pass
        try:
            codec.decode_event_index(codec.num_classes)
            raise AssertionError(codec.num_classes)
        except ValueError:
            pass
        out[str(nvb)] = {
            "num_classes": codec.num_classes,
            "ranges": {t: list(codec.event_type_range(t)) for t in ("shift", "pitch", "velocity", "tie", "program", "drum")},
            "events": [[e.type, e.value] for e in events],
            "is_shift": [int(codec.is_shift_event_index(i)) for i in range(codec.num_classes)],
            "encode_raises": bad_events,
            "decode_raises": [codec.num_classes],
        }
    with open(os.path.join(HERE, "event_codec_tables.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))


def make_gin_golden():
    """The model surface gin_lite reads from the reference's unmodified gin/model.gin + gin/<model>.gin."""
    from mt3_b200 import gin_lite
    out = {}
    for mt in ("mt3", "ismir2021"):
        c = gin_lite.parse_config_files_and_bindings([os.path.join(REF, "gin", f) for f in ("model.gin", mt + ".gin")],
                                                     GIN_BINDINGS)
        p = c.params('network.T5Config')
        out[mt] = {"T5Config": {k: list(p[k]) if k == 'mlp_activations' else p[k] for k in GIN_T5_KEYS},
                   "TASK_FEATURE_LENGTHS": c.macro('TASK_FEATURE_LENGTHS'),
                   "num_velocity_bins": c.binding('vocabularies.VocabularyConfig', 'num_velocity_bins')}
    with open(os.path.join(HERE, "gin_reference.json"), "w") as f:
        json.dump(out, f, indent=1)


def make_logmel_golden():
    x = O.sine_mix(32768, seed=7)
    lm = O.compute_spectrogram(x.astype(np.float64), np.float64)
    rows = np.array([0, 1, 2, 100, 101, 239, 240, 241, 254, 255])
    np.savez_compressed(os.path.join(HERE, "logmel_sine_seed7.npz"), seed=7, rows=rows, logmel=lm[rows].astype(np.float64))
    rng = np.random.default_rng(11)
    noise = rng.uniform(-1, 1, 5000).astype(np.float32)     # ragged length: not a multiple of hop
    ln = O.compute_spectrogram(noise.astype(np.float64), np.float64)
    np.savez_compressed(os.path.join(HERE, "logmel_noise_5000.npz"), audio=noise, logmel=ln)


def make_model_golden():
    """mt3-config layer sizes but 1+1 layers and T=32 so the fixture stays small (<1 MB)."""
    cfg = O.T5Config(vocab_size=1536, num_encoder_layers=1, num_decoder_layers=1)
    params = O.init_params(cfg, seed=5, norm_scale_jitter=0.1)
    rng = np.random.default_rng(1)
    x = rng.standard_normal((2, 32, 512)).astype(np.float32)
    enc = O.encode(params, cfg, x, np.float64)
    toks, logits = O.greedy_decode(params, cfg, enc, 6, np.float64, stop_at_eos=False, return_logits=True)
    np.savez_compressed(os.path.join(HERE, "model_tiny.npz"), x=x, encoded=enc[:, ::8, ::16],
                        tokens=toks[:, :6], logits=logits[:, :, ::16], weight_seed=5, jitter=0.1)


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isfile(os.path.join(sys.argv[1], "event_codec.py")):
        sys.exit(__doc__)
    REF = sys.argv[1]
    make_codec_golden()
    make_codec_tables_golden()
    make_gin_golden()
    make_logmel_golden()
    make_model_golden()
    for f in sorted(os.listdir(HERE)):
        print(f, os.path.getsize(os.path.join(HERE, f)))

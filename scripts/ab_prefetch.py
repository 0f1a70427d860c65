#!/usr/bin/env python
"""A/B of value-neutral scheduling / cache knobs of the decode step in ONE process: every setting builds its own model
handle (the switches are read from the environment at mt3_model_create), runs bench.py's device-resident pass (log-mel +
encoder + cross-K/V + 1024 greedy steps, batch 64, L2 flushed between passes) and must reproduce the first setting's
token streams bit for bit.

The study it was written for (profiles/r02_call63_ab_l2_prefetch.txt, library at commit a136618): L2 prefetch of the K/V
tiles beyond the attention ring by the attention kernel itself (MT3_PF_ATTN, kept: -1.6 % at 16 tiles), by the GEMMs of
the previous layer (MT3_PF_GEMM: +0.8 .. +3.4 %) and a persisting-L2 window over the decoder weights (MT3_L2_PERSIST_MB:
0 .. +1.2 %); the last two and the evict_first hint (MT3_PF_HINT, neutral) were removed from the library afterwards.

  python scripts/ab_prefetch.py [--kv p24] [--reps 3] [--settings "name:K=V,K=V;..."] > gpurun_out/ab_prefetch.txt
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

KNOBS = ("MT3_PF_ATTN", "MT3_PDL", "MT3_DEC_FUSE", "MT3_DEC_CLUSTER", "MT3_DEC_PIPE")

DEFAULT = ";".join(["off:MT3_PF_ATTN=0", "attn4:MT3_PF_ATTN=4", "attn8:MT3_PF_ATTN=8", "default:", "attn32:MT3_PF_ATTN=32",
                    "attn64:MT3_PF_ATTN=64", "off2:MT3_PF_ATTN=0"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kv", default="p24", choices=["f32", "f16", "p24"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dec-steps", type=int, default=1024)
    ap.add_argument("--settings", default=DEFAULT)
    args = ap.parse_args()

    import torch
    import bench
    from mt3_b200 import _lib, network, spectrograms, weights

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B = bench.BATCH_PER_GPU
    cfg = network.T5Config(vocab_size=1536, emb_dim=512, num_heads=6, num_encoder_layers=8, num_decoder_layers=8, head_dim=64,
                           mlp_dim=1024, mlp_activations=('gelu', 'linear'))
    params = weights.synthetic_params(cfg, 0)
    spec_cfg = spectrograms.SpectrogramConfig()
    audio = torch.from_numpy(bench.synth_audio(B, 1234)).to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    kvf = {'f32': _lib.KV_F32, 'f16': _lib.KV_F16, 'p24': _lib.KV_P24}[args.kv]
    ref_tokens = None
    rows = []
    for item in args.settings.split(";"):
        name, _, kvs = item.partition(":")
        for k in KNOBS:
            os.environ.pop(k, None)
        for kv in filter(None, kvs.split(",")):
            k, v = kv.split("=")
            assert k in KNOBS, k
            os.environ[k] = v
        model = network.Transformer(cfg, params, device=dev, max_batch=B, max_input_length=256, max_decode_length=1024,
                                    gemm_mode=_lib.GEMM_TF32X3, kv_format=kvf)
        tokens = torch.empty((B, 1024), dtype=torch.int32, device=dev)

        def one_pass():
            spec = spectrograms.compute_spectrogram(audio, spec_cfg)
            model.generate(spec, num_steps=args.dec_steps, stop_at_eos=False, use_graph=True, out=tokens)

        for _ in range(2):
            one_pass()
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(args.reps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            one_pass()
            e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        tok = tokens.cpu().numpy().copy()
        if ref_tokens is None:
            ref_tokens = tok
        same = bool((tok == ref_tokens).all())
        row = {"setting": name, "env": kvs, "ms_mean": float(np.mean(ts)), "ms_min": float(np.min(ts)), "tokens_equal_first": same}
        rows.append(row)
        print(json.dumps(row), flush=True)
        del model
        torch.cuda.empty_cache()
    base = rows[0]["ms_mean"]
    print("\n%-28s %9s %9s %8s  tokens==first" % ("setting", "ms mean", "ms min", "vs first"))
    for r in rows:
        print("%-28s %9.2f %9.2f %+7.2f%%  %s" % (r["setting"], r["ms_mean"], r["ms_min"], 100.0 * (r["ms_mean"] / base - 1.0),
                                                  r["tokens_equal_first"]))
    return 0 if all(r["tokens_equal_first"] for r in rows) else 1


if __name__ == "__main__":
    sys.exit(main())

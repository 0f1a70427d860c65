"""MT3_DEC_PIPE (bitmask, decode.cuh dec_cluster_body): bit 0 stages the split-K decode GEMM's operand loads so the FMAs
start on the first 16 k-steps while the rest are in flight; bit 1 replaces the cluster-wide exchange barrier with one
bulk DSMEM copy per peer, completing on the receiver's mbarrier.  Neither touches an FMA or the order of any sum, so
graph-replayed greedy tokens and step-by-step logits are bit-identical to MT3_DEC_PIPE=0 for every bit combination.

The cases cover every cluster kernel instantiation the decode step launches: K chunks of 48 and 112 (fused
out-projection + cross-query launch), 64 (QKV, MLP-in, logits, and the unfused out / cross-query pair), the 16-CTA
MLP-out cluster (K = 1024, N = 512), and 128 (emb_dim 1024: QKV, MLP-in, MLP-out with N = 1024, logits); every K/V row
format; the exact-fp32 and the 3xTF32 encoder; full (64), ragged (33) and tiny (5) row counts."""
import numpy as np
import pytest
import torch

from oracle import mt3_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SMALL = dict(num_encoder_layers=1, num_decoder_layers=2)

# id: (gemm mode, K/V rows, batch rows, MT3_DEC_FUSE, config overrides)
CASES = {
    "mt3-b64-p24-tf32x3": ("tf32x3", "p24", 64, "1", {}),
    "mt3-b64-p24-unfused": ("tf32x3", "p24", 64, "0", {}),
    "small-b33-f32-tf32x3": ("tf32x3", "f32", 33, "1", SMALL),
    "small-b5-f16-tf32x3-unfused": ("tf32x3", "f16", 5, "0", SMALL),
    "small-b5-f32-simt": ("simt", "f32", 5, "1", SMALL),
    "small-b33-p24-simt-unfused": ("simt", "p24", 33, "0", SMALL),
    "d1024-b33-f16-tf32x3": ("tf32x3", "f16", 33, "1", dict(SMALL, emb_dim=1024)),
    "d1024-b64-p24-simt": ("simt", "p24", 64, "1", dict(SMALL, emb_dim=1024)),
}


def _mode_ids(gm, kv):
    from mt3_b200 import _lib
    return ({"simt": _lib.GEMM_FP32_SIMT, "tf32x3": _lib.GEMM_TF32X3}[gm],
            {"f32": _lib.KV_F32, "f16": _lib.KV_F16, "p24": _lib.KV_P24}[kv])


def _inputs(b, t=64, seed=0):
    audio = np.stack([O.sine_mix(t * 128, seed=1234 + seed + i) for i in range(b)])
    return O.compute_spectrogram(audio, np.float32)


@pytest.mark.parametrize("case", list(CASES))
def test_dec_pipe_bit_identical(case, monkeypatch):
    from mt3_b200 import network
    gm, kv, rows, fuse, over = CASES[case]
    kw = dict(vocab_size=1536, emb_dim=512, num_heads=6, num_encoder_layers=8, num_decoder_layers=8, head_dim=64, mlp_dim=1024,
              mlp_activations=('gelu', 'linear'))
    kw.update(over)
    ocfg = O.T5Config(**kw)
    cfg = network.T5Config(**kw)
    params = O.init_params(ocfg, seed=41)
    x = torch.from_numpy(_inputs(rows, seed=900)).to(DEV)
    forced = torch.from_numpy(np.random.default_rng(7).integers(3, 1500, size=(rows, 12)).astype(np.int32)).to(DEV)
    gmode, kvf = _mode_ids(gm, kv)
    monkeypatch.setenv("MT3_DEC_FUSE", fuse)

    def run(pipe):
        monkeypatch.setenv("MT3_DEC_PIPE", str(pipe))
        m = network.Transformer(cfg, params, device=DEV, max_batch=rows, max_input_length=64, max_decode_length=40, gemm_mode=gmode,
                                kv_format=kvf)
        toks = m.generate(x, stop_at_eos=False, use_graph=True).cpu().numpy()
        lg = m.teacher_forced_logits(m.encode(x), forced).cpu().numpy()
        del m
        return toks, lg

    base_t, base_l = run(0)
    assert np.isfinite(base_l).all()
    for pipe in (1, 2, 3):
        t, lg = run(pipe)
        np.testing.assert_array_equal(t, base_t, err_msg=f"MT3_DEC_PIPE={pipe}: tokens")
        np.testing.assert_array_equal(lg, base_l, err_msg=f"MT3_DEC_PIPE={pipe}: logits")

"""Multi-GPU parity (-m gpu, skipped below 2 GPUs; run on a machine with 2 or more GPUs: `python -m pytest tests/test_gpu_multi.py -m gpu`).

BASELINE configs[4]: 3 minutes of audio -> 88 segments -> tokens -> stitched NoteSequence, with the segments sharded over
one process per GPU (torch.distributed / NCCL): ONE weight broadcast at load, ONE all-gather of the token streams, no
other collective (SURVEY 8e; notebook :283-308, metrics_utils.py:119-146).  The sharded result must be identical to the
single-GPU one: segments never interact."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import mt3_oracle as O

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _audio():
    n = 3 * 60 * 16000
    return np.concatenate([O.sine_mix(32768, 100 + i) for i in range(-(-n // 32768))])[:n]


def _notes(ns):
    return [(n.pitch, n.start_time, n.end_time, n.program, n.velocity) for n in ns.notes]


def _worker(rank, world, port, steps, q):
    import torch.distributed as dist
    from mt3_b200 import _lib, inference, note_decoding
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        # only rank 0 has the checkpoint: the other ranks receive the weights through the one broadcast
        im = inference.InferenceModel("synthetic:0" if rank == 0 else None, "mt3", device=dev, batch_size=32)
        im.outputs_length = 1024
        audio = _audio()
        ds = im.preprocess(im.audio_to_dataset(audio))
        hop = im.spectrogram_config.hop_width
        segs = np.zeros((len(ds), 256 * hop), np.float32)
        nv = np.zeros((len(ds),), np.int32)
        for i, ex in enumerate(ds):
            flat = np.asarray(ex['inputs'], np.float32).reshape(-1)
            segs[i, :flat.size] = flat
            nv[i] = flat.size // hop
        toks = im.transcribe_segments_sharded(segs, n_valid_frames=nv, num_steps=steps, stop_at_eos=False)
        preds = [im.postprocess(t, ex) for t, ex in zip(toks, ds)]
        ns = note_decoding.event_predictions_to_ns(preds, im.codec, im.encoding_spec)['est_ns']
        out = {"rank": rank, "segments": len(ds), "tokens_shape": tuple(toks.shape), "notes": _notes(ns)}
        if rank == 0:      # the whole list on this GPU alone, outside the sharding
            ref = im.transcribe_segments(segs, n_valid_frames=nv, num_steps=steps, stop_at_eos=False)
            out["tokens_equal"] = bool(np.array_equal(ref, toks))
            rpreds = [im.postprocess(t, ex) for t, ex in zip(ref, ds)]
            out["ref_notes"] = _notes(note_decoding.event_predictions_to_ns(rpreds, im.codec, im.encoding_spec)['est_ns'])
        q.put(out)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_longform_three_minutes_sharded_over_gpus():
    n_gpus = torch.cuda.device_count()
    if n_gpus < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    world = min(n_gpus, 8)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, 96, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=900) for _ in procs), key=lambda r: r["rank"])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    r0 = res[0]
    assert r0["segments"] == 88 and r0["tokens_shape"] == (88, 1024)
    assert r0["tokens_equal"], "sharded token streams differ from the single-GPU run"
    assert r0["notes"] == r0["ref_notes"]
    for r in res[1:]:                       # every rank holds the same stitched result after the all-gather
        assert r["notes"] == r0["notes"]

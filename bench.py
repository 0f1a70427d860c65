#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on its configs[1]: audio-seconds transcribed per second,
mt3 config, batch = 64 x 2.048 s synthetic segments per GPU, log-mel + encoder + greedy decode.

A "step" is one pass of the hot path over one batch (64 segments/GPU): log-mel kernel ->
8-layer encoder -> cross-K/V -> DEC_STEPS greedy decode steps (default 1024 = the reference's
outputs_length with EOS never stopping the loop: random weights make EOS timing meaningless,
so the worst case is what is timed; nothing is skipped).

  python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
  python bench.py --impl reference ...                     (the CPU restatement on host cores)
  python bench.py ... --dump-outputs DIR                   (also saves the last timed step's tokens: DIR/tokens.npy)

`value`  device-resident inputs, timed with CUDA events per step (L2 flushed between steps),
         max over ranks, whole-job aggregate over N GPUs (weak scaling: 64 segments per GPU).
         Arithmetic is float32 everywhere; the decoder's K/V rows are STORED with 24 bits per element by
         default (--kv p24: three quarters of the bytes the decode step streams; logit error ~5e-6 of the
         scale against the float64 oracle at cache lengths up to 1024, the level of the float32
         arithmetic).  The same pass with fp32 and with fp16 rows is timed too and reported as
         `value_kv_f32` / `value_kv_f16` (fp16 rows leave the 5e-4 bar when attention is sharp: DESIGN.md 4).
`e2e`    same metric through InferenceModel.transcribe_segments with pinned HOST audio in and
         HOST tokens out (H2D + D2H inside the timed region).
`roofline` the dominant kernel (decode self-attention over the KV cache), algorithmic bytes per
         launch / CUDA-event time per launch, against MEASURED_PEAKS.json's HBM copy bandwidth;
         `roofline.job`: the whole pass -- algorithmic bytes of one step (all K/V rows read once per
         decode step + the decoder weights once per decode step) / the measured step time.
`cpu_baseline` the torch-CPU port of the reference semantics (oracle/torch_cpu.py; the JAX/T5X
         reference itself is not installable here) on a bounded sample, rank 0, N=1 only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEG_SAMPLES = 32768
SEG_SECONDS = SEG_SAMPLES / 16000.0
BATCH_PER_GPU = 64


def synth_audio(n, seed0):
    """SURVEY 8d sine-mix, numpy default_rng seeded per segment (vectorised; the product never
    imports oracle/, so this is bench's own generator)."""
    out = np.zeros((n, SEG_SAMPLES), np.float32)
    t = np.arange(SEG_SAMPLES, dtype=np.float64) / 16000.0
    for i in range(n):
        rng = np.random.default_rng(seed0 + i)
        x = np.zeros(SEG_SAMPLES)
        for _ in range(int(rng.integers(3, 9))):
            pitch = int(rng.integers(36, 97))
            f = 440.0 * 2.0 ** ((pitch - 69) / 12.0)
            x += rng.uniform(0.05, 0.3) * np.sin(2 * np.pi * f * t + rng.uniform(0, 2 * np.pi))
        out[i] = (x * (0.9 / max(1e-12, np.abs(x).max()))).astype(np.float32)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.p, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """CPU threads this process may really use: affinity mask and cgroup quota, not os.cpu_count()
    (a container on a 200-core host may own 8 of them; oversubscribing torch's pool stalls it)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, min(n, 64))


def workload_config(dec_steps):
    """`config` is IDENTICAL in both arms (the driver compares them): what is computed, not how."""
    return {"workload": "mt3 config (BASELINE configs[1]): batch=64 x 2.048 s synthetic sine-mix segments per GPU, "
                        f"log-mel + 8-layer encoder + greedy decode, {dec_steps} decode steps, EOS never stops the loop; "
                        "GPU arm: L2 flushed between timed steps (256 MB write)",
            "segments_per_gpu": BATCH_PER_GPU, "dec_steps": dec_steps}


def log(msg):
    sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')}] {msg}\n")
    sys.stderr.flush()


def cpu_port_sample(params, audio, nb, dec_steps, budget_s):
    """Times the torch-CPU port on `nb` segments: log-mel + encoder fully, then greedy decode until
    `budget_s` of wall time; the decode is extrapolated linearly to `dec_steps` (the per-step cost grows
    with the cache, so this favours the CPU).  Returns (audio-s/s, cores, description, ms)."""
    import torch
    from oracle import mt3_oracle as O
    from oracle import torch_cpu as TC
    cores = host_threads()
    torch.set_num_threads(cores)
    cm = TC.TorchCpuModel(params, O.T5Config())
    a = audio[:nb].clone()
    with torch.no_grad():
        t0 = time.perf_counter()
        spec = TC.compute_logmel(a)
        enc = cm.encode(spec)
        t_fixed = time.perf_counter() - t0
        log(f"cpu port: log-mel+encoder {t_fixed:.2f} s on {cores} threads")
        t0 = time.perf_counter()
        cm.greedy_decode(enc, dec_steps, time_budget_s=budget_s)
        t_dec = time.perf_counter() - t0
        ran = max(1, cm.last_steps_run)
    log(f"cpu port: {ran} decode steps in {t_dec:.2f} s")
    full = t_fixed + t_dec / ran * dec_steps
    desc = (f"{nb} segments: log-mel + encoder in full ({t_fixed:.2f} s), {ran} of {dec_steps} greedy steps ({t_dec:.2f} s) "
            f"extrapolated linearly to {dec_steps} (favours the CPU); torch-CPU fp32 port of the reference semantics "
            f"with hoisted cross-K/V (the JAX/T5X reference is not installable here)")
    return nb * SEG_SECONDS / full, cores, desc, 1000.0 * (t_fixed + t_dec)


def KV_FORMATS():
    from mt3_b200 import _lib
    return {'f32': _lib.KV_F32, 'f16': _lib.KV_F16, 'p24': _lib.KV_P24}


def load_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return float(json.load(f)[kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------------------------
def ref_budget(args):
    """Wall-time budget of one CPU sample's decode loop: the whole `--steps K --warmup W` run must end within a few
    minutes, so the per-sample budget shrinks with K + W (the decode is extrapolated linearly from the steps that fit,
    which favours the CPU: the per-step cost grows with the cache)."""
    return max(2.0, min(args.ref_budget_s, 200.0 / max(1, args.steps + args.warmup)))


def run_reference(args):
    """The reference arm: the CPU restatement (torch-CPU port of the oracle) on the host cores, on the SAME workload
    as the GPU arm (64 segments per batch).  Each step is one bounded sample (see cpu_port_sample); `value` is the mean."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    from oracle import mt3_oracle as O
    params = O.init_params(O.T5Config(), seed=0)
    audio = torch.from_numpy(synth_audio(args.ref_batch, 1234))
    vals, mss = [], []
    budget = ref_budget(args)
    for i in range(args.warmup + args.steps):
        v, cores, desc, ms = cpu_port_sample(params, audio, args.ref_batch, args.dec_steps, budget if i >= args.warmup else min(3.0, budget))
        if i >= args.warmup:
            vals.append(v)
            mss.append(ms)
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(mss)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.dec_steps),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": desc,
                         "sample_batch": args.ref_batch, "decode_budget_s": budget},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from mt3_b200 import _lib, inference, spectrograms, weights

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = BATCH_PER_GPU
    from mt3_b200 import distributed as mt3_dist
    # ---- weights: rank 0 draws them, ONE NCCL broadcast at load (north_star) -------------------
    # (InferenceModel.restore_from_checkpoint: only rank 0 materialises the checkpoint, then broadcast_params)
    gm = {'simt': _lib.GEMM_FP32_SIMT, 'tf32x3': _lib.GEMM_TF32X3, 'tf32': _lib.GEMM_TF32}[args.gemm_mode]
    kvf = KV_FORMATS()[args.kv]
    im = inference.InferenceModel('synthetic:0', 'mt3', device=dev, batch_size=B, use_graph=True, gemm_mode=gm, kv_format=kvf)

    # ---- inputs: contiguous shard of the global segment list ---------------------------------
    audio_host = torch.from_numpy(synth_audio(B, 1234 + rank * B)).pin_memory()
    audio_dev = audio_host.to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2
    tokens = torch.empty((B, 1024), dtype=torch.int32, device=dev)
    dec_steps = args.dec_steps

    def one_pass():
        spec = spectrograms.compute_spectrogram(audio_dev, im.spectrogram_config)
        im.model.generate(spec, num_steps=dec_steps, stop_at_eos=False, use_graph=True, out=tokens)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    log(f"model ready; warm-up x{args.warmup}")
    for _ in range(args.warmup):
        one_pass()
    barrier()
    log("timed region")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    evs = []
    barrier()
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        one_pass()
        e1.record()
        evs.append((e0, e1))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = _lib.launch_count() - launches0
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # the legs below reuse `tokens`: take the last timed step's ids now, every rank's segments in global order
        dump = mt3_dist.gather_tokens(tokens.clone(), world * B).cpu().numpy()
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "tokens.npy"), dump.astype(np.float32))   # ids < 2^24: exact
            log(f"wrote {args.dump_outputs}/tokens.npy {dump.shape}")

    log(f"timed {args.steps} steps: {total_ms / args.steps:.1f} ms/step; e2e leg")
    # ---- e2e: public API with HOST buffers (H2D + D2H inside the timed region) ----------------
    out_host = im.transcribe_segments(audio_host, num_steps=dec_steps, stop_at_eos=False)   # warm the API path ...
    if world > 1:                                                                            # ... and the collective
        mt3_dist.gather_tokens(torch.from_numpy(out_host).to(dev), world * B)
    barrier()
    e2e_times = []
    for _ in range(max(3, min(args.steps, 5))):
        flush.fill_(1)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        out_host = im.transcribe_segments(audio_host, num_steps=dec_steps, stop_at_eos=False)
        if world > 1:      # the job's one data-path collective: all-gather of the token streams, inside the timed region
            all_tokens = mt3_dist.gather_tokens(torch.from_numpy(out_host).to(dev), world * B)
            torch.cuda.synchronize(dev)
            assert all_tokens.shape == (world * B, 1024)
        e2e_times.append(time.perf_counter() - t0)
    e2e_ms = 1000.0 * float(np.median(e2e_times))

    # ---- the same device-resident pass with the OTHER K/V storage formats (fp32 and fp16 rows when the headline uses 24-bit rows) ----
    alt_ms = {}
    for alt_name in ([] if args.no_alt_kv else [n for n in ('f32', 'p24', 'f16') if n != args.kv]):
        im_alt = inference.InferenceModel('synthetic:0', 'mt3', device=dev, batch_size=B, use_graph=True, gemm_mode=gm,
                                          kv_format=KV_FORMATS()[alt_name])

        def alt_pass():
            spec = spectrograms.compute_spectrogram(audio_dev, im_alt.spectrogram_config)
            im_alt.model.generate(spec, num_steps=dec_steps, stop_at_eos=False, use_graph=True, out=tokens)
        for _ in range(2):
            alt_pass()
        barrier()
        ts = []
        for _ in range(3):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            alt_pass()
            e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        alt_ms[alt_name] = float(np.mean(ts))
        del im_alt
        torch.cuda.empty_cache()

    # ---- the same pass at T_dec = 256 (SURVEY 8d reports both decode lengths) ----------------------------------------
    d256_ms = None
    if dec_steps == 1024 and not args.no_alt_kv:
        def pass256():
            spec = spectrograms.compute_spectrogram(audio_dev, im.spectrogram_config)
            im.model.generate(spec, num_steps=256, stop_at_eos=False, use_graph=True, out=tokens)
        pass256()
        ts = []
        for _ in range(3):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            pass256()
            e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        d256_ms = float(np.mean(ts))

    # ---- all-gather of the decoded token streams at the end (north_star) -----------------------
    if world > 1:
        alt_names = sorted(alt_ms)
        t = torch.tensor([total_ms, e2e_ms, d256_ms or 0.0] + [alt_ms[n] for n in alt_names], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms = float(t[0]), float(t[1])
        d256_ms = float(t[2]) if d256_ms is not None else None
        alt_ms = {n: float(t[3 + i]) for i, n in enumerate(alt_names)}
        ln = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(ln)
        launches = int(ln[0])

    ms_per_step = total_ms / args.steps
    value = world * B * SEG_SECONDS / (ms_per_step / 1000.0)
    e2e_value = world * B * SEG_SECONDS / (e2e_ms / 1000.0)

    log(f"e2e {e2e_ms:.1f} ms/step; roofline leg")
    # ---- roofline of the dominant kernel: decode self-attention over the KV cache --------------
    roofline = None
    cpu_baseline = None
    if rank == 0:
        peak, peak_src = load_peaks()
        lib = _lib.load()
        h = im.model._h
        stream = torch.cuda.current_stream(dev).cuda_stream
        pos = 511                                   # mean cache length of a 1024-step decode
        H, D = 6, 64
        elt = {'f32': 4, 'f16': 2, 'p24': 3}[args.kv]   # bytes per stored K/V element
        alg_bytes = B * H * (pos + 1) * D * elt * 2 + B * H * D * 4 * 2   # K and V rows read once + q in, o out
        iters = 64
        for _ in range(2):
            _lib.check(lib.mt3_debug_launch(h, _lib.K_DEC_SELF_ATTN, pos, 8, stream))
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(lib.mt3_debug_launch(h, _lib.K_DEC_SELF_ATTN, pos, iters, stream))   # cycles over 8 layers' caches (805 MB > L2)
        e1.record()
        torch.cuda.synchronize(dev)
        us = 1000.0 * e0.elapsed_time(e1) / iters
        ach = alg_bytes / (us * 1e-6) / 1e9
        roofline = {"kernel": f"dec_attention_bulk_kernel (decode self-attention, cache length 512, B=64, 6 heads, {args.kv} K/V rows)", "bound": "hbm",
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": load_traffic("dec_attention_bulk_kernel_" + args.kv),
                    "peak_source": peak_src, "us_per_launch": us, "algorithmic_bytes_per_launch": alg_bytes}
        # the whole pass against the same peak: every decode step reads all K/V rows written so far (self) and the 256
        # hoisted rows (cross) of 8 layers once, plus the decoder's 103.9 MB of fp32 weights (L2-resident across steps
        # when they fit, counted anyway); encoder + frontend traffic (< 1 %) is left out, so the fraction is a lower bound
        Ld, T = 8, 256
        kv_bytes = sum(B * H * D * elt * 2 * (l_ + T) for l_ in range(1, dec_steps + 1)) * Ld
        w_bytes = 103.9e6 * dec_steps
        job_bytes = kv_bytes + w_bytes
        job_ach = job_bytes / (ms_per_step * 1e-3) / 1e9
        roofline["job"] = {"bytes_per_step": job_bytes, "kv_bytes": kv_bytes, "weight_bytes": w_bytes, "achieved": job_ach, "peak": peak,
                           "unit": "GB/s", "frac": job_ach / peak, "ms_per_step": ms_per_step,
                           "floor_ms": job_bytes / (peak * 1e9) * 1e3}
        # back-to-back launch time of the other hot kernels at the bench shapes (device events, stream order)
        kernels_us = {}
        for name, kind, p_, it_ in (("dec_self_attention_len512", _lib.K_DEC_SELF_ATTN, 511, 64),
                                    ("dec_self_attention_len32", _lib.K_DEC_SELF_ATTN, 31, 64),
                                    ("dec_self_attention_len128", _lib.K_DEC_SELF_ATTN, 127, 64),
                                    ("dec_self_attention_len1024", _lib.K_DEC_SELF_ATTN, 1023, 64),
                                    ("dec_cross_attention_len256", _lib.K_DEC_CROSS_ATTN, 0, 64),
                                    ("dec_qkv_gemm_64x1152x512", _lib.K_DEC_QKV_GEMM, 0, 64),
                                    ("enc_qkv_gemm_16384x1152x512", _lib.K_ENC_QKV_GEMM, 0, 16),
                                    ("enc_attention_64x6x256x256", _lib.K_ENC_ATTN, 0, 16)):
            _lib.check(lib.mt3_debug_launch(h, kind, p_, 4, stream))
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(lib.mt3_debug_launch(h, kind, p_, it_, stream))
            e1.record()
            torch.cuda.synchronize(dev)
            kernels_us[name] = 1000.0 * e0.elapsed_time(e1) / it_
        # K1 at the bench shape (64 segments) and BASELINE configs[3]: 10 min stream, FFT 1024 / 2048 / 4096 at hop 128
        from mt3_b200 import spectral_ops
        def time_logmel(a, fft, iters=5):
            kw = dict(lo_hz=20.0, hi_hz=7600.0, bins=512, fft_size=fft, overlap=1.0 - 128.0 / fft)
            spectral_ops.compute_logmel(a, **kw)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                spectral_ops.compute_logmel(a, **kw)
            e1.record()
            torch.cuda.synchronize(dev)
            return 1000.0 * e0.elapsed_time(e1) / iters
        kernels_us["logmel_fft2048_64x2.048s"] = time_logmel(audio_dev, 2048, 20)
        # encoder + cross-K/V alone (SURVEY 8d: 10.603 + 1.611 GFLOP per segment) against the tensor roof: the tf32 peak is
        # nominally half of the measured bf16 throughput; TF32X3 issues 3 MMAs per algorithmic one
        spec_dev = spectrograms.compute_spectrogram(audio_dev, im.spectrogram_config)
        enc_out = im.model.encode(spec_dev)
        im.model.init_cache(enc_out)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            enc_out = im.model.encode(spec_dev)
            im.model.init_cache(enc_out)
        e1.record()
        torch.cuda.synchronize(dev)
        enc_ms = e0.elapsed_time(e1) / 5
        try:
            bf16_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
        except Exception:
            bf16_peak = 1664.5
        enc_tflops = (10.603e9 + 1.611e9) * B / (enc_ms * 1e-3) / 1e12
        passes = 3 if args.gemm_mode == "tf32x3" else 1
        roofline["encoder"] = {"ms": enc_ms, "algorithmic_tflops": enc_tflops, "mma_tflops": enc_tflops * passes,
                               "tf32_peak_tflops": bf16_peak / 2, "frac_algorithmic": enc_tflops / (bf16_peak / 2),
                               "frac_mma_work": enc_tflops * passes / (bf16_peak / 2),
                               "note": "encode + cross-K/V of 64 segments; tf32 peak taken as half of the measured bf16 throughput"}
        stream10 = torch.from_numpy(synth_audio(293, 99)).to(dev)          # 293 x 32768 samples = 10 min
        sweep = {}
        for fft in (1024, 2048, 4096):
            us = time_logmel(stream10, fft, 3)
            alg = 293 * (32768 * 4 + 256 * 512 * 4)
            # the roof that binds K1 is fp32 issue, not HBM (hop 128: every sample feeds fft/128 frames): radix-2 work of the
            # packed real FFT, 5 NC log2(NC) + 20 NC flops per frame with NC = fft / 2, against 148 SMs x 128 lanes x 2 x f_SM
            nc = fft // 2
            flops = 293 * 256 * (5 * nc * np.log2(nc) + 20 * nc)
            fp32_peak = 148 * 128 * 2 * 1.965e9
            sweep[f"fft{fft}"] = {"us": us, "algorithmic_GBps": alg / (us * 1e-6) / 1e9, "frac_of_hbm_peak": alg / (us * 1e-6) / 1e9 / peak,
                                  "fft_tflops": flops / (us * 1e-6) / 1e12, "frac_of_fp32_peak": flops / (us * 1e-6) / fp32_peak}
        del stream10
        roofline["logmel_10min_stream_sweep"] = sweep
        roofline["other_kernels_us_per_launch"] = kernels_us
        log("kernel microbench: " + ", ".join(f"{k}={v:.1f}us" for k, v in kernels_us.items()))
        if world == 1 and not args.no_cpu_baseline:
            log("cpu baseline (torch-CPU port) ...")
            cpu_params = weights.synthetic_params(im._model_config(), 0)
            cpu_port_sample(cpu_params, audio_host, args.ref_batch, dec_steps, 2.0)          # warm (thread pool, allocator)
            v, cores, desc, _ = cpu_port_sample(cpu_params, audio_host, args.ref_batch, dec_steps, args.ref_budget_s)
            cpu_baseline = {"value": v, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": desc,
                            "sample_batch": args.ref_batch}

    if rank == 0:
        line = {
            "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(dec_steps),
            "impl_config": {"gemm_mode": args.gemm_mode, "kv_cache": args.kv + " rows, fp32 arithmetic",
                            "l2": "flushed between steps (256 MB write)",
                            "kv_l2_prefetch_tiles": os.environ.get("MT3_PF_ATTN", "16 (library default)"),
                            "parallelism": f"dp{world} (segments sharded, 1 weight broadcast, 1 token all-gather)"},
            "segments_per_second": value / SEG_SECONDS,
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": int(B * SEG_SAMPLES * 4),
                    "d2h_bytes_per_step": int(B * 1024 * 4), "ms_per_step": e2e_ms,
                    "api": "InferenceModel.transcribe_segments (pinned host audio -> host tokens)"},
            "gpu_launches": int(launches), "wall_s_timed_region": t_wall,
            "clocks": clocks, "roofline": roofline,
        }
        for alt_name, ms in sorted(alt_ms.items()):
            line["value_kv_" + alt_name] = world * B * SEG_SECONDS / (ms / 1000.0)
            line["ms_per_step_kv_" + alt_name] = ms
        if d256_ms is not None:
            line["dec_steps_256"] = {"ms_per_step": d256_ms, "value": world * B * SEG_SECONDS / (d256_ms / 1000.0), "unit": "audio-s/s"}
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_longform(args):
    """BASELINE configs[4]: 3 minutes of audio -> 88 segments of 2.048 s -> tokens -> stitched NoteSequence, the segments
    sharded over the N GPUs (strong scaling: the work is fixed).  Timed end to end through InferenceModel.__call__'s
    pieces: host framing, H2D, log-mel + encoder + greedy decode, D2H, all-gather, host stitch."""
    import torch
    import torch.distributed as dist
    from mt3_b200 import _lib, inference, note_decoding
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    kvf = KV_FORMATS()[args.kv]
    im = inference.InferenceModel('synthetic:0' if rank == 0 else None, 'mt3', device=dev, batch_size=BATCH_PER_GPU, kv_format=kvf)
    n = 3 * 60 * 16000
    audio = synth_audio(-(-n // SEG_SAMPLES), 100).reshape(-1)[:n]
    launches0 = _lib.launch_count()

    def one():
        preds = im.predict_segments(audio)
        return note_decoding.event_predictions_to_ns(preds, im.codec, im.encoding_spec)['est_ns'], len(preds)

    for _ in range(max(1, args.warmup)):
        one()
    times = []
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        ns, nseg = one()
        torch.cuda.synchronize(dev)
        times.append(time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    ms = 1000.0 * float(np.mean(times))
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
    if rank == 0:
        v = (n / 16000.0) / (ms / 1000.0)
        print(json.dumps({
            "metric": "audio_seconds_per_second", "value": v, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "mt3 config long-form (BASELINE configs[4]): 3 min of 16 kHz audio -> 88 segments -> greedy decode "
                                   "(1024 steps, synthetic weights never emit EOS) -> event_codec stitch to a NoteSequence",
                       "segments": nseg, "segments_per_gpu": -(-nseg // world)},
            "impl_config": {"kv_cache": args.kv + " rows, fp32 arithmetic", "parallelism": f"dp{world}: segments sharded, 1 all-gather"},
            "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": int(nseg * SEG_SAMPLES * 4), "d2h_bytes_per_step": int(nseg * 1024 * 4),
                    "ms_per_step": ms, "api": "InferenceModel.predict_segments + note_decoding.event_predictions_to_ns"},
            "gpu_launches": int(_lib.launch_count() - launches0), "clocks": clocks, "notes_out": len(ns.notes)}))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dec-steps", type=int, default=1024)
    ap.add_argument("--ref-batch", type=int, default=BATCH_PER_GPU, help="CPU sample: segments per batch (the GPU arm's 64)")
    ap.add_argument("--kv", default="p24", choices=["f32", "f16", "p24"], help="storage format of the decoder's K/V rows")
    ap.add_argument("--no-alt-kv", action="store_true", help="skip timing the other K/V storage format")
    ap.add_argument("--ref-budget-s", type=float, default=15.0, help="CPU sample: wall-time budget of the decode loop")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gemm-mode", default="tf32x3", choices=["simt", "tf32x3", "tf32"],
                    help="encoder/cross-K/V GEMMs: exact fp32 CUDA cores, or tcgen05 tf32 (x3 = fp32-faithful split)")
    ap.add_argument("--workload", default="batch", choices=["batch", "longform"],
                    help="batch: BASELINE configs[1]/[2] (64 segments per GPU, the headline); longform: configs[4] (3 min of audio, strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="batch workload: write the raw token ids of the last timed step, all segments of all GPUs, "
                         "to DIR/tokens.npy (float32 [segments, 1024], 0 past --dec-steps)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "batch"):
        ap.error("--dump-outputs needs --impl ours --workload batch")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "longform":
        return run_longform(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

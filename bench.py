#!/usr/bin/env python
"""bench.py -- Diffsound hot path on B200: text->wav clips/s for 10 s clips at 100 diffusion steps.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 16] [--codebook 256] [--precision f16x3]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference algorithm's CPU path (oracle port) on the host cores

One "step" = one caption batch through the whole hot path (BASELINE.json configs[1] extended to audio, i.e. configs[2]'s pipeline at
configs[1]'s batch): DiffusionTransformer.sample() (100 sequential p_sample steps, top0.85r) -> SpecVQGAN decoder -> MelGAN vocoder,
`batch` clips per GPU.  `value` times it with the caption embeddings resident in HBM; `e2e` times pipeline.synthesize() from pinned
host embeddings to pinned host waveforms.  Weak scaling over ranks (independent captions), finished waveforms all-gathered over NCCL
inside the timed region.  The denoiser runs in the parity-grade 'f16x3' mode by default (split-fp16, three tcgen05 passes, fp32-class
logits); the single-pass 'f16' throughput mode is reported under "modes".  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "clips/sec (10s audio, 100 diffusion steps)"
FLOP_PER_CLIP_STEP = {256: 158.25e9, 512: 158.39e9}  # SURVEY.md section 8(d): denoiser FLOPs per clip per diffusion step
DECODER_FLOP_PER_CLIP = 0.2613e12                    # SURVEY.md 8(d): SpecVQGAN decoder
VOCODER_FLOP_PER_CLIP = 0.0766e12                    # MelGAN generator
VOCODER_BYTES_PER_CLIP = 0.73e9                      # algorithmic activation traffic of the MelGAN stack (fp32), SURVEY.md 8(d)
DECODER_BYTES_PER_CLIP = 0.81e9                      # conv input + output activations in fp32, SURVEY.md 8(d)
L_TOK, WAV_LEN = 265, 217088
DUMP_LIMIT_BYTES = 64 << 20                          # --dump-outputs: at most this much in all


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, parsed by tools/ncu_traffic.py from the committed
    `ncu --set full` capture of THIS build (profiles/r2_traffic.json); None when the capture is absent."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) >= 7 and r[3 + i].lower().startswith("active")})
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def synthetic_cond(B, seed, cond_dim=512):
    g = torch.Generator().manual_seed(seed)
    c = torch.randn(B, 77, cond_dim, generator=g)
    return c / c.norm(dim=-1, keepdim=True)  # normalize: True (clip_text_embedding.py:78-79)


# ------------------------------------------------------------------------------------------------ CPU leg (oracle port = checker + baseline)
def best_thread_count(O, sd, B):
    """"All the host threads it can use": torch's intra-op pool stops scaling long before 100+ threads on M = B*265 row GEMMs, so probe a
    few pool sizes on one layer and keep the fastest."""
    ncpu = os.cpu_count() or 1
    x = torch.randn(B, L_TOK, 1024)
    cond = synthetic_cond(B, 1)
    tt = torch.full((B,), 50, dtype=torch.long)
    best = (float("inf"), 1)
    for n in sorted({min(n, ncpu) for n in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(n)
        with torch.no_grad():
            O.transformer_block(sd, "transformer.blocks.0.", x, cond, tt, 16)
            t0 = time.perf_counter()
            for _ in range(2):
                O.transformer_block(sd, "transformer.blocks.0.", x, cond, tt, 16)
            best = min(best, (time.perf_counter() - t0, n))
    return best[1]


def cpu_leg(sd_t, sd_codec, sd_voc, *, K, n_layer, B, n_steps, seed=77):
    """The reference algorithm (oracle port) on the host cores for a BOUNDED sample of the workload: `n_steps` of the 100 p_sample steps
    (t = 99 ..), then SpecVQGAN decode and MelGAN vocode of the resulting grids, at batch B.  Returns the extrapolated text->wav clips/s and the
    tensors the GPU leg is checked against (same weights, same caption embeddings, same uniforms)."""
    from oracle import diffsound_oracle as O
    threads = best_thread_count(O, sd_t, B)
    torch.set_num_threads(threads)
    cond = synthetic_cond(B, seed)
    g = torch.Generator().manual_seed(seed + 1)
    us = [torch.rand(B, K + 1, L_TOK, generator=g) for _ in range(n_steps)]
    steps = list(range(99, 99 - n_steps, -1))
    with torch.no_grad():
        t99 = torch.full((B,), 99, dtype=torch.long)
        logits0 = O.transformer_forward(sd_t, torch.full((B, L_TOK), K, dtype=torch.long), cond, t99, n_layer=n_layer, n_head=16, spatial=(5, 53))  # also the warm-up
        t0 = time.perf_counter()
        tok = O.sample(sd_t, cond, lambda i: us[i], n_layer=n_layer, n_head=16, spatial=(5, 53), steps=steps)
        t_samp = time.perf_counter() - t0
        tok_dec = tok.clamp(max=K - 1)  # a partially denoised grid still holds [MASK] = K: decode a valid id instead (same on both sides)
        t0 = time.perf_counter()
        mel = O.decode_to_img(sd_codec, tok_dec)
        t_dec = time.perf_counter() - t0
        t0 = time.perf_counter()
        wav = O.melgan_forward(sd_voc, (mel[:, 0] + 1) / 2)
        t_voc = time.perf_counter() - t0
    per_batch = t_samp / n_steps * 100.0 + t_dec + t_voc
    sample = (f"B={B}: {n_steps} of 100 p_sample steps (t=99..{steps[-1]}, {t_samp:.1f} s, x{100 / n_steps:g} linear extrapolation) + SpecVQGAN decode "
              f"({t_dec:.1f} s) + MelGAN ({t_voc:.1f} s); fp32 torch on {threads} threads")
    return {"value": B / per_batch, "cores": threads, "sample": sample, "cond": cond, "us": us, "steps": steps, "tok": tok, "tok_dec": tok_dec,
            "mel": mel, "wav": wav, "logits0": logits0}


def random_state_dicts(K, n_layer):
    """CPU-only weights for `--impl reference` (no GPU module to take them from)."""
    from oracle import diffsound_oracle as O
    sd_t = O.make_transformer_state_dict(K=K, D=1024, n_layer=n_layer, n_head=16, cond_dim=512, seed=0)
    sd_c = O.make_decoder_state_dict(n_embed=K, seed=4)
    ck = os.path.join(ROOT, "oracle", "_ref", "best_netG.pt")
    sd_v = torch.load(ck, map_location="cpu") if os.path.exists(ck) else O.make_melgan_state_dict(seed=1)
    return sd_t, sd_c, sd_v


def run_reference_arm(args):
    """CPU arm: the reference algorithm (oracle port -- the reference itself is Python under /root/reference and cannot travel to the GPU box;
    its transformer also hard-requires CUDA, SURVEY.md section 0 fact 3) on the host cores, same workload, bounded sample."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    sd_t, sd_c, sd_v = random_state_dicts(args.codebook, args.layers)
    r = cpu_leg(sd_t, sd_c, sd_v, K=args.codebook, n_layer=args.layers, B=min(args.batch, 4), n_steps=max(5, min(50, 2 * args.steps)))
    v = r["value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "clips/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * args.batch / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.batch, args.codebook, args.layers) + " [CPU port of the reference algorithm]"},
            "cpu_baseline": {"value": v, "unit": "clips/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": v, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_name(B, K, layers):
    return (f"Diffsound text->wav: batch {B}/GPU, 100 diffusion steps (top0.85r), K={K} codebook, 265-token grid -> SpecVQGAN decoder -> MelGAN, 9.85 s "
            f"clips @22.05 kHz (BASELINE.json configs[1] batch with configs[2]'s full pipeline); {layers}-layer D=1024 denoiser, random-init weights, "
            f"shipped MelGAN weights, synthetic caption embeddings")


# ------------------------------------------------------------------------------------------------ GPU arm
def build_models(K, n_layer, precision):
    import _pkg
    _pkg.load()
    from diffsound_b200.utils import builders
    dalle = builders.build_dalle(K=K, NL=n_layer, precision=precision, seed=0)
    voc = builders.build_vocoder(os.path.join(ROOT, "oracle", "_ref", "best_netG.pt"))
    return dalle, voc


def time_events(fn, iters):
    st = torch.cuda.current_stream()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(st)
    for _ in range(iters):
        fn()
    e.record(st)
    e.synchronize()
    return s.elapsed_time(e) / iters  # ms


def gemm_roofline(eng, B, peaks, peaks_src, traffic):
    """Average device time of the dominant kernel (the tcgen05 GEMM) over the launches of one denoiser pass, CUDA events on the launching
    stream, 19 launches per shape replayed from a CUDA graph (every launch reads a different layer's weights: nothing is L2-warm).
    `achieved` counts ALGORITHMIC flops (2*M*N*K of the fp32 nn.Linear being replaced); in 'f16x3' mode the tensor pipe executes three
    fp16 passes per algorithmic product, reported separately as `tensor_pipe`."""
    L, D = L_TOK, eng.D
    ws = eng.workspace(B, L)
    M = B * L
    split = eng.precision == "f16x3"
    w = 2 if split else 1
    h2, x2 = ws["h"].view(M, w * D), ws["x"].view(M, D)
    lin = eng._linear
    so = dict(split_out=True) if split else {}
    shapes = [("qkv", lambda l: lin(h2, l["wqkv"], l["bqkv"], out=ws["qkv"], **so), 3 * D, D),
              ("proj1", lambda l: lin(ws["att"], l["wo1"], l["bo1"], residual=x2, out=x2), D, D),
              ("q2", lambda l: lin(h2, l["wq2"], l["bq2"], out=ws["q2"], **so), D, D),
              ("proj2", lambda l: lin(ws["att"], l["wo2"], l["bo2"], residual=x2, out=x2), D, D),
              ("mlp1", lambda l: lin(h2, l["w1"], l["b1"], out=ws["hid"], gelu=True, **so), 4 * D, D),
              ("mlp2", lambda l: lin(ws["hid"], l["w2"], l["bm2"], residual=x2, out=x2), D, 4 * D)]
    ws["x"].normal_()
    for k in ("h", "att", "hid"):
        ws[k].normal_(std=0.5)
    per = {}
    tot_ms, tot_flop = 0.0, 0.0
    for name, fn, N, Kd in shapes:
        def run_all():
            for lay in eng.layers:
                fn(lay)
        run_all()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            run_all()
        g.replay()
        torch.cuda.synchronize()
        ms = time_events(g.replay, 5) / len(eng.layers)
        fl = 2.0 * M * N * Kd
        per[name] = {"us": round(ms * 1e3, 2), "tflops": round(fl / (ms * 1e-3) / 1e12, 1)}
        tot_ms += ms
        tot_flop += fl
    n_shapes = len(shapes)
    achieved = tot_flop / (tot_ms * 1e-3) / 1e12
    peak_bf16 = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    peak = peak_bf16 / 2.0 if eng.precision == "tf32" else peak_bf16
    passes = 3 if split else 1
    tr = traffic.get(f"gemm_{eng.precision}_B{B}")
    return {"bound": "tensor", "kernel": ("gemm_f16x3_pair_kernel<256> (fused split-fp16, tcgen05 cta_group::2)" if split else f"gemm_tcgen05_kernel<f16> ({eng.precision})"), "achieved": round(achieved, 1), "peak": round(peak, 1),
            "unit": "TFLOP/s", "frac": round(achieved / peak, 4),
            "tensor_pipe": {"mma_passes_per_product": passes, "executed_tflops": round(achieved * passes, 1), "frac_of_peak": round(achieved * passes / peak, 4),
                            "note": "f16x3 = lo*hi + hi*lo + hi*hi fp16 passes per fp32-equivalent product; executed = algorithmic x passes"},
            "traffic": tr["dram_bytes_per_launch"] if tr else None, "traffic_unit": "bytes/launch",
            "traffic_source": tr.get("source") if tr else "no ncu --set full capture of this build/mode committed (profiles/r2_traffic.json)",
            "algorithmic_bytes_per_launch_avg": round(sum((M * Kd * w * 2 + N * Kd * w * 2 + M * N * 4) for _, _, N, Kd in shapes) / n_shapes),
            "peak_source": f"{peaks_src} MEASURED_PEAKS.json bf16_tflops_sustained={peak_bf16} (cuBLAS bf16 GEMM inside a long loop; kind::f16 fp16 operands issue at the same rate)",
            "per_gemm": per, "flop_per_launch_avg": tot_flop / n_shapes, "us_per_launch_avg": round(tot_ms * 1e3 / n_shapes, 2)}


def stage_times(dalle, voc, cond_dev, B):
    """One extra pass with CUDA events between the three stages."""
    tr = dalle.transformer
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    st = torch.cuda.current_stream()
    torch.cuda.synchronize()
    ev[0].record(st)
    tok = tr.sample(condition_token=None, condition_mask=None, condition_embed=cond_dev, filter_ratio=0, batch_size=B)["content_token"]
    ev[1].record(st)
    mel = dalle.decode_to_img(tok, (B, 256, 5, 53))
    ev[2].record(st)
    voc((mel[:, 0] + 1) / 2)
    ev[3].record(st)
    torch.cuda.synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]


def gpu_parity(dalle, voc, ref, K):
    """Checker: the GPU path on the CPU leg's inputs (same weights, caption embeddings and uniforms).  Token agreement of the free-running
    chain, logits of the first step, mel of the decoder and waveform of the vocoder (both fed the oracle's tensors)."""
    from diffsound_b200 import ops
    tr = dalle.transformer
    eng = tr.transformer.engine
    cond = ref["cond"].cuda()
    B = cond.shape[0]
    kv = eng.encode_condition(cond)
    x = torch.full((B, L_TOK), K, dtype=torch.long, device="cuda")
    mode, r, k = 1, 0.85, 0
    logits_err = None
    for i, ti in enumerate(ref["steps"]):
        t = torch.full((B,), ti, dtype=torch.long, device="cuda")
        logits = eng.forward(x, kv, t, cond.shape[1])
        if i == 0:
            a, b = logits.permute(0, 2, 1).double().cpu(), ref["logits0"].double()
            logits_err = float((a - b).abs().max() / b.abs().max())
        x = ops.posterior_sample(logits, x, t, ref["us"][i].cuda(), tr._sched(), T=100, trunc_mode=mode, trunc_r=r, trunc_k=k)
    tok = x.cpu()
    agree = float((tok == ref["tok"]).float().mean())
    mel = dalle.decode_to_img(ref["tok_dec"].cuda(), (B, 256, 5, 53)).cpu()
    wav = voc(((ref["mel"][:, 0] + 1) / 2).cuda()).cpu()
    rel = lambda a, b: float((a.double() - b.double()).abs().max() / b.double().abs().max())
    return {"checked_against": "oracle port of the reference (CPU fp32), same weights / caption embeddings / uniforms",
            "chain": f"B={B}, {len(ref['steps'])} free-running p_sample steps from all-[MASK]",
            "token_agreement": agree, "tokens_compared": int(tok.numel()), "unmasked_by_oracle": int((ref["tok"] != K).sum()),
            "logits_rel_err_step0": logits_err, "mel_mse": float(((mel - ref["mel"]) ** 2).mean()), "mel_rel_err": rel(mel, ref["mel"]),
            "wav_rel_err": rel(wav, ref["wav"]), "tolerance": "token ids bit-exact; mel / wav 1e-3 relative (north_star)"}


def dump_outputs(directory, out, limit=DUMP_LIMIT_BYTES):
    """What pipeline.synthesize returned -- tokens (B,265), mel (B,1,80,848), wav (B,1,217088) -- as <directory>/<name>.npy in float32 (token
    ids are exact).  Two builds run with the same arguments get the same inputs, so their dumps compare output for output.  A batch larger than
    `limit` bytes is cut to a subset of clips drawn with a fixed seed, the same clips for every build, kept in batch order."""
    import numpy as np
    arrs = {k: v.detach().float().cpu() for k, v in out.items() if v is not None}
    B = arrs["tokens"].shape[0]
    keep = min(B, limit // sum(a[0].numel() * 4 for a in arrs.values()))
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    os.makedirs(directory, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(directory, f"{k}.npy"), a[idx].numpy())


def run_gpu_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: everything else that writes to fd 1 (NCCL's INFO log, library chatter) is routed to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    dist = None
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    B, K = args.batch, args.codebook
    dalle, voc = build_models(K, args.layers, args.precision)
    import _pkg
    _pkg.load()
    from diffsound_b200 import pipeline
    tr = dalle.transformer
    cond_host = synthetic_cond(B, 1 + rank).pin_memory()
    cond_dev = cond_host.to(dev)
    wav_host = torch.empty(B, 1, WAV_LEN, dtype=torch.float32).pin_memory()
    tok_host = torch.empty(B, L_TOK, dtype=torch.int64).pin_memory()
    gathered = torch.empty(world * B, 1, WAV_LEN, dtype=torch.float32, device=dev) if world > 1 else None

    def one_clip_batch(model, e2e: bool):
        c = cond_host.to(dev, non_blocking=True) if e2e else cond_dev
        out = pipeline.synthesize(model, voc, c, sample_type="top0.85r", codec_batch=args.codec_batch)
        if world > 1:
            dist.all_gather_into_tensor(gathered, out["wav"])  # the only collective of the path: gather finished clips (SURVEY.md 8e)
        if e2e:
            wav_host.copy_(out["wav"], non_blocking=True)
            tok_host.copy_(out["tokens"], non_blocking=True)
        return out

    def timed(model, e2e: bool, steps: int):
        """(ms, what the last step returned)"""
        torch.manual_seed(1234 + rank)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        st = torch.cuda.current_stream()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(st)
        for _ in range(steps):
            out = one_clip_batch(model, e2e)
        e.record(st)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    warm = max(args.warmup, 3)
    for _ in range(warm):
        one_clip_batch(dalle, False)
    torch.cuda.synchronize()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms_dev, last = timed(dalle, False, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)  # before the next pass can reuse the engines' buffers
    ms_e2e, _ = timed(dalle, True, args.steps)
    clk = clocks.stop() if rank == 0 else None
    clips = B * world * args.steps
    value, e2e_v = clips / (ms_dev * 1e-3), clips / (ms_e2e * 1e-3)
    launches_per_batch = tr.last_gpu_launches + dalle.content_codec.engine.launches + voc.engine.launches
    st_ms = stage_times(dalle, voc, cond_dev, B)

    # ---- the single-pass fp16 throughput mode on the same workload (shares the codec and the vocoder)
    modes = None
    if args.precision == "f16x3" and not args.no_modes:
        from diffsound_b200.utils import builders
        fast = builders.build_dalle(K=K, NL=args.layers, precision="f16", seed=0)
        fast.content_codec = dalle.content_codec
        for _ in range(2):
            one_clip_batch(fast, False)
        n_fast = max(3, args.steps // 2)
        ms_fast, _ = timed(fast, False, n_fast)
        f_ms = stage_times(fast, voc, cond_dev, B)
        modes = {"f16": {"value": B * world * n_fast / (ms_fast * 1e-3), "unit": "clips/s", "steps": n_fast, "sampler_only_clips_per_s": B / (f_ms[0] * 1e-3),
                         "note": "single-pass fp16 GEMM / attention operands (11-bit significand): logits ~1e-3 of fp32, ~99.6 % free-running token agreement "
                                 "-- NOT parity-grade, reported for reference only"}}
        if rank == 0 and world == 1:
            peaks, src = load_peaks()
            modes["f16"]["roofline"] = gemm_roofline(fast.transformer.transformer.engine, B, peaks, src, load_traffic())
        del fast
        torch.cuda.empty_cache()

    if rank == 0:
        peaks, src = load_peaks()
        traffic = load_traffic()
        roof = gemm_roofline(tr.transformer.engine, B, peaks, src, traffic)
        flops = FLOP_PER_CLIP_STEP.get(K, 158.3e9) * 100 * (args.layers / 19.0)
        roof["pipeline_tflops"] = round(value * (flops + DECODER_FLOP_PER_CLIP + VOCODER_FLOP_PER_CLIP) / 1e12 / world, 1)
        hbm = float(peaks["hbm_gbs"])
        peak_bf16 = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
        stages = {"sampler_100_steps": {"ms": round(st_ms[0], 2), "clips_per_s": round(B / (st_ms[0] * 1e-3), 2),
                                         "algorithmic_tflops": round(B * flops / (st_ms[0] * 1e-3) / 1e12, 1),
                                         "frac_of_bf16_peak": round(B * flops / (st_ms[0] * 1e-3) / 1e12 / peak_bf16, 4)},
                  "decoder": {"ms": round(st_ms[1], 2), "algorithmic_tflops": round(B * DECODER_FLOP_PER_CLIP / (st_ms[1] * 1e-3) / 1e12, 1),
                              "frac_of_bf16_peak": round(B * DECODER_FLOP_PER_CLIP / (st_ms[1] * 1e-3) / 1e12 / peak_bf16, 4),
                              "algorithmic_gbs": round(B * DECODER_BYTES_PER_CLIP / (st_ms[1] * 1e-3) / 1e9, 1),
                              "frac_of_hbm_peak": round(B * DECODER_BYTES_PER_CLIP / (st_ms[1] * 1e-3) / 1e9 / hbm, 4), "launches": dalle.content_codec.engine.launches},
                  "vocoder": {"ms": round(st_ms[2], 2), "bound": "hbm", "algorithmic_gbs": round(B * VOCODER_BYTES_PER_CLIP / (st_ms[2] * 1e-3) / 1e9, 1),
                              "frac_of_hbm_peak": round(B * VOCODER_BYTES_PER_CLIP / (st_ms[2] * 1e-3) / 1e9 / hbm, 4),
                              "algorithmic_tflops": round(B * VOCODER_FLOP_PER_CLIP / (st_ms[2] * 1e-3) / 1e12, 1), "launches": voc.engine.launches}}
        cpu = parity = None
        if not (args.no_cpu_baseline or world > 1):  # the CPU leg is timed at N=1 only; its outputs double as the parity reference
            sd_t = {k: v.detach().float().cpu() for k, v in tr.state_dict().items()}
            sd_c = {k: v.detach().float().cpu() for k, v in dalle.state_dict().items() if k.startswith("content_codec.")}
            sd_v = {k: v.detach().float().cpu() for k, v in voc.state_dict().items()}
            ref = cpu_leg(sd_t, sd_c, sd_v, K=K, n_layer=args.layers, B=2, n_steps=args.cpu_steps)
            cpu = {"value": ref["value"], "unit": "clips/s", "cores": ref["cores"], "kind": "port", "sample": ref["sample"]}
            parity = gpu_parity(dalle, voc, ref, K)
            parity["mode"] = args.precision
        extras = run_extras(args, rank, world, dev, dist, voc) if not args.no_extras else None
        line = {"metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms_dev / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
                "config": {"workload": workload_name(B, K, args.layers),
                           "arithmetic": {"f16x3": "denoiser GEMM / attention operands are fp16 (hi | lo) pairs (22 significand bits), three tcgen05 kind::f16 passes per product, "
                                                   "fp32 TMEM accumulation = fp32-class logits (the reference's nn.Linear is fp32); residual stream / LayerNorm / softmax fp32; "
                                                   "log_softmax fp64; decoder / vocoder convs split-fp16 pairs (3 passes, fp32 accumulation), the decoder AttnBlocks split-TF32",
                                          "f16": "denoiser operands single-pass fp16; decoder / vocoder split-TF32", "tf32": "tf32", "fp32": "FFMA"}[args.precision],
                           "global_batch": B * world, "parallelism": f"dp{world} (independent captions per rank, all_gather of waveforms)",
                           "l2_policy": "working set per diffusion step (3.1 GB of (hi | lo) fp16 weights) exceeds the 126 MB L2; no explicit flush"},
                "e2e": {"value": e2e_v, "unit": "clips/s", "h2d_bytes_per_step": cond_host.numel() * 4, "d2h_bytes_per_step": wav_host.numel() * 4 + tok_host.numel() * 8,
                        "api": "pipeline.synthesize(DALLE, Generator, <pinned host caption embeddings -> device>) -> waveforms + token grids copied to pinned host"},
                "gpu_launches": launches_per_batch * args.steps, "gpu_launches_per_step": launches_per_batch,
                "stages": stages, "roofline": roof, "cpu_baseline": cpu, "parity": parity, "modes": modes, "clocks": clk, "extras": extras}
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
    elif not args.no_extras:
        run_extras(args, rank, world, dev, dist, voc)
    if world > 1:
        print(f"[bench] NCCL process group: nranks={dist.get_world_size()} backend={dist.get_backend()}", file=sys.stderr)
        dist.destroy_process_group()


def run_extras(args, rank, world, dev, dist, voc):
    """Driver-visible numbers for the other BASELINE configs, measured in the same run (one timed pass each, after a short warm-up):
    configs[2]: B=64 per GPU text->wav;  configs[4]: B=512 TOTAL, K=512 codebook, sharded 512/N per rank (strong scaling), waveforms all-gathered."""
    import _pkg
    _pkg.load()
    from diffsound_b200 import pipeline
    from diffsound_b200.utils import builders
    out = {}

    def one(tag, K, B_local, total, note):
        model = builders.build_dalle(K=K, NL=args.layers, precision=args.precision, seed=0)
        cond = synthetic_cond(B_local, 100 + rank).to(dev)
        gathered = torch.empty(world * B_local, 1, WAV_LEN, dtype=torch.float32, device=dev) if world > 1 else None

        mid = torch.cuda.Event(enable_timing=True)

        def go(sample_type):
            o = pipeline.synthesize(model, voc, cond, sample_type=sample_type, codec_batch=args.codec_batch)
            mid.record(torch.cuda.current_stream())
            if world > 1:
                dist.all_gather_into_tensor(gathered, o["wav"])
        go("top0.85r,fast24")  # warm-up: 5 denoiser calls (graph capture, workspaces, NCCL buffers)
        torch.manual_seed(4321 + rank)
        clk = ClockSampler(dev.index) if rank == 0 else None
        if clk is not None:
            clk.start()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        st = torch.cuda.current_stream()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(st)
        go("top0.85r")
        e.record(st)
        torch.cuda.synchronize()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        ms_gather = round(mid.elapsed_time(e), 2)  # this rank: end of its own synthesis -> gather complete (includes waiting for slower ranks)
        per_rank = [round(float(ms.item()), 1)]
        if world > 1:
            allms = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(allms, ms)
            per_rank = [round(float(v.item()), 1) for v in allms]
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        out[tag] = {"clips_per_s": total / (float(ms.item()) * 1e-3), "ms": round(float(ms.item()), 1), "ms_per_rank": per_rank, "ms_gather_rank0": ms_gather, "clips_total": total,
                    "clips_per_gpu": B_local, "K": K, "n_gpus": world, "timed_passes": 1, "note": note,
                    "clocks": clk.stop() if clk is not None else None}
        del model
        torch.cuda.empty_cache()

    sel = set(args.extras.split(","))
    if "train" in sel:
        out["configs3_train_ddp"] = train_extra(args, rank, world, dev, dist)
    if "configs2" in sel:
        one("configs2_b64_text_to_wav", 256, 64, 64 * world, "BASELINE.json configs[2]: batch 64 per GPU, full pipeline (weak scaling over ranks)")
    if "configs4" in sel and 512 % world == 0:
        one("configs4_b512_k512_sharded", 512, 512 // world, 512, "BASELINE.json configs[4]: 512 clips TOTAL sharded over the ranks (strong scaling), K=512 codebook, "
            "full pipeline, NCCL all_gather of the waveforms inside the timed pass")
    return out


def train_extra(args, rank, world, dev, dist, per_gpu_batch=20, warm=3, steps=8):
    """BASELINE.json configs[3]: diffusion-transformer training step on synthetic tokens, bf16 GEMM operands, per-GPU batch 20 (configs/audioset.yaml:140),
    stock torch DistributedDataParallel over NCCL when N > 1 (the reference's own wrapper, engine/solver_spec.py:109) + fused AdamW; whole-job samples/s."""
    import _pkg
    _pkg.load()
    from diffsound_b200.utils import builders
    K, L = 256, L_TOK
    torch.manual_seed(0)
    m = builders.build_diffusion_transformer(K, 1024, args.layers, 16, 512).train()
    for p in m.parameters():
        p.requires_grad_(True)
    g = torch.Generator().manual_seed(100 + rank)
    batch = {"content_token": torch.randint(0, K, (per_gpu_batch, L), generator=g).to(dev),
             "condition_embed_token": torch.nn.functional.normalize(torch.randn(per_gpu_batch, 77, 512, generator=g), dim=-1).to(dev)}
    net = torch.nn.parallel.DistributedDataParallel(m, device_ids=[dev.index]) if world > 1 else m
    opt = torch.optim.AdamW(m.parameters(name="transformer"), lr=3e-6, betas=(0.9, 0.96), fused=True)

    def step():
        out = net(batch, return_loss=True, return_logits=False)
        opt.zero_grad(set_to_none=True)
        out["loss"].backward()
        opt.step()
        return out["loss"]
    for _ in range(warm):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    st = torch.cuda.current_stream()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(st)
    for _ in range(steps):
        loss = step()
    e.record(st)
    torch.cuda.synchronize()
    ms = torch.tensor([s.elapsed_time(e)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms.item()) / steps
    res = {"samples_per_s": world * per_gpu_batch / ms_step * 1e3, "ms_per_step": round(ms_step, 2), "per_gpu_batch": per_gpu_batch, "n_gpus": world,
           "steps": steps, "loss": float(loss.detach()), "dtype": "bf16 GEMM operands, fp32 master weights / residual stream / loss",
           "algorithmic_tflops": round(3 * 158.25e9 * per_gpu_batch * (args.layers / 19.0) / (ms_step * 1e-3) / 1e12, 1),
           "note": "BASELINE.json configs[3]: forward + fused loss + hand-written backward + AdamW" + (", torch DDP bucketed gradient all-reduce overlapped with the "
                   "remaining backward segments (one autograd node per layer)" if world > 1 else "")}
    del net, m, opt
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=16, help="clips per GPU per step (BASELINE configs[1]: 16)")
    ap.add_argument("--codebook", type=int, default=256)
    ap.add_argument("--layers", type=int, default=19)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="f16x3", choices=["f16x3", "f16", "tf32", "fp32"])
    ap.add_argument("--codec-batch", type=int, default=32, help="clips per SpecVQGAN-decoder / MelGAN sub-batch (bounds activation memory)")
    ap.add_argument("--cpu-steps", type=int, default=20, help="p_sample steps of the CPU leg's bounded sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-modes", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--extras", default="train,configs2,configs4", help="which of the other BASELINE configs to measure in the same run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's tokens / mel / wav of the last timed step to DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU arm)")
        run_gpu_arm(args)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- headline benchmark: audio-seconds/second of Conformer-CTC training on synthetic
LibriSpeech-shape 16 kHz waveforms (BASELINE.json configs[2]: Conformer encoder 17 x 512, conv-k31, CTC, bf16,
on-the-fly fbank + SpecAugment, data parallel with one gradient all-reduce).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference ...                      CPU arm: the oracle port of the reference path on host cores

One "step" = one full update: front end -> conv front -> 17 Conformer layers -> fc_out -> CTC -> backward ->
gradient all-reduce -> clip + Adam.  `value` times K steps with the step's waveforms already in HBM; `e2e`
times the same K steps from pinned HOST buffers (H2D copy of every step's inputs inside the timed region)
and reads the step's loss back (D2H).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

V = 5004  # 5000 sentencepiece units + <s>(blank) <pad> </s> <unk>   (SURVEY.md §8, run_torchaudio.sh:25)
MAX_TOKENS, MAX_SENTENCES = 26000, 24  # frames / sentences per GPU batch (conformer_librispeech.yaml:29-30)
MODEL = dict(embed_dim=512, ffn_embed_dim=2048, layers=17, attention_heads=8, normalize_before=True, learned_pos=False,
             relative_positional_embeddings=True, layer_type="conformer", depthwise_conv_kernel_size=31)
SPECAUG = {"time_warp_W": 0, "freq_mask_F": 27, "freq_mask_N": 2, "time_mask_pm": 0.04, "time_mask_ps": 0.04}


def synth_wave(rs, n):
    """noise + sine in int16 range (SURVEY.md §8d), float32."""
    t = np.arange(n, dtype=np.float32) / 16000.0
    x = np.round(3000.0 * rs.standard_normal(n).astype(np.float32) + 1500.0 * np.sin(2 * np.pi * rs.uniform(80, 400) * t))
    return np.clip(x, -32767, 32767).astype(np.float32)


def make_batches(n_batches, seed=7, pool=4000):
    """LibriSpeech-shape durations Gamma(6.1, 2.0) clipped to [1, 35] s, sorted by length, packed under
    max_tokens/max_sentences (fairseq batch_by_size), batch order shuffled with a fixed seed.

    EVERY rank gets the SAME list (same shapes, same order) at every world size: per-GPU work per step is then
    identical for N = 1, 2, 4, 8, so the driver's scaling efficiency isolates the gradient collective instead of
    mixing in batch composition (round-1 VERDICT).  Length-bucket straggling between ranks is therefore not in the
    number; the reference bounds it with grouped shuffling (fairseq/data/iterators.py:537-545)."""
    from espresso_b200.data import batching, specaugment as SA

    rs = np.random.RandomState(seed)
    durs = np.clip(rs.gamma(6.1, 2.0, size=pool), 1.0, 35.0)
    n_samples = np.round(durs * 16000).astype(np.int64)
    frames = 1 + (n_samples - 400) // 160
    order = batching.ordered_indices(frames)
    batches = batching.batch_by_size(order, frames, MAX_TOKENS, MAX_SENTENCES)
    batches = [b for b in batches if frames[b].sum() >= 0.8 * MAX_TOKENS or len(b) == MAX_SENTENCES]  # drop the ragged tail
    np.random.RandomState(seed + 1).shuffle(batches)
    cfg = SA.AdaptiveSpecAugmentConfig.from_config_dict(SPECAUG)
    out = []
    for gi in range(n_batches):
        idx = batches[gi % len(batches)]
        idx = idx[np.argsort(-frames[idx], kind="mergesort")]  # collate: sort by length descending (asr_dataset.py:60-70)
        B = len(idx)
        n = n_samples[idx]
        wave = np.zeros((B, int(n.max())), dtype=np.float32)
        fms, tms, tgts = [], [], []
        for b, i in enumerate(idx):
            wrs = np.random.RandomState(1000 + int(i))
            wave[b, : n[b]] = synth_wave(wrs, int(n[b]))
            with SA.numpy_seed(1, 1, int(i)):
                fm, tm = SA.draw_masks(cfg, int(frames[i]), 80)
            fms.append(fm)
            tms.append(tm)
            u = max(1, int(round(4.0 * durs[i])))
            tgts.append(np.random.RandomState(11 + int(i)).randint(4, V, size=u))
        fmp, tmp = SA.pack_masks(fms, tms)
        U = max(len(t) for t in tgts) + 1
        target = np.full((B, U), 1, dtype=np.int64)
        for b, t in enumerate(tgts):
            target[b, : len(t)] = t
            target[b, len(t)] = 2
        out.append(dict(wave=wave, n_samples=n.astype(np.int32), fm=fmp, tm=tmp, target=target,
                        audio_s=float(n.sum() / 16000.0), ntokens=int(sum(len(t) for t in tgts)),
                        frames=frames[idx].astype(np.int64)))
    return out


def useful_gemm_flops(frames, d=512, ffn=2048, layers=17, in_dim=2560):
    """Flops of one update that land on REAL (unpadded) frames, split by where they execute (SURVEY.md section 8d accounting;
    the conv front and the depthwise conv are left out).  `frames`: input frames per utterance.  Returns (gemm, attn_fwd,
    attn_bwd):
      gemm      what the tcgen05 GEMM launches execute -- per encoder frame and layer: FFN 2 x (2 x 2 d ffn), q/k/v/out 8 d^2,
                point-wise convs 6 d^2 (x3: forward, dgrad, wgrad); pos_proj 2 d^2 (2 T'max - 1) per layer (x2: no dgrad);
                fc0 and fc_out per frame (x3); and the attention-backward products that are still plain GEMMs:
                dq_u = dS k (2 d T'^2), dq_v = dBD pos and dpos = dBD^T q_v (2 d T'(2T'-1) each) per utterance and layer;
      attn_fwd  the fused attention forward kernel: scores 2 d T'^2, position logits 2 d T'(2T'-1), P v 2 d T'^2;
      attn_bwd  the fused attention backward kernel: dPd, dV, dK, 2 d T'^2 each."""
    tp = -(-(-(-np.asarray(frames, dtype=np.float64) // 2)) // 2)   # T' = ceil(ceil(T/2)/2)
    per_frame = layers * (8.0 * d * ffn + 14.0 * d * d) + 2.0 * in_dim * d + 2.0 * d * V
    pos = layers * 2.0 * d * d * (2.0 * tp.max() - 1.0)
    attn_fwd = layers * 2.0 * d * (4.0 * tp * tp - tp)
    attn_bwd_fused = layers * 2.0 * d * (3.0 * tp * tp)
    attn_bwd_gemm = layers * 2.0 * d * (tp * tp + 2.0 * tp * (2.0 * tp - 1.0))
    return 3.0 * per_frame * tp.sum() + 2.0 * pos + attn_bwd_gemm.sum(), attn_fwd.sum(), attn_bwd_fused.sum()


def effective_cores():
    """CPU cores this process may really use: affinity mask and cgroup quota, not just os.cpu_count()."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = max(1, min(n, int(float(q[0]) / float(q[1]))))
    except Exception:
        pass
    return n


class _Dict:
    def __len__(self):
        return V

    def pad(self):
        return 1

    def eos(self):
        return 2

    def unk(self):
        return 3

    def index(self, s):
        return 0


class _Task:
    feat_dim, feat_in_channels, target_dictionary = 80, 1, _Dict()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 6 and r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


ORACLE_CFG = dict(embed_dim=512, ffn_dim=2048, heads=8, layers=17, layer_type="conformer", dw_kernel=31, dropout=0.1,
                  attention_dropout=0.1, activation_dropout=0.1, layernorm_embedding=True, final_layer_norm=False, vocab=V)
CPU_SAMPLE_DURS = (10.0, 10.0, 10.0, 10.0)   # BASELINE.md section 4.2: a reduced batch of 4 x 10 s for the CPU leg


class OracleStep:
    """One full update of the reference's path as restated by the oracle (oracle/conformer.py: functional PyTorch keyed
    by the reference's parameter names, pinned bit-exactly against the real reference model): fwd + CTC + bwd + 1/B
    normalisation + clip 2.0 + Adam.  Used by the two BASELINE legs only (CPU fp32; GPU eager bf16) -- never by the
    product path.  bf16 mode follows fairseq --bf16 (fairseq/trainer.py:105-107, fairseq/optim/fp16_optimizer.py:
    109-168): bf16 parameters and gradients, fp32 master copy updated by Adam, copied back."""

    def __init__(self, device, bf16):
        from oracle import conformer as OC

        self.OC, self.dev, self.bf16 = OC, device, bf16
        dt = torch.bfloat16 if bf16 else torch.float32
        sd = OC.random_state_dict(ORACLE_CFG, seed=1)
        self.sd = {k: v.to(device=device, dtype=dt) for k, v in sd.items()}  # model.bfloat16() casts the BN buffers too
        self.params = [v.requires_grad_(True) for k, v in self.sd.items() if "running_" not in k]
        self.master = [p.detach().float().clone() for p in self.params] if bf16 else self.params
        self.opt = torch.optim.Adam(self.master, lr=1e-4, betas=(0.9, 0.98), eps=1e-8)
        if device.type == "cuda":  # the reference caches its sinusoidal table on the device; give the oracle the same
            cache, orig = {}, OC.rel_pos_table

            def cached(T, d, dtype=torch.float32):
                k = (T, d, dtype)
                if k not in cache:
                    cache[k] = orig(T, d, dtype).to(device)
                return cache[k]

            OC.rel_pos_table = cached

    def __call__(self, feats, lens, target):
        OC = self.OC
        for p in self.params:
            p.grad = None
        logits, ol, _ = OC.encoder_forward(self.sd, ORACLE_CFG, feats, lens, training=True)
        with torch.backends.cudnn.flags(enabled=False):  # espresso/criterions/ctc_loss.py:85-94
            loss = OC.ctc_criterion(logits, ol, target, 1, 2, 0)
        loss.backward()
        if self.bf16:
            for m, p in zip(self.master, self.params):
                m.grad = p.grad.float()
        torch._foreach_mul_([m.grad for m in self.master], 1.0 / feats.shape[0])   # sentence_avg: sample_size = B
        torch.nn.utils.clip_grad_norm_(self.master, 2.0)
        self.opt.step()
        if self.bf16:
            torch._foreach_copy_([p.data for p in self.params], self.master)
        return loss.detach()


def cpu_sample(it=0):
    """The bounded CPU sample: 4 x 10 s utterances through the oracle's numpy front end (Kaldi fbank + CMVN + adaptive
    SpecAugment), collated like the reference."""
    from oracle import frontend as OF

    feats = []
    for i, d in enumerate(CPU_SAMPLE_DURS):
        x = OF.global_cmvn(OF.kaldi_fbank(OF.synth_waveform(i, d)), np.full(80, 15.0), np.full(80, 4.0))
        with OF.numpy_seed(1, it, i):
            x = OF.adaptive_specaugment(x)
        feats.append(torch.from_numpy(x).float())
    T = max(f.shape[0] for f in feats)
    batch = torch.zeros(len(feats), T, 80)
    for b, f_ in enumerate(feats):
        batch[b, : f_.shape[0]] = f_
    lens = torch.tensor([f_.shape[0] for f_ in feats])
    tgt = torch.full((len(feats), 41), 1, dtype=torch.long)
    g = torch.Generator().manual_seed(it)
    tgt[:, :40] = torch.randint(4, V, (len(feats), 40), generator=g)
    tgt[:, 40] = 2
    return batch, lens, tgt


def cpu_sample_label(cores):
    return ("%d x %.0f s utterances per step (a bounded sample of the 24-utterance / 26000-frame batch): numpy fbank + CMVN "
            "+ SpecAugment, fp32 fwd + CTC + bwd + clip + Adam, %d torch threads" % (len(CPU_SAMPLE_DURS), CPU_SAMPLE_DURS[0], cores))


def run_reference(args):
    """CPU arm: the oracle port of the reference path on the host cores; one bounded sample (4 x 10 s) per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(effective_cores(), 32)  # per-op work is small: more threads only add synchronisation cost
    torch.set_num_threads(cores)
    stepper = OracleStep(torch.device("cpu"), bf16=False)
    audio_s = float(sum(CPU_SAMPLE_DURS))
    for i in range(args.warmup):
        stepper(*cpu_sample(i))
    t0 = time.perf_counter()
    for i in range(args.steps):
        stepper(*cpu_sample(args.warmup + i))
    dt = time.perf_counter() - t0
    val = audio_s * args.steps / dt
    cfg = workload_config(args.gpus)
    cfg["sample"] = cpu_sample_label(cores)
    print(json.dumps({
        "impl": "reference", "metric": "training throughput (audio-seconds/second)", "value": val, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": cfg["sample"]},
        "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def gpu_eager_baseline(dev, host_batches, steps=6, warmup=2):
    """The number to beat (BASELINE.md section 4.4): the reference's PyTorch-eager bf16 path on THIS B200 -- the oracle
    restatement of the reference model (bit-exact to it on CPU) run with cuda tensors under fairseq --bf16 semantics, on
    the SAME batches as the product arm.  The baseline is given every advantage the product does not get: features are
    already on the device (the reference's CPU DataLoader front end and its H2D copy are NOT timed) and nothing is
    read back."""
    stepper = OracleStep(dev, bf16=True)
    data = []
    for b in host_batches[: max(1, min(len(host_batches), steps))]:
        fr = torch.from_numpy(b["frames"])
        T = int(fr.max())
        g = torch.Generator().manual_seed(int(fr.sum()))
        feats = torch.randn(len(fr), T, 80, generator=g)
        feats = feats * (torch.arange(T)[None, :] < fr[:, None])[:, :, None]
        data.append((feats.to(dev).bfloat16(), fr.to(dev), torch.from_numpy(b["target"]).to(dev), b["audio_s"]))
    for i in range(warmup):
        stepper(*data[i % len(data)][:3])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    audio = 0.0
    e0.record()
    for i in range(steps):
        d = data[i % len(data)]
        loss = stepper(*d[:3])
        audio += d[3]
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    assert bool(torch.isfinite(loss)), "eager baseline diverged"
    mem = torch.cuda.max_memory_allocated() / 2 ** 30
    return {"value": audio / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms / steps, "steps": steps, "dtype": "bf16",
            "kind": "port of the reference model (oracle/conformer.py, pinned bit-exact to it) as eager PyTorch on cuda, "
                    "fairseq --bf16 optimizer semantics; features resident on the device (front end and H2D not timed)",
            "peak_mem_gib": mem}


def run_reference_gpu(args):
    """`--impl reference-gpu`: only the eager-PyTorch baseline leg, same batches as the product arm (1 GPU)."""
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if int(os.environ.get("RANK", "0")) != 0:
        return
    res = gpu_eager_baseline(dev, make_batches(min(8, args.steps)), steps=args.steps, warmup=args.warmup)
    print(json.dumps({"impl": "reference-gpu", "metric": "training throughput (audio-seconds/second)", "value": res["value"],
                      "unit": "audio-s/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": res["ms_per_step"], "higher_is_better": True, "dtype": "bf16", "data": "synthetic",
                      "config": workload_config(1), "gpu_eager_baseline": res}))


def decode_rtf(dev, n_utts=1000, per_batch=50, seconds=10.0):
    """Second half of the headline metric (BASELINE.json configs[4]): batched beam-5 decoding with Transformer-LM
    shallow fusion, 1000 synthetic 10 s utterances from raw waveforms, through espresso_b200.SequenceGenerator
    (the reference's speech_recognize.py path: fairseq/sequence_generator.py:212-621).  RTF = decode seconds / audio
    seconds, timed with CUDA events around generate() calls (host bookkeeping and the final D2H included); decode
    settings of examples/asr_librispeech/run_torchaudio.sh:180-198 (lm-weight 0.47, eos-factor 1.5, max-len-a 0.08)."""
    from espresso_b200.data.frontend import OnTheFlyFbank
    from espresso_b200.models import SpeechTransformerConfig, SpeechTransformerModelBase
    from espresso_b200.models.transformer_lm import TransformerLanguageModel
    from espresso_b200.sequence_generator import SequenceGenerator

    torch.manual_seed(5)
    cfg = SpeechTransformerConfig.from_dict(dict(
        dropout=0.0, attention_dropout=0.0, activation_dropout=0.0, layernorm_embedding=False, max_target_positions=1024,
        encoder=dict(embed_dim=256, ffn_embed_dim=1024, layers=12, attention_heads=4, normalize_before=True,
                     learned_pos=False, relative_positional_embeddings=True, layer_type="transformer"),
        decoder=dict(embed_dim=256, ffn_embed_dim=1024, layers=6, attention_heads=4, normalize_before=True,
                     learned_pos=False, relative_positional_embeddings=False, input_dim=256, output_dim=256)))
    model = SpeechTransformerModelBase.build_model(cfg, _Task()).finalize_(dev)
    model.frontend = OnTheFlyFbank(np.full(80, 15.0), np.full(80, 4.0))
    model.eval()
    lm = TransformerLanguageModel(_Dict(), embed_dim=512, ffn_embed_dim=2048, layers=6, attention_heads=8,
                                  max_target_positions=1024).finalize_(dev)
    gen = SequenceGenerator([model], _Dict(), beam_size=5, max_len_a=0.08, max_len_b=0, lm_model=lm, lm_weight=0.47,
                            eos_factor=1.5)
    n = int(seconds * 16000)
    rs = np.random.RandomState(3)
    waves = [torch.from_numpy(np.stack([synth_wave(rs, n) for _ in range(per_batch)]).astype(np.float32)).pin_memory()
             for _ in range(2)]
    lens_h = torch.full((per_batch,), n, dtype=torch.int32)

    def one(i):
        w = waves[i % 2].to(dev, non_blocking=True)
        sample = {"net_input": {"src_tokens": w, "src_lengths": lens_h.to(dev, non_blocking=True),
                                "src_lengths_cpu": lens_h.long()}}
        return gen.generate([model], sample)

    for i in range(2):  # warm-up
        hyp = one(i)
    torch.cuda.synchronize()
    n_batches = max(1, n_utts // per_batch)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ntok = 0
    e0.record()
    for i in range(n_batches):
        hyp = one(i)
        ntok += sum(len(h[0]["tokens"]) for h in hyp)
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) * 1e-3
    audio = n_batches * per_batch * seconds
    # HBM roofline of the per-step search kernels at this leg's shape (bsz*beam = 250 rows, V = 5004): 16 rotating
    # operand sets (160 MB together, beyond the 126 MB L2)
    from espresso_b200 import ops
    N_, beam_ = per_batch * 5, 5
    Vp = (V + 7) // 8 * 8
    sets = [(torch.randn(N_, Vp, device=dev).bfloat16(), torch.randn(N_, Vp, device=dev).bfloat16(),
             torch.empty(N_, V, device=dev, dtype=torch.float32), torch.randn(N_, device=dev)) for _ in range(16)]

    def search_step(x, lm_, cand, prev):
        ops.beam_merge(x, V, True, cand, prev_scores=prev, lm=lm_, lm_is_logits=True, lm_weight=0.47, eos_factor=1.5)
        ops.beam_topk(cand, per_batch, beam_ * V, beam_ * V, 2 * beam_, V)

    for st_ in sets:
        search_step(*st_)
    torch.cuda.synchronize()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(int(1e8))
    b0.record()
    for _ in range(4):
        for st_ in sets:
            search_step(*st_)
    b1.record()
    torch.cuda.synchronize()
    us_beam = b0.elapsed_time(b1) * 1e3 / (4 * len(sets))
    nb = N_ * V * (2 + 2 + 4 + 4)  # model + LM logits read (bf16), candidates written and read once (fp32)
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        hbm_peak = 6575.8
    beam_roof = {"kernel": "beam_merge + beam_topk (one search step)", "bound": "hbm", "us_per_launch": us_beam,
                 "achieved": nb / us_beam / 1e3, "peak": hbm_peak, "unit": "GB/s", "frac": nb / us_beam / 1e3 / hbm_peak,
                 "algorithmic_bytes_per_launch": nb, "per_unit": "12 V B per hypothesis and step",
                 "shape": "bsz*beam=%d V=%d" % (N_, V), "note": "two launches; latency-bound at this size, judged on RTF"}
    del sets
    cpu_ref = None
    try:
        cpu_ref = cpu_decode_reference(model, lm, waves[0][:2].numpy(), one(0)[:2], seconds)
    except Exception as ex:  # the comparison leg must never cost the main line
        cpu_ref = {"error": repr(ex)[:300]}
    return {"cpu_reference": cpu_ref, "roofline_hbm": [beam_roof], "metric": "beam-5 decode real-time factor (decode seconds / audio second)", "rtf": sec / audio,
            "audio_s_per_s": audio / sec, "utterances": n_batches * per_batch, "utterance_s": seconds, "batch": per_batch,
            "beam": 5, "lm_weight": 0.47, "eos_factor": 1.5, "max_len_a": 0.08, "ms_per_batch": 1e3 * sec / n_batches,
            "best_hyp_tokens_per_utt": ntok / (n_batches * per_batch),
            "model": "SpeechTransformerModel 12-enc/6-dec d=256 (rel-pos encoder) + Transformer LM 6x512 shallow fusion, "
                     "V=%d, random init, raw 16 kHz waveforms in pinned host memory" % V}


def cpu_decode_reference(model, lm, waves, gpu_hyps, seconds):
    """CPU leg of the decode metric: the reference's search as restated by the oracle (oracle/frontend.py numpy Kaldi fbank,
    oracle/conformer.py encoder, oracle/decoder.py decoder and LM recomputed per step, oracle/beam.py = fairseq
    SequenceGenerator incl. eos_factor and LM shallow fusion; fp32, the product model's weights) on a bounded sample of
    the same workload: the first utterances of the first batch, one at a time.  Returns its RTF and how far the GPU
    hypotheses (bf16) follow the fp32 ones: with RANDOM-INIT weights the top-2 logit margin is of the order of the bf16
    logit error (~6 % of the steps are near-ties), so a token-identical 80-step search is not expected here -- token
    bit-exactness is tested where it is well defined, on identical log-probs (tests/test_beam_search.py,
    tests/test_gpu_beam.py: 69 reference hypotheses reproduced exactly)."""
    import torch.nn.functional as F

    from oracle import beam as OB
    from oracle import conformer as OC
    from oracle import decoder as OD
    from oracle import frontend as OF

    cores = min(effective_cores(), 32)
    torch.set_num_threads(cores)
    sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
    sd_lm = {k: v.detach().float().cpu() for k, v in lm.state_dict().items()}
    ecfg = dict(embed_dim=256, ffn_dim=1024, heads=4, layers=12, layer_type="transformer", dropout=0.0, attention_dropout=0.0,
                activation_dropout=0.0, layernorm_embedding=False, final_layer_norm=True, vocab=None)
    dcfg = dict(dec_embed_dim=256, dec_heads=4, dec_layers=6, pad=1, dropout=0.0, attention_dropout=0.0, activation_dropout=0.0,
                dec_layernorm_embedding=False, share_decoder_input_output_embed="decoder.output_projection.weight" not in sd)
    lcfg = dict(dec_embed_dim=512, dec_heads=8, dec_layers=6, pad=1, dropout=0.0, attention_dropout=0.0, activation_dropout=0.0,
                dec_layernorm_embedding=False, share_decoder_input_output_embed="decoder.output_projection.weight" not in sd_lm)
    t0 = time.perf_counter()
    hyps = []
    with torch.no_grad():
        for w in waves:
            x = OF.global_cmvn(OF.kaldi_fbank(w), np.full(80, 15.0), np.full(80, 4.0))
            feats = torch.from_numpy(x).float()[None]
            enc, ol, pad = OC.encoder_forward(sd, ecfg, feats, torch.tensor([feats.shape[1]]), training=False)

            def lprobs_fn(step, toks, reorder_state):
                rows = toks.shape[0]
                lg = OD.decoder_forward(sd, dcfg, toks, enc.expand(rows, -1, -1), None)[:, -1]
                ll = OD.decoder_forward(sd_lm, lcfg, toks, None, None)[:, -1]
                return F.log_softmax(lg.float(), -1) + 0.47 * F.log_softmax(ll.float(), -1)

            hyps.append(OB.generate(lprobs_fn, 1, feats.shape[1], V, 1, 3, 2, beam_size=5, max_len_a=0.08, max_len_b=0,
                                    model_max_len=1024, eos_factor=1.5)[0])
    dt = time.perf_counter() - t0
    same, frac = 0, []
    for h_cpu, h_gpu in zip(hyps, gpu_hyps):
        a, b = h_cpu[0]["tokens"].tolist(), h_gpu[0]["tokens"].tolist()
        n = 0
        while n < min(len(a), len(b)) and a[n] == b[n]:
            n += 1
        same += int(a == b)
        frac.append(n / max(len(a), 1))
    return {"rtf": dt / (len(waves) * seconds), "utterances": len(waves), "cores": cores, "kind": "port",
            "sample": "%d x %.0f s utterances, beam 5 + LM fusion, fp32, decoder and LM recomputed per step" % (len(waves), seconds),
            "best_hypothesis_identical_to_gpu": same, "mean_common_prefix_fraction": float(np.mean(frac)),
            "note": "random-init weights: top-2 margins are of the order of the bf16 logit error, see cpu_decode_reference.__doc__"}


DUMP_SAMPLE = 1 << 20  # entries drawn from each parameter-sized buffer for --dump-outputs (4 MB each in float32)


def step_outputs(trainer):
    """What the last update handed its caller, copied on the device: the stats row [sample_size, ntokens, nsentences,
    loss], the gradient norm, and the same fixed, seeded sample of the updated fp32 master weights, the gradients and
    Adam's two moments (the full buffers are ~0.4 GB each).  Two runs of the same build agree to rounding, not bit for
    bit: with --steps 20 --warmup 5 on a B200 (1000 W limit) they differed by 3e-5 (weights) and 1e-3 (gradients) in
    relative Frobenius norm, so compare builds with a tolerance."""
    flat = trainer.flat
    idx = np.unique(np.random.RandomState(0).randint(0, flat.numel, size=DUMP_SAMPLE))
    idx = torch.from_numpy(idx).to(flat.p32.device)
    out = {"stats": trainer.last_stats[:4], "grad_norm": trainer._gnorm, "sample_index": idx}
    for name, t in (("params", flat.p32), ("grads", flat.grads), ("adam_m", flat.m), ("adam_v", flat.v)):
        out[name + "_sample"] = t.index_select(0, idx)
    return {k: v.detach().clone() for k, v in out.items()}


def dump_outputs(outputs, out_dir):
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().double().numpy() if name == "sample_index" else t.float().cpu().numpy())


def workload_config(n):
    return {"workload": "Conformer encoder 17x512 (ffn 2048, 8 heads, conv-k31, sinusoidal rel-pos) + CTC, V=5004, on-the-fly "
                        "fbank80+CMVN+adaptive SpecAugment from raw 16 kHz waveforms, Adam + clip 2.0, dropout 0.1",
            "max_tokens": MAX_TOKENS, "batch_size": MAX_SENTENCES, "length_distribution": "Gamma(6.1,2.0) s clipped [1,35]",
            "parallelism": "dp%d" % n, "l2": "per-step working set (activations+weights > 1 GB) exceeds the 126 MB L2",
            "per_rank_batches": "the same list of distinct LibriSpeech-shape batches on every rank at every N (per-GPU work is "
                                "identical across N; length-bucket straggling between ranks is not measured)"}


def cpu_baseline_quick(budget_s=14.0):
    """Oracle (port) timed on the host cores on the bounded sample: full updates of the same model on 4 x 10 s."""
    cores = min(effective_cores(), 32)
    torch.set_num_threads(cores)
    stepper = OracleStep(torch.device("cpu"), bf16=False)
    stepper(*cpu_sample(0))  # warm-up (allocator, thread pool)
    t0 = time.perf_counter()
    reps = 0
    while time.perf_counter() - t0 < budget_s or reps < 2:
        stepper(*cpu_sample(1 + reps))
        reps += 1
    dt = time.perf_counter() - t0
    return {"value": float(sum(CPU_SAMPLE_DURS)) * reps / dt, "unit": "audio-s/s", "cores": cores, "kind": "port",
            "sample": "%d steps of: %s" % (reps, cpu_sample_label(cores))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--layers", type=int, default=None, help="debug only: override layer count (invalidates the number)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager", action="store_true", help="disable CUDA-graph capture of the step")
    ap.add_argument("--no-decode", action="store_true", help="skip the beam-5 decode RTF leg")
    ap.add_argument("--decode-only", action="store_true", help="run only the beam-5 decode RTF leg (debugging)")
    ap.add_argument("--distinct", type=int, default=48, help="distinct batches (shapes) cycled through")
    ap.add_argument("--sustain", type=int, default=200, help="extra timed steps after the K-step measurement (clocks settle)")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the eager-PyTorch bf16 baseline leg")
    ap.add_argument("--no-hbm-roofline", action="store_true", help="skip the per-kernel HBM roofline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the K timed steps, write what the last of them computed to DIR/<name>.npy (a fixed, seeded "
                         "sample of the parameter-sized buffers) so that two builds can be compared")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "reference-gpu":
        return run_reference_gpu(args)

    import torch.distributed as dist

    from espresso_b200 import lib, ops
    from espresso_b200.criterions import CtcLossCriterion
    from espresso_b200.data.frontend import OnTheFlyFbank
    from espresso_b200.models import SpeechTransformerConfig, SpeechTransformerEncoderModel
    from espresso_b200.optim import NoamLRScheduler
    from espresso_b200.trainer import Trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, "--gpus must equal WORLD_SIZE (launch N > 1 under torchrun)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib.load()

    if args.decode_only:
        print(json.dumps({"decode": decode_rtf(dev)}))
        return
    torch.manual_seed(1)
    enc = dict(MODEL)
    if args.layers is not None:
        enc["layers"] = args.layers
    cfg = SpeechTransformerConfig.from_dict(dict(dropout=0.1, attention_dropout=0.1, activation_dropout=0.1,
                                                 layernorm_embedding=True, encoder=enc))
    model = SpeechTransformerEncoderModel.build_model(cfg, _Task()).finalize_(dev)
    model.frontend = OnTheFlyFbank(np.full(80, 15.0), np.full(80, 4.0))
    trainer = Trainer(model, CtcLossCriterion(_Task()), NoamLRScheduler(5.0, 25000, 512, 1e-6), adam_betas=(0.9, 0.98),
                      clip_norm=2.0, use_cuda_graphs=not args.eager)

    n_distinct = max(1, args.distinct)
    host = make_batches(n_distinct)
    pinned = [{k: (torch.from_numpy(v).pin_memory() if isinstance(v, np.ndarray) else v) for k, v in b.items()} for b in host]

    def to_dev(b):
        return {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in b.items()}

    def sample_of(d, n_cpu):
        return {"net_input": {"src_tokens": d["wave"], "src_lengths": d["n_samples"], "freq_masks": d["fm"],
                              "time_masks": d["tm"], "src_lengths_cpu": n_cpu},
                "target": d["target"]}

    resident = [to_dev(b) for b in pinned]
    n_cpu = [b["n_samples"].clone().long() for b in pinned]
    h2d_bytes = int(np.mean([sum(v.numel() * v.element_size() for v in b.values() if torch.is_tensor(v)) for b in pinned]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    copy_stream = torch.cuda.Stream()

    def upload(j):
        """H2D of step inputs from pinned host memory on the copy stream (like the reference's pinned DataLoader +
        non_blocking move_to_cuda, fairseq/trainer.py:1298-1338); returns (tensors, event)."""
        with torch.cuda.stream(copy_stream):
            d = to_dev(pinned[j])
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return d, ev

    loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event() for _ in range(2)]

    def timed(nsteps, from_host, do_upload=True, read_loss=True, sync_each=False):
        losses = []
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        audio = 0.0
        e0.record()
        nxt = upload(0) if (from_host and do_upload) else None
        for i in range(nsteps):
            j = i % n_distinct
            if from_host and not do_upload:
                d = resident[j]
            elif from_host:
                d, ev = nxt
                torch.cuda.current_stream().wait_event(ev)
                for t in d.values():
                    if torch.is_tensor(t):
                        t.record_stream(torch.cuda.current_stream())
                if i + 1 < nsteps:
                    nxt = upload((i + 1) % n_distinct)  # overlaps with this step's compute
            else:
                d = resident[j]
            trainer.train_step([sample_of(d, n_cpu[j])])
            audio += pinned[j]["audio_s"]
            if from_host and sync_each:
                _ = trainer.last_stats[3].item()
            elif from_host and read_loss:
                # D2H read of EVERY step's loss into pinned memory; the host consumes it one step late (after the next
                # step has been queued), as a training loop that logs asynchronously does, so the GPU never idles
                # waiting for Python between steps.
                slot = i % 2
                loss_host[slot].copy_(trainer.last_stats[3:4], non_blocking=True)
                loss_ev[slot].record()
                if i > 0:
                    loss_ev[1 - slot].synchronize()
                    losses.append(float(loss_host[1 - slot][0]))
        if from_host and read_loss and not sync_each and nsteps > 0:
            loss_ev[(nsteps - 1) % 2].synchronize()
            losses.append(float(loss_host[(nsteps - 1) % 2][0]))
            assert len(losses) == nsteps and all(np.isfinite(losses))
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms, audio], dtype=torch.float64, device=dev)
        if world > 1:
            mx = t.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return float(mx[0]), float(t[1])
        return float(t[0]), float(t[1])

    def note(msg):
        if rank == 0:
            print("[bench] " + msg, file=sys.stderr, flush=True)

    note("model + data ready (world=%d)" % world)
    if not args.eager:  # every shape bucket: one eager pass + one capture pass (not timed, not warm-up)
        for p_ in range(2):
            for j in range(n_distinct):
                trainer.train_step([sample_of(resident[j], n_cpu[j])])
            torch.cuda.synchronize()
            note("prepare pass %d done (%d graphs for %d distinct batches)" % (p_, len(trainer._graphs), n_distinct))
    trainer.graph_hits = trainer.graph_misses = 0
    timed(args.warmup, False)
    note("warm-up done")
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = lib.launch_count()
    ms, audio = timed(args.steps, False)
    launches = lib.launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(step_outputs(trainer), args.dump_outputs)
    timed(max(3, args.warmup), True)  # warm the host-buffer path too (copy-stream allocator pool, pinned staging)
    ms_e2e, audio_e2e = timed(args.steps, True)
    clk = clocks.stop() if rank == 0 else None
    sustained = None
    if args.sustain > 0:  # a seconds-long run: clocks settle to their sustained value, all distinct shapes are visited
        ms_s, audio_s_ = timed(args.sustain, True)
        sustained = {"steps": args.sustain, "ms_per_step": ms_s / args.sustain, "value": audio_s_ / (ms_s * 1e-3),
                     "unit": "audio-s/s", "from": "pinned host buffers (same path as e2e)"}
    graph_stats = {"graphs": len(trainer._graphs), "distinct_batches": n_distinct, "hits": trainer.graph_hits,
                   "misses": trainer.graph_misses, "bucket_frames": trainer.bucket_frames}
    if not args.eager and world == 1:
        # the same step WITHOUT graph replay (every kernel launched from Python): what a batch whose shape bucket has no
        # captured graph yet costs, on the same resident batches
        trainer.use_cuda_graphs = False
        timed(3, False)
        ms_eager, _ae = timed(10, False)
        trainer.use_cuda_graphs = True
        graph_stats["eager_ms_per_step"] = ms_eager / 10
        graph_stats["note"] = ("a bucket's first occurrence runs eagerly, its second captures; %d buckets cover the %d distinct "
                               "LibriSpeech-shape batches of this run" % (len(trainer._graphs), n_distinct))
    if os.environ.get("ESP_BENCH_E2E_DEBUG"):
        for name, kw in (("upload+lagged read", {}), ("upload only", dict(read_loss=False)), ("lagged read only", dict(do_upload=False)),
                         ("upload+item()", dict(sync_each=True)), ("item() only", dict(do_upload=False, sync_each=True))):
            m_, _a = timed(args.steps, True, **kw)
            note("e2e variant %-20s %.2f ms/step" % (name, m_ / args.steps))

    # ---- rooflines: the dominant kernel (tcgen05 GEMM, tensor-bound) and the HBM-bound front end / CTC kernels ------
    roof, roof_hbm = None, []
    if rank == 0:
        import json as _json
        peaks = {}
        try:
            peaks = _json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6575.8)

        def replay_us(calls, reps=1):
            """Device time per call of `calls` (zero-argument launchers) run back to back between ONE pair of CUDA
            events on the launching stream: kernel time without launch gaps or per-launch event overhead."""
            for c in calls:
                c()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(int(2e8))  # let the host run ahead so the GPU never waits for a launch
            e0.record()
            for _ in range(reps):
                for c in calls:
                    c()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e3 / (reps * len(calls))

        # Record every GEMM / CTC call of one eager step (arguments + operand tensors kept alive), then replay them.
        recs, ctc_recs, af_recs, ab_recs = [], [], [], []
        orig, orig_ctc, orig_af, orig_ab = ops.gemm, ops.ctc_loss, ops.attn_fused_fwd, ops.attn_fused_bwd

        def rec_gemm(A, B, C_out, M, N, K, *a, **kw):
            recs.append(((A, B, C_out, M, N, K) + a, dict(kw), 2.0 * M * N * K * kw.get("nb1", 1) * kw.get("nb2", 1)))
            return orig(A, B, C_out, M, N, K, *a, **kw)

        def rec_ctc(*a, **kw):
            ctc_recs.append((a, dict(kw)))
            return orig_ctc(*a, **kw)

        def rec_af(*a, **kw):
            af_recs.append((a, dict(kw)))
            return orig_af(*a, **kw)

        def rec_ab(*a, **kw):
            ab_recs.append((a, dict(kw)))
            return orig_ab(*a, **kw)

        ops.gemm, ops.ctc_loss, ops.attn_fused_fwd, ops.attn_fused_bwd = rec_gemm, rec_ctc, rec_af, rec_ab
        trainer.use_cuda_graphs = False
        trainer.world = 1  # rank-0-only pass: no collective (the other ranks are not in this code path)
        try:
            trainer.train_step([sample_of(resident[0], n_cpu[0])])
            torch.cuda.synchronize()
        finally:
            ops.gemm, ops.ctc_loss, ops.attn_fused_fwd, ops.attn_fused_bwd = orig, orig_ctc, orig_af, orig_ab
        us_gemm = replay_us([(lambda a_=a_, kw_=kw_: orig(*a_, **kw_)) for a_, kw_, _ in recs])
        tot_ms = us_gemm * len(recs) * 1e-3
        tot_fl = sum(f_ for _, _, f_ in recs)
        useful, fl_af, fl_ab = (float(x_) for x_ in useful_gemm_flops(host[0]["frames"]))
        model.flat.zero_grad()
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        ach = useful / (tot_ms * 1e-3) / 1e12 if tot_ms > 0 else 0.0
        roof = {"kernel": "gemm_tcgen05_kernel (all %d launches of one step, replayed back to back)" % len(recs),
                "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s",
                "achieved_is": "useful flops executed by the step's tcgen05 GEMM launches (padded frames EXCLUDED, SURVEY 8d "
                               "accounting; the fused attention kernels' flops are NOT counted here, see tensor_other) / summed "
                               "device time of those launches",
                "achieved_incl_padding": tot_fl / (tot_ms * 1e-3) / 1e12, "useful_tflop_per_step": useful / 1e12,
                "launched_tflop_per_step": tot_fl / 1e12,
                "gemm_ms_per_step": tot_ms, "gemm_share_of_step": tot_ms / (ms / args.steps), "traffic": None,
                "launches": len(recs),
                "whole_step_frac": (useful + fl_af + fl_ab) / ((ms / args.steps) * 1e-3) / 1e12 / peak}
        # the other tensor-core kernels of the step: fused attention forward / backward, replayed the same way
        other = []
        for nm, rl, fn_, fl_ in (("attn_fused_fwd_kernel", af_recs, orig_af, fl_af),
                                 ("attn_fused_bwd_kernel (+ row-dot and skew kernels)", ab_recs, orig_ab, fl_ab)):
            if rl:
                us_ = replay_us([(lambda a_=a_, kw_=kw_, fn_=fn_: fn_(*a_, **kw_)) for a_, kw_ in rl])
                t_ms = us_ * len(rl) * 1e-3
                other.append({"kernel": nm, "launches": len(rl), "ms_per_step": t_ms, "useful_tflop_per_step": fl_ / 1e12,
                              "achieved": fl_ / (t_ms * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s",
                              "frac": fl_ / (t_ms * 1e-3) / 1e12 / peak,
                              "bound": "instruction issue of the softmax / dS warps and TMA latency, not the tensor pipe (DESIGN.md 4)"})
        roof["tensor_other"] = other
        try:  # DRAM bytes per launch from the committed ncu capture of the same command (profiles/)
            tr = _json.load(open(os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")))
            roof["traffic"] = tr["dram_bytes_per_launch"]
            roof["traffic_unit"] = ("bytes per launch (dram read+write, mean over the %d GEMM launches of a step, ncu capture "
                                    "profiles/r02_gemm_traffic.json taken before the attention-backward fusion removed 51 of them)" % tr["launches"])
            roof["algorithmic_bytes_per_launch"] = sum(
                2.0 * (a_[3] * a_[5] + a_[4] * a_[5] + a_[3] * a_[4]) * kw_.get("nb1", 1) * kw_.get("nb2", 1)
                for a_, kw_, _ in recs) / max(len(recs), 1)
        except Exception:
            pass
        if not args.no_hbm_roofline:
            # front end: every distinct batch once per repetition (inputs 15 MB each: together far beyond the 126 MB L2)
            fe = model.frontend
            calls = [(lambda d=d: fe(d["wave"], d["n_samples"], d["fm"], d["tm"])) for d in resident]
            us = replay_us(calls, reps=2)
            audio_mean = float(np.mean([b["audio_s"] for b in host]))
            nbytes = 80000.0 * audio_mean   # SURVEY 8d: 16 000 x 4 B in + 100 x 80 x 2 B out per audio-second
            roof_hbm.append({"kernel": "frontend_kernel (fbank+CMVN+SpecAugment)", "bound": "hbm", "us_per_launch": us,
                             "achieved": nbytes / us / 1e3, "peak": hbm_peak, "unit": "GB/s", "frac": nbytes / us / 1e3 / hbm_peak,
                             "algorithmic_bytes_per_launch": nbytes, "per_unit": "80 000 B per audio-second (f32 wave in, bf16 out)",
                             "inputs": "%d distinct batches cycled (> L2)" % len(resident)})
            # CTC (log-softmax + alpha/beta + gradient): the recorded call on 3 rotating logits buffers (> L2 together)
            if ctc_recs:
                a_, kw_ = ctc_recs[0]
                lg = [a_[0]] + [a_[0].clone() for _ in range(2)]
                calls = [(lambda l_=l_: orig_ctc(l_, *a_[1:], **kw_)) for l_ in lg]
                us = replay_us(calls, reps=4)
                Bc, Tc = a_[0].shape[0], a_[0].shape[1]
                cells_valid = int(a_[2].sum().item())  # encoder frames that belong to an utterance
                nbytes = 6.0 * V * cells_valid
                roof_hbm.append({"kernel": "ctc_prep + ctc_scan + ctc_grad (esp_ctc_loss)", "bound": "hbm", "us_per_launch": us,
                                 "achieved": nbytes / us / 1e3, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": nbytes / us / 1e3 / hbm_peak, "algorithmic_bytes_per_launch": nbytes,
                                 "per_unit": "6 V B per valid encoder frame (logits read twice, gradient written once)",
                                 "shape": "B=%d T'=%d V=%d valid_frames=%d" % (Bc, Tc, V, cells_valid),
                                 "inputs": "3 rotating logits buffers of %.0f MB" % (a_[0].numel() * 2 / 1e6)})
                del lg
        del recs, ctc_recs, af_recs, ab_recs

    if rank == 0:
        val = audio / (ms * 1e-3)
        out = {
            "metric": "training throughput (audio-seconds/second)", "value": val, "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(world), "clocks": clk, "gpu_launches": int(launches),
            "e2e": {"value": audio_e2e / (ms_e2e * 1e-3), "unit": "audio-s/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
            "roofline": roof, "roofline_hbm": roof_hbm, "sustained": sustained, "cuda_graphs": graph_stats,
            "audio_s_per_gpu_step": audio / args.steps / world,
        }
        if args.layers is not None:
            out["INVALID"] = "layer count overridden for debugging"
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_quick()
        if world == 1:
            del trainer, resident
            model.flat.g32 = model.flat.p32 = model.flat.m = model.flat.v = None
            torch.cuda.empty_cache()
        if world == 1 and not args.no_gpu_eager:
            try:
                out["gpu_eager_baseline"] = gpu_eager_baseline(dev, host)
                out["gpu_eager_baseline"]["speedup_e2e_over_eager"] = out["e2e"]["value"] / out["gpu_eager_baseline"]["value"]
            except Exception as ex:  # never lose the main line over the comparison leg
                out["gpu_eager_baseline"] = {"error": repr(ex)[:300]}
            torch.cuda.empty_cache()
        if world == 1 and not args.no_decode:  # configs[4] is a 1xB200 measurement
            out["decode"] = decode_rtf(dev)
            out["roofline_hbm"] += out["decode"].pop("roofline_hbm", [])
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

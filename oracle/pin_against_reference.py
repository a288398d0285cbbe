"""Pin the oracle against the REAL reference and (re)generate tests/golden/*.npz.

Runs only in the authoring container (needs /root/reference; imported through oracle/refshim).
    python -m oracle.pin_against_reference [frontend] [ctc] [conformer] ...
Each section (1) runs the reference's own code on seeded synthetic inputs, (2) asserts the oracle
restatement agrees, (3) stores inputs + reference outputs as a small fixture.  The GPU tests compare
the CUDA path against those fixtures (and against the oracle on fresh seeded inputs).
"""
import os
import sys

import numpy as np
import torch

from oracle import refshim

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
SPECAUG_CFG = {"time_warp_W": 0, "freq_mask_F": 27, "freq_mask_N": 2, "time_mask_pm": 0.04, "time_mask_ps": 0.04}


def pin_frontend():
    from espresso.data.feature_transforms.adaptive_specaugment import AdaptiveSpecAugmentTransform
    from espresso.tools.utils import get_torchaudio_fbank_or_mfcc
    from fairseq.data import data_utils
    from fairseq.data.audio.feature_transforms.global_cmvn import GlobalCMVN  # noqa: F401

    from oracle import frontend as O

    durs = [1.0, 2.35, 0.5, 3.17, 0.03]
    waves = [O.synth_waveform(i, d) for i, d in enumerate(durs)]
    # CMVN stats with the reference formula (espresso/tools/compute_global_cmvn_stats.py:94-118)
    feats_ref = [get_torchaudio_fbank_or_mfcc(w[None, :], 16000, n_bins=80) for w in waves[:4]]
    allf = np.concatenate(feats_ref, axis=0).astype(np.float64)
    mean = allf.mean(axis=0)
    var = (allf ** 2).mean(axis=0) - mean ** 2
    std = np.sqrt(np.maximum(var, 1e-8))
    aug = AdaptiveSpecAugmentTransform.from_config_dict(SPECAUG_CFG)
    out = {"durs": np.array(durs), "cmvn_mean": mean, "cmvn_std": std}
    worst = 0.0
    for i, w in enumerate(waves):
        n = len(w)
        if O.num_frames(n) == 0:
            continue
        ref_fb = get_torchaudio_fbank_or_mfcc(w[None, :], 16000, n_bins=80)      # float32 [m,80]
        ref_cm = (ref_fb - mean) / std                                            # GlobalCMVN.__call__
        with data_utils.numpy_seed(1, 1, i):
            ref_sa = aug(ref_cm)
        # oracle restatement
        o_fb = O.kaldi_fbank(w)
        o_cm = O.global_cmvn(o_fb, mean, std)
        with O.numpy_seed(1, 1, i):
            o_sa, fm, tm = O.adaptive_specaugment(o_cm, return_masks=True)
        d_fb = np.abs(o_fb - ref_fb).max()
        d_sa = np.abs(o_sa - ref_sa).max()
        worst = max(worst, d_fb, d_sa)
        print("frontend utt %d: m=%d |fbank diff|=%.3g |specaug diff|=%.3g masks f=%s t=%d" % (
            i, ref_fb.shape[0], d_fb, d_sa, fm, len(tm)))
        assert d_fb < 2e-3 and d_sa < 2e-3, "oracle front end disagrees with the reference"
        out["wave_%d" % i] = w
        out["fbank_%d" % i] = ref_fb.astype(np.float32)
        out["final_%d" % i] = ref_sa.astype(np.float32)
        out["fmask_%d" % i] = np.array(fm, dtype=np.int32).reshape(-1, 2)
        out["tmask_%d" % i] = np.array(tm, dtype=np.int32).reshape(-1, 2)
    np.savez_compressed(os.path.join(GOLDEN, "frontend.npz"), **out)
    print("frontend pinned (worst abs diff %.3g) -> tests/golden/frontend.npz" % worst)


def pin_ctc():
    import torch.nn.functional as F

    from oracle import ctc as O

    rs = np.random.RandomState(3)
    B, T, V, blank = 4, 23, 11, 0
    logits = torch.from_numpy(rs.randn(B, T, V).astype(np.float32) * 2.0).to(torch.bfloat16)
    in_lens = np.array([23, 17, 9, 3], dtype=np.int32)
    tgts = [rs.randint(1, V, size=u) for u in (7, 5, 4, 5)]  # last one infeasible (U > T)
    tgts[1][1] = tgts[1][0]  # repeated label
    u_max = max(len(t) for t in tgts)
    targets = np.zeros((B, u_max), dtype=np.int32)
    for b, t in enumerate(tgts):
        targets[b, :len(t)] = t
    tgt_lens = np.array([len(t) for t in tgts], dtype=np.int32)
    # the reference call (espresso/criterions/ctc_loss.py:85-94) on [T,B,V] fp32 log-probs
    x = logits.float().transpose(0, 1).contiguous().requires_grad_(True)
    lprobs = F.log_softmax(x, dim=-1)
    flat = torch.from_numpy(np.concatenate(tgts)).long()
    loss = F.ctc_loss(lprobs, flat, torch.from_numpy(in_lens).long(), torch.from_numpy(tgt_lens).long(),
                      blank=blank, reduction="none", zero_infinity=True)
    loss.sum().backward()
    ref_loss = loss.detach().numpy()
    ref_grad = x.grad.transpose(0, 1).numpy()  # [B,T,V]
    for b in range(B):
        nll, g = O.ctc_loss_and_grad(logits[b].float().numpy(), in_lens[b], tgts[b], blank)
        assert abs(nll - ref_loss[b]) < 1e-4 * max(1.0, abs(ref_loss[b])), (b, nll, ref_loss[b])
        assert np.abs(g - ref_grad[b]).max() < 1e-5, (b, np.abs(g - ref_grad[b]).max())
    print("ctc losses", ref_loss)
    np.savez_compressed(os.path.join(GOLDEN, "ctc.npz"), logits=logits.float().numpy(), in_lens=in_lens,
                        targets=targets, tgt_lens=tgt_lens, blank=blank, loss=ref_loss, grad=ref_grad)
    print("ctc pinned -> tests/golden/ctc.npz")


def _ref_model(layer_type, layers=2, d=64, ffn=128, heads=4, V=50, learned_pos=False, share_heads=False,
               conv_channels="[64, 64, 128, 128]"):
    from espresso.models.transformer.speech_transformer_config import SpeechTransformerConfig
    from espresso.models.transformer.speech_transformer_encoder_model import SpeechTransformerEncoderModel

    cfg = SpeechTransformerConfig()
    cfg.max_source_positions, cfg.max_target_positions, cfg.tpu = 3600, 200, False
    e = cfg.encoder
    e.conv_channels = conv_channels
    e.conv_kernel_sizes = "[(3, 3), (3, 3), (3, 3), (3, 3)]"
    e.conv_strides = "[(1, 1), (2, 2), (1, 1), (2, 2)]"
    e.embed_dim, e.ffn_embed_dim, e.layers, e.attention_heads = d, ffn, layers, heads
    e.normalize_before, e.learned_pos, e.relative_positional_embeddings = True, learned_pos, True
    e.share_learned_relative_positional_embeddings_across_heads = share_heads
    e.layer_type, e.depthwise_conv_kernel_size = layer_type, 31
    cfg.layernorm_embedding = True
    cfg.dropout = cfg.attention_dropout = cfg.activation_dropout = 0.0

    class _Dict:
        def __len__(self):
            return V

        def pad(self):
            return 1

    class _Task:
        feat_dim, feat_in_channels, target_dictionary = 80, 1, _Dict()

    torch.manual_seed(1)
    return SpeechTransformerEncoderModel.build_model(cfg, _Task())


def pin_conformer():
    """Reference model forward + CtcLossCriterion-equivalent loss/grad vs oracle/conformer.py; fixtures for both
    layer types (conformer = cfg 3/4 encoder, transformer = cfg 2 encoder)."""
    import torch.nn.functional as F

    from oracle import conformer as O

    for variant in ("conformer", "transformer", "transformer_learned", "conformer_learned_sh"):
        layer_type = variant.split("_")[0]
        learned = "learned" in variant
        m = _ref_model(layer_type, learned_pos=learned, share_heads=variant.endswith("_sh"))
        if learned:  # max_source_positions 3600 -> tables of 2*900-1 rows; keep the fixture small
            assert any("positional_embedding.weight" in k for k in m.state_dict())
        # make LayerNorm/BatchNorm affine params and biases non-trivial so every gradient path is exercised
        g = torch.Generator().manual_seed(5)
        with torch.no_grad():
            for n, p_ in m.named_parameters():
                if p_.dim() == 1:
                    p_.add_(0.1 * torch.randn(p_.shape, generator=g))
        rs = np.random.RandomState(11)
        B, T = 3, 61
        lens = torch.tensor([61, 50, 37])
        feats = torch.from_numpy(rs.randn(B, T, 80).astype(np.float32))
        for b in range(B):
            feats[b, lens[b]:] = 0.0
        V, pad_idx, eos_idx, blank = 50, 1, 2, 0
        tgt = torch.full((B, 7), pad_idx, dtype=torch.long)
        for b, u in enumerate((6, 4, 3)):
            tgt[b, :u] = torch.from_numpy(rs.randint(4, V, size=u))
            tgt[b, u] = eos_idx
        cfg = dict(embed_dim=64, ffn_dim=128, heads=4, layers=2, layer_type=layer_type, dw_kernel=31, dropout=0.0,
                   attention_dropout=0.0, activation_dropout=0.0, layernorm_embedding=True,
                   final_layer_norm=(layer_type != "conformer"), vocab=V)
        out = {}
        for mode in ("train", "eval"):
            m.train(mode == "train")
            sd0 = {k: v.clone() for k, v in m.state_dict().items()}
            m.zero_grad()
            net = m(feats, lens)
            logits = net["encoder_out"][0]                      # T' x B x V
            olens = net["src_lengths"][0]
            lprobs = m.get_normalized_probs(net, log_probs=True).contiguous()
            keep = (tgt != pad_idx) & (tgt != eos_idx)
            with torch.backends.cudnn.flags(enabled=False):
                loss = F.ctc_loss(lprobs, tgt.masked_select(keep), olens, keep.sum(-1), blank=blank, reduction="sum",
                                  zero_infinity=True)              # espresso/criterions/ctc_loss.py:85-94
            # oracle on the same weights (state before this forward: BN running stats are updated in train mode)
            sd = {k: v.clone().requires_grad_(v.is_floating_point() and k in dict(m.named_parameters()))
                  for k, v in sd0.items()}
            o_logits, o_lens, _ = O.encoder_forward(sd, cfg, feats, lens, training=(mode == "train"))
            o_loss = O.ctc_criterion(o_logits, o_lens, tgt, pad_idx, eos_idx, blank)
            d_log = (o_logits.transpose(0, 1) - logits).abs().max().item()
            assert torch.equal(o_lens, olens)
            assert d_log < 2e-4, (layer_type, mode, d_log)
            assert abs(o_loss.item() - loss.item()) < 1e-3 * abs(loss.item())
            print("%s/%s: |logits diff|=%.3g loss ref=%.6f oracle=%.6f" % (layer_type, mode, d_log, loss.item(), o_loss.item()))
            if mode == "train":
                loss.backward()
                o_loss.backward()
                worst = 0.0
                for n, p_ in m.named_parameters():
                    # biases feeding a BatchNorm have an analytically zero gradient (pure rounding noise): compare
                    # against the largest gradient magnitude in the model, not the tensor's own
                    dg = (sd[n].grad - p_.grad).abs().max().item() / max(p_.grad.abs().max().item(), 1e-3)
                    if dg > 2e-3:
                        print("   ", n, dg, p_.grad.abs().max().item())
                    worst = max(worst, dg)
                print("   worst relative grad diff %.3g" % worst)
                assert worst < 2e-3
                for k, v in sd0.items():
                    out["sd." + k] = v.numpy()
                for n, p_ in m.named_parameters():
                    out["grad." + n] = p_.grad.numpy()
                # BN running stats after the training forward (momentum update incl. padded frames)
                for k, v in m.state_dict().items():
                    if "running_" in k:
                        out["after." + k] = v.numpy()
                        assert (sd[k] - v).abs().max().item() < 1e-4
            out["logits_" + mode] = logits.detach().transpose(0, 1).numpy()   # B x T' x V
            out["loss_" + mode] = np.float64(loss.item())
        out.update(feats=feats.numpy(), lens=lens.numpy(), target=tgt.numpy(), out_lens=olens.numpy())
        np.savez_compressed(os.path.join(GOLDEN, "encoder_%s.npz" % variant), **out)
        print("%s encoder pinned -> tests/golden/encoder_%s.npz" % (variant, variant))


def pin_encdec():
    """Reference SpeechTransformerModelBase (Transformer encoder + Transformer decoder) with the reference's
    label_smoothed_nll_loss vs oracle/conformer.py + oracle/decoder.py; fixture for the enc-dec path (cfg 2/5)."""
    from espresso.criterions.label_smoothed_cross_entropy_v2 import label_smoothed_nll_loss
    from espresso.models.transformer.speech_transformer_base import SpeechTransformerModelBase
    from espresso.models.transformer.speech_transformer_config import SpeechTransformerConfig

    from oracle import conformer as OC
    from oracle import decoder as OD

    V, pad_idx, eos_idx = 50, 1, 2
    cfg = SpeechTransformerConfig()
    cfg.max_source_positions, cfg.max_target_positions, cfg.tpu = 3600, 200, False
    e = cfg.encoder
    e.conv_channels = conv_channels
    e.conv_kernel_sizes = "[(3, 3), (3, 3), (3, 3), (3, 3)]"
    e.conv_strides = "[(1, 1), (2, 2), (1, 1), (2, 2)]"
    e.embed_dim, e.ffn_embed_dim, e.layers, e.attention_heads = 64, 128, 2, 4
    e.normalize_before, e.learned_pos, e.relative_positional_embeddings, e.layer_type = True, False, True, "transformer"
    d = cfg.decoder
    d.embed_dim, d.ffn_embed_dim, d.layers, d.attention_heads = 64, 128, 2, 4
    d.normalize_before, d.learned_pos, d.relative_positional_embeddings = True, False, False
    d.input_dim, d.output_dim = 64, 64
    cfg.dropout = cfg.attention_dropout = cfg.activation_dropout = 0.0

    class _Dict:
        def __len__(self):
            return V

        def pad(self):
            return pad_idx

        def eos(self):
            return eos_idx

    class _Task:
        feat_dim, feat_in_channels, target_dictionary = 80, 1, _Dict()

    torch.manual_seed(2)
    m = SpeechTransformerModelBase.build_model(cfg, _Task())
    g = torch.Generator().manual_seed(6)
    with torch.no_grad():
        for n, p_ in m.named_parameters():
            if p_.dim() == 1:
                p_.add_(0.1 * torch.randn(p_.shape, generator=g))
    rs = np.random.RandomState(12)
    B, T = 3, 61
    lens = torch.tensor([61, 50, 37])
    feats = torch.from_numpy(rs.randn(B, T, 80).astype(np.float32))
    for b in range(B):
        feats[b, lens[b]:] = 0.0
    U = 8
    tgt = torch.full((B, U), pad_idx, dtype=torch.long)
    prev = torch.full((B, U), pad_idx, dtype=torch.long)
    for b, u in enumerate((7, 5, 3)):
        toks = torch.from_numpy(rs.randint(4, V, size=u))
        tgt[b, :u] = toks
        tgt[b, u] = eos_idx
        prev[b, 0] = eos_idx          # fairseq feeds </s> first (move_eos_to_beginning)
        prev[b, 1:u + 1] = toks
    ecfg = dict(embed_dim=64, ffn_dim=128, heads=4, layers=2, layer_type="transformer", dropout=0.0, attention_dropout=0.0,
                activation_dropout=0.0, layernorm_embedding=False, final_layer_norm=True, vocab=None)
    dcfg = dict(dec_embed_dim=64, dec_heads=4, dec_layers=2, pad=pad_idx, dropout=0.0, attention_dropout=0.0,
                activation_dropout=0.0)
    eps = 0.1
    m.train()
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    m.zero_grad()
    logits, extra = m(feats, lens, prev)
    lprobs = m.get_normalized_probs((logits, extra), log_probs=True)
    loss, nll = label_smoothed_nll_loss(lprobs.view(-1, lprobs.size(-1)), tgt.view(-1), eps, ignore_index=pad_idx, reduce=True,
                                        smoothing_type="uniform")
    loss.backward()
    pnames = dict(m.named_parameters())
    sd = {k: v.clone().requires_grad_(k in pnames) for k, v in sd0.items()}
    enc, ol, pad = OC.encoder_forward(sd, ecfg, feats, lens, training=True)
    o_logits = OD.decoder_forward(sd, dcfg, prev, enc, pad if bool(pad.any()) else None, training=True)
    o_loss, o_nll = OD.label_smoothed_ce(o_logits, tgt, eps, pad_idx)
    o_loss.backward()
    dl = (o_logits - logits).abs().max().item()
    print("encdec: |logits diff|=%.3g loss ref=%.6f oracle=%.6f nll ref=%.6f oracle=%.6f" % (dl, loss.item(), o_loss.item(), nll.item(), o_nll.item()))
    assert dl < 2e-4 and abs(loss.item() - o_loss.item()) < 1e-3 * abs(loss.item())
    worst = 0.0
    for n, p_ in m.named_parameters():
        dg = (sd[n].grad - p_.grad).abs().max().item() / max(p_.grad.abs().max().item(), 1e-3)
        worst = max(worst, dg)
    print("   worst relative grad diff %.3g" % worst)
    assert worst < 2e-3
    out = {"sd." + k: v.numpy() for k, v in sd0.items()}
    out.update({"grad." + n: p_.grad.numpy() for n, p_ in m.named_parameters()})
    out.update(feats=feats.numpy(), lens=lens.numpy(), target=tgt.numpy(), prev_output_tokens=prev.numpy(),
               logits=logits.detach().numpy(), loss=np.float64(loss.item()), nll=np.float64(nll.item()), eps=np.float64(eps))
    np.savez_compressed(os.path.join(GOLDEN, "encdec_transformer.npz"), **out)
    print("encdec pinned -> tests/golden/encdec_transformer.npz")


def pin_scheduled_sampling():
    """Scheduled sampling of the Transformer decoder (espresso/models/transformer/speech_transformer_decoder.py:254-324): the
    REAL reference model of the encdec fixture (same weights), sampling probability 0.4, torch seed 77, training mode,
    dropout 0.  Stores the returned logits and the tokens that were fed (reconstructed from the logits' arg-max and a
    replay of the coin flips -- the only RNG consumers of that pass)."""
    from espresso.models.transformer.speech_transformer_base import SpeechTransformerModelBase
    from espresso.models.transformer.speech_transformer_config import SpeechTransformerConfig
    from espresso.tools.scheduled_sampling_rate_scheduler import ScheduledSamplingRateScheduler

    gfix = np.load(os.path.join(GOLDEN, "encdec_transformer.npz"))
    V, pad_idx, eos_idx = 50, 1, 2
    cfg = SpeechTransformerConfig()
    cfg.max_source_positions, cfg.max_target_positions, cfg.tpu = 3600, 200, False
    e = cfg.encoder
    e.conv_channels = "[64, 64, 128, 128]"
    e.conv_kernel_sizes = "[(3, 3), (3, 3), (3, 3), (3, 3)]"
    e.conv_strides = "[(1, 1), (2, 2), (1, 1), (2, 2)]"
    e.embed_dim, e.ffn_embed_dim, e.layers, e.attention_heads = 64, 128, 2, 4
    e.normalize_before, e.learned_pos, e.relative_positional_embeddings, e.layer_type = True, False, True, "transformer"
    d = cfg.decoder
    d.embed_dim, d.ffn_embed_dim, d.layers, d.attention_heads = 64, 128, 2, 4
    d.normalize_before, d.learned_pos, d.relative_positional_embeddings = True, False, False
    d.input_dim, d.output_dim = 64, 64
    cfg.dropout = cfg.attention_dropout = cfg.activation_dropout = 0.0

    class _Dict:
        def __len__(self):
            return V

        def pad(self):
            return pad_idx

        def eos(self):
            return eos_idx

    class _Task:
        feat_dim, feat_in_channels, target_dictionary = 80, 1, _Dict()

    m = SpeechTransformerModelBase.build_model(cfg, _Task())
    sd = {k[3:]: torch.from_numpy(gfix[k]) for k in gfix.files if k.startswith("sd.")}
    torch.nn.Module.load_state_dict(m, sd, strict=False)
    feats, lens, prev = torch.from_numpy(gfix["feats"]), torch.from_numpy(gfix["lens"]), torch.from_numpy(gfix["prev_output_tokens"])
    out = {}
    for tag, prob, seed in (("p04", 0.4, 77), ("p00", 0.0, 5)):
        m.decoder.scheduled_sampling_rate_scheduler = ScheduledSamplingRateScheduler([prob], 1)
        m.train()
        torch.manual_seed(seed)
        with torch.no_grad():
            logits, _ = m(feats, lens, prev, epoch=1)
        B, U = prev.shape
        torch.manual_seed(seed)
        feed = prev.clone()
        for step in range(1, U):
            coin = torch.rand([B, 1]).lt(prob)[:, 0]
            feed[:, step] = torch.where(coin, prev[:, step], logits[:, step - 1].argmax(-1))
        # self-check: a plain teacher-forced pass over the fed tokens reproduces the logits of the sampled pass -- with ONE
        # quirk of the reference: its sampled pass feeds a [B, 1] token tensor per step, so the sinusoidal position module
        # (incremental branch, sinusoidal_positional_embedding.py:78-87: pos = seq_len = 1) gives EVERY step the embedding of
        # the first position
        m.decoder.scheduled_sampling_rate_scheduler = ScheduledSamplingRateScheduler([1.0], 1)
        pe = m.decoder.embed_positions
        orig_fwd = pe.forward

        def const_pos(input, incremental_state=None, timestep=None, positions=None):
            full = orig_fwd(input[:, :1], incremental_state={}, timestep=None)   # [B, 1, d]: position padding_idx + 1
            return full.expand(-1, input.size(1), -1)

        pe.forward = const_pos
        with torch.no_grad():
            again, _ = m(feats, lens, feed, epoch=1)
        pe.forward = orig_fwd
        # (positions of the padded tail are not comparable: the incremental pass builds its key-padding mask from the ONE
        # token it is fed, the full pass from the whole row -- they only feed the ignored tail of the loss)
        valid = prev.ne(pad_idx)
        top2 = logits.topk(2, dim=-1).values
        dmax = (again - logits)[valid].abs().max().item()
        print("scheduled sampling %s: fed != truth at %d of %d valid positions; teacher-forced replay |diff| %.2e; min top-2 margin %.3f"
              % (tag, int(((feed != prev) & valid).sum()), int(valid.sum()), dmax, (top2[..., 0] - top2[..., 1])[valid].min().item()))
        assert dmax < 1e-4
        out.update({tag + "_prob": np.float64(prob), tag + "_seed": np.int64(seed), tag + "_logits": logits.numpy(),
                    tag + "_feed": feed.numpy(), tag + "_valid": valid.numpy()})
    np.savez_compressed(os.path.join(GOLDEN, "scheduled_sampling.npz"), **out)
    print("scheduled sampling pinned -> tests/golden/scheduled_sampling.npz")


def pin_transducer():
    """Reference SpeechTransformerTransducerModelBase (Conformer encoder + LSTM predictor + joint) with the criterion's
    torchaudio rnnt_loss call vs oracle/conformer.py + oracle/transducer.py; fixture for the RNN-T path (cfg 4)."""
    import torchaudio

    from espresso.models.transformer.speech_transformer_transducer_base import SpeechTransformerTransducerModelBase
    from espresso.models.transformer.speech_transformer_transducer_config import SpeechTransformerTransducerConfig

    from oracle import conformer as OC
    from oracle import transducer as OT

    V, pad_idx, eos_idx, blank = 50, 1, 2, 0
    cfg = SpeechTransformerTransducerConfig()
    cfg.max_source_positions, cfg.max_target_positions, cfg.tpu = 3600, 200, False
    e = cfg.encoder
    e.conv_channels = conv_channels
    e.conv_kernel_sizes = "[(3, 3), (3, 3), (3, 3), (3, 3)]"
    e.conv_strides = "[(1, 1), (2, 2), (1, 1), (2, 2)]"
    e.embed_dim, e.ffn_embed_dim, e.layers, e.attention_heads = 64, 128, 2, 4
    e.normalize_before, e.learned_pos, e.relative_positional_embeddings, e.layer_type = True, False, True, "conformer"
    e.depthwise_conv_kernel_size = 31
    d = cfg.decoder
    d.embed_dim, d.hidden_size, d.layers, d.dropout_in, d.dropout_out, d.residual = 64, 64, 2, 0.0, 0.0, False
    cfg.joint_dim = 64
    cfg.layernorm_embedding = True
    cfg.dropout = cfg.attention_dropout = cfg.activation_dropout = 0.0

    class _Dict:
        def __len__(self):
            return V

        def pad(self):
            return pad_idx

        def eos(self):
            return eos_idx

    class _Task:
        feat_dim, feat_in_channels, target_dictionary = 80, 1, _Dict()

    torch.manual_seed(3)
    m = SpeechTransformerTransducerModelBase.build_model(cfg, _Task())
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for n, p_ in m.named_parameters():
            if p_.dim() == 1:
                p_.add_(0.1 * torch.randn(p_.shape, generator=g))
    rs = np.random.RandomState(13)
    B, T = 3, 61
    lens = torch.tensor([61, 50, 37])
    feats = torch.from_numpy(rs.randn(B, T, 80).astype(np.float32))
    for b in range(B):
        feats[b, lens[b]:] = 0.0
    U = 6
    tgt = torch.full((B, U + 1), pad_idx, dtype=torch.long)
    prev = torch.full((B, U + 1), pad_idx, dtype=torch.long)
    for b, u in enumerate((6, 4, 2)):
        toks = torch.from_numpy(rs.randint(4, V, size=u))
        tgt[b, :u] = toks
        tgt[b, u] = eos_idx
        prev[b, 0] = eos_idx
        prev[b, 1:u + 1] = toks
    m.train()
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    m.zero_grad()
    logits, enc_lens = m(feats, lens, prev)
    u_lens = ((tgt != pad_idx) & (tgt != eos_idx)).sum(-1).int()
    loss = torchaudio.functional.rnnt_loss(logits, tgt[:, :-1].int().contiguous(), enc_lens.int(), u_lens, blank=blank, clamp=-1.0,
                                           reduction="sum")  # espresso/criterions/transducer_loss.py:130-140
    loss.backward()
    pnames = dict(m.named_parameters())
    sd = {k: v.clone().requires_grad_(k in pnames) for k, v in sd0.items()}
    ecfg = dict(embed_dim=64, ffn_dim=128, heads=4, layers=2, layer_type="conformer", dw_kernel=31, dropout=0.0,
                attention_dropout=0.0, activation_dropout=0.0, layernorm_embedding=True, final_layer_norm=False, vocab=None)
    enc, ol, _ = OC.encoder_forward(sd, ecfg, feats, lens, training=True)
    dec = OT.predictor(sd, prev, 2, pad_idx)
    o_logits = OT.joint_logits(sd, enc, dec)
    o_loss = OT.transducer_loss(o_logits, ol, tgt, pad_idx, eos_idx, blank)
    o_loss.backward()
    dl = (o_logits - logits).abs().max().item()
    print("transducer: |logits diff|=%.3g loss ref=%.6f oracle=%.6f" % (dl, loss.item(), o_loss.item()))
    assert dl < 2e-4 and abs(loss.item() - o_loss.item()) < 1e-4 * abs(loss.item())
    worst = 0.0
    for n, p_ in m.named_parameters():
        dg = (sd[n].grad - p_.grad).abs().max().item() / max(p_.grad.abs().max().item(), 1e-3)
        worst = max(worst, dg)
    print("   worst relative grad diff %.3g" % worst)
    assert worst < 1e-2  # fp32 recurrences (LSTM, RNN-T lattice) accumulate in a different order
    out = {"sd." + k: v.numpy() for k, v in sd0.items()}
    out.update({"grad." + n: p_.grad.numpy() for n, p_ in m.named_parameters()})
    out.update(feats=feats.numpy(), lens=lens.numpy(), target=tgt.numpy(), prev_output_tokens=prev.numpy(),
               logits=logits.detach().numpy(), loss=np.float64(loss.item()), enc_lens=enc_lens.numpy())
    np.savez_compressed(os.path.join(GOLDEN, "transducer_conformer.npz"), **out)
    print("transducer pinned -> tests/golden/transducer_conformer.npz")

    # ---- greedy decoding (validation decoder): the reference's TransducerGreedyDecoder vs oracle/transducer.greedy_decode
    from espresso.tools.transducer_greedy_decoder import TransducerGreedyDecoder

    class _DDict(_Dict):
        def bos(self):
            return blank

    torch.nn.Module.load_state_dict(m, sd0)  # (plain nn.Module load: fairseq's override trips on Conformer layers) fixture weights + running stats
    m.eval()
    gout = {}
    for name, kw in (("e2", dict(max_num_expansions_per_step=2)), ("e1_eos", dict(max_num_expansions_per_step=1, model_predicts_eos=True))):
        dec = TransducerGreedyDecoder([m], _DDict(), blank=blank, **kw)
        r_tok, r_sc, _ = dec.decode([m], {"net_input": {"src_tokens": feats, "src_lengths": lens}})
        with torch.no_grad():
            sde = {k: v.clone() for k, v in sd0.items()}
            enc_e, ol_e, _ = OC.encoder_forward(sde, ecfg, feats, lens, training=False)
            o_tok, o_sc, o_mar = OT.greedy_decode(sde, enc_e, ol_e, 2, pad_idx, blank, eos_idx, eos_idx, **kw)
        assert torch.equal(o_tok, r_tok), (name, o_tok, r_tok)
        assert (o_sc - r_sc).abs().max().item() < 1e-3, (o_sc, r_sc)
        print("transducer greedy %-7s: tokens identical (%d non-blank), |score diff| %.3g"
              % (name, int((r_tok != blank).sum()), (o_sc - r_sc).abs().max().item()))
        gout["tokens_" + name], gout["scores_" + name], gout["margins_" + name] = r_tok.numpy(), r_sc.numpy(), o_mar.numpy()
    # ---- with LSTM-LM shallow fusion (the reference requires an LSTM LM here: masked_copy_cached_state)
    from argparse import Namespace

    from espresso.models.lstm_lm import LSTMLanguageModelEspresso

    class _LmTask:
        source_dictionary = target_dictionary = _DDict()

    largs = Namespace(dropout=0.0, decoder_embed_path=None, decoder_freeze_embed=False, decoder_layers=2, decoder_embed_dim=24,
                      decoder_hidden_size=32, decoder_out_embed_dim=40, share_embed=False, decoder_rnn_residual=False,
                      adaptive_softmax_cutoff=None, is_wordlm=False, decoder_dropout_in=0.0, decoder_dropout_out=0.0,
                      criterion_name="cross_entropy", max_target_positions=64, tokens_per_sample=64)
    chosen = None
    for lm_seed in range(70, 130):  # pick an LM whose fusion changes many decisions while none of them is a near-tie
        torch.manual_seed(lm_seed)
        lm = LSTMLanguageModelEspresso.build_model(largs, _LmTask())
        with torch.no_grad():
            for p_ in lm.parameters():
                p_.mul_(6.0)
            lm.decoder.fc_out.weight.mul_(12.0)  # a peaky LM, so that fusion actually changes decisions
        lm_sd = {k: v.clone() for k, v in lm.state_dict().items()}
        with torch.no_grad():
            o_tok, o_sc, o_mar = OT.greedy_decode(sde, enc_e, ol_e, 2, pad_idx, blank, eos_idx, eos_idx, max_num_expansions_per_step=2,
                                                  lm_sd=lm_sd, lm_weight=1.0)
        fin = o_mar[torch.isfinite(o_mar)]
        changed = int((o_tok != torch.from_numpy(gout["tokens_e2"])).sum())
        if float(fin.min()) > 0.3 and changed >= 20:
            chosen = lm_seed
            break
    assert chosen is not None, "no LM seed with clear margins found"
    lm.decoder.dictionary = _DDict()
    lm.eval()
    dec = TransducerGreedyDecoder([m], _DDict(), blank=blank, max_num_expansions_per_step=2, lm_model=lm, lm_weight=1.0)
    r_tok, r_sc, _ = dec.decode([m], {"net_input": {"src_tokens": feats, "src_lengths": lens}})
    assert torch.equal(o_tok, r_tok), (o_tok, r_tok)
    assert (o_sc - r_sc).abs().max().item() < 1e-3
    print("transducer greedy + LM fusion (LM seed %d): tokens identical (%d non-blank, %d differ from no-LM), min margin %.3f"
          % (chosen, int((r_tok != blank).sum()), changed, float(fin.min())))
    gout["tokens_lm"], gout["scores_lm"], gout["margins_lm"] = r_tok.numpy(), r_sc.numpy(), o_mar.numpy()

    # ---- beam search ("adaptive expansion search", the recipes' decoder): the reference TransducerBeamSearchDecoder vs
    # espresso_b200's host search driven by fp32 oracle callbacks -- n-best token sequences and scores must be identical
    from espresso.tools.transducer_beam_search_decoder import TransducerBeamSearchDecoder as RefBeam

    from espresso_b200.tools.transducer_beam_search_decoder import AdaptiveExpansionSearch

    for name, kw, use_lm in (("beam5", dict(beam_size=5, max_num_expansions_per_step=3, expansion_beta=2, expansion_gamma=2.3,
                                            prefix_alpha=1, temperature=1.3), False),
                             ("beam3_lm", dict(beam_size=3, max_num_expansions_per_step=2, expansion_beta=1, expansion_gamma=4.0,
                                               prefix_alpha=2, temperature=1.0), True),
                             ("beam4_eos", dict(beam_size=4, max_num_expansions_per_step=2, expansion_beta=0, expansion_gamma=None,
                                                prefix_alpha=None, temperature=1.0, model_predicts_eos=True), False)):
        rdec = RefBeam([m], _DDict(), blank=blank, lm_model=lm if use_lm else None, lm_weight=0.3, **kw)
        r_seqs, r_scores, _ = rdec._generate({"net_input": {"src_tokens": feats, "src_lengths": lens}})
        core = AdaptiveExpansionSearch(V, blank, pad_idx, eos_idx, eos_idx, kw["beam_size"], kw["max_num_expansions_per_step"],
                                       kw["expansion_beta"], kw["expansion_gamma"], kw["prefix_alpha"], True,
                                       kw.get("model_predicts_eos", False), 0.3, False)
        n_h = 0
        for b in range(feats.size(0)):
            cb = OT.search_callbacks(sde, enc_e[b], 2, pad_idx, temperature=kw["temperature"], lm_sd=lm_sd if use_lm else None)
            with torch.no_grad():
                seqs, scores = core.search(int(ol_e[b]), cb, torch.device("cpu"), use_lm=use_lm)
            assert seqs.shape == r_seqs[b].shape and torch.equal(seqs, r_seqs[b]), (name, b, seqs, r_seqs[b])
            assert (scores - r_scores[b]).abs().max().item() < 1e-4, (name, b)
            gout["%s_b%d_seqs" % (name, b)], gout["%s_b%d_scores" % (name, b)] = r_seqs[b].numpy(), r_scores[b].numpy()
            n_h += seqs.size(0)
        print("transducer beam search %-9s: %d hypotheses identical to the reference (tokens and scores)" % (name, n_h))
    for k, v in lm_sd.items():
        gout["lm.sd." + k] = v.numpy()
    np.savez_compressed(os.path.join(GOLDEN, "transducer_greedy.npz"), **gout)
    print("transducer greedy decoder pinned -> tests/golden/transducer_greedy.npz")


def pin_label_smoothing():
    """label_smoothed_nll_loss + temporal_label_smoothing_prob_mask of the reference on seeded logits, for the three
    smoothing types (espresso/criterions/label_smoothed_cross_entropy_v2.py:49-120) vs oracle/ops_ref.lsce_loss."""
    from espresso.criterions.label_smoothed_cross_entropy_v2 import label_smoothed_nll_loss, temporal_label_smoothing_prob_mask

    from oracle import ops_ref as O

    rs = np.random.RandomState(4)
    B, U, V, pad, eps = 3, 7, 40, 1, 0.1
    logits = torch.from_numpy((2.0 * rs.randn(B, U, V)).astype(np.float32)).to(torch.bfloat16).float()
    target = torch.from_numpy(rs.randint(2, V, size=(B, U)))
    target[1, 5:] = pad
    target[2, 2:] = pad
    target[0, 3] = target[0, 2]  # a repeated neighbour
    counts = torch.from_numpy(rs.randint(0, 50, size=V).astype(np.float32))
    uni = (counts + 1.0) / (counts + 1.0).sum()
    out = dict(logits=logits.numpy(), target=target.numpy(), unigram=uni.numpy(), eps=np.float32(eps), pad=np.int64(pad))
    for name, mode in (("uniform", 0), ("unigram", 1), ("temporal", 2)):
        x = logits.clone().requires_grad_(True)
        lp = torch.log_softmax(x, dim=-1)
        pm = temporal_label_smoothing_prob_mask(lp, target, padding_index=pad) if name == "temporal" else None
        loss, nll = label_smoothed_nll_loss(lp.view(-1, V), target.view(-1, 1), eps, ignore_index=pad, reduce=True,
                                            smoothing_type=name, prob_mask=pm, unigram_tensor=uni[:, None])
        loss.backward()
        ol, on, og = O.lsce_loss(logits.view(-1, V).to(torch.bfloat16), V, target.view(-1).int(), pad, eps, smoothing=mode,
                                 unigram=uni, U=U)
        assert abs(ol.sum().item() - loss.item()) < 1e-4 * abs(loss.item()), (name, ol.sum().item(), loss.item())
        assert abs(on.sum().item() - nll.item()) < 1e-4 * abs(nll.item())
        assert (og.float().view(B, U, V) - x.grad).abs().max().item() < 4e-3  # bf16 gradient storage
        out["loss_" + name], out["nll_" + name], out["grad_" + name] = np.float64(loss.item()), np.float64(nll.item()), x.grad.numpy()
        print("label smoothing %-8s loss ref=%.6f oracle=%.6f" % (name, loss.item(), ol.sum().item()))
    np.savez_compressed(os.path.join(GOLDEN, "label_smoothing.npz"), **out)
    print("label smoothing pinned -> tests/golden/label_smoothing.npz")


def _table_lprobs(seed, V, step, tokens):
    """Deterministic pseudo-random log-prob rows that depend on the hypothesis prefix (same function as
    tests/test_beam_search.py::_RandomModel.lprobs)."""
    rows = tokens.shape[0]
    out = torch.empty(rows, V)
    for r in range(rows):
        h = hash((seed, step) + tuple(int(t) for t in tokens[r, : step + 1].tolist())) % (2 ** 31)
        g = torch.Generator().manual_seed(h)
        out[r] = torch.log_softmax(torch.randn(V, generator=g) * 2.0, dim=-1)
    return out


def pin_beam():
    """The REAL reference SequenceGenerator (fairseq/sequence_generator.py, Espresso's version with lm_model /
    lm_weight / eos_factor) on table-driven fake models, incl. LM shallow fusion, eos_factor, unk penalty, min_len and
    length penalty -- paths the reference's own known-answer tests do not exercise -- vs oracle/beam.generate."""
    import argparse

    from fairseq.sequence_generator import SequenceGenerator
    from tests import utils as ref_test_utils

    from oracle import beam as OB

    PAD, EOS, UNK = 1, 2, 3
    out = {}
    cases = [dict(seed=1, beam=2, bsz=3, V=9, eos_factor=None, lenpen=1.0, lm=None),
             dict(seed=2, beam=5, bsz=4, V=17, eos_factor=1.5, lenpen=1.0, lm=0.47),
             dict(seed=3, beam=3, bsz=2, V=8, eos_factor=None, lenpen=0.5, lm=0.3),
             dict(seed=4, beam=4, bsz=3, V=6, eos_factor=2.0, lenpen=1.0, lm=None),
             dict(seed=5, beam=5, bsz=5, V=40, eos_factor=1.5, lenpen=1.0, lm=1.0)]
    for ci, c in enumerate(cases):
        V, seed = c["V"], c["seed"]
        d = ref_test_utils.dummy_dictionary(vocab_size=V - 4)
        assert len(d) == V and d.pad() == PAD and d.eos() == EOS and d.unk() == UNK

        class Dec(ref_test_utils.TestIncrementalDecoder):
            def forward(self, prev_output_tokens, encoder_out=None, incremental_state=None):
                step = prev_output_tokens.size(1) - 1
                lp = _table_lprobs(seed, V, step, prev_output_tokens)
                return lp[:, None, :], {"attn": [None]}

            def get_normalized_probs(self, net_output, log_probs, _):
                return net_output[0]

        class LM:
            """FairseqLanguageModel stand-in (plain object): log-probs from a second table keyed by the prefix."""
            def __init__(self):
                self.decoder = self

            def eval(self):
                return self

            def reorder_incremental_state_scripting(self, state, order):
                pass

            def __call__(self, tokens, incremental_state=None):
                return (_table_lprobs(seed + 1000, V, tokens.size(1) - 1, tokens)[:, None, :], None)

            def get_normalized_probs(self, net_output, log_probs, sample=None):
                return net_output[0]

        args = argparse.Namespace(beam_probs=[], max_decoder_positions=40)
        model = ref_test_utils.TestModel(ref_test_utils.TestEncoder(args, d), Dec(args, d))
        kw = dict(beam_size=c["beam"], max_len_a=0.0, max_len_b=12, min_len=2, len_penalty=c["lenpen"], unk_penalty=0.3)
        gen = SequenceGenerator([model], d, lm_model=LM() if c["lm"] is not None else None,
                                lm_weight=c["lm"] if c["lm"] is not None else 1.0, eos_factor=c["eos_factor"], **kw)
        src = torch.full((c["bsz"], 7), 5, dtype=torch.long)
        src[:, -1] = EOS
        sample = {"net_input": {"src_tokens": src, "src_lengths": torch.full((c["bsz"],), 7)}}
        ref = gen.forward(sample)

        def fn(step, tokens, ro):
            lp = _table_lprobs(seed, V, step, tokens)
            if c["lm"] is not None:
                lp = lp + c["lm"] * _table_lprobs(seed + 1000, V, step, tokens)
            return lp

        ours = OB.generate(fn, c["bsz"], 7, V, PAD, UNK, EOS, model_max_len=40, eos_factor=c["eos_factor"], **kw)
        n_h = 0
        for b, (rh, oh) in enumerate(zip(ref, ours)):
            assert len(rh) == len(oh), (ci, b, len(rh), len(oh))
            for k, (r_, o_) in enumerate(zip(rh, oh)):
                assert r_["tokens"].tolist() == o_["tokens"].tolist(), (ci, b, k)
                assert abs(float(r_["score"]) - float(o_["score"])) < 1e-5
                out["c%d_b%d_k%d_tokens" % (ci, b, k)] = r_["tokens"].numpy()
                out["c%d_b%d_k%d_score" % (ci, b, k)] = np.float32(float(r_["score"]))
                n_h += 1
            out["c%d_b%d_n" % (ci, b)] = np.int64(len(rh))
        print("beam case %d (beam %d, V %d, lm %s, eos_factor %s): %d hypotheses identical" % (ci, c["beam"], V, c["lm"], c["eos_factor"], n_h))
    out["cases"] = np.array([[c["seed"], c["beam"], c["bsz"], c["V"], -1.0 if c["eos_factor"] is None else c["eos_factor"], c["lenpen"],
                              -1.0 if c["lm"] is None else c["lm"]] for c in cases], dtype=np.float64)
    np.savez_compressed(os.path.join(GOLDEN, "beam_reference.npz"), **out)
    print("beam search pinned -> tests/golden/beam_reference.npz")


def pin_optimizer():
    """fairseq's Adam (fairseq/optim/adam.py:110-239, decoupled weight decay, bias-corrected step) after
    fairseq.utils.clip_grad_norm_ (fairseq/utils.py:347-397) and the division by sample_size that
    Trainer.train_step applies (fairseq/trainer.py:950-975), over several updates, vs oracle/ops_ref.adam_step on flat
    buffers; plus the noam / tri_stage learning-rate schedules of the reference at a spread of update counts."""
    from argparse import Namespace

    from fairseq.optim.adam import Adam
    from fairseq.utils import clip_grad_norm_

    from oracle import ops_ref as O

    g = torch.Generator().manual_seed(9)
    shapes = [(7, 5), (13,), (4, 3, 2)]
    params = [torch.nn.Parameter(torch.randn(*s_, generator=g)) for s_ in shapes]
    n = sum(p_.numel() for p_ in params)
    lr, betas, eps, wd, clip = 3e-3, (0.9, 0.98), 1e-8, 0.01, 0.5
    opt = Adam(params, lr=lr, betas=betas, eps=eps, weight_decay=wd)
    p32 = torch.cat([p_.detach().reshape(-1) for p_ in params]).clone()
    m, v = torch.zeros(n), torch.zeros(n)
    p16 = p32.to(torch.bfloat16)
    out = {"p0": p32.numpy().copy()}
    for step in range(1, 5):
        grads = [torch.randn(*s_, generator=g) * (3.0 if step == 2 else 0.2) for s_ in shapes]
        sample_size = float(2 + step)
        flat_g = torch.cat([x.reshape(-1) for x in grads]).clone()
        for p_, gr in zip(params, grads):
            p_.grad = gr / sample_size                      # multiply_grads(1 / sample_size)
        gnorm = clip_grad_norm_(params, clip)
        opt.step()
        sumsq = (flat_g * flat_g).sum().reshape(1)
        gn_out = torch.zeros(1)
        O.adam_step(p32, m, v, flat_g, p16, lr, betas[0], betas[1], eps, wd, step, sumsq, denom_const=sample_size,
                    clip_norm=clip, gnorm_out=gn_out)
        ref_flat = torch.cat([p_.detach().reshape(-1) for p_ in params])
        assert abs(gn_out.item() - gnorm.item()) < 1e-5 * gnorm.item(), (gn_out.item(), gnorm.item())
        assert (ref_flat - p32).abs().max().item() < 1e-6, (step, (ref_flat - p32).abs().max().item())
        out["g%d" % step], out["ss%d" % step], out["p%d" % step], out["gnorm%d" % step] = (
            flat_g.numpy(), np.float64(sample_size), ref_flat.numpy().copy(), np.float64(gnorm.item()))
    out["hyper"] = np.array([lr, betas[0], betas[1], eps, wd, clip])
    print("optimizer: 4 clipped AdamW-style updates identical to fairseq's Adam (max diff < 1e-6)")

    # ---- learning-rate schedules
    from espresso.optim.lr_scheduler.noam_lr_scheduler import NoamLRScheduler
    from fairseq.optim.lr_scheduler.tri_stage_lr_scheduler import TriStageLRSchedule

    from espresso_b200.optim import NoamLRScheduler as OurNoam
    from espresso_b200.optim import TriStageLRScheduler as OurTri

    steps = [0, 1, 10, 99, 100, 101, 5000, 24999, 25000, 25001, 100000]
    ref = NoamLRScheduler.__new__(NoamLRScheduler)
    ref.cfg, ref.optimizer, ref.best = None, Namespace(set_lr=lambda x: None, get_lr=lambda: 0.0), None
    ref.factor, ref.warmup_steps, ref.model_size, ref.final_lr = 5.0, 25000, 512, 1e-6
    ours = OurNoam(5.0, 25000, 512, 1e-6)
    noam = []
    for s_ in steps:
        a, b = ref.step_update(s_), ours.step_update(s_)
        assert abs(a - b) <= 1e-12 * max(abs(a), 1e-12), (s_, a, b)
        noam.append(a)
    tcfg = Namespace(lr=[5e-4], init_lr_scale=0.01, final_lr_scale=0.05, phase_ratio=None, warmup_steps=100, hold_steps=200,
                     decay_steps=300, max_update=0)
    # run the reference constructor body without its FairseqOptimizer type check
    import fairseq.optim.lr_scheduler.fairseq_lr_scheduler as _fl
    _orig = _fl.FairseqLRScheduler.__init__
    _fl.FairseqLRScheduler.__init__ = lambda self, cfg, optimizer: (setattr(self, "cfg", cfg), setattr(self, "optimizer", optimizer),
                                                                    setattr(self, "best", None)) and None
    try:
        tref = TriStageLRSchedule(tcfg, Namespace(set_lr=lambda x: None, get_lr=lambda: 0.0))
    finally:
        _fl.FairseqLRScheduler.__init__ = _orig
    tours = OurTri(5e-4, 100, 200, 300, init_lr_scale=0.01, final_lr_scale=0.05)
    tsteps = [0, 1, 50, 99, 100, 150, 299, 300, 301, 450, 599, 600, 601, 5000]
    tri = []
    for s_ in tsteps:
        a, b = tref.step_update(s_), tours.step_update(s_)
        assert abs(a - b) <= 1e-12 * max(abs(a), 1e-12), (s_, a, b)
        tri.append(a)
    out.update(noam_steps=np.array(steps), noam_lr=np.array(noam), tri_steps=np.array(tsteps), tri_lr=np.array(tri))
    print("lr schedules: noam and tri_stage identical to the reference at %d + %d update counts" % (len(steps), len(tsteps)))
    np.savez_compressed(os.path.join(GOLDEN, "optimizer.npz"), **out)
    print("optimizer + schedules pinned -> tests/golden/optimizer.npz")


def pin_lr_schedules_v2():
    """The schedules of the speech_lstm recipes -- reduce_lr_on_plateau_v2 (espresso/optim/lr_scheduler/
    reduce_lr_on_plateau_v2.py over fairseq's reduce_lr_on_plateau and torch's ReduceLROnPlateau) and polynomial_decay_v2 --
    run with the REAL reference classes on recorded validation curves / update counts; espresso_b200.optim must replay them."""
    from argparse import Namespace

    import fairseq.optim.lr_scheduler.fairseq_lr_scheduler as _fl
    from espresso.optim.lr_scheduler.polynomial_decay_schedule import PolynomialDecayV2LRSchedule
    from espresso.optim.lr_scheduler.reduce_lr_on_plateau_v2 import ReduceLROnPlateauLRScheduleV2

    from espresso_b200.optim.lr_scheduler import PolynomialDecayV2LRScheduler, ReduceLROnPlateauV2LRScheduler

    class _Opt:  # what the schedules need from a FairseqOptimizer: one param group with an lr
        def __init__(self, lr):
            self.optimizer = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=lr)

        def set_lr(self, lr):
            for gp in self.optimizer.param_groups:
                gp["lr"] = lr

        def get_lr(self):
            return self.optimizer.param_groups[0]["lr"]

    _orig = _fl.FairseqLRScheduler.__init__
    _fl.FairseqLRScheduler.__init__ = lambda self, cfg, optimizer: (setattr(self, "cfg", cfg), setattr(self, "optimizer", optimizer),
                                                                    setattr(self, "best", None)) and None
    out = {}
    try:
        rs = np.random.RandomState(4)
        cases = [dict(lr=1e-3, lr_shrink=0.5, lr_threshold=1e-4, lr_patience=0, warmup_updates=0, warmup_init_lr=-1.0,
                      start_reduce_lr_epoch=4, final_lr_scale=0.01, maximize_best_checkpoint_metric=False),
                 dict(lr=2e-3, lr_shrink=0.1, lr_threshold=1e-2, lr_patience=1, warmup_updates=50, warmup_init_lr=1e-5,
                      start_reduce_lr_epoch=0, final_lr_scale=0.05, maximize_best_checkpoint_metric=True),
                 dict(lr=5e-4, lr_shrink=0.5, lr_threshold=1e-4, lr_patience=0, warmup_updates=0, warmup_init_lr=-1.0,
                      start_reduce_lr_epoch=11, final_lr_scale=1e-4, maximize_best_checkpoint_metric=False)]  # asr_wsj run.sh
        for ci, c in enumerate(cases):
            cfg = Namespace(lr=[c["lr"]], **{k: v for k, v in c.items() if k != "lr"})
            ref = ReduceLROnPlateauLRScheduleV2(cfg, _Opt(c["lr"]))
            ours = ReduceLROnPlateauV2LRScheduler(**c)
            E = 30
            base = np.linspace(5.0, 3.0, E) if not c["maximize_best_checkpoint_metric"] else np.linspace(0.5, 0.8, E)
            vals = base + rs.randn(E) * 0.05
            vals[12:18] = vals[12]  # a plateau
            lrs, n = [], 0
            for ep in range(1, E + 1):
                for _ in range(20):  # updates of the epoch
                    n += 1
                    a, b = ref.step_update(n), ours.step_update(n)
                    assert abs(a - b) <= 1e-12 * max(abs(a), 1e-12), (ci, ep, n, a, b)
                a, b = ref.step(ep, float(vals[ep - 1])), ours.step(ep, float(vals[ep - 1]))
                assert abs(a - b) <= 1e-12 * max(abs(a), 1e-12), (ci, ep, a, b)
                lrs.append(a)
            sd = ref.state_dict()
            assert abs(sd["best"] - ours.state_dict()["best"]) < 1e-12 and sd["last_epoch"] == ours.state_dict()["last_epoch"]
            out["plateau%d_cfg" % ci] = np.array([c["lr"], c["lr_shrink"], c["lr_threshold"], c["lr_patience"], c["warmup_updates"],
                                                  c["warmup_init_lr"], c["start_reduce_lr_epoch"], c["final_lr_scale"],
                                                  float(c["maximize_best_checkpoint_metric"])])
            out["plateau%d_vals" % ci] = vals
            out["plateau%d_lr" % ci] = np.array(lrs)
            print("reduce_lr_on_plateau_v2 case %d: %d distinct rates over %d epochs, identical to the reference" % (ci, len(set(lrs)), E))
        pcfg = Namespace(lr=[3e-4], warmup_updates=100, end_learning_rate=1e-6, total_num_update=2000, power=2.0, force_anneal=None)
        pref = PolynomialDecayV2LRSchedule(pcfg, _Opt(3e-4))
        pours = PolynomialDecayV2LRScheduler(3e-4, 2000, warmup_updates=100, end_learning_rate=1e-6, power=2.0)
        psteps = [0, 1, 50, 100, 101, 500, 1999, 2000, 2001, 9999]
        plr = []
        for s_ in psteps:
            a, b = pref.step_update(s_), pours.step_update(s_)
            assert abs(a - b) <= 1e-12 * max(abs(a), 1e-12), (s_, a, b)
            plr.append(a)
        out.update(poly_steps=np.array(psteps), poly_lr=np.array(plr))
        print("polynomial_decay_v2: identical to the reference at %d update counts" % len(psteps))
    finally:
        _fl.FairseqLRScheduler.__init__ = _orig
    np.savez_compressed(os.path.join(GOLDEN, "lr_schedules_v2.npz"), **out)
    print("schedules pinned -> tests/golden/lr_schedules_v2.npz")


def pin_wer_scorer():
    """espresso/tools/wer.py Scorer (+ edit_distance / aligned_print of espresso/tools/utils.py) on random token strings with
    non-linguistic symbols and a word filter file: edit counts, rates and the printed blocks, recorded for
    espresso_b200.tools.wer.Scorer (tests/golden/wer_scorer.json)."""
    import json
    import tempfile

    from espresso.tools.wer import Scorer as RefScorer

    from espresso_b200.tools.wer import Scorer as OurScorer

    class _D:
        non_lang_syms = ["<noise>", "<laugh>"]

        @staticmethod
        def wordpiece_decode(x):
            return x.replace(" ", "").replace("\u2581", " ").strip()

    rs = np.random.RandomState(17)
    pieces = ["\u2581the", "\u2581a", "\u2581cat", "\u2581sat", "s", "ing", "\u2581on", "\u2581mat", "ter", "\u2581uh", "\u2581um", "\u2581it's",
              "\u2581dog", "\u2581ran", "<noise>", "<laugh>", "\u2581far", "ther", "\u2581", "\u2581x"]
    filt = tempfile.NamedTemporaryFile("w", suffix=".filt", delete=False, encoding="utf-8")
    filt.write("#!/bin/sed -f\ns/\\buh\\b//g\ns:\\bum\\b::g\nthis line is ignored\n")
    filt.close()
    ref, ours = RefScorer(_D(), wer_output_filter=filt.name), OurScorer(_D(), wer_output_filter=filt.name)
    utts = []
    for u in range(60):
        n = int(rs.randint(0, 14))
        r = [pieces[i] for i in rs.randint(0, len(pieces), size=n)]
        h = list(r)
        for _ in range(int(rs.randint(0, 5))):  # corrupt: substitute / insert / delete
            k = rs.randint(0, 3)
            if k == 0 and h:
                h[int(rs.randint(0, len(h)))] = pieces[int(rs.randint(0, len(pieces)))]
            elif k == 1:
                h.insert(int(rs.randint(0, len(h) + 1)), pieces[int(rs.randint(0, len(pieces)))])
            elif h:
                del h[int(rs.randint(0, len(h)))]
        uid = "utt%03d" % u
        rstr, hstr = " ".join(r), " ".join(h)
        for sc in (ref, ours):
            sc.add_prediction(uid, hstr)
            sc.add_evaluation(uid, rstr, hstr)
        utts.append([uid, rstr, hstr])
    order = [u[0] for u in utts][::-1]
    for sc in (ref, ours):
        sc.add_ordered_utt_list(order)
    exp = {"utts": utts, "order": order, "filter": open(filt.name, encoding="utf-8").read(),
           "char_counter": dict(ref.char_counter), "word_counter": dict(ref.word_counter), "cer": list(ref.cer()), "wer": list(ref.wer()),
           "print_char_results": ref.print_char_results(), "print_results": ref.print_results(),
           "print_aligned_results": ref.print_aligned_results()}
    assert dict(ours.char_counter) == exp["char_counter"] and dict(ours.word_counter) == exp["word_counter"]
    assert list(ours.cer()) == exp["cer"] and list(ours.wer()) == exp["wer"]
    assert ours.print_char_results() == exp["print_char_results"] and ours.print_results() == exp["print_results"]
    assert ours.print_aligned_results() == exp["print_aligned_results"]
    assert ours.tot_word_error() == ref.tot_word_error() and ours.tot_char_count() == ref.tot_char_count()
    os.unlink(filt.name)
    with open(os.path.join(GOLDEN, "wer_scorer.json"), "w", encoding="utf-8") as f:
        json.dump(exp, f, ensure_ascii=False, indent=0)
    print("wer scorer: %d utterances, WER %.2f%% CER %.2f%%, counters / rates / printed blocks identical to the reference -> tests/golden/wer_scorer.json"
          % (len(utts), exp["wer"][0], exp["cer"][0]))


def pin_global_cmvn():
    """Global CMVN statistics as espresso/tools/compute_global_cmvn_stats.py computes them: the reference's fbank per utterance
    (get_torchaudio_fbank_or_mfcc) and its pooling of per-utterance sums / unnormalised variances (:93-116, restated here
    because the script's own main() reads files through libsndfile); the seeds of the synthetic int16 utterances are
    stored so the test regenerates them."""
    from espresso.tools.utils import get_torchaudio_fbank_or_mfcc

    from oracle import frontend as OF

    durs = [1.3, 0.03, 4.0, 2.25, 0.6, 7.1]
    total_sum, total_var, total_frames = np.zeros(80), np.zeros(80), 0
    for i, dsec in enumerate(durs):
        w = OF.synth_waveform(300 + i, dsec)
        feat = get_torchaudio_fbank_or_mfcc(w[None, :], 16000, n_bins=80)
        if feat.shape[0] == 0:
            continue
        cur_sum, cur_frames = feat.sum(axis=0), feat.shape[0]
        cur_var = np.var(feat, axis=0) * cur_frames
        if total_frames > 0:
            ratio = total_frames / cur_frames
            total_var = total_var + cur_var + ratio / (total_frames + cur_frames) * (total_sum / ratio - cur_sum) ** 2
        else:
            total_var = cur_var
        total_sum, total_frames = total_sum + cur_sum, total_frames + cur_frames
    np.savez_compressed(os.path.join(GOLDEN, "global_cmvn.npz"), durs=np.array(durs), seed0=np.int64(300),
                        mean=total_sum / total_frames, std=np.sqrt(total_var / total_frames), frames=np.int64(total_frames))
    print("global CMVN: %d frames of %d utterances pinned -> tests/golden/global_cmvn.npz" % (total_frames, len(durs)))


def pin_batching():
    """The reference's native batch packer (fairseq/data/data_utils_fast.pyx, compiled from /root/reference into
    oracle/_ref/ by oracle/build_ref.sh) vs espresso_b200.data.batching.batch_by_size (esp_batch_by_size in the C ABI)
    on random size lists, max_tokens / max_sentences / batch-size multiples incl. the tail-overflow corner."""
    import subprocess
    import sys as _sys

    ref_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
    subprocess.check_call(["bash", os.path.join(os.path.dirname(os.path.abspath(__file__)), "build_ref.sh")])
    _sys.path.insert(0, ref_dir)
    import data_utils_fast as R

    from espresso_b200.data import batching as Bt

    rs = np.random.RandomState(21)
    out, n_cases = {}, 0
    for trial in range(400):
        n = int(rs.randint(1, 120))
        sizes = rs.randint(1, 400, size=n).astype(np.int64)
        order = np.argsort(sizes, kind="mergesort").astype(np.int64) if rs.rand() < 0.7 else rs.permutation(n).astype(np.int64)
        mt = int(rs.choice([0, 400, 1000, 4000]))
        ms = int(rs.choice([0, 1, 5, 24]))
        mult = int(rs.choice([1, 1, 8, 4, 3]))
        if mt and sizes.max() > mt:
            mt = int(sizes.max())
        ref = R.batch_by_size_vec(order, sizes[order], mt if mt else -1, ms if ms else -1, mult)
        got = Bt.batch_by_size(order, sizes, mt or None, ms or None, mult)
        assert len(ref) == len(got) and all(np.array_equal(a, b) for a, b in zip(ref, got)), (trial, mt, ms, mult)
        if trial < 60:  # a committed subset for hosts without /root/reference
            out["c%d_sizes" % n_cases], out["c%d_order" % n_cases] = sizes, order
            out["c%d_cfg" % n_cases] = np.array([mt, ms, mult], dtype=np.int64)
            out["c%d_ends" % n_cases] = np.cumsum([len(b) for b in ref]).astype(np.int64)
            n_cases += 1
    out["n_cases"] = np.int64(n_cases)
    np.savez_compressed(os.path.join(GOLDEN, "batching.npz"), **out)
    print("batching: 400 random cases identical to the reference's compiled Cython packer; %d cases -> tests/golden/batching.npz" % n_cases)
    # 100 cases at the recipe's limits (3000 frames, 24 sentences); the test redraws the inputs from the same seed
    rs, ends = np.random.RandomState(3), {}
    for c in range(100):
        n = int(rs.randint(1, 200))
        sizes = rs.randint(1, 300, size=n).astype(np.int64)
        order = rs.permutation(n).astype(np.int64)
        mult = int(rs.choice([1, 8]))
        ends["c%d_ends" % c] = np.cumsum([len(b) for b in R.batch_by_size_vec(order, sizes[order], 3000, 24, mult)]).astype(np.int64)
    np.savez_compressed(os.path.join(GOLDEN, "batching_seeded.npz"), **ends)
    print("batching: 100 seeded cases at max_tokens 3000 / max_sentences 24 -> tests/golden/batching_seeded.npz")


def pin_collate():
    """espresso.data.asr_dataset.collate (the reference's batch assembly) vs espresso_b200.data.collate.collate on random
    samples with distinct source lengths (torch.sort is not stable, so ties are outside the contract)."""
    from espresso.data.asr_dataset import collate as ref_collate

    from espresso_b200.data.collate import collate as our_collate

    rs = np.random.RandomState(17)
    n_checked = 0
    gold = {}
    for trial in range(20):
        B = int(rs.randint(1, 9))
        lens = rs.choice(np.arange(5, 60), size=B, replace=False)
        samples = []
        for i in range(B):
            u = int(rs.randint(1, 8))
            tgt = torch.cat([torch.from_numpy(rs.randint(4, 50, size=u)), torch.tensor([2])]).long()
            samples.append({"id": int(rs.randint(0, 1000)), "utt_id": "utt%d" % i, "source": torch.from_numpy(rs.randn(int(lens[i]), 80).astype(np.float32)),
                            "target": tgt, "text": "t%d" % i})
        for bos in (None, 0):
            for mult in (1, 8):
                a = ref_collate(samples, pad_idx=1, eos_idx=2, left_pad_source=False, left_pad_target=False, input_feeding=True,
                                maybe_bos_idx=bos, pad_to_multiple=mult)
                b = our_collate(samples, pad_idx=1, eos_idx=2, maybe_bos_idx=bos, pad_to_multiple=mult)
                assert torch.equal(a["id"], b["id"]) and a["utt_id"] == b["utt_id"] and a["text"] == b["text"]
                assert a["nsentences"] == b["nsentences"] and a["ntokens"] == b["ntokens"]
                for k in ("src_tokens", "src_lengths", "prev_output_tokens"):
                    assert torch.equal(a["net_input"][k], b["net_input"][k]), (k, trial)
                    assert a["net_input"][k].dtype == b["net_input"][k].dtype, k
                assert torch.equal(a["target"], b["target"])
                n_checked += 1
                if trial < 3 and mult == 1:  # small committed cases (feature width cut to 4 to keep the file tiny)
                    key = "c%d_bos%d_" % (trial, -1 if bos is None else bos)
                    gold[key + "lens"] = np.array([s_["source"].size(0) for s_ in samples])
                    gold[key + "ids"] = np.array([s_["id"] for s_ in samples])
                    for j, s_ in enumerate(samples):
                        gold[key + "tgt%d" % j] = s_["target"].numpy()
                    gold[key + "out_id"], gold[key + "out_src_lengths"] = a["id"].numpy(), a["net_input"]["src_lengths"].numpy()
                    gold[key + "out_target"], gold[key + "out_prev"] = a["target"].numpy(), a["net_input"]["prev_output_tokens"].numpy()
                    gold[key + "ntokens"] = np.int64(a["ntokens"])
    np.savez_compressed(os.path.join(GOLDEN, "collate.npz"), **gold)
    print("collate: %d batches identical to espresso.data.asr_dataset.collate -> tests/golden/collate.npz" % n_checked)


def pin_sharding():
    """fairseq.data.iterators.ShardedIterator (rank r takes batches r, r+W, ...; the tail is filled so every rank gets
    the same count) vs espresso_b200.data.batching.shard_batches; AsrDataset.ordered_indices' double stable sort
    (espresso/data/asr_dataset.py:392-408) vs batching.ordered_indices."""
    from fairseq.data.iterators import ShardedIterator

    from espresso_b200.data import batching as Bt

    rs = np.random.RandomState(5)
    for n in (0, 1, 7, 8, 9, 31):
        batches = [rs.randint(0, 100, size=rs.randint(1, 5)).tolist() for _ in range(n)]
        for W in (1, 2, 4, 8):
            for r in range(W):
                ref = list(ShardedIterator(batches, W, r, fill_value=[]))
                ours = Bt.shard_batches(batches, W, r, fill_value=[])
                assert ref == ours, (n, W, r)
    for _ in range(20):
        n = int(rs.randint(1, 200))
        src, tgt = rs.randint(1, 50, size=n), rs.randint(1, 10, size=n)
        seed = int(rs.randint(0, 10000))
        np.random.seed(seed)
        idx = np.random.permutation(n)
        idx = idx[np.argsort(tgt[idx], kind="mergesort")]
        ref = idx[np.argsort(src[idx], kind="mergesort")]           # asr_dataset.py:392-408 with shuffle=True
        assert np.array_equal(ref, Bt.ordered_indices(src, tgt, shuffle_seed=seed))
    print("sharding: ShardedIterator and ordered_indices semantics reproduced")


def pin_dictionary():
    """espresso.data.asr_dictionary.AsrDictionary (load with / without <s>, index order, counts, string(), encode_line)
    vs espresso_b200.data.asr_dictionary.AsrDictionary on a temporary vocabulary file."""
    import tempfile

    from espresso.data.asr_dictionary import AsrDictionary as Ref

    from espresso_b200.data.asr_dictionary import AsrDictionary as Ours

    words = ["\u2581the", "\u2581a", "s", "ing", "<space>", "\u2581speech", "@@x", "q|", "'"]
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "dict.txt")
        with open(path, "w", encoding="utf-8") as f:
            for i, w in enumerate(words):
                f.write("%s %d\n" % (w, 100 - 7 * i))
        for enable_bos in (False, True):
            a, b = Ref.load(path, enable_bos=enable_bos), Ours.load(path, enable_bos=enable_bos)
            assert len(a) == len(b) and a.symbols == b.symbols and a.count == b.count and a.indices == b.indices
            assert (a.pad(), a.eos(), a.unk(), a.space(), a.nspecial) == (b.pad(), b.eos(), b.unk(), b.space(), b.nspecial)
            if enable_bos:
                assert a.bos() == b.bos() == 0
            ids = torch.tensor([a.index(w) for w in ["\u2581the", "s", "zzz", "\u2581speech", "ing"]] + [a.eos()])
            for kw in (dict(), dict(bpe_symbol="sentencepiece"), dict(escape_unk=True), dict(include_eos=True),
                       dict(extra_symbols_to_ignore={a.pad()}), dict(bpe_symbol="@@ ")):
                assert a.string(ids, **kw) == b.string(ids, **kw), kw
            assert a.string(torch.stack([ids, ids])) == b.string(torch.stack([ids, ids]))
            line = "\u2581the s zzz ing"
            assert a.encode_line(line, add_if_not_exist=False).tolist() == b.encode_line(line, add_if_not_exist=False).tolist()
            assert a.encode_line(line, add_if_not_exist=False, append_eos=False).tolist() == b.encode_line(line, append_eos=False).tolist()
    print("dictionary: AsrDictionary layout, string() and encode_line identical to the reference")


def pin_speech_lstm():
    """The reference `speech_lstm` model (espresso/models/speech_lstm.py; BASELINE configs[0] family: conv front, BiLSTM
    encoder, attention LSTM decoder with input feeding and residuals) + label_smoothed_nll_loss: teacher-forced logits,
    loss and every parameter gradient -> tests/golden/speech_lstm.npz for espresso_b200.models.SpeechLSTMModel."""
    from argparse import Namespace

    from espresso.criterions.label_smoothed_cross_entropy_v2 import label_smoothed_nll_loss
    from espresso.models.speech_lstm import SpeechLSTMModel

    V, pad_idx, eos_idx = 50, 1, 2

    class _Dict:
        def __len__(self):
            return V

        def pad(self):
            return pad_idx

        def eos(self):
            return eos_idx

    class _Task:
        feat_dim, feat_in_channels, target_dictionary = 80, 1, _Dict()
        cfg = Namespace(num_batch_buckets=0)

    args = Namespace(
        dropout=0.0, encoder_conv_channels="[64, 64, 128, 128]", encoder_conv_kernel_sizes="[(3, 3), (3, 3), (3, 3), (3, 3)]",
        encoder_conv_strides="[(1, 1), (2, 2), (1, 1), (2, 2)]", encoder_rnn_hidden_size=32, encoder_rnn_layers=2,
        encoder_rnn_bidirectional=True, encoder_rnn_residual=True, encoder_multilayer_rnn_as_single_module=False,
        decoder_embed_path=None, decoder_embed_dim=24, decoder_freeze_embed=False, decoder_hidden_size=32, decoder_layers=2,
        decoder_out_embed_dim=40, decoder_rnn_residual=True, attention_type="bahdanau", attention_dim=16, need_attention=False,
        adaptive_softmax_cutoff=None, share_decoder_input_output_embed=False, pretrained_lm_checkpoint=None,
        encoder_rnn_dropout_in=0.0, encoder_rnn_dropout_out=0.0, decoder_dropout_in=0.0, decoder_dropout_out=0.0,
        scheduled_sampling_probs=[1.0], start_scheduled_sampling_epoch=1, criterion_name="label_smoothed_cross_entropy_v2",
        max_source_positions=3600, max_target_positions=200)
    torch.manual_seed(11)
    m = SpeechLSTMModel.build_model(args, _Task())
    g = torch.Generator().manual_seed(12)
    with torch.no_grad():
        for n, p_ in m.named_parameters():
            if p_.dim() == 1:
                p_.add_(0.1 * torch.randn(p_.shape, generator=g))
    rs = np.random.RandomState(19)
    B, T = 3, 61
    lens = torch.tensor([61, 50, 37])
    feats = torch.from_numpy(rs.randn(B, T, 80).astype(np.float32))
    for b in range(B):
        feats[b, lens[b]:] = 0.0
    U = 6
    tgt = torch.full((B, U + 1), pad_idx, dtype=torch.long)
    prev = torch.full((B, U + 1), pad_idx, dtype=torch.long)
    for b, u in enumerate((6, 4, 2)):
        toks = torch.from_numpy(rs.randint(4, V, size=u))
        tgt[b, :u], tgt[b, u] = toks, eos_idx
        prev[b, 0], prev[b, 1:u + 1] = eos_idx, toks
    out = {"sd." + k: v.clone().numpy() for k, v in m.state_dict().items()}
    m.train()
    m.zero_grad()
    logits, _ = m(feats, lens, prev)
    lp = torch.log_softmax(logits.float(), dim=-1)
    loss, nll = label_smoothed_nll_loss(lp.view(-1, V), tgt.view(-1, 1), 0.1, ignore_index=pad_idx, reduce=True)
    loss.backward()
    out.update({"grad." + n: p_.grad.numpy() for n, p_ in m.named_parameters()})
    for k, v in m.state_dict().items():
        if "running_" in k:
            out["after." + k] = v.numpy()
    out.update(feats=feats.numpy(), lens=lens.numpy(), target=tgt.numpy(), prev_output_tokens=prev.numpy(),
               logits=logits.detach().numpy(), loss=np.float64(loss.item()), nll=np.float64(nll.item()))
    np.savez_compressed(os.path.join(GOLDEN, "speech_lstm.npz"), **out)
    print("speech_lstm: loss %.6f, %d parameters -> tests/golden/speech_lstm.npz" % (loss.item(), sum(p_.numel() for p_ in m.parameters())))


def pin_lstm_lm():
    """The reference LSTM language model (espresso/models/lstm_lm.py, the LM the LibriSpeech recipe fuses): teacher-forced
    logits with residual layers, additional_fc and shared / separate output embeddings -> tests/golden/lstm_lm.npz."""
    from argparse import Namespace

    from espresso.models.lstm_lm import LSTMLanguageModelEspresso

    V = 50

    class _Dict:
        def __len__(self):
            return V

        def pad(self):
            return 1

        def eos(self):
            return 2

    class _Task:
        source_dictionary = target_dictionary = _Dict()

    out = {}
    for name, kw in (("shared", dict(decoder_embed_dim=32, decoder_hidden_size=32, decoder_out_embed_dim=32, share_embed=True,
                                     decoder_rnn_residual=True)),
                     ("proj", dict(decoder_embed_dim=24, decoder_hidden_size=32, decoder_out_embed_dim=40, share_embed=False,
                                   decoder_rnn_residual=False))):
        args = Namespace(dropout=0.0, decoder_embed_path=None, decoder_freeze_embed=False, decoder_layers=2,
                         adaptive_softmax_cutoff=None, is_wordlm=False, decoder_dropout_in=0.0, decoder_dropout_out=0.0,
                         criterion_name="cross_entropy", max_target_positions=64, tokens_per_sample=64, **kw)
        torch.manual_seed(31)
        m = LSTMLanguageModelEspresso.build_model(args, _Task())
        m.eval()
        rs = np.random.RandomState(8)
        toks = torch.from_numpy(rs.randint(2, V, size=(3, 9)))
        with torch.no_grad():
            logits = m(toks)[0]
        for k, v in m.state_dict().items():
            out["%s.sd.%s" % (name, k)] = v.numpy()
        out[name + ".tokens"], out[name + ".logits"] = toks.numpy(), logits.numpy()
        print("lstm_lm %-6s: logits %s, %d parameters" % (name, tuple(logits.shape), sum(p_.numel() for p_ in m.parameters())))
    np.savez_compressed(os.path.join(GOLDEN, "lstm_lm.npz"), **out)
    print("lstm_lm pinned -> tests/golden/lstm_lm.npz")


def pin_text():
    """Character tokenisation (espresso/tools/utils.py:36-58, espresso/data/encoders/characters_asr.py) and the word /
    character error counting behind validation WER (espresso/tools/utils.py:265-330 edit_distance) vs
    espresso_b200.data.encoders / espresso_b200.tasks.speech_recognition.edit_counts."""
    from espresso.data.encoders.characters_asr import CharactersAsr as RefChars
    from espresso.tools.utils import edit_distance

    from espresso_b200.data.encoders import CharactersAsr
    from espresso_b200.tasks.speech_recognition import edit_counts

    nls = ["<noise>", "[laughter]", "<unk>"]
    sents = ["hello  world", " a <noise> b[laughter]c ", "", "x", "<noise><noise> y  z ", "it's <unk> o'clock"]
    for ends in (True, False):
        for syms in (None, [], nls):
            a, b = RefChars(None, ends_with_space=ends, non_lang_syms=syms), CharactersAsr(ends_with_space=ends, non_lang_syms=syms)
            for s_ in sents:
                assert a.encode(s_) == b.encode(s_), (s_, a.encode(s_), b.encode(s_))
                assert a.decode(a.encode(s_)) == b.decode(b.encode(s_))
    rs = np.random.RandomState(2)
    vocab = ["a", "b", "c", "dd", "e"]
    for _ in range(200):
        ref = [vocab[i] for i in rs.randint(0, 5, size=rs.randint(0, 12))]
        hyp = [vocab[i] for i in rs.randint(0, 5, size=rs.randint(0, 12))]
        _, _, counter = edit_distance(ref, hyp)
        assert edit_counts(ref, hyp) == (counter["sub"] + counter["ins"] + counter["del"], counter["words"]), (ref, hyp)
    print("text: characters_asr encode/decode and edit-distance error counts identical to the reference")


from oracle.fullsize import (FULLSIZE_CFG, FULLSIZE_GRADS, FULLSIZE_GRADS_SUB, fullsize_cotangent,  # noqa: E402
                             fullsize_inputs)


def pin_streaming():
    """Chunk-streaming / limited-context self-attention.  (1) espresso_b200.tools.utils.chunk_streaming_bounds and
    context_bounds against the reference's chunk_streaming_mask (espresso/tools/utils.py:131-194) and get_attn_mask
    (speech_transformer_encoder.py:226-263) over a grid, same numpy seeds; (2) the reference encoder model with
    chunk_size > 0 (train at two num_updates -> both coin outcomes, and eval) against oracle/conformer.py with the mask,
    stored as tests/golden/encoder_streaming.npz for the GPU parity test."""
    import types

    import torch.nn.functional as F
    from espresso.models.transformer.speech_transformer_encoder import SpeechTransformerEncoder
    from espresso.tools import utils as RU
    from fairseq.data import data_utils

    from espresso_b200.tools.utils import bounds_to_mask, chunk_streaming_bounds, context_bounds
    from oracle import conformer as O

    n = 0
    for max_len in (1, 2, 7, 18, 37, 64, 131):
        for chunk in (1, 4, 18, 40):
            for lw, rw in ((0, 0), (1, 0), (2, 1), (0, 3), (100, 100)):
                for partial_last in (True, False):
                    for seed in range(4):
                        with data_utils.numpy_seed(seed):
                            ref = RU.chunk_streaming_mask(torch.tensor([max_len, max(max_len // 2, 1)]), chunk, left_window=lw,
                                                          right_window=rw, always_partial_in_last=partial_last).numpy()
                        with data_utils.numpy_seed(seed):
                            lo, hi = chunk_streaming_bounds(max_len, chunk, lw, rw, always_partial_in_last=partial_last)
                        assert np.array_equal(bounds_to_mask(lo, hi), ref), (max_len, chunk, lw, rw, partial_last, seed)
                        n += 1
    class _Lengths(torch.Tensor):
        """speech_transformer_encoder.py:255 calls `in_lengths.ones(...)`, which torch.Tensor does not have (the
        reference raises AttributeError there, so `transformer_context` is dead upstream); supplying the evidently
        intended new_ones lets the rest of the reference's band-mask expression run unmodified."""
        def ones(self, *a, **k):
            return torch.ones(*a, **k)

    for max_len in (1, 5, 33):
        for ctx in ((None, 0), (0, None), (3, 2), (0, 0), (40, 1), (2, 50)):
            fake = types.SimpleNamespace(cfg=types.SimpleNamespace(encoder=types.SimpleNamespace(chunk_size=0)),
                                         transformer_context=ctx)
            ref = SpeechTransformerEncoder.get_attn_mask(fake, torch.tensor([max_len, 1]).as_subclass(_Lengths)).numpy()   # True = hidden
            lo, hi = context_bounds(max_len, *ctx)
            assert np.array_equal(~bounds_to_mask(lo, hi), ref), (max_len, ctx)
            n += 1
    print("streaming masks: %d reference masks reproduced as key ranges" % n)

    # (2) model-level fixture: head_dim 64 (the fused attention kernel's shape)
    V, pad_idx, eos_idx, blank = 50, 1, 2, 0
    m = _ref_model("conformer", d=128, ffn=128, heads=2, V=V, conv_channels="[16, 16, 32, 32]")
    enc_cfg = m.encoder.cfg.encoder
    enc_cfg.chunk_size, enc_cfg.chunk_left_window, enc_cfg.chunk_right_window = 6, 2, 1
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for _, p_ in m.named_parameters():
            if p_.dim() == 1:
                p_.add_(0.1 * torch.randn(p_.shape, generator=g))
    rs = np.random.RandomState(12)
    B, T = 3, 163
    lens = torch.tensor([163, 140, 75])
    feats = torch.from_numpy(rs.randn(B, T, 80).astype(np.float32))
    for b in range(B):
        feats[b, lens[b]:] = 0.0
    tgt = torch.full((B, 9), pad_idx, dtype=torch.long)
    for b, u in enumerate((8, 6, 3)):
        tgt[b, :u] = torch.from_numpy(rs.randint(4, V, size=u))
        tgt[b, u] = eos_idx
    cfg = dict(embed_dim=128, ffn_dim=128, heads=2, layers=2, layer_type="conformer", dw_kernel=31, dropout=0.0,
               attention_dropout=0.0, activation_dropout=0.0, layernorm_embedding=True, final_layer_norm=False, vocab=V)
    out = dict(feats=feats.numpy(), lens=lens.numpy(), target=tgt.numpy(), chunk=np.array([6, 2, 1]))
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    coins = set()
    # num_updates 0 and 1 give different first-or-last-partial coins under numpy_seed(num_updates)
    cases = [("train", 0), ("train", 1), ("eval", 7)]
    for mode, nu in cases:
        torch.nn.Module.load_state_dict(m, sd0)   # the Conformer layer has no upgrade_state_dict_named upstream
        m.train(mode == "train")
        m.set_num_updates(nu)
        m.zero_grad()
        net = m(feats, lens)
        logits = net["encoder_out"][0]
        olens = net["src_lengths"][0]
        hidden = m.encoder.get_attn_mask(olens)                      # deterministic given num_updates
        if mode == "train":
            coins.add(int((~hidden[0]).sum()))
        lprobs = m.get_normalized_probs(net, log_probs=True).contiguous()
        keep = (tgt != pad_idx) & (tgt != eos_idx)
        loss = F.ctc_loss(lprobs, tgt.masked_select(keep), olens, keep.sum(-1), blank=blank, reduction="sum",
                          zero_infinity=True)
        sd = {k: v.clone().requires_grad_(v.is_floating_point() and k in dict(m.named_parameters())) for k, v in sd0.items()}
        o_logits, o_lens, _ = O.encoder_forward(sd, cfg, feats, lens, training=(mode == "train"), attn_mask=hidden)
        o_loss = O.ctc_criterion(o_logits, o_lens, tgt, pad_idx, eos_idx, blank)
        d_log = (o_logits.transpose(0, 1) - logits).abs().max().item()
        assert d_log < 2e-4 and abs(o_loss.item() - loss.item()) < 1e-3 * abs(loss.item()), (mode, nu, d_log)
        tag = "%s%d" % (mode, nu)
        if mode == "train":
            loss.backward()
            o_loss.backward()
            worst = max((sd[k].grad - p_.grad).abs().max().item() / max(p_.grad.abs().max().item(), 1e-3)
                        for k, p_ in m.named_parameters())
            assert worst < 2e-3, worst
            if nu == 0:   # one gradient set keeps the fixture small; train1 is covered through loss + logits
                for k, p_ in m.named_parameters():
                    out["grad_%s.%s" % (tag, k)] = p_.grad.numpy().copy()
        # the unmasked model must differ visibly, or the fixture would not test the mask
        enc_cfg.chunk_size = 0
        with torch.no_grad():
            torch.nn.Module.load_state_dict(m, sd0)
            free = m(feats, lens)["encoder_out"][0]
        enc_cfg.chunk_size = 6
        sep = (free - logits).abs().max().item() / logits.abs().max().item()
        assert sep > 0.05, sep
        out["hidden_" + tag] = hidden.numpy()
        out["logits_" + tag] = logits.detach().transpose(0, 1).numpy()
        out["loss_" + tag] = np.float64(loss.item())
        out["out_lens"] = olens.numpy()
        print("streaming %s: |logits diff|=%.3g loss %.5f, masked vs free logits differ by %.2f of range" % (tag, d_log, loss.item(), sep))
    assert len(coins) == 2, "both partial-chunk placements must be covered"
    for k, v in sd0.items():
        out["sd." + k] = v.numpy()
    np.savez_compressed(os.path.join(GOLDEN, "encoder_streaming.npz"), **out)
    print("streaming encoder pinned -> tests/golden/encoder_streaming.npz")


def _lookahead_vocab():
    """Character subwords and a word list in lexical order with shared prefixes, words ending inside other words, a word
    with an unknown character (stays out of the tree) -- shared by the pin and the tests through the fixture."""
    chars = list("abcdeghilnorst'")
    words = sorted({"a", "an", "and", "ant", "are", "art", "as", "at", "be", "bed", "bee", "been", "best", "bet", "can",
                    "cat", "do", "dog", "done", "door", "eat", "go", "god", "gold", "good", "he", "hen", "her", "here", "his",
                    "in", "is", "it", "its", "no", "nor", "not", "note", "on", "one", "or", "so", "son", "the", "then",
                    "there", "to", "toe", "ton", "too", "don't", "quiz"})    # "quiz": q, u, z are not subwords
    return chars, words


def pin_lookahead():
    """Look-ahead word-LM fusion: the REAL TensorizedLookaheadLanguageModel over the reference LSTM word LM, driven step by
    step like the beam search does (forward on the growing prefix, then reorder_incremental_state), vs (1) oracle/lookahead.py
    fed with the reference LM's word distributions and (2) espresso_b200's prefix tree walked on the host.  Inputs, LM
    weights, the per-step word distributions and the reference outputs -> tests/golden/lookahead_lm.npz."""
    from argparse import Namespace

    from espresso.data import AsrDictionary as RefDict
    from espresso.models.lstm_lm import LSTMLanguageModelEspresso
    from espresso.models.tensorized_lookahead_language_model import TensorizedLookaheadLanguageModel as RefLookahead

    from espresso_b200.data.asr_dictionary import AsrDictionary as OurDict
    from espresso_b200.tools.tensorized_prefix_tree import TensorizedPrefixTree
    from oracle import lookahead as OL

    chars, words = _lookahead_vocab()

    def dicts(cls):
        sd, wd = cls(), cls()
        for c in chars + ["<space>"]:
            sd.add_symbol(c)
        for w in words:
            wd.add_symbol(w)
        if cls is OurDict:
            sd.space_index = sd.indices.get(sd.space_word, -1)
        else:
            sd.space_index = sd.indices.get(sd.space_word, -1)
        return sd, wd

    sub, wrd = dicts(RefDict)
    Vs, Vw = len(sub), len(wrd)

    class _Task:
        source_dictionary = target_dictionary = word_dictionary = wrd

    args = Namespace(dropout=0.0, decoder_embed_path=None, decoder_freeze_embed=False, decoder_layers=2,
                     adaptive_softmax_cutoff=None, is_wordlm=True, decoder_dropout_in=0.0, decoder_dropout_out=0.0,
                     criterion_name="cross_entropy", max_target_positions=64, tokens_per_sample=64, decoder_embed_dim=24,
                     decoder_hidden_size=32, decoder_out_embed_dim=32, share_embed=False, decoder_rnn_residual=False)
    torch.manual_seed(77)
    lm = LSTMLanguageModelEspresso.build_model(args, _Task())
    with torch.no_grad():      # peaky word distributions: the tree ratios are far from uniform
        for n_, p_ in lm.named_parameters():
            if "fc_out" in n_ or "embed" in n_:
                p_.mul_(6.0)
    lm.eval()
    assert lm.decoder.dictionary is wrd

    # hypotheses as strings over the subword alphabet: "_" = <space>, "$" = </s>; the beam reordering between steps is
    # explicit (new_orders[t] is applied after step t)
    texts = ["the_cat_$", "then_go_$", "be_been_$", "xq_not_$", "goldx_a_$", "do_n't_$", "a_an_ant_$", "there_$"]
    N = len(texts)
    L = max(len(t) for t in texts)
    sym = lambda ch: sub.space() if ch == "_" else sub.eos() if ch == "$" else sub.index(ch)  # noqa: E731
    assert sub.index("x") == sub.unk()     # "x" / "q" exercise out-of-vocabulary subwords

    out = {}
    for variant, (open_vocab, oov_pen) in {"open": (True, 1e-4), "closed": (False, 1e-4), "open_pen": (True, 0.3)}.items():
        ref = RefLookahead(lm, sub, oov_penalty=oov_pen, open_vocab=open_vocab)
        ref.eval()
        dec = ref.decoder
        # capture the word distributions the reference's LM produces inside forward()
        seen = []
        orig = dec.lm_decoder.get_normalized_probs

        def spy(net_output, log_probs, sample=None, _orig=orig):
            r = _orig(net_output, log_probs, sample)
            seen.append(r.detach().clone())
            return r

        dec.lm_decoder.get_normalized_probs = spy
        rs = np.random.RandomState(3)
        rows = [list(t) for t in texts]           # current text per hypothesis SLOT (slots get permuted)
        inc = {}
        toks = torch.full((N, 1), sub.eos(), dtype=torch.long)
        tok_hist, order_hist, ref_out, lm_hist = [], [], [], []
        tree = dec.tree
        state = OL.LookaheadState(OL.build_tree([wrd[i] for i in range(Vw)], {wrd.pad(), wrd.eos(), wrd.unk()}, sub.index,
                                                sub.unk()), N)
        ours = TensorizedPrefixTree.build(*dicts(OurDict)[::-1])
        our_nodes = [ours.root_id] * N
        for t in range(L + 1):
            seen.clear()
            lp, _ = dec(toks, incremental_state=inc)                       # [N, 1, Vs]
            lm_probs = seen[0][:, 0].numpy()                                # word distribution of this step
            prev = toks[:, -1].numpy()
            o = OL.step(state, prev, lm_probs, t == 0, Vs, sub.space(), sub.eos(), sub.pad(), wrd.unk(), wrd.eos(), oov_pen,
                        open_vocab)
            ref_lp = lp[:, 0].numpy()
            big = ref_lp > -15          # below: differences of float32 cumulative sums are cancellation noise
            err = np.abs(o - ref_lp)[big].max() if big.any() else 0.0
            assert err < 2e-4 and np.abs(o - ref_lp).max() < 1.0, (variant, t, err)
            # the oracle walked its own tree; the reference's node ids agree in the words they end / ranges they span
            rn = dec.get_incremental_state(inc, "nodes").numpy()
            for n in range(N):
                nd = state.nodes[n]
                assert (nd is None) == (rn[n] == 0)
                if nd is not None and nd is not state.root:
                    assert (int(tree.word_idx[rn[n]]), tuple(tree.word_set_idx[rn[n]].tolist())) == (nd.word, (nd.lo, nd.hi))
                # and so does the product's CSR tree
                if t > 0:
                    our_nodes[n] = ours.root_id if prev[n] == sub.space() else ours.step(our_nodes[n], int(prev[n]))
                assert (nd is None) == (our_nodes[n] == 0)
                if nd is not None and nd is not state.root:
                    k = our_nodes[n]
                    assert (int(ours.node_word[k]), int(ours.node_lo[k]), int(ours.node_hi[k])) == (nd.word, nd.lo, nd.hi)
            tok_hist.append(prev.copy())
            ref_out.append(ref_lp.copy())
            lm_hist.append(lm_probs.copy())
            if t == L:
                break
            # beam-search style permutation with duplicates, then each surviving slot emits its next symbol
            order = rs.randint(0, N, size=N) if t in (2, 4, 5) else np.arange(N)
            order_hist.append(order.copy())
            # the generator's entry point: walks every sub-module, i.e. also the wrapped LSTM LM's cached state
            # (fairseq/sequence_generator.py:368-371)
            dec.reorder_incremental_state_scripting(inc, torch.from_numpy(order))
            state.reorder(order)
            our_nodes = [our_nodes[i] for i in order]
            rows = [rows[i] for i in order]
            toks = toks[torch.from_numpy(order)]
            nxt = [sym(r[t]) if t < len(r) else sub.eos() for r in rows]
            toks = torch.cat([toks, torch.tensor(nxt)[:, None]], dim=1)
        dec.lm_decoder.get_normalized_probs = orig
        out[variant + ".prev_tokens"] = np.stack(tok_hist)                   # [L+1, N]
        out[variant + ".new_orders"] = np.stack(order_hist)                  # [L, N]
        out[variant + ".out"] = np.stack(ref_out).astype(np.float32)         # [L+1, N, Vs]
        out[variant + ".lm_probs"] = np.stack(lm_hist).astype(np.float32)    # [L+1, N, Vw]
        out[variant + ".tokens_final"] = toks.numpy()
        print("lookahead %-8s: %d steps x %d hypotheses, oracle within %.1e of the reference" % (variant, L + 1, N, 2e-4))
    for k, v in lm.state_dict().items():
        out["sd." + k] = v.numpy()
    out["chars"], out["words"] = np.array(chars), np.array(words)
    out["lm_cfg"] = np.array([24, 32, 32, 2])
    np.savez_compressed(os.path.join(GOLDEN, "lookahead_lm.npz"), **out)
    print("look-ahead LM pinned -> tests/golden/lookahead_lm.npz (|subwords| %d, |words| %d)" % (Vs, Vw))


def pin_multilevel():
    """MultiLevelLanguageModel (subword LSTM LM + word LSTM LM): the REAL reference class driven step by step (forward, then
    reorder_incremental_state_scripting) vs oracle/lookahead.py::multilevel_step fed with the two reference LMs' recorded
    log-probabilities -> tests/golden/multilevel_lm.npz."""
    from argparse import Namespace

    from espresso.data import AsrDictionary as RefDict
    from espresso.models.external_language_model import MultiLevelLanguageModel as RefML
    from espresso.models.lstm_lm import LSTMLanguageModelEspresso

    from oracle import lookahead as OL

    chars, words = _lookahead_vocab()
    sub, wrd = RefDict(), RefDict()
    for c in chars + ["<space>"]:
        sub.add_symbol(c)
    sub.space_index = sub.indices.get(sub.space_word, -1)
    for w in words:
        wrd.add_symbol(w)
    Vs, Vw = len(sub), len(wrd)

    def build(d, seed, is_wordlm, e, h):
        class _Task:
            source_dictionary = target_dictionary = word_dictionary = d

        args = Namespace(dropout=0.0, decoder_embed_path=None, decoder_freeze_embed=False, decoder_layers=1,
                         adaptive_softmax_cutoff=None, is_wordlm=is_wordlm, decoder_dropout_in=0.0, decoder_dropout_out=0.0,
                         criterion_name="cross_entropy", max_target_positions=64, tokens_per_sample=64, decoder_embed_dim=e,
                         decoder_hidden_size=h, decoder_out_embed_dim=h, share_embed=False, decoder_rnn_residual=False)
        torch.manual_seed(seed)
        m = LSTMLanguageModelEspresso.build_model(args, _Task())
        with torch.no_grad():
            for n_, p_ in m.named_parameters():
                if "fc_out" in n_ or "embed" in n_:
                    p_.mul_(5.0)
        return m.eval()

    wlm, slm = build(wrd, 5, True, 16, 24), build(sub, 6, False, 12, 20)
    texts = ["the_cat_$", "then_go_$", "be_been_$", "xq_not_$", "goldx_a_$", "do_n't_$", "a_an_ant_$", "there_$"]
    N, L = len(texts), max(len(t) for t in texts)
    sym = lambda ch: sub.space() if ch == "_" else sub.eos() if ch == "$" else sub.index(ch)  # noqa: E731
    out = {}
    for variant, (open_vocab, pen, weight) in {"open": (True, 1.0, 0.8), "open_pen": (True, 0.05, 0.5), "open_w1": (True, 0.3, 1.0)}.items():
        # open_vocab=False cannot be recorded: the reference raises TypeError at external_language_model.py:484
        # (`~batch_is_child_mask` on a Python list) on the first non-initial step
        ref = RefML(wlm, slm, subwordlm_weight=weight, oov_penalty=pen, open_vocab=open_vocab).eval()
        dec = ref.decoder
        seen = {"w": [], "s": []}

        def spy(key, orig):
            def f(net_output, log_probs, sample=None):
                r = orig(net_output, log_probs, sample)
                seen[key].append(r.detach().clone())
                return r
            return f

        ow, os_ = dec.wordlm_decoder.get_normalized_probs, dec.subwordlm_decoder.get_normalized_probs
        dec.wordlm_decoder.get_normalized_probs, dec.subwordlm_decoder.get_normalized_probs = spy("w", ow), spy("s", os_)
        rs = np.random.RandomState(4)
        rows = [list(t) for t in texts]
        inc = {}
        toks = torch.full((N, 1), sub.eos(), dtype=torch.long)
        state = OL.MultiLevelState(OL.build_tree([wrd[i] for i in range(Vw)], {wrd.pad(), wrd.eos(), wrd.unk()}, sub.index,
                                                 sub.unk()), N)
        tok_hist, order_hist, ref_out, w_hist, s_hist = [], [], [], [], []
        for t in range(L + 1):
            seen["w"].clear(), seen["s"].clear()
            lp, _ = dec(toks, incremental_state=inc)
            ref_lp = lp[:, 0].numpy().copy()        # the reference keeps mutating this tensor as state
            wl, sl = seen["w"][0][:, 0].numpy(), seen["s"][0][:, 0].numpy()
            prev = toks[:, -1].numpy()
            o = OL.multilevel_step(state, prev, wl, sl, t == 0, sub.space(), sub.eos(), wrd.unk(), wrd.eos(), weight, pen, open_vocab)
            err = np.abs(o - ref_lp).max()
            assert err < 1e-4, (variant, t, err)
            tok_hist.append(prev.copy()), ref_out.append(ref_lp), w_hist.append(wl.copy()), s_hist.append(sl.copy())
            if t == L:
                break
            order = rs.randint(0, N, size=N) if t in (2, 4, 5) else np.arange(N)
            order_hist.append(order.copy())
            dec.reorder_incremental_state_scripting(inc, torch.from_numpy(order))
            state.reorder(order)
            rows = [rows[i] for i in order]
            toks = toks[torch.from_numpy(order)]
            nxt = [sym(r[t]) if t < len(r) else sub.eos() for r in rows]
            toks = torch.cat([toks, torch.tensor(nxt)[:, None]], dim=1)
        dec.wordlm_decoder.get_normalized_probs, dec.subwordlm_decoder.get_normalized_probs = ow, os_
        out[variant + ".prev_tokens"], out[variant + ".new_orders"] = np.stack(tok_hist), np.stack(order_hist)
        out[variant + ".out"] = np.stack(ref_out).astype(np.float32)
        out[variant + ".word_logprobs"] = np.stack(w_hist).astype(np.float32)
        out[variant + ".sub_logprobs"] = np.stack(s_hist).astype(np.float32)
        out[variant + ".params"] = np.array([float(open_vocab), pen, weight])
        print("multilevel %-8s: %d steps x %d hypotheses, oracle within 1e-4 of the reference" % (variant, L + 1, N))
    for k, v in wlm.state_dict().items():
        out["wsd." + k] = v.numpy()
    for k, v in slm.state_dict().items():
        out["ssd." + k] = v.numpy()
    out["chars"], out["words"] = np.array(chars), np.array(words)
    out["wlm_cfg"], out["slm_cfg"] = np.array([16, 24, 24, 1]), np.array([12, 20, 20, 1])
    np.savez_compressed(os.path.join(GOLDEN, "multilevel_lm.npz"), **out)
    print("multi-level LM pinned -> tests/golden/multilevel_lm.npz")


def pin_fullsize():
    """The BENCHMARKED configuration (17 x 512 Conformer, ffn 2048, 8 heads, conv-k31, V = 5004) through the REAL
    reference model in fp32 and in bf16 (`model.bfloat16()`, fairseq --bf16 semantics, fairseq/trainer.py:105-107).
    Weights come from oracle.conformer.random_state_dict(FULLSIZE_CFG, seed=1) -- reproducible on the GPU box, so the
    fixture only stores outputs: sub-sampled logits, per-frame log-normalisers, the CTC loss and a set of gradients (small
    tensors whole, matrices sub-sampled), each from the fp32 run (truth) and from the bf16 run (the reference's own
    bf16 error, the yardstick for ours)."""
    import torch.nn.functional as F

    from oracle import conformer as O

    feats_np, lens_np, tgt_np = fullsize_inputs()
    feats, lens, tgt = torch.from_numpy(feats_np), torch.from_numpy(lens_np), torch.from_numpy(tgt_np)
    sd = O.random_state_dict(FULLSIZE_CFG, seed=1)
    out = {}
    for mode in ("fp32", "bf16"):
        m = _ref_model("conformer", layers=17, d=512, ffn=2048, heads=8, V=5004)
        # plain nn.Module loading: the reference's upgrade_state_dict hook does not exist on its Conformer layers
        missing = torch.nn.Module.load_state_dict(m, {k: v.clone() for k, v in sd.items()}, strict=False)
        assert not missing.unexpected_keys and all("num_batches_tracked" in k or k.endswith("version") or k.endswith("_float_tensor") for k in missing.missing_keys), missing
        if mode == "bf16":
            m = m.bfloat16()
        m.train()
        x = feats.bfloat16() if mode == "bf16" else feats
        net = m(x, lens)
        logits = net["encoder_out"][0]                      # T' x B x V
        olens = net["src_lengths"][0]
        lprobs = m.get_normalized_probs(net, log_probs=True).contiguous()
        assert lprobs.dtype == torch.float32
        keep = (tgt != 1) & (tgt != 2)
        with torch.backends.cudnn.flags(enabled=False):
            loss = F.ctc_loss(lprobs, tgt.masked_select(keep), olens, keep.sum(-1), blank=0, reduction="sum", zero_infinity=True)
        # gradients: of the linear functional sum(G * logits) (well conditioned; see fullsize_cotangent), not of the CTC
        # loss -- the CTC value itself is stored and its kernel gradient is tested against autograd on identical logits
        G = torch.from_numpy(fullsize_cotangent(olens.tolist()))
        (logits.transpose(0, 1).float() * G).sum().backward()
        lg = logits.detach().float().transpose(0, 1)        # B x T' x V
        out["logits_sub_" + mode] = lg[:, ::5, ::11].numpy()
        out["lse_" + mode] = torch.logsumexp(lg, dim=-1).numpy()
        out["loss_" + mode] = np.float64(loss.item())
        grads = dict(m.named_parameters())
        for n in FULLSIZE_GRADS:
            out["grad_%s.%s" % (mode, n)] = grads[n].grad.float().numpy()
        for n in FULLSIZE_GRADS_SUB:
            g = grads[n].grad.float()
            g2 = g.reshape(g.shape[0], -1)
            out["gradsub_%s.%s" % (mode, n)] = g2[::8, ::8].contiguous().numpy()
        out["gnorm_" + mode] = np.float64(torch.sqrt(sum((p.grad.float() ** 2).sum() for p in m.parameters())).item())
        print("fullsize/%s: loss %.6f  |g| %.5f  out_lens %s" % (mode, loss.item(), out["gnorm_" + mode], olens.tolist()))
        if mode == "fp32":
            out["out_lens"] = olens.numpy()
            # the oracle restatement at this size too (forward only: it is what bench.py times as the baselines)
            with torch.no_grad():
                o_logits, o_lens, _ = O.encoder_forward({k: v.clone() for k, v in sd.items()}, FULLSIZE_CFG, feats, lens, training=True)
            d_log = (o_logits - lg).abs().max().item()
            print("   oracle vs reference |logits diff| = %.3g" % d_log)
            assert d_log < 5e-3 and torch.equal(o_lens, olens)
    rel = lambda a, b: float(np.linalg.norm(a - b) / np.linalg.norm(b))  # noqa: E731
    print("   reference bf16 vs fp32: logits rel-Frobenius %.3g, loss rel %.3g" % (
        rel(out["logits_sub_bf16"], out["logits_sub_fp32"]), abs(out["loss_bf16"] - out["loss_fp32"]) / out["loss_fp32"]))
    np.savez_compressed(os.path.join(GOLDEN, "fullsize_conformer.npz"), **out)
    print("full-size encoder pinned -> tests/golden/fullsize_conformer.npz")


CKPT_ENC = dict(layers=1, d=32, ffn=64, heads=4, conv_channels="[8, 8, 16, 16]")  # small enough for a stored checkpoint


def pin_checkpoint():
    """Checkpoint interchange with the real fairseq loader, in both directions, on a small Conformer encoder.
    (1) A checkpoint written by espresso_b200.checkpoint_utils.save_checkpoint loads through
    fairseq.checkpoint_utils.load_checkpoint_to_cpu into the reference model, whose encoder output then equals that of the
    same weights put in directly; the layout of that file is recorded.  (2) A checkpoint in the reference's own layout,
    with a pickled reference config object that is not importable without fairseq, is stored for the reverse
    direction.  -> tests/golden/checkpoint_interchange.npz, tests/golden/checkpoint_reference.pt"""
    import tempfile

    from espresso.models.transformer.speech_transformer_config import SpeechTransformerConfig as RefConfig
    from fairseq import checkpoint_utils as RCU

    from espresso_b200 import checkpoint_utils as CU
    from espresso_b200.models import SpeechTransformerConfig, SpeechTransformerEncoderModel

    c = CKPT_ENC
    ref0 = _ref_model("conformer", **c)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for _, p_ in ref0.named_parameters():
            if p_.dim() == 1:
                p_.add_(0.1 * torch.randn(p_.shape, generator=g))
    ref0.eval()

    class _Dict:
        def __len__(self):
            return 50

        def pad(self):
            return 1

    class _Task:
        feat_dim, feat_in_channels, target_dictionary = 80, 1, _Dict()

    cfg = SpeechTransformerConfig.from_dict(dict(
        dropout=0.0, attention_dropout=0.0, activation_dropout=0.0, layernorm_embedding=True, max_source_positions=3600,
        encoder=dict(embed_dim=c["d"], ffn_embed_dim=c["ffn"], layers=c["layers"], attention_heads=c["heads"],
                     conv_channels=c["conv_channels"], normalize_before=True, learned_pos=False,
                     relative_positional_embeddings=True, layer_type="conformer", depthwise_conv_kernel_size=31)))
    ours = SpeechTransformerEncoderModel.build_model(cfg, _Task())
    ours.load_state_dict(ref0.state_dict(), strict=False)
    rs = np.random.RandomState(11)
    feats, lens = torch.from_numpy(rs.randn(2, 41, 80).astype(np.float32)), torch.tensor([41, 30])
    feats[1, 30:] = 0.0
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "from_b200.pt")
        CU.save_checkpoint(path, ours)
        written = torch.load(path, weights_only=False)
        rstate = RCU.load_checkpoint_to_cpu(path)
    ref = _ref_model("conformer", **c)
    missing, unexpected = torch.nn.Module.load_state_dict(ref, rstate["model"], strict=False)
    assert not unexpected, unexpected
    ref.eval()
    with torch.no_grad():
        out = ref(feats, lens)["encoder_out"][0]
        out0 = ref0(feats, lens)["encoder_out"][0]
    assert torch.equal(out, out0)
    np.savez_compressed(os.path.join(GOLDEN, "checkpoint_interchange.npz"),
                        file_keys=np.array(sorted(written)), model_keys=np.array(sorted(written["model"])),
                        missing_in_reference=np.array(sorted(missing), dtype=str),
                        optimizer_history_keys=np.array(sorted(written["optimizer_history"][-1])))
    torch.save({"cfg": {"model": RefConfig()}, "args": None, "model": ref0.state_dict(),
                "optimizer_history": [{"criterion_name": "CtcLossCriterion", "optimizer_name": "FP16Optimizer",
                                       "lr_scheduler_state": {"best": None}, "num_updates": 7}],
                "extra_state": {"train_iterator": {"epoch": 3, "iterations_in_epoch": 11}}, "last_optimizer_state": None},
               os.path.join(GOLDEN, "checkpoint_reference.pt"))
    print("checkpoint interchange: a b200 checkpoint loads into the reference model (same encoder output); layout -> "
          "tests/golden/checkpoint_interchange.npz, reference-layout checkpoint -> tests/golden/checkpoint_reference.pt")


SECTIONS = {"checkpoint": pin_checkpoint, "global_cmvn": pin_global_cmvn, "wer_scorer": pin_wer_scorer, "lr_schedules_v2": pin_lr_schedules_v2, "scheduled_sampling": pin_scheduled_sampling, "multilevel": pin_multilevel, "lookahead": pin_lookahead, "streaming": pin_streaming, "fullsize": pin_fullsize, "text": pin_text, "lstm_lm": pin_lstm_lm, "speech_lstm": pin_speech_lstm, "dictionary": pin_dictionary, "sharding": pin_sharding, "collate": pin_collate, "batching": pin_batching, "optimizer": pin_optimizer, "beam": pin_beam, "label_smoothing": pin_label_smoothing, "frontend": pin_frontend, "ctc": pin_ctc, "conformer": pin_conformer, "encdec": pin_encdec,
            "transducer": pin_transducer}


def main(argv):
    refshim.activate()
    torch.manual_seed(0)
    os.makedirs(GOLDEN, exist_ok=True)
    for name in (argv or list(SECTIONS)):
        SECTIONS[name]()


if __name__ == "__main__":
    main(sys.argv[1:])

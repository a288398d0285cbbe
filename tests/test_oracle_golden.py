"""CPU: the oracle restatements reproduce the fixtures generated from the real reference
(oracle/pin_against_reference.py), and the host mask-drawing logic consumes the RNG like the reference."""
import os

import numpy as np

from espresso_b200.data import specaugment as SA
from oracle import ctc as octc
from oracle import frontend as ofe


def test_frontend_oracle_matches_reference_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "frontend.npz"))
    mean, std = g["cmvn_mean"], g["cmvn_std"]
    for i in range(len(g["durs"])):
        if "wave_%d" % i not in g:
            continue
        w = g["wave_%d" % i]
        fb = ofe.kaldi_fbank(w)
        assert fb.shape == g["fbank_%d" % i].shape
        # two fp32 FFT implementations (numpy pocketfft vs torch) differ by a few 1e-4 on log-mel
        assert np.abs(fb - g["fbank_%d" % i]).max() < 2e-3
        # ... and both sit that close to the float64 evaluation of the same formula
        fb64 = ofe.kaldi_fbank(w, dtype=np.float64)
        assert np.abs(fb64 - g["fbank_%d" % i]).max() < 2e-3
        with ofe.numpy_seed(1, 1, i):
            out, fm, tm = ofe.adaptive_specaugment(ofe.global_cmvn(fb, mean, std), return_masks=True)
        assert np.abs(out - g["final_%d" % i]).max() < 2e-3
        assert np.array_equal(np.array(fm, dtype=np.int32).reshape(-1, 2), g["fmask_%d" % i])
        assert np.array_equal(np.array(tm, dtype=np.int32).reshape(-1, 2), g["tmask_%d" % i])


def test_host_mask_draws_match_reference_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "frontend.npz"))
    cfg = SA.AdaptiveSpecAugmentConfig.from_config_dict(
        {"time_warp_W": 0, "freq_mask_F": 27, "freq_mask_N": 2, "time_mask_pm": 0.04, "time_mask_ps": 0.04})
    for i in range(len(g["durs"])):
        if "wave_%d" % i not in g:
            continue
        m = g["fbank_%d" % i].shape[0]
        with SA.numpy_seed(1, 1, i):
            fm, tm = SA.draw_masks(cfg, m, 80)
        assert np.array_equal(np.array(fm, dtype=np.int32).reshape(-1, 2), g["fmask_%d" % i])
        assert np.array_equal(np.array(tm, dtype=np.int32).reshape(-1, 2), g["tmask_%d" % i])
    fmp, tmp = SA.pack_masks([[(1, 2)], []], [[], [(3, 4), (5, 6)]])
    assert fmp.shape == (2, 1, 2) and tmp.shape == (2, 2, 2) and tmp[0].sum() == 0


def test_num_frames_edges():
    assert ofe.num_frames(399) == 0 and ofe.num_frames(400) == 1 and ofe.num_frames(559) == 1
    assert ofe.num_frames(560) == 2 and ofe.num_frames(160000) == 998


def test_ctc_oracle_matches_reference_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "ctc.npz"))
    for b in range(g["logits"].shape[0]):
        tgt = g["targets"][b, : g["tgt_lens"][b]]
        nll, grad = octc.ctc_loss_and_grad(g["logits"][b], g["in_lens"][b], tgt, int(g["blank"]))
        assert abs(nll - g["loss"][b]) < 1e-4 * max(1.0, abs(g["loss"][b]))
        assert np.abs(grad - g["grad"][b]).max() < 1e-5


def test_ctc_oracle_edge_cases():
    x = np.zeros((4, 3))
    nll, grad = octc.ctc_loss_and_grad(x, 4, [], 0)  # empty target: all-blank path
    assert abs(nll - 4 * np.log(3.0)) < 1e-9
    nll, grad = octc.ctc_loss_and_grad(x, 1, [1, 2], 0)  # infeasible -> zero_infinity
    assert nll == 0.0 and not grad.any()


def test_label_smoothing_variants_match_reference_fixture(golden_dir):
    """oracle/ops_ref.lsce_loss (uniform / unigram / temporal) vs the reference's label_smoothed_nll_loss +
    temporal_label_smoothing_prob_mask outputs recorded by oracle/pin_against_reference.py."""
    import torch

    from oracle import ops_ref as O

    g = np.load(os.path.join(golden_dir, "label_smoothing.npz"))
    logits = torch.from_numpy(g["logits"])
    B, U, V = logits.shape
    tgt = torch.from_numpy(g["target"]).view(-1).int()
    uni = torch.from_numpy(g["unigram"])
    for name, mode in (("uniform", 0), ("unigram", 1), ("temporal", 2)):
        loss, nll, grad = O.lsce_loss(logits.view(-1, V).to(torch.bfloat16), V, tgt, int(g["pad"]), float(g["eps"]),
                                      smoothing=mode, unigram=uni, U=U)
        assert abs(loss.sum().item() - float(g["loss_" + name])) < 1e-4 * abs(float(g["loss_" + name])), name
        assert abs(nll.sum().item() - float(g["nll_" + name])) < 1e-4 * abs(float(g["nll_" + name])), name
        assert np.abs(grad.float().view(B, U, V).numpy() - g["grad_" + name]).max() < 4e-3, name


def test_adam_clip_and_lr_schedules_match_fairseq_fixture(golden_dir):
    """oracle/ops_ref.adam_step (the restatement the CUDA optimizer kernel is tested against) replays the trajectory of
    fairseq's Adam + clip_grad_norm_ + 1/sample_size scaling recorded in tests/golden/optimizer.npz; the host LR
    schedules reproduce the reference's noam / tri_stage values."""
    import torch

    from espresso_b200.optim import NoamLRScheduler, TriStageLRScheduler
    from oracle import ops_ref as O

    g = np.load(os.path.join(golden_dir, "optimizer.npz"))
    lr, b1, b2, eps, wd, clip = g["hyper"].tolist()
    p32 = torch.from_numpy(g["p0"]).clone()
    m, v = torch.zeros_like(p32), torch.zeros_like(p32)
    p16 = p32.to(torch.bfloat16)
    for step in range(1, 5):
        grad = torch.from_numpy(g["g%d" % step])
        gn = torch.zeros(1)
        O.adam_step(p32, m, v, grad, p16, lr, b1, b2, eps, wd, step, (grad * grad).sum().reshape(1),
                    denom_const=float(g["ss%d" % step]), clip_norm=clip, gnorm_out=gn)
        assert np.abs(p32.numpy() - g["p%d" % step]).max() < 1e-6
        assert abs(gn.item() - float(g["gnorm%d" % step])) < 1e-5 * float(g["gnorm%d" % step])
        assert torch.equal(p16, p32.to(torch.bfloat16))
    noam = NoamLRScheduler(5.0, 25000, 512, 1e-6)
    for s_, ref in zip(g["noam_steps"].tolist(), g["noam_lr"].tolist()):
        assert abs(noam.step_update(int(s_)) - ref) <= 1e-12 * max(abs(ref), 1e-12)
    tri = TriStageLRScheduler(5e-4, 100, 200, 300, init_lr_scale=0.01, final_lr_scale=0.05)
    for s_, ref in zip(g["tri_steps"].tolist(), g["tri_lr"].tolist()):
        assert abs(tri.step_update(int(s_)) - ref) <= 1e-12 * max(abs(ref), 1e-12)


def test_batch_packer_matches_reference_cython_fixture(golden_dir):
    """esp_batch_by_size (C ABI, host code) vs the batches produced by the reference's compiled Cython packer
    (fairseq/data/data_utils_fast.pyx) recorded in tests/golden/batching.npz, and at the recipe's limits on the seeded
    cases recorded in tests/golden/batching_seeded.npz."""
    from espresso_b200.data import batching as Bt

    g = np.load(os.path.join(golden_dir, "batching.npz"))
    for c in range(int(g["n_cases"])):
        sizes, order = g["c%d_sizes" % c], g["c%d_order" % c]
        mt, ms, mult = (int(x) for x in g["c%d_cfg" % c])
        got = Bt.batch_by_size(order, sizes, mt or None, ms or None, mult)
        assert np.array_equal(np.cumsum([len(b) for b in got]), g["c%d_ends" % c]), c
        assert np.array_equal(np.concatenate(got), order)
    assert Bt.batch_by_size(np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64), 100, None, 1) == []
    try:
        Bt.batch_by_size(np.arange(3), np.array([5, 500, 7]), 100, None, 1)
        raise RuntimeError("oversized sample must be rejected")
    except AssertionError:
        pass
    ref = np.load(os.path.join(golden_dir, "batching_seeded.npz"))
    rs = np.random.RandomState(3)
    for c in range(100):
        n = int(rs.randint(1, 200))
        sizes = rs.randint(1, 300, size=n).astype(np.int64)
        order = rs.permutation(n).astype(np.int64)
        mult = int(rs.choice([1, 8]))
        got = Bt.batch_by_size(order, sizes, 3000, 24, mult)
        assert np.array_equal(np.cumsum([len(b) for b in got]), ref["c%d_ends" % c]), c
        assert np.array_equal(np.concatenate(got), order)


def test_collate_matches_reference_fixture(golden_dir):
    """espresso_b200.data.collate vs batches assembled by the reference's espresso.data.asr_dataset.collate
    (tests/golden/collate.npz): ordering by length, padding, target / prev_output_tokens layout, ntokens."""
    import torch

    from espresso_b200.data.collate import collate

    g = np.load(os.path.join(golden_dir, "collate.npz"))
    keys = sorted({k[: k.index("_", k.index("bos")) + 1] for k in g.files})
    assert keys
    for key in keys:
        bos = int(key.split("bos")[1].rstrip("_"))
        lens, ids = g[key + "lens"], g[key + "ids"]
        samples = [{"id": int(ids[j]), "utt_id": "u%d" % j, "source": torch.full((int(lens[j]), 4), float(j + 1)),
                    "target": torch.from_numpy(g[key + "tgt%d" % j]), "text": "t%d" % j} for j in range(len(lens))]
        b = collate(samples, pad_idx=1, eos_idx=2, maybe_bos_idx=None if bos < 0 else bos)
        assert np.array_equal(b["id"].numpy(), g[key + "out_id"])
        assert np.array_equal(b["net_input"]["src_lengths"].numpy(), g[key + "out_src_lengths"])
        assert b["net_input"]["src_lengths"].dtype == torch.int32
        assert np.array_equal(b["target"].numpy(), g[key + "out_target"])
        assert np.array_equal(b["net_input"]["prev_output_tokens"].numpy(), g[key + "out_prev"])
        assert b["ntokens"] == int(g[key + "ntokens"]) and b["nsentences"] == len(lens)
        src = b["net_input"]["src_tokens"]
        for r in range(len(lens)):  # rows carry their own sample, zero padded on the right
            n = int(b["net_input"]["src_lengths"][r])
            assert (src[r, :n] == src[r, 0, 0]).all() and (src[r, n:] == 0).all()
    assert collate([], 1, 2) == {}


def test_asr_dictionary_layout(tmp_path):
    """Index order and text round trip of the dictionary mirror (pinned against the reference class by
    oracle/pin_against_reference.py::pin_dictionary): specials first ([<s>] <pad> </s> <unk>), file order after."""
    import torch

    from espresso_b200.data.asr_dictionary import AsrDictionary

    p = tmp_path / "dict.txt"
    p.write_text("▁the 50\n▁a 40\ns 30\n<space> 3\n", encoding="utf-8")
    d = AsrDictionary.load(str(p))
    assert (d.pad(), d.eos(), d.unk(), len(d), d.nspecial, d.space()) == (0, 1, 2, 7, 3, 6)
    db = AsrDictionary.load(str(p), enable_bos=True)
    assert (db.bos(), db.pad(), db.eos(), db.unk(), len(db)) == (0, 1, 2, 3, 8) and db.index("s") == 6 and db.index("nope") == 3
    ids = db.encode_line("▁the s zz ▁a")
    assert ids.tolist() == [4, 6, 3, 5, 2]
    assert db.string(ids) == "▁the s <unk> ▁a" and db.string(ids, bpe_symbol="sentencepiece") == "thes<unk> a"
    assert db.count[4] == 50 and db.count[:4] == [1, 0, 0, 0]
    try:
        d.bos()
        raise RuntimeError("bos must not exist without enable_bos")
    except NotImplementedError:
        pass
    out = tmp_path / "saved.txt"
    db.save(str(out))
    assert AsrDictionary.load(str(out), enable_bos=True).symbols == db.symbols


def test_character_encoder_and_edit_counts():
    """Known answers for the text utilities pinned against the reference by oracle/pin_against_reference.py::pin_text."""
    from espresso_b200.data.encoders import CharactersAsr, tokenize
    from espresso_b200.tasks.speech_recognition import edit_counts

    assert tokenize("ab c") == "a b <space> c"
    enc = CharactersAsr(non_lang_syms=["<noise>"])
    assert enc.encode(" hi <noise> yo ") == "h i <space> <noise> <space> y o <space>"
    assert enc.decode(enc.encode("hi <noise> yo")) == "hi <noise> yo"
    assert CharactersAsr(ends_with_space=False).encode("a b") == "a <space> b"
    assert edit_counts(list("kitten"), list("sitting")) == (3, 6)
    assert edit_counts([], ["a", "b"]) == (2, 0) and edit_counts(["a"], []) == (1, 1)

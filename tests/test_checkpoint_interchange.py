"""Checkpoint interchange with the reference (SURVEY 8(f)4): a checkpoint written here loads through the REAL
fairseq.checkpoint_utils.load_checkpoint_to_cpu into the REAL reference model (same logits), a checkpoint written in the
reference's layout (with pickled config objects that are not importable without fairseq) loads here, and Adam's moments
survive the round trip through fairseq's flat-fp32 optimizer layout."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import ops_ref, refshim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def cpu_ops(monkeypatch):
    from espresso_b200 import ops

    for name in dir(ops_ref):
        if name.startswith("_") or not callable(getattr(ops_ref, name)) or not hasattr(ops, name):
            continue
        monkeypatch.setattr(ops, name, getattr(ops_ref, name))
    return ops


def _ours(golden_dir):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_host_orchestration import _Task, _build

    g = np.load(os.path.join(golden_dir, "encoder_conformer.npz"))
    return g, _build("conformer", g), _Task


def test_round_trip_and_optimizer_state(golden_dir, tmp_path, cpu_ops):
    from espresso_b200 import checkpoint_utils as CU
    from espresso_b200.criterions import CtcLossCriterion
    from espresso_b200.optim import NoamLRScheduler
    from espresso_b200.trainer import Trainer

    g, m, Task = _ours(golden_dir)
    m.finalize_(torch.device("cpu"))
    tr = Trainer(m, CtcLossCriterion(Task(50)), NoamLRScheduler(5.0, 100, 64, 1e-6), clip_norm=2.0)
    sample = {"net_input": {"src_tokens": torch.from_numpy(g["feats"]), "src_lengths": torch.from_numpy(g["lens"])},
              "target": torch.from_numpy(g["target"])}
    for _ in range(2):
        tr.train_step([sample])
    path = str(tmp_path / "checkpoint_last.pt")
    CU.save_checkpoint(path, m, tr)
    state = CU.load_checkpoint_to_cpu(path)
    assert state["optimizer_history"][-1]["num_updates"] == 2
    n_params = sum(p.numel() for p in m.parameters())
    assert state["last_optimizer_state"]["state"][0]["exp_avg"].numel() == n_params   # fairseq's flat layout: no padding
    # a fresh model + trainer resumes to the same weights and moments
    _, m2, _ = _ours(golden_dir)
    m2.finalize_(torch.device("cpu"))
    tr2 = Trainer(m2, CtcLossCriterion(Task(50)), NoamLRScheduler(5.0, 100, 64, 1e-6), clip_norm=2.0)
    CU.load_model_state(m2, state)
    CU.optimizer_state_from_fairseq(tr2, state["last_optimizer_state"])
    assert tr2.num_updates == 2
    assert torch.equal(m2.flat.p32, m.flat.p32) and torch.equal(m2.flat.m, m.flat.m) and torch.equal(m2.flat.v, m.flat.v)
    tr.train_step([sample])
    tr2.train_step([sample])
    assert torch.allclose(m2.flat.p32, m.flat.p32, atol=1e-6)


def test_interchange_with_reference_fixture(golden_dir, tmp_path):
    """Both directions against what the real reference did when the fixtures were made
    (oracle/pin_against_reference.py::pin_checkpoint): checkpoint_reference.pt was written by the reference, with its own
    pickled config object inside, and a file of checkpoint_interchange.npz's layout loaded through the real
    fairseq.checkpoint_utils.load_checkpoint_to_cpu into the reference model with none of its weights missing."""
    from espresso_b200 import checkpoint_utils as CU
    from espresso_b200.models import SpeechTransformerConfig, SpeechTransformerEncoderModel

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_host_orchestration import _Task

    from oracle.pin_against_reference import CKPT_ENC as c

    g = np.load(os.path.join(golden_dir, "checkpoint_interchange.npz"))
    cfg = SpeechTransformerConfig.from_dict(dict(
        dropout=0.0, attention_dropout=0.0, activation_dropout=0.0, layernorm_embedding=True, max_source_positions=3600,
        encoder=dict(embed_dim=c["d"], ffn_embed_dim=c["ffn"], layers=c["layers"], attention_heads=c["heads"],
                     conv_channels=c["conv_channels"], normalize_before=True, learned_pos=False,
                     relative_positional_embeddings=True, layer_type="conformer", depthwise_conv_kernel_size=31)))
    # reference -> ours: the reference's layout, with a config object that only unpickles where fairseq is installed
    state = CU.load_checkpoint_to_cpu(os.path.join(golden_dir, "checkpoint_reference.pt"))
    assert state["optimizer_history"][-1]["num_updates"] == 7 and state["extra_state"]["train_iterator"]["epoch"] == 3
    m = SpeechTransformerEncoderModel.build_model(cfg, _Task(50))
    with torch.no_grad():
        for p in m.parameters():
            p.zero_()
    missing, unexpected = CU.load_model_state(m, state)
    assert not missing and not unexpected
    for k, v in state["model"].items():
        if k in m.state_dict() and not k.endswith("num_batches_tracked"):
            assert torch.equal(m.state_dict()[k].float(), v.float()), k
    # ours -> reference: the file has the layout the real loader accepted, every weight the reference model has, and
    # the reference's own values back
    path = str(tmp_path / "from_b200.pt")
    CU.save_checkpoint(path, m)
    written = torch.load(path, weights_only=False)
    assert sorted(written) == g["file_keys"].tolist()
    assert sorted(written["optimizer_history"][-1]) == g["optimizer_history_keys"].tolist()
    assert sorted(written["model"]) == g["model_keys"].tolist() and g["missing_in_reference"].size == 0
    for k, v in written["model"].items():
        assert torch.equal(v, state["model"][k]), k


@pytest.mark.skipif(not refshim.available(), reason="needs the reference sources (ESPRESSO_REFERENCE_ROOT)")
def test_interchange_with_the_real_reference(golden_dir, tmp_path):
    from espresso_b200 import checkpoint_utils as CU

    refshim.activate()
    from fairseq import checkpoint_utils as RCU

    from oracle.pin_against_reference import _ref_model

    g, m, _ = _ours(golden_dir)
    # ours -> reference: the real fairseq loader and the real reference model accept the file
    path = str(tmp_path / "from_b200.pt")
    CU.save_checkpoint(path, m)
    rstate = RCU.load_checkpoint_to_cpu(path)
    ref = _ref_model("conformer")
    torch.nn.Module.load_state_dict(ref, rstate["model"], strict=False)
    ref.eval()
    ref0 = _ref_model("conformer")          # the same weights put in directly
    torch.nn.Module.load_state_dict(ref0, {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}, strict=False)
    ref0.eval()
    with torch.no_grad():
        out = ref(torch.from_numpy(g["feats"]), torch.from_numpy(g["lens"]))["encoder_out"][0]
        out0 = ref0(torch.from_numpy(g["feats"]), torch.from_numpy(g["lens"]))["encoder_out"][0]
    assert torch.equal(out, out0)
    # reference -> ours: a checkpoint in the reference's layout, with a pickled (reference-only) config object inside
    from espresso.models.transformer.speech_transformer_config import SpeechTransformerConfig

    rpath = str(tmp_path / "from_reference.pt")
    torch.save({"cfg": {"model": SpeechTransformerConfig()}, "args": None, "model": ref.state_dict(),
                "optimizer_history": [{"criterion_name": "CtcLossCriterion", "optimizer_name": "FP16Optimizer",
                                       "lr_scheduler_state": {"best": None}, "num_updates": 7}],
                "extra_state": {"train_iterator": {"epoch": 3, "iterations_in_epoch": 11}}, "last_optimizer_state": None}, rpath)
    state = CU.load_checkpoint_to_cpu(rpath)
    assert state["optimizer_history"][-1]["num_updates"] == 7 and state["extra_state"]["train_iterator"]["epoch"] == 3
    _, m3, _ = _ours(golden_dir)
    with torch.no_grad():
        for p in m3.parameters():
            p.zero_()
    missing, unexpected = CU.load_model_state(m3, state)
    assert not missing and not unexpected
    for k, v in ref.state_dict().items():
        if k in m3.state_dict() and not k.endswith("num_batches_tracked"):
            assert torch.equal(m3.state_dict()[k].float(), v.float()), k

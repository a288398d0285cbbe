"""The drop-in boundary under the REAL fairseq (CPU, authoring container only: needs /root/reference through
oracle/refshim): `utils.import_user_module` loads espresso_b200_plugin, fairseq's own registries accept the B200 model and
criterion (they extend BaseFairseqModel / FairseqCriterion), `task.build_model` / `task.build_criterion` construct them and
the unmodified `FairseqTask.train_step` (fairseq/tasks/fairseq_task.py:490-522) runs forward + backward, leaving
gradients in `.grad` that match the reference model's own autograd gradients.  CUDA ops are replaced by oracle/ops_ref."""
import argparse
import os

import numpy as np
import pytest
import torch

from oracle import ops_ref, refshim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.skipif(not refshim.available(), reason="needs the reference sources (ESPRESSO_REFERENCE_ROOT)")


@pytest.fixture()
def cpu_ops(monkeypatch):
    from espresso_b200 import ops

    for name in dir(ops_ref):
        if name.startswith("_") or not callable(getattr(ops_ref, name)) or not hasattr(ops, name):
            continue
        monkeypatch.setattr(ops, name, getattr(ops_ref, name))
    return ops


def _load_plugin():
    refshim.activate()
    from fairseq import utils

    utils.import_user_module(argparse.Namespace(user_dir=os.path.join(ROOT, "espresso_b200_plugin")))


def test_plugin_registers_with_fairseq_and_trains_through_fairseq_task(golden_dir, cpu_ops):
    _load_plugin()
    from fairseq import criterions, models
    from fairseq.criterions import FairseqCriterion
    from fairseq.models import ARCH_MODEL_REGISTRY, MODEL_REGISTRY, BaseFairseqModel
    from fairseq.tasks import FairseqTask

    assert "speech_transformer_encoder_model_b200" in MODEL_REGISTRY
    assert "speech_conformer_encoder_model_b200" in ARCH_MODEL_REGISTRY
    assert "ctc_loss_b200" in criterions.CRITERION_REGISTRY
    cls = MODEL_REGISTRY["speech_transformer_encoder_model_b200"]
    assert issubclass(cls, BaseFairseqModel) and issubclass(criterions.CRITERION_REGISTRY["ctc_loss_b200"], FairseqCriterion)
    # a duplicate registration is refused by fairseq itself (fairseq/models/__init__.py:128-129)
    with pytest.raises(ValueError):
        models.register_model("speech_transformer_encoder_model_b200")(cls)

    g = np.load(os.path.join(golden_dir, "encoder_conformer.npz"))

    class _Dict:
        def __len__(self):
            return 50

        def pad(self):
            return 1

        def eos(self):
            return 2

        def index(self, sym):
            return 0

    class _Task(FairseqTask):
        feat_dim, feat_in_channels, blank_symbol = 80, 1, "<s>"

        def __init__(self):
            super().__init__(None)

        @property
        def target_dictionary(self):
            return _Dict()

        @property
        def source_dictionary(self):
            return None

    task = _Task()
    # the reference's own config dataclass drives the B200 model (same yaml / CLI as the reference recipe)
    from espresso.models.transformer.speech_transformer_config import SpeechTransformerConfig

    cfg = SpeechTransformerConfig()
    cfg._name = "speech_transformer_encoder_model_b200"
    cfg.max_source_positions, cfg.max_target_positions, cfg.tpu = 3600, 200, False
    e = cfg.encoder
    e.conv_channels, e.conv_kernel_sizes = "[64, 64, 128, 128]", "[(3, 3), (3, 3), (3, 3), (3, 3)]"
    e.conv_strides = "[(1, 1), (2, 2), (1, 1), (2, 2)]"
    e.embed_dim, e.ffn_embed_dim, e.layers, e.attention_heads = 64, 128, 2, 4
    e.normalize_before, e.learned_pos, e.relative_positional_embeddings = True, False, True
    e.layer_type, e.depthwise_conv_kernel_size = "conformer", 31
    cfg.layernorm_embedding = True
    cfg.dropout = cfg.attention_dropout = cfg.activation_dropout = 0.0
    cfg.__dict__["_parent"] = None             # what a real DictConfig node carries (fairseq/dataclass/utils.py:500)
    model = task.build_model(cfg)              # FairseqTask.build_model -> fairseq.models.build_model -> MODEL_REGISTRY
    assert type(model) is cls
    assert isinstance(model, BaseFairseqModel)
    ref_keys = sorted(k[3:] for k in g.files if k.startswith("sd."))
    assert sorted(model.state_dict().keys()) == ref_keys          # checkpoints interchange with the reference
    model.load_state_dict({k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}, strict=True)
    model = model.bfloat16()                                      # what fairseq's trainer does under --bf16

    ccfg = argparse.Namespace(criterion="ctc_loss_b200", zero_infinity=True, sentence_avg=True)   # the argparse route
    criterion = task.build_criterion(ccfg)     # FairseqTask.build_criterion -> fairseq.criterions.build_criterion -> registry
    assert isinstance(criterion, FairseqCriterion)

    class _Opt:  # FairseqOptimizer.backward (fairseq/optim/fairseq_optimizer.py:97-99)
        def backward(self, loss):
            loss.backward()

    sample = {"net_input": {"src_tokens": torch.from_numpy(g["feats"]), "src_lengths": torch.from_numpy(g["lens"])},
              "target": torch.from_numpy(g["target"]), "ntokens": 13, "nsentences": 3}
    loss, sample_size, log = task.train_step(sample, model, criterion, _Opt(), update_num=0)
    assert sample_size == 3
    assert abs(float(loss) - float(g["loss_train"])) < 0.03 * float(g["loss_train"])
    # gradients arrived in .grad (bf16, the slots fairseq's optimizers read) and follow the reference's
    worst = []
    for n, p in model.named_parameters():
        assert p.grad is not None and p.grad.dtype == p.dtype, n
        if ("pre_encoder.convolutions" in n and n.endswith(".bias")) or n.endswith("k_proj.bias"):
            continue
        ref = g["grad." + n]
        worst.append((np.linalg.norm(p.grad.float().numpy() - ref) / max(np.linalg.norm(ref), 1e-3), n))
    worst.sort(reverse=True)
    assert np.median([w[0] for w in worst]) < 0.04 and worst[0][0] < 0.3, worst[:5]
    # a second micro-batch accumulates (update_freq > 1), zero_grad semantics stay fairseq's
    before = {n: p.grad.clone() for n, p in model.named_parameters()}
    task.train_step(sample, model, criterion, _Opt(), update_num=0)
    for n, p in model.named_parameters():
        if "pre_encoder.convolutions" in n and n.endswith(".bias"):
            continue
        assert torch.allclose(p.grad.float(), 2 * before[n].float(), rtol=0.05, atol=1e-3 * float(before[n].float().abs().max() + 1e-6)), n
    # logging contract: reduce_metrics is the reference's
    from fairseq.logging import metrics

    with metrics.aggregate() as agg:
        criterion.reduce_metrics([{k: (float(v) if torch.is_tensor(v) else v) for k, v in log.items()}])
    assert "loss" in agg.get_smoothed_values()

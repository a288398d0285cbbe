"""CPU, world_size 2 over gloo: the data-parallel update (one all-reduce of the flat gradient buffer with the
stats tail) is equivalent to a single rank accumulating both micro-batches (update_freq = 2), like
legacy_ddp + trainer semantics (fairseq/trainer.py:903-953); plus ShardedIterator-style batch sharding."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# torch threads of every rank and of the single-process reference: CPU reductions split their sums by thread count, so
# the two sides only add in the same order with the same setting (hosts with many cores differ otherwise)
THREADS = 2


def _patch_ops():
    from espresso_b200 import ops
    from oracle import ops_ref

    for name in dir(ops_ref):
        if not name.startswith("_") and callable(getattr(ops_ref, name)) and hasattr(ops, name):
            setattr(ops, name, getattr(ops_ref, name))


def _make(golden_dir, reduce_dtype="fp32"):
    for pth in (ROOT, os.path.join(ROOT, "tests")):
        if pth not in sys.path:
            sys.path.insert(0, pth)
    from test_host_orchestration import _Task, _build
    from espresso_b200.criterions import CtcLossCriterion
    from espresso_b200.optim import NoamLRScheduler
    from espresso_b200.trainer import Trainer

    g = np.load(os.path.join(golden_dir, "encoder_conformer.npz"))
    m = _build("conformer", g).finalize_(torch.device("cpu"))
    tr = Trainer(m, CtcLossCriterion(_Task(50)), NoamLRScheduler(5.0, 100, 64, 1e-6), clip_norm=2.0, reduce_dtype=reduce_dtype)
    feats, lens, tgt = torch.from_numpy(g["feats"]), torch.from_numpy(g["lens"]), torch.from_numpy(g["target"])
    s0 = {"net_input": {"src_tokens": feats[:2], "src_lengths": lens[:2]}, "target": tgt[:2]}
    s1 = {"net_input": {"src_tokens": feats[2:, :40].contiguous(), "src_lengths": lens[2:].clamp(max=40)}, "target": tgt[2:]}
    return tr, m, (s0, s1)


def _worker(rank, world, port, golden_dir, out_dir, reduce_dtype):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(THREADS)
    _patch_ops()
    tr, m, samples = _make(golden_dir, reduce_dtype)
    tail = tr.train_step([samples[rank]])
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), p32=m.flat.p32.numpy(), tail=tail.numpy())
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.timeout(600)
@pytest.mark.parametrize("reduce_dtype", ["fp32", "bf16"])
def test_two_rank_update_equals_accumulated_update(golden_dir, tmp_path, reduce_dtype):
    """fp32: one all-reduce of the flat fp32 buffer (+ stats tail); bf16: the reference's exchange dtype (bf16 gradients,
    fp32 stats in a second tiny all-reduce)."""
    mp.spawn(_worker, args=(2, _free_port(), golden_dir, str(tmp_path), reduce_dtype), nprocs=2, join=True)
    r0 = np.load(os.path.join(str(tmp_path), "rank0.npz"))
    r1 = np.load(os.path.join(str(tmp_path), "rank1.npz"))
    assert np.array_equal(r0["p32"], r1["p32"])  # both ranks hold the same parameters after the update
    assert r0["tail"][0] == 3 and r0["tail"][2] == 3  # global sample_size / nsentences through the tail
    # single process, both micro-batches in one update
    import importlib

    from espresso_b200 import ops
    saved = {n: getattr(ops, n) for n in dir(ops)}
    threads = torch.get_num_threads()
    try:
        torch.set_num_threads(THREADS)
        _patch_ops()
        tr, m, samples = _make(golden_dir)
        tr.train_step(list(samples))
        ref = m.flat.p32.numpy()
    finally:
        torch.set_num_threads(threads)
        for n, v in saved.items():
            setattr(ops, n, v)
        importlib.reload(ops)
    # Adam's first step moves every weight by ~lr * g/(|g|+eps): elements whose gradient is at the fp32-rounding
    # floor are ill-conditioned, so compare the bulk tightly and bound the rest by the step size
    diff = np.abs(r0["p32"] - ref)
    lr = tr.get_lr()
    assert diff.max() <= 2.0 * lr, (diff.max(), lr)
    # (bf16 exchange rounds every gradient once more: a few more sign flips at the rounding floor)
    assert (diff > 1e-6).mean() < (2e-3 if reduce_dtype == "fp32" else 1e-2), (diff > 1e-6).mean()


def test_shard_batches_round_robin_with_padding():
    from espresso_b200.data.batching import batch_by_size, ordered_indices, shard_batches

    sizes = np.array([10, 50, 20, 40, 30, 60, 70])
    order = ordered_indices(sizes)
    assert list(sizes[order]) == sorted(sizes)
    batches = batch_by_size(order, sizes, max_tokens=100, max_sentences=3)
    flat = np.concatenate(batches)
    assert sorted(flat.tolist()) == list(range(7))
    for b in batches:
        assert len(b) <= 3 and len(b) * sizes[b].max() <= 100
    shards = [shard_batches(batches, 2, r) for r in range(2)]
    assert len(shards[0]) == len(shards[1]) == (len(batches) + 1) // 2
    got = [x for i in range(len(shards[0])) for r in range(2) for x in shards[r][i].tolist()]
    assert sorted(got) == list(range(7))

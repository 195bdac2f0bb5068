"""GPU, 2 ranks over NCCL (skipped when fewer than 2 GPUs are visible): the data-parallel step through the REAL fused
backward hook (fused.GatedXattnBlockFn -> train.GradBucket.on_block_backward_done), with the reference's step shape --
two backward passes per optimizer step (LAION + MMC4, train_utils.py:109-118,153-172; the first under no_sync()).

Each rank runs its own two micro-batches; the all-reduced flat gradient must equal the sum of the gradients a single
process computes for all four (rank, micro-batch) pairs, and a second backward WITHOUT no_sync() must be refused."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

VIT = dict(image_size=56, patch_size=14, width=128, layers=2, heads=2, output_dim=128)
MPT = dict(d_model=128, n_heads=2, n_layers=4, vocab_size=61, max_seq_len=64, expansion_ratio=2)


def _build():
    from open_flamingo_b200.testing import build_flamingo
    model, _, tok = build_flamingo(VIT, MPT, device="cuda", gate_init=1.0, seed=0)
    return model.train(), tok


def _batch(tok, seed):
    from open_flamingo_b200.testing import synthetic_batch
    media_id, eoc_id = tok.encode("<image>")[-1], tok.encode("<|endofchunk|>")[-1]
    return {k: v.cuda() for k, v in synthetic_batch(3, 2, 24, media_id, eoc_id, 61, image_size=56, seed=seed).items()}


def _fwd_bwd(model, batch):
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = model(vision_x=batch["vision_x"], lang_x=batch["lang_x"], attention_mask=batch["attention_mask"], labels=batch["labels"])
    out.loss.backward()


def worker():
    import torch.distributed as dist
    from open_flamingo_b200.train import FlatTrainer
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    model, tok = _build()
    trainer = FlatTrainer(model, lr=1e-3, num_chunks=3)
    launched_during_first = None
    trainer.zero_grad()
    with trainer.no_sync():
        _fwd_bwd(model, _batch(tok, 10 * rank + 1))
        launched_during_first = len(trainer.bucket._launched)
    _fwd_bwd(model, _batch(tok, 10 * rank + 2))
    launched_during_second = len(trainer.bucket._launched)
    trainer.bucket.finish()
    torch.cuda.synchronize()
    got = trainer.bucket.grads.detach().clone()
    # single-process reference on this rank: all four (rank, micro-batch) batches, no collectives
    trainer.bucket.zero()
    with trainer.no_sync():
        for r in range(world):
            for mb in (1, 2):
                _fwd_bwd(model, _batch(tok, 10 * r + mb))
    torch.cuda.synchronize()
    want = trainer.bucket.grads.detach().clone()
    rel = ((got - want).norm() / want.norm()).item()
    # misuse: second backward after the chunks went out
    trainer.bucket.zero()
    _fwd_bwd(model, _batch(tok, 3))
    refused = False
    try:
        _fwd_bwd(model, _batch(tok, 4))
    except RuntimeError as e:
        refused = "no_sync" in str(e)
    trainer.bucket.finish()
    torch.cuda.synchronize()
    ok = launched_during_first == 0 and launched_during_second >= 1 and rel <= 2e-3 and refused
    print(f"rank {rank}: launched {launched_during_first}/{launched_during_second} rel {rel:.3e} refused {refused} -> {'OK' if ok else 'FAIL'}",
          flush=True)
    dist.barrier()
    os._exit(0 if ok else 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (NCCL)")
def test_two_micro_batches_two_ranks_nccl():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.abspath(__file__), "--worker"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("OK") == 2, r.stdout[-2000:]


def test_two_micro_batches_single_gpu_equals_concatenated_batch():
    """World 1 through the real fused hook: backward(A) under no_sync + backward(B) == gradient of the summed losses."""
    from open_flamingo_b200.train import FlatTrainer
    model, tok = _build()
    trainer = FlatTrainer(model, lr=1e-3, num_chunks=3)
    a, b = _batch(tok, 1), _batch(tok, 2)
    trainer.zero_grad()
    with trainer.no_sync():
        _fwd_bwd(model, a)
    _fwd_bwd(model, b)
    trainer.bucket.finish()
    got = trainer.bucket.grads.detach().clone()
    ga, gb = [], []
    for dst, batch in ((ga, a), (gb, b)):
        trainer.bucket.zero()
        _fwd_bwd(model, batch)
        trainer.bucket.finish()
        dst.append(trainer.bucket.grads.detach().clone())
    want = ga[0] + gb[0]
    assert ((got - want).norm() / want.norm()).item() <= 2e-3
    trainer.close()


if __name__ == "__main__" and "--worker" in sys.argv:
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    worker()

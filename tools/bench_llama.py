"""OF-9B v1 shape (ViT-L/14 + LLaMA-7B dims, cross_attn_every_n_layers=4): the CUDA-graphed training step with the
frozen LLaMA blocks on libofk (lm_blocks.ENABLED = True) against HF's eager blocks (False), in one process, the two
arms alternating window by window.  Per arm: median tokens/s and ms/step, the step loss on the same weights and
batch, and one frozen block's forward + backward (fast path against HF under autocast) at R = B * T rows.  Prints one
JSON line.

    python tools/bench_llama.py --steps 5 --reps 3 [--out profiles/r03_bench_llama.json]
"""
import argparse
import contextlib
import gc
import io
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
# the two arms' graphs and eager activations at 7B size fragment the caching allocator's fixed-size segments
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

import torch  # noqa: E402

VIT_L14 = dict(image_size=224, patch_size=14, width=1024, layers=24, heads=16, output_dim=768)


def gpu_info():
    """Card name and power limit, read in the same process as the measurement."""
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clk = [s.strip() for s in r.stdout.strip().split(",")]
        return dict(gpu=name, power_limit=power, clocks_max_sm=clk)
    except Exception as e:  # noqa: BLE001 - the measurement stands; say what could not be read
        return dict(gpu=torch.cuda.get_device_name(), power_limit=f"unavailable ({e!r})")


def time_ms(fn, n):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def block_times(llama_kw, B, T, reps, iters):
    """One frozen LlamaDecoderLayer at the model's dims: forward + backward (input gradient), fast against HF."""
    from transformers import LlamaConfig
    from transformers.models.llama.modeling_llama import LlamaDecoderLayer, LlamaRotaryEmbedding
    from open_flamingo_b200 import lm_blocks
    cfg = LlamaConfig(**llama_kw)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(0)
    with torch.device("cuda"):
        blk = LlamaDecoderLayer(cfg, 0).requires_grad_(False)
        rot = LlamaRotaryEmbedding(cfg)
    fast = lm_blocks.accelerate(blk)
    x = torch.randn(B, T, cfg.hidden_size, device="cuda").requires_grad_(True)
    pe = rot(x, torch.arange(T, device="cuda").view(1, T))
    dy = torch.randn_like(x)

    def run(use_fast):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = fast(x, position_embeddings=pe) if use_fast else blk(x, position_embeddings=pe)
        assert y is not None
        y.backward(dy)
        x.grad = None

    out = {}
    for arm in (True, False):
        run(arm)
    samples = {True: [], False: []}
    for _ in range(reps):
        for arm in (True, False):
            samples[arm].append(time_ms(lambda: run(arm), iters))
    out["block_fwd_bwd_ms_fast"] = statistics.median(samples[True])
    out["block_fwd_bwd_ms_hf"] = statistics.median(samples[False])
    out["block_rows"] = B * T
    del blk, fast, x
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5, help="graphed steps per timed window")
    ap.add_argument("--reps", type=int, default=3, help="timed windows per arm (alternating)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--t-img", type=int, default=5)
    ap.add_argument("--t-txt", type=int, default=512)
    ap.add_argument("--layers", type=int, default=32, help="LLaMA decoder layers (32 = LLaMA-7B)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_llama.py measures on the GPU; there is no CPU fallback"
    torch.cuda.set_device(0)

    from open_flamingo_b200 import lm_blocks
    from open_flamingo_b200.testing import LLAMA_7B, build_flamingo, build_llama, synthetic_batch
    from open_flamingo_b200.train import FlatTrainer, GraphedTrainStep

    llama_kw = dict(LLAMA_7B, num_hidden_layers=args.layers, max_position_embeddings=2048)
    res = dict(model="OF-9B-v1 (ViT-L/14 + LLaMA-7B dims, random init)", layers=args.layers, every=4,
               batch=args.batch, t_img=args.t_img, t_txt=args.t_txt, steps=args.steps, reps=args.reps,
               precision="amp_bf16", **gpu_info())
    res.update(block_times(llama_kw, args.batch, args.t_txt, args.reps, 3))

    with contextlib.redirect_stdout(io.StringIO()):
        model, _, tok = build_flamingo(VIT_L14, llama_kw, cross_attn_every_n_layers=4, device="cuda", seed=0,
                                       gate_init=1.0, lm_builder=build_llama)
    model.train()
    media_id, eoc_id = tok.encode("<image>")[-1], tok.encode("<|endofchunk|>")[-1]
    batch = {k: v.cuda() for k, v in synthetic_batch(args.batch, args.t_img, args.t_txt, media_id, eoc_id,
                                                     llama_kw["vocab_size"], image_size=224, seed=100).items()}
    trainer = FlatTrainer(model, lr=1e-4, weight_decay=0.1, max_grad_norm=1.0)

    # the same weights and batch through both arms: the losses must agree
    arms = {"fast": True, "hf": False}
    for name, on in arms.items():
        lm_blocks.ENABLED = on
        trainer.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = model(vision_x=batch["vision_x"], lang_x=batch["lang_x"], attention_mask=batch["attention_mask"],
                         labels=batch["labels"]).loss
        loss.backward()
        res[f"loss_{name}"] = loss.item()
    trainer.zero_grad()
    res["loss_rel_diff"] = abs(res["loss_fast"] - res["loss_hf"]) / abs(res["loss_hf"])

    # Both arms' captured graphs do not fit in memory together at this size (each holds a private pool of its
    # activations), so every timed window captures its arm afresh and frees it afterwards; the arms alternate.
    samples = {n: [] for n in arms}
    last_loss = {}
    for _ in range(args.reps):
        for name, on in arms.items():
            lm_blocks.ENABLED = on
            g = GraphedTrainStep(model, trainer, batch, warmup=args.warmup)
            res[f"graphed_{name}"] = g.ok
            if not g.ok:
                res[f"graph_error_{name}"] = g.error
            g(batch)

            def step():
                last_loss[name] = g(batch)
            samples[name].append(time_ms(step, args.steps))
            last_loss[name] = float(last_loss[name].item())
            del g, step
            gc.collect()                # the graph's private memory pool goes with the last reference to it
            torch.cuda.empty_cache()
    lm_blocks.ENABLED = True
    tokens = args.batch * args.t_txt
    for name in arms:
        ms = statistics.median(samples[name])
        res[f"ms_step_{name}"] = ms
        res[f"tokens_per_s_{name}"] = tokens / (ms / 1e3)
        res[f"ms_step_samples_{name}"] = samples[name]
        res[f"last_step_loss_{name}"] = last_loss[name]
    res["speedup"] = res["tokens_per_s_fast"] / res["tokens_per_s_hf"]
    res["peak_mem_gb"] = torch.cuda.max_memory_allocated() / 1e9
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

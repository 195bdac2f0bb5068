#!/usr/bin/env python
"""bench.py -- OF-3B training tokens/sec on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]      # CPU port of the reference (oracle), host cores

Workload (BASELINE.json configs[1], SURVEY.md C2): OF-3B = ViT-L/14 + MPT-1B-shaped LM (HF MptForCausalLM,
random init -- there is no network for checkpoints) with a gated cross-attention block before every decoder
block; per GPU batch 32 sequences x (2 images 224x224, 256 text tokens); amp_bf16 numerics (fp32 master
weights, bf16 GEMM operands); a step = zero_grad + forward + backward (+ NCCL all-reduce of the resampler and
gated-xattn gradients when N > 1) + global-norm clip + AdamW.  Synthetic data.  Weak scaling.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

VIT_L14 = dict(image_size=224, patch_size=14, width=1024, layers=24, heads=16, output_dim=768)
METRIC = "OF-3B training tokens/sec"          # BASELINE.json's metric (the default --model of3b)
LM_NAME = {"of3b": "MPT-1B", "of9b": "MPT-7B"}


def metric_name(model):
    return METRIC if model == "of3b" else f"{model.upper().replace('OF', 'OF-')} training tokens/sec"
UNIT = "tokens/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gemm-shapes", default=None, help="write the per-shape GEMM table of the instrumented pass here")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--t_img", type=int, default=2)
    ap.add_argument("--t_txt", type=int, default=256)
    ap.add_argument("--model", default="of3b", choices=["of3b", "of9b", "tiny"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graph", default="auto", choices=["auto", "off"],
                    help="capture the whole training step into one CUDA graph (falls back to eager if capture fails)")
    ap.add_argument("--lm", default="fused", choices=["fused", "eager"],
                    help="frozen-LM decoder blocks: 'fused' = libofk kernels (lm_blocks.py), 'eager' = HF PyTorch "
                         "modules as in the reference")
    ap.add_argument("--cpu-sample-batch", type=int, default=1)
    ap.add_argument("--no-gpu-eager-ref", action="store_true",
                    help="skip timing the reference's eager-PyTorch path (oracle restatement) on the same GPU")
    ap.add_argument("--micro-batches", type=int, default=1,
                    help="backward passes per optimizer step (the reference's step is LAION + MMC4 = 2, "
                         "train_utils.py:118,172); all but the last run under trainer.no_sync(); tokens/s counts all of them")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32): "
                         "its loss and a fixed seeded sample of the updated fp32 master weights")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def model_dims(name):
    from open_flamingo_b200.testing import MPT_1B, MPT_7B
    if name == "of3b":
        return VIT_L14, dict(MPT_1B), 1
    if name == "of9b":
        return VIT_L14, dict(MPT_7B), 4
    return (dict(image_size=56, patch_size=14, width=128, layers=2, heads=2, output_dim=128),
            dict(d_model=128, n_heads=2, n_layers=2, vocab_size=61, max_seq_len=512, expansion_ratio=2), 1)


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons = [], set()
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    out["sm_max_mhz"] = float(parts[2])
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out["sm_mhz"] = statistics.median(sm)
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


# ----------------------------------------------------------------------------------------------- GEMM timing hook
class GemmTimer:
    """CUDA-event timing of every tcgen05 GEMM launch inside the timed region (events are recorded on the stream
    the kernel is launched on; the overhead is two event records per launch)."""

    def __init__(self):
        self.records = []

    def wrap(self, ops_mod):
        timer = self

        def make(orig):
            def timed(a, b, **kw):
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
                out = orig(a, b, **kw)
                e1.record()
                a_mn, b_mn = kw.get("a_mn", False), kw.get("b_mn", False)
                m, k = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
                n = b.shape[1] if b_mn else b.shape[0]
                m, n, k = kw.get("M") or m, kw.get("N") or n, kw.get("K") or k
                timer.records.append((e0, e1, 2.0 * m * n * k, kw.get("epi", 0), int(a_mn), int(b_mn),
                                      (m, n, k, kw.get("splits", 1))))
                return out
            return timed

        self._mod = ops_mod
        self._orig = {name: getattr(ops_mod, name) for name in ("gemm", "gemm_grouped")}
        for name, fn in self._orig.items():   # fused.py / vit.py call these through the module, so this covers them
            setattr(ops_mod, name, make(fn))

    def unwrap(self):
        for name, fn in self._orig.items():
            setattr(self._mod, name, fn)

    def by_shape(self, steps):
        """Per (variant, M, N, K, splits): launches/step, mean us, TFLOP/s, tiles and waves of the 2-CTA 256x256 grid."""
        acc = {}
        for e0, e1, flop, epi, a_mn, b_mn, shape in self.records:
            d = acc.setdefault((epi, a_mn, b_mn) + shape, [0.0, 0.0, 0])
            d[0] += e0.elapsed_time(e1); d[1] += flop; d[2] += 1
        rows = []
        for (epi, a_mn, b_mn, m, n, k, splits), (ms, flop, cnt) in acc.items():
            tiles = ((m + 255) // 256) * ((n + 255) // 256) * splits
            rows.append({"epi": epi, "a_mn": a_mn, "b_mn": b_mn, "M": m, "N": n, "K": k, "splits": splits,
                         "launches_per_step": cnt / steps, "ms_per_step": ms / steps, "us_per_launch": 1e3 * ms / cnt,
                         "TFLOP/s": flop / (ms * 1e-3) / 1e12 if ms else 0.0, "tiles": tiles, "waves_74": tiles / 74.0})
        return sorted(rows, key=lambda r: -r["ms_per_step"])

    def summary(self):
        tot_ms, tot_flop = 0.0, 0.0
        by = {}
        for e0, e1, flop, epi, a_mn, b_mn, _shape in self.records:
            ms = e0.elapsed_time(e1)
            tot_ms += ms
            tot_flop += flop
            key = f"epi{epi}_a{a_mn}b{b_mn}"
            d = by.setdefault(key, [0.0, 0.0, 0])
            d[0] += ms; d[1] += flop; d[2] += 1
        return tot_ms, tot_flop, len(self.records), by


class GraphGemmTimer:
    """Per-GEMM device times INSIDE a captured CUDA graph of the training step: an event-record node with the
    cudaEventRecordExternal flag before and after every tcgen05 GEMM launch (cudart called directly on the capturing
    stream; torch.cuda.Event cannot be recorded during capture).  Inside a graph there is no CPU between the nodes, so
    the pairs bracket exactly the kernel (plus one node-to-node gap), unlike event pairs in an eager pass, which also
    contain whatever time the host needs to enqueue the launch when the step is CPU-bound."""

    def __init__(self):
        import ctypes
        self.ct = ctypes
        self.rt = None
        for name in ("libcudart.so.12", "libcudart.so"):
            try:
                self.rt = ctypes.CDLL(name)
                break
            except OSError:
                continue
        if self.rt is None:
            raise RuntimeError("libcudart not loadable")
        self.rt.cudaEventCreate.argtypes = [ctypes.POINTER(ctypes.c_void_p)]
        self.rt.cudaEventRecordWithFlags.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint]
        self.rt.cudaEventElapsedTime.argtypes = [ctypes.POINTER(ctypes.c_float), ctypes.c_void_p, ctypes.c_void_p]
        self.rt.cudaEventDestroy.argtypes = [ctypes.c_void_p]
        self.pairs = []      # (ev0, ev1, flop, epi, a_mn, b_mn, shape)
        self.acc = {}        # index -> accumulated ms
        self.replays = 0

    def _event(self):
        ev = self.ct.c_void_p()
        if self.rt.cudaEventCreate(self.ct.byref(ev)) != 0:
            raise RuntimeError("cudaEventCreate failed")
        return ev

    def _record(self, ev):
        rc = self.rt.cudaEventRecordWithFlags(ev, self.ct.c_void_p(torch.cuda.current_stream().cuda_stream), 1)  # 1 = External
        if rc != 0:
            raise RuntimeError(f"cudaEventRecordWithFlags failed ({rc})")

    def wrap(self, ops_mod):
        timer = self

        def make(orig):
            def timed(a, b, **kw):
                if not torch.cuda.is_current_stream_capturing():      # warm-up passes: the External flag is capture-only
                    return orig(a, b, **kw)
                e0, e1 = timer._event(), timer._event()
                timer._record(e0)
                out = orig(a, b, **kw)
                timer._record(e1)
                a_mn, b_mn = kw.get("a_mn", False), kw.get("b_mn", False)
                m, k = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
                n = b.shape[1] if b_mn else b.shape[0]
                m, n, k = kw.get("M") or m, kw.get("N") or n, kw.get("K") or k
                timer.pairs.append((e0, e1, 2.0 * m * n * k, kw.get("epi", 0), int(a_mn), int(b_mn), (m, n, k, kw.get("splits", 1))))
                return out
            return timed

        self._mod = ops_mod
        self._orig = {name: getattr(ops_mod, name) for name in ("gemm", "gemm_grouped")}
        for name, fn in self._orig.items():
            setattr(ops_mod, name, make(fn))

    def unwrap(self):
        for name, fn in self._orig.items():
            setattr(self._mod, name, fn)

    def collect(self):
        """Call after each replay + synchronize: accumulate the elapsed time of every pair."""
        ms = self.ct.c_float()
        for i, (e0, e1, *_rest) in enumerate(self.pairs):
            if self.rt.cudaEventElapsedTime(self.ct.byref(ms), e0, e1) != 0:
                raise RuntimeError("cudaEventElapsedTime failed")
            self.acc[i] = self.acc.get(i, 0.0) + ms.value
        self.replays += 1

    def records_ms(self):
        return [(self.acc[i] / self.replays, flop, epi, a_mn, b_mn, shape)
                for i, (_e0, _e1, flop, epi, a_mn, b_mn, shape) in enumerate(self.pairs)]


# ----------------------------------------------------------------------------------------------- reference arm (CPU port)
def build_cpu_oracle(model_name, seed=0):
    """Oracle (CPU fp32 port of the reference) with the bench model's architecture, random init."""
    from oracle import flamingo_oracle as O
    from open_flamingo_b200.testing import build_mpt
    from open_flamingo_b200.src.helpers import PerceiverResampler, GatedCrossAttentionBlock
    from open_flamingo_b200.src.vit import VisionTransformer
    vit_cfg, mpt_kw, every = model_dims(model_name)
    torch.manual_seed(seed)
    lm = build_mpt(mpt_kw, seed=seed + 1)
    for p in lm.parameters():
        p.requires_grad_(False)
    sd = {}
    vit = VisionTransformer(**vit_cfg)
    for k, v in vit.state_dict().items():
        sd["vision_encoder." + k] = v.detach()
    per = PerceiverResampler(dim=vit_cfg["width"])
    for k, v in per.state_dict().items():
        sd["perceiver." + k] = v.detach().requires_grad_(True)
    n_layers = mpt_kw["n_layers"]
    g = torch.Generator().manual_seed(seed + 2)
    for i in range(n_layers):
        if (i + 1) % every:
            continue
        blk = GatedCrossAttentionBlock(dim=mpt_kw["d_model"], dim_visual=vit_cfg["width"])
        for k, v in blk.state_dict().items():
            v = v.detach()
            if k.endswith("_gate"):
                v = torch.rand(1, generator=g) * 2 - 1
            sd[f"lang_encoder.gated_cross_attn_layers.{i}.{k}"] = v.requires_grad_(True)
    media_id, eoc_id = mpt_kw["vocab_size"] + 1, mpt_kw["vocab_size"]
    lm.resize_token_embeddings(mpt_kw["vocab_size"] + 3)
    orc = O.OracleFlamingo(lm, lm.transformer.blocks, sd, media_id, xattn_every=every, vit_heads=vit_cfg["heads"],
                           vit_patch=vit_cfg["patch_size"])
    trainable = [v for v in sd.values() if v.requires_grad]
    return orc, trainable, media_id, eoc_id, mpt_kw["vocab_size"], vit_cfg["image_size"]


def cpu_oracle_step(orc, trainable, batch):
    for t in trainable:
        t.grad = None
    out = orc.forward(batch["vision_x"], batch["lang_x"], attention_mask=batch["attention_mask"], labels=batch["labels"])
    out.loss.backward()
    return float(out.loss.detach())


def usable_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def time_cpu_oracle(model_name, sample_batch, t_img, t_txt, steps, warmup):
    from open_flamingo_b200.testing import synthetic_batch
    cores = usable_cores()
    torch.set_num_threads(cores)
    orc, trainable, media_id, eoc_id, vocab, image_size = build_cpu_oracle(model_name)
    batch = synthetic_batch(sample_batch, t_img, t_txt, media_id, eoc_id, vocab, image_size=image_size, seed=1)
    for _ in range(warmup):
        cpu_oracle_step(orc, trainable, batch)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_oracle_step(orc, trainable, batch)
    dt = (time.perf_counter() - t0) / max(1, steps)
    return dict(value=sample_batch * t_txt / dt, unit=UNIT, cores=cores, kind="port",
                sample=f"{steps} fwd+bwd step(s) of {sample_batch} sequence(s) x ({t_img} images, {t_txt} tokens), "
                       f"fp32, torch.set_num_threads({cores}), {dt*1e3:.0f} ms/step"), dt


def time_gpu_eager_reference(model, every, batch, steps):
    """The like-for-like bar (SURVEY.md section 2a / 8d): the reference's eager-PyTorch forward + backward -- the oracle
    restatement, module for module the reference's ops (oracle/flamingo_oracle.py, pinned to the unmodified reference by
    tests/golden) around the same HF LM -- on THIS GPU, same weights, same batch, fp32 and torch.autocast(bf16)
    (train_utils.py:34-43).  No optimizer / clip in its timed region (ours includes them), so the ratio is conservative."""
    from oracle.harness import oracle_from_model, oracle_train_step
    out = {}
    orc, sd, trainable = oracle_from_model(model, every)
    tokens = batch["lang_x"].numel()
    for name, dt in (("amp_bf16", torch.bfloat16), ("fp32", None)):
        try:
            for _ in range(2):
                oracle_train_step(orc, sd, trainable, batch, amp_dtype=dt)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                oracle_train_step(orc, sd, trainable, batch, amp_dtype=dt)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"value": tokens / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms}
        except Exception as e:  # pragma: no cover - e.g. out of memory on a smaller part
            out[name] = {"error": repr(e)[:200]}
            torch.cuda.empty_cache()
    out["what"] = ("reference eager PyTorch path (oracle restatement of open_flamingo/src on the same HF LM), fwd+bwd only, "
                   f"same GPU / weights / batch, {steps} steps after 2 warm-up")
    del orc, sd
    torch.cuda.empty_cache()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb, dt = time_cpu_oracle(args.model, args.cpu_sample_batch, args.t_img, args.t_txt, args.steps, args.warmup)
    line = {"impl": "reference", "metric": metric_name(args.model), "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.model.upper()} train step (CPU port of the reference, oracle/)",
                       "global_batch": args.cpu_sample_batch, "t_img": args.t_img, "seq_len": args.t_txt},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- output dump
DUMP_SAMPLE = 1 << 22      # sampled weights: 16 MB of float32


def dump_outputs(out_dir, loss, bucket, sample=DUMP_SAMPLE, seed=0):
    """What one training step hands back to its caller: the loss, and the fp32 master weights its AdamW update left.
    The flat weight buffer holds ~1e9 values at OF-3B, so it is sampled at positions drawn from a fixed seed (the same
    positions for the same --model); a buffer no larger than `sample` is written whole.

    The step's gradient is not written: a single step reproduces its gradient to ~3e-8 (float atomics), but the
    training steps before the dump amplify that about tenfold per step, so two runs of the same build differ by ~0.8
    relative L2 in the last step's gradient against ~2e-3 in the loss and ~6e-4 in the weights (OF-3B, --steps 8,
    B200 at 1000 W)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().float().reshape(()), "params": bucket.params}
    if bucket.total > sample:
        pos = np.sort(np.random.default_rng(seed).choice(bucket.total, size=sample, replace=False))
        arrays["params"] = bucket.params.index_select(0, torch.from_numpy(pos).to(bucket.device))
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy().astype(np.float32))


# ----------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch.distributed as dist
    from open_flamingo_b200 import _lib, ops
    from open_flamingo_b200.testing import build_flamingo, synthetic_batch
    from open_flamingo_b200.train import FlatTrainer, GraphedTrainStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        from open_flamingo_b200.train import configure_nccl_for_overlap
        configure_nccl_for_overlap()
        dist.init_process_group("nccl", device_id=dev)

    from open_flamingo_b200 import lm_blocks
    lm_blocks.ENABLED = args.lm == "fused"
    vit_cfg, mpt_kw, every = model_dims(args.model)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        model, _, tok = build_flamingo(vit_cfg, mpt_kw, cross_attn_every_n_layers=every, device=dev,
                                       freeze_lm_embeddings=True, seed=0, gate_init=1.0)
    model.train()
    media_id, eoc_id = tok.encode("<image>")[-1], tok.encode("<|endofchunk|>")[-1]
    trainer = FlatTrainer(model, lr=1e-4, weight_decay=0.1, max_grad_norm=1.0)
    B, T_img, T_txt = args.batch, args.t_img, args.t_txt
    host = synthetic_batch(B, T_img, T_txt, media_id, eoc_id, mpt_kw["vocab_size"], image_size=vit_cfg["image_size"],
                           seed=100 + rank, pin=True)
    MB = max(1, args.micro_batches)
    hosts = [host] + [synthetic_batch(B, T_img, T_txt, media_id, eoc_id, mpt_kw["vocab_size"], image_size=vit_cfg["image_size"],
                                      seed=1000 * (i + 1) + rank, pin=True) for i in range(MB - 1)]
    residents = [{k: v.to(dev) for k, v in hb.items()} for hb in hosts]
    resident = residents[0] if MB == 1 else residents
    host = hosts[0] if MB == 1 else hosts
    h2d_bytes = sum(v.numel() * v.element_size() for hb in hosts for v in hb.values())

    def fwd_bwd(batch):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model(vision_x=batch["vision_x"], lang_x=batch["lang_x"], attention_mask=batch["attention_mask"],
                        labels=batch["labels"])
        out.loss.backward()
        return out.loss

    def train_step(batch):
        batches = batch if isinstance(batch, (list, tuple)) else [batch]
        trainer.zero_grad()
        loss = None
        for i, b_ in enumerate(batches):
            if i + 1 < len(batches):
                with trainer.no_sync():     # gradient accumulation: chunks are reduced during the LAST backward only
                    l_ = fwd_bwd(b_)
            else:
                l_ = fwd_bwd(b_)
            loss = l_ if loss is None else loss + l_
        trainer.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # warm-up (also materialises bf16 caches, TMA descriptors, allocator pools)
    for _ in range(max(3, args.warmup)):
        train_step(resident)
    barrier()
    l0 = _lib.launch_count()
    train_step(resident)
    launches = _lib.launch_count() - l0          # libofk kernels per step (a graph replays exactly these nodes)
    graphed = None
    if args.graph == "auto":
        graphed = GraphedTrainStep(model, trainer, resident, warmup=1)
        if not graphed.ok:
            if rank == 0:
                print(f"[bench] CUDA-graph capture unavailable, running eagerly: {graphed.error}", file=sys.stderr)
                if os.environ.get("OFK_DEBUG"):
                    print(graphed.traceback, file=sys.stderr)
            graphed = None
        else:
            for _ in range(2):
                graphed(resident)
    barrier()
    run_step = (lambda batch: graphed(batch)) if graphed is not None else train_step
    graph_used = graphed is not None

    # ---- device-resident timing (value), clocks sampled during the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last = {}

    def timed_step():
        last["loss"] = run_step(resident)

    ms_total = timed(timed_step, args.steps)
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        # before anything below runs the step again: the graph's loss buffer and the weights would move on
        dump_outputs(args.dump_outputs, last["loss"], trainer.bucket)
    ms_step = ms_total / args.steps
    tokens = world * B * T_txt * MB
    # host time needed to ENQUEUE one step (no sync inside): must stay well below ms_step or the GPU starves
    torch.cuda.synchronize()
    t_cpu0 = time.perf_counter()
    run_step(resident)
    cpu_enqueue_ms = (time.perf_counter() - t_cpu0) * 1e3
    torch.cuda.synchronize()

    # ---- same K steps again with a CUDA-event pair around every tcgen05 GEMM launch (roofline numerator/denominator)
    timer = GemmTimer()
    timer.wrap(ops)
    ms_instr = timed(lambda: train_step(resident), args.steps)
    timer.unwrap()
    gemm_ms, gemm_flop, gemm_n, gemm_by = timer.summary()
    gemm_steps = args.steps
    gemm_method = "CUDA-event pair around every GEMM launch of an eager pass of the same K steps (contains host enqueue gaps when CPU-bound)"
    shape_rows = timer.by_shape(args.steps)
    if graphed is not None:
        # preferred: the same pairs as external-event nodes inside a second captured graph of the step
        try:
            gt = GraphGemmTimer()
            gt.wrap(ops)
            try:
                g2 = GraphedTrainStep(model, trainer, resident, warmup=1)
            finally:
                gt.unwrap()
            if not g2.ok:
                raise RuntimeError(g2.error)
            for _ in range(2):
                g2(resident)
            torch.cuda.synchronize()
            gt.acc, gt.replays = {}, 0
            for _ in range(args.steps):
                g2(resident)
                torch.cuda.synchronize()
                gt.collect()
            recs = gt.records_ms()
            gemm_ms = sum(r[0] for r in recs)
            gemm_flop = sum(r[1] for r in recs)
            gemm_n = len(recs)
            gemm_steps = 1
            gemm_by = {}
            acc = {}
            for ms_, flop, epi, a_mn, b_mn, shape in recs:
                d = gemm_by.setdefault(f"epi{epi}_a{a_mn}b{b_mn}", [0.0, 0.0, 0])
                d[0] += ms_; d[1] += flop; d[2] += 1
                d2 = acc.setdefault((epi, a_mn, b_mn) + shape, [0.0, 0.0, 0])
                d2[0] += ms_; d2[1] += flop; d2[2] += 1
            shape_rows = []
            for (epi, a_mn, b_mn, m, n, k, splits), (ms_, flop, cnt) in acc.items():
                tiles = ((m + 255) // 256) * ((n + 255) // 256) * splits
                shape_rows.append({"epi": epi, "a_mn": a_mn, "b_mn": b_mn, "M": m, "N": n, "K": k, "splits": splits,
                                   "launches_per_step": cnt, "ms_per_step": ms_, "us_per_launch": 1e3 * ms_ / cnt,
                                   "TFLOP/s": flop / (ms_ * 1e-3) / 1e12 if ms_ else 0.0, "tiles": tiles, "waves_74": tiles / 74.0})
            shape_rows.sort(key=lambda r: -r["ms_per_step"])
            gemm_method = ("cudaEventRecordExternal node pair around every GEMM launch INSIDE a captured CUDA graph of the step, "
                           f"mean of {args.steps} replays")
            del g2
        except Exception as e:  # noqa: BLE001 - keep the eager numbers
            if rank == 0:
                print(f"[bench] in-graph GEMM timing unavailable ({e!r}); using the eager event pairs", file=sys.stderr)
    if args.gemm_shapes and rank == 0:
        with open(args.gemm_shapes, "w") as f:
            json.dump(shape_rows, f, indent=1)

    # ---- end-to-end timing: pinned host inputs -> device every step, loss read back every step
    def e2e_step():
        if graphed is not None:
            loss = graphed(host)                 # pinned host tensors -> static device buffers (async H2D) -> replay
        else:
            hb = host if isinstance(host, list) else [host]
            loss = train_step([{k: v.to(dev, non_blocking=True) for k, v in h_.items()} for h_ in hb])
        return float(loss.item())

    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps) / args.steps

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else \
            "fallback 1.4 PF sustained (B200_PROFILING.md)"
        achieved_tf = gemm_flop / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        traffic = None
        try:  # mean DRAM bytes per launch of the FFN GEMMs from the committed `ncu --set full` capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "gemm_traffic.json")))
            traffic = tj.get("mean_dram_bytes_per_launch")
        except Exception:
            pass
        roofline = {"bound": "tensor", "kernel": "ofk::gemm2_kernel<A_MN,B_MN,EPI> / gemm_kernel<BN,...> (tcgen05 cta_group::2 / ::1, every launch in the timed region)",
                    "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                    "peak_source": peak_src, "traffic": traffic,
                    "traffic_source": "STATIC: mean dram__bytes_read+write per launch of the FFN GEMMs in the committed ncu --set full "
                                      "capture profiles/gemm_traffic.json (see its `build` field), not re-measured by this run",
                    "launches_per_step": gemm_n / gemm_steps, "gemm_ms_per_step": gemm_ms / gemm_steps,
                    "share_of_step": (gemm_ms / gemm_steps) / ms_step if ms_step else None,
                    "method": gemm_method,
                    "eager_instrumented_ms_per_step": ms_instr / args.steps,
                    "by_variant": {k: {"TFLOP/s": v[1] / (v[0] * 1e-3) / 1e12 if v[0] else 0.0, "ms_per_step": v[0] / gemm_steps,
                                       "launches_per_step": v[2] / gemm_steps} for k, v in sorted(gemm_by.items())}}
        gpu_eager = None
        if not args.no_gpu_eager_ref and world == 1:
            try:
                graphed = None                  # release the captured graph's private pool before the eager run
                torch.cuda.empty_cache()
                gpu_eager = time_gpu_eager_reference(model, every, residents[0], steps=3)
                for k_ in ("amp_bf16", "fp32"):
                    if "value" in gpu_eager.get(k_, {}):
                        gpu_eager[k_]["ours_over_this"] = (tokens / (ms_step * 1e-3)) / gpu_eager[k_]["value"]
            except Exception as e:  # pragma: no cover
                gpu_eager = {"error": repr(e)[:200]}
        cpu_baseline = None
        if not args.no_cpu_baseline and world == 1:
            try:
                cpu_baseline, _ = time_cpu_oracle(args.model, args.cpu_sample_batch, T_img, T_txt, steps=1, warmup=0)
            except Exception as e:  # pragma: no cover
                cpu_baseline = {"error": repr(e)}
        line = {"metric": metric_name(args.model), "value": tokens / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"{args.model.upper()} (ViT-L/14 + {LM_NAME.get(args.model, 'tiny')}-shaped HF MptForCausalLM, xattn_every={every}) "
                                       "amp_bf16 train step: fwd+bwd+grad all-reduce+clip+AdamW",
                           "global_batch": world * B * MB, "per_gpu_batch": B, "micro_batches": MB, "t_img": T_img, "seq_len": T_txt,
                           "parallelism": f"dp{world}", "frozen_lm_blocks": args.lm, "cuda_graph": graph_used, "l2": "per-step working set (>10 GB weights+activations) exceeds the 126 MB L2; no explicit flush",
                           "trainable_params": sum(p.numel() for p in model.parameters() if p.requires_grad)},
                "e2e": {"value": tokens / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
                "gpu_launches": launches, "cpu_enqueue_ms_per_step": cpu_enqueue_ms, "clocks": clocks,
                "roofline": roofline}
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if gpu_eager is not None:
            line["gpu_eager_reference"] = gpu_eager
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear down in a hang-proof order: release the captured graph (it holds NCCL kernels) before touching the
        # communicator, synchronise, and leave without running NCCL's destructor-time collectives.
        graphed = None
        torch.cuda.synchronize()
        try:
            dist.barrier()
        except Exception:
            pass
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

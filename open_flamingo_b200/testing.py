"""Offline construction helpers (no hub / no open_clip): a tokenizer-like object and random-init model builders
with the OF-3B / OF-9B shapes (MPT, and LLaMA for the first OF-9B release).  Used by tests, __graft_entry__.smoke() and bench.py."""
import torch

from .src.factory import create_model_and_transforms
from .src.vit import CLIPVisionStandIn, VisionTransformer


class SimpleTokenizer:
    """Minimal tokenizer-like object for create_model_and_transforms: ids 0..base_vocab-1 are ordinary tokens,
    special tokens are appended in the order they are added (as HF tokenizers do, factory.py:57-63)."""

    def __init__(self, base_vocab, pad_token=None):
        self.base_vocab = base_vocab
        self.special = {}
        self.pad_token = pad_token
        self.padding_side = "right"

    def add_special_tokens(self, d):
        added = 0
        toks = list(d.get("additional_special_tokens", []))
        if "pad_token" in d:
            toks.append(d["pad_token"])
            self.pad_token = d["pad_token"]
        for t in toks:
            if t not in self.special:
                self.special[t] = self.base_vocab + len(self.special)
                added += 1
        return added

    def encode(self, text):
        if text in self.special:
            return [self.special[text]]
        raise KeyError(f"SimpleTokenizer only encodes its special tokens, got {text!r}")

    @property
    def pad_token_id(self):
        return None if self.pad_token is None else self.special[self.pad_token]

    def __len__(self):
        return self.base_vocab + len(self.special)


MPT_1B = dict(d_model=2048, n_heads=16, n_layers=24, vocab_size=50277, max_seq_len=2048, expansion_ratio=4)
MPT_7B = dict(d_model=4096, n_heads=32, n_layers=32, vocab_size=50277, max_seq_len=2048, expansion_ratio=4)


def build_mpt(mpt_kw, dtype=torch.float32, device="cpu", seed=0):
    """Random-init HF MptForCausalLM (the stand-in for anas-awadalla/mpt-1b-redpajama-200b: same dims, 1.31 B
    params; the hub checkpoint's remote code is unavailable offline)."""
    from transformers import MptConfig, MptForCausalLM
    torch.manual_seed(seed)
    cfg = MptConfig(**mpt_kw)
    with torch.device(device):
        lm = MptForCausalLM(cfg)
    return lm.to(dtype).eval()


# LLaMA-7B, the language model of the first OpenFlamingo-9B release
LLAMA_7B = dict(hidden_size=4096, num_hidden_layers=32, num_attention_heads=32, num_key_value_heads=32,
                intermediate_size=11008, vocab_size=32000)


def build_llama(llama_kw, dtype=torch.float32, device="cpu", seed=0):
    """Random-init HF LlamaForCausalLM with the given LlamaConfig fields (SDPA attention, HF's default)."""
    from transformers import LlamaConfig, LlamaForCausalLM
    torch.manual_seed(seed)
    cfg = LlamaConfig(**llama_kw)
    cfg._attn_implementation = "sdpa"
    with torch.device(device):
        lm = LlamaForCausalLM(cfg)
    return lm.to(dtype).eval()


def build_flamingo(vit_cfg, mpt_kw, cross_attn_every_n_layers=1, device="cuda", freeze_lm_embeddings=True, seed=0,
                   lm_dtype=torch.float32, gate_init=None, lm_builder=build_mpt):
    """Random-init Flamingo through the public factory.  gate_init: None keeps the reference's zero gates
    (helpers.py:255,258); a float f draws gates ~ U(-f, f) so the gated path is actually exercised.
    lm_builder(mpt_kw, dtype=, device=, seed=) makes the language model: build_mpt (default) or build_llama, with
    `mpt_kw` the matching config fields."""
    torch.manual_seed(seed)
    with torch.device(device):
        vit = VisionTransformer(**vit_cfg)
    lm = lm_builder(mpt_kw, dtype=lm_dtype, device=device, seed=seed + 1)
    base_vocab = mpt_kw["vocab_size"]
    tok = SimpleTokenizer(base_vocab)
    model, image_processor, tok = create_model_and_transforms(
        CLIPVisionStandIn(vit), None, lm, tok, cross_attn_every_n_layers=cross_attn_every_n_layers,
        freeze_lm_embeddings=freeze_lm_embeddings)
    model = model.to(device)
    if gate_init is not None:
        g = torch.Generator().manual_seed(seed + 2)
        with torch.no_grad():
            for name, p in model.named_parameters():
                if name.endswith("attn_gate") or name.endswith("ff_gate"):
                    p.copy_(((torch.rand(1, generator=g) * 2 - 1) * gate_init).to(p.device))
    return model, image_processor, tok


def synthetic_batch(B, T_img, T_txt, media_id, eoc_id, vocab, image_size=224, device="cpu", seed=0, pin=False):
    """Synthetic interleaved batch with the shapes the MMC4 pipeline produces (data.py:138-268): `<image>` at
    positions k*T_txt/T_img, `<|endofchunk|>` before every `<image>` but the first, labels mask `<image>`
    (train_utils.py:102-106,149)."""
    g = torch.Generator().manual_seed(seed)
    vision_x = torch.randn(B, T_img, 1, 3, image_size, image_size, generator=g)
    lang_x = torch.randint(0, vocab, (B, T_txt), generator=g)
    for k in range(T_img):
        pos = (k * T_txt) // T_img
        lang_x[:, pos] = media_id
        if k > 0:
            lang_x[:, pos - 1] = eoc_id
    labels = lang_x.clone()
    labels[labels == media_id] = -100
    attention_mask = torch.ones_like(lang_x)
    out = dict(vision_x=vision_x, lang_x=lang_x, attention_mask=attention_mask, labels=labels)
    if pin:
        out = {k: v.pin_memory() for k, v in out.items()}
    return out

"""Benchmark harness: a Llama-architecture decoder whose every base linear is `bitsandbytes.nn.Linear4bit`
(NF4 + double quant, frozen) wrapped by a LoRA adapter — the model `qlora.py` builds, minus the parts the
image cannot run (peft / accelerate are not installed; SURVEY.md Appendix C).

This is CALLER-side scaffolding for bench.py, not part of the product package:
  * architecture = HF `LlamaForCausalLM` (RMSNorm -> q/k/v/o -> RoPE -> causal SDPA -> SwiGLU MLP);
  * the base model is quantized THE WAY THE REFERENCE DOES IT (qlora.py:310-330): a `transformers.BitsAndBytesConfig(
    load_in_4bit, nf4, double_quant, compute_dtype=bf16)` drives HF's own `replace_with_bnb_linear`, which instantiates
    `bitsandbytes.nn.Linear4bit` (here: `shims/bitsandbytes` -> qlora_b200) on the meta device; every weight is then
    materialised as HF's `Bnb4bitQuantize.convert` does — `Params4bit(value, requires_grad=False, **old.__dict__)
    .to(device)` — from random-init N(0, 0.02) values generated per layer ON DEVICE (never a bf16 7B anywhere);
  * LoRA targets = `find_all_linear_names` (qlora.py:248-259); wrapper = peft's `lora.Linear4bit.forward`:
    `base(x) + lora_B(lora_A(dropout(x))) * (alpha / r)` (qlora.py:386-394), A kaiming-uniform / B zeros, bf16
    (qlora.py:396-399);
  * norms hold fp32 weights and compute in fp32 (qlora.py:400-401).  By default they emit bf16 — the value Linear4bit
    would cast to anyway (`x.to(compute_dtype)`), so the GEMM inputs are identical; `norm_out_fp32=True` keeps the
    reference's dtype flow instead (fp32 norm output -> Linear4bit sees fp32 in, returns fp32);
  * lm_head / embed_tokens bf16 and frozen, never quantized (qlora.py:257-258, 402-405);
  * gradient checkpointing per decoder layer (qlora.py:206,377) => every Linear4bit forward runs twice
    and the dX kernel once per step; no dW for the frozen base.
"""
from __future__ import annotations

import math
import os
import sys
import warnings
from dataclasses import dataclass

import torch
import torch.nn.functional as F
from torch import nn
from torch.utils.checkpoint import checkpoint

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SHIMS = os.path.join(_ROOT, "shims")
if _SHIMS not in sys.path:  # `import bitsandbytes` -> shims/bitsandbytes -> qlora_b200 (INTEGRATION.md)
    sys.path.insert(0, _SHIMS)

import bitsandbytes as bnb  # noqa: E402  (the shim; the product package under the reference's import name)

from . import fused_ops  # noqa: E402

try:   # the cuDNN frontend (pip: nvidia-cudnn-frontend) builds the deterministic attention backward (CausalAttention)
    import cudnn as _cudnn
except ImportError:
    _cudnn = None
    warnings.warn("harness: nvidia-cudnn-frontend is not installed; attention uses torch's SDPA backward, whose dQ is not "
                  "bit-repeatable, so training steps will differ in the last bits from run to run")

# caller-side elementwise fusions (RoPE on q+k in one launch, SwiGLU fwd/bwd in one launch each); plain torch otherwise
USE_FUSED_OPS = True


@dataclass
class LlamaShape:
    name: str
    hidden: int
    inter: int
    layers: int
    heads: int
    vocab: int = 32000
    rope_theta: float = 10000.0
    rms_eps: float = 1e-5  # Llama-2 (1e-6 for LLaMA-1; irrelevant to throughput)


SHAPES = {
    "llama2-7b": LlamaShape("llama2-7b", 4096, 11008, 32, 32),
    "llama2-13b": LlamaShape("llama2-13b", 5120, 13824, 40, 40),
    "llama-65b": LlamaShape("llama-65b", 8192, 22016, 80, 64),
    "tiny": LlamaShape("tiny", 256, 704, 2, 4, vocab=512),
}


class RMSNorm(nn.Module):
    def __init__(self, dim, eps, device=None, out_fp32=False):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(dim, dtype=torch.float32, device=device), requires_grad=False)
        self.eps = eps
        self.out_fp32 = out_fp32

    def forward(self, x):
        # fp32 weight (qlora.py:400-401); fp32 statistics
        if self.out_fp32:  # HF LlamaRMSNorm with an fp32 weight: `weight * hidden.to(input_dtype)` promotes to fp32
            return F.rms_norm(x.float(), (x.shape[-1],), None, self.eps).to(x.dtype) * self.weight
        if USE_FUSED_OPS and x.is_cuda and x.dtype == torch.bfloat16 and not self.weight.requires_grad and fused_ops.available():
            return fused_ops.rmsnorm(x, self.weight, self.eps)
        return F.rms_norm(x, (x.shape[-1],), self.weight.to(x.dtype), self.eps)


class LoRALinear4bit(nn.Module):
    """peft.tuners.lora.Linear4bit restated (the caller of the hot path; SURVEY.md 8a row a12)."""

    _next_salt = [1]

    def __init__(self, base, r: int, alpha: int, dropout: float, device=None, seed_tensor=None):
        super().__init__()
        self.base_layer = base
        self.lora_A = nn.Linear(base.in_features, r, bias=False, dtype=torch.bfloat16, device=device)
        self.lora_B = nn.Linear(r, base.out_features, bias=False, dtype=torch.bfloat16, device=device)
        nn.init.kaiming_uniform_(self.lora_A.weight, a=math.sqrt(5))
        nn.init.zeros_(self.lora_B.weight)
        self.scaling = alpha / r
        self.p = float(dropout)
        self.dropout = nn.Dropout(dropout) if dropout > 0 else nn.Identity()
        self.fused = True
        self.salt = LoRALinear4bit._next_salt[0]     # call-site id of the seeded dropout
        LoRALinear4bit._next_salt[0] += 1
        self._seed = [seed_tensor]                   # in a list: not a registered buffer, shared by every adapter

    def lora_input(self, x):
        """The LoRA branch's input `dropout(x)`, or None when it is x itself (p = 0 / eval)."""
        if self.p <= 0.0 or not self.training:
            return None
        xb = x if x.dtype == torch.bfloat16 else x.to(torch.bfloat16)
        if USE_FUSED_OPS and x.is_cuda and self._seed[0] is not None and fused_ops.available() and xb.numel() % 8 == 0:
            return fused_ops.seeded_dropout(xb, self.p, self._seed[0], self.salt)
        return self.dropout(xb)

    def is_fusable(self):
        return self.fused and isinstance(self.base_layer, bnb.nn.Linear4bit)

    def forward(self, x):
        if self.is_fusable():
            # SURVEY.md 8f-1: the low-rank update rides in the NF4 GEMM as one extra bf16 contraction step
            return bnb.lora_linear4bit(x, self.base_layer, self.lora_A.weight, self.lora_B.weight, self.scaling, self.lora_input(x))
        result = self.base_layer(x)
        xl = self.lora_input(x)
        a = self.lora_A(x.to(torch.bfloat16) if xl is None else xl)
        if result.dtype != torch.bfloat16:   # fp32 flow (peft: result += lora_out.to(result.dtype))
            return result + (F.linear(a, self.lora_B.weight) * self.scaling).to(result.dtype)
        # result + (a @ B^T) * scaling as ONE cuBLAS GEMM with a beta=1 epilogue (no separate scale / add passes)
        out = torch.addmm(result.reshape(-1, result.shape[-1]), a.reshape(-1, a.shape[-1]), self.lora_B.weight.t(),
                          alpha=self.scaling)
        return out.view(result.shape)


def lora_group(mods, x):
    """q/k/v (gate/up): LoRA-wrapped Linear4bit of one shape on one input -> ONE grouped launch per direction."""
    if GROUP_LINEARS and all(isinstance(m, LoRALinear4bit) and m.is_fusable() for m in mods) and len({m.scaling for m in mods}) == 1:
        xls = [m.lora_input(x) for m in mods]
        return bnb.lora_linear4bit_group(x, [m.base_layer for m in mods], [m.lora_A.weight for m in mods],
                                         [m.lora_B.weight for m in mods], mods[0].scaling,
                                         None if all(t is None for t in xls) else xls)
    return tuple(m(x) for m in mods)


GROUP_LINEARS = True


def _rope_tables(seq, head_dim, theta, device):
    """cos / sign-folded sin tables, shape [seq, 1, head_dim] (broadcast over heads in the [b, s, h, d] layout).
    HF's rotate_half form:  x*cos + cat(-x2, x1)*sin  ==  x*cos + cat(x2, x1) * cat(-sin_half, sin_half)."""
    inv_freq = 1.0 / (theta ** (torch.arange(0, head_dim, 2, device=device, dtype=torch.float32) / head_dim))
    t = torch.arange(seq, device=device, dtype=torch.float32)
    freqs = torch.outer(t, inv_freq)
    cos = torch.cat((freqs.cos(), freqs.cos()), dim=-1)
    sin_signed = torch.cat((-freqs.sin(), freqs.sin()), dim=-1)
    return cos.to(torch.bfloat16)[:, None, :].contiguous(), sin_signed.to(torch.bfloat16)[:, None, :].contiguous()


def _apply_rope(x, cos, sin_signed):
    """x: [b, s, h, d] contiguous.  3 contiguous elementwise kernels (swap halves, mul, addcmul)."""
    half = x.shape[-1] // 2
    swapped = torch.cat((x[..., half:], x[..., :half]), dim=-1)
    return torch.addcmul(x * cos, swapped, sin_signed)


_CUDNN_HANDLES = {}
_CUDNN_BWD_GRAPHS = {}


def _cudnn_sdpa_backward(q, k, v, o, do, lse):
    """dQ, dK, dV of causal attention from cuDNN's flash backward with its deterministic algorithm.  The backward PyTorch
    runs for SDPA accumulates dQ over key blocks with atomics, so the same step would not give the same gradients twice."""
    cudnn = _cudnn
    dev = q.device.index
    if dev not in _CUDNN_HANDLES:
        with torch.cuda.device(dev):
            _CUDNN_HANDLES[dev] = cudnn.create_handle()
    handle = _CUDNN_HANDLES[dev]
    b, h, s, d = q.shape
    lse = lse.reshape(b, h, s, 1)
    if do.stride(-1) != 1:
        do = do.contiguous()
    grads = [torch.empty_like(t) for t in (q, k, v)]
    key = (dev, q.dtype) + tuple((tuple(t.shape), t.stride()) for t in (q, k, v, o, do, lse, *grads))
    if key not in _CUDNN_BWD_GRAPHS:
        g = cudnn.pygraph(io_data_type=cudnn.data_type.BFLOAT16, intermediate_data_type=cudnn.data_type.FLOAT,
                          compute_data_type=cudnn.data_type.FLOAT, handle=handle)
        ins = [g.tensor_like(t) for t in (q, k, v, o, do, lse)]
        outs = g.sdpa_backward(*ins, attn_scale=1.0 / math.sqrt(d), use_causal_mask=True, use_deterministic_algorithm=True)
        for gt, t in zip(outs, grads):
            gt.set_output(True).set_dim(list(t.shape)).set_stride(list(t.stride())).set_data_type(cudnn.data_type.BFLOAT16)
        g.validate()
        g.build_operation_graph()
        g.create_execution_plans([cudnn.heur_mode.A, cudnn.heur_mode.FALLBACK])
        g.check_support()
        g.build_plans()
        _CUDNN_BWD_GRAPHS[key] = (g, ins + list(outs), g.get_workspace_size())
    g, tensors, ws = _CUDNN_BWD_GRAPHS[key]
    workspace = torch.empty(max(ws, 1), device=q.device, dtype=torch.uint8)
    cudnn.set_stream(handle=handle, stream=torch.cuda.current_stream(q.device).cuda_stream)
    g.execute(dict(zip(tensors, (q, k, v, o, do, lse, *grads))), workspace, handle=handle)
    return grads


class CausalAttention(torch.autograd.Function):
    """Causal SDPA on bf16 [b, h, s, d]: the cuDNN flash forward F.scaled_dot_product_attention runs on this GPU, and a
    backward that gives the same bits on every run (_cudnn_sdpa_backward)."""

    @staticmethod
    def forward(ctx, q, k, v):
        assert q.dtype == torch.bfloat16 and q.is_cuda, (q.dtype, q.device)
        out, lse = torch.ops.aten._scaled_dot_product_cudnn_attention(q, k, v, None, True, 0.0, True, False)[:2]
        ctx.save_for_backward(q, k, v, out, lse)
        return out

    @staticmethod
    def backward(ctx, do):
        q, k, v, out, lse = (t.detach() for t in ctx.saved_tensors)
        return tuple(_cudnn_sdpa_backward(q, k, v, out, do.detach(), lse))


class DecoderLayer(nn.Module):
    """Submodule names follow HF's LlamaDecoderLayer leaves (q_proj ... down_proj), which is what
    `find_all_linear_names` (qlora.py:248-259) keys on."""

    def __init__(self, shape: LlamaShape, device=None, norm_out_fp32=False):
        super().__init__()
        h, i = shape.hidden, shape.inter
        self.heads = shape.heads
        self.head_dim = h // shape.heads
        self.input_layernorm = RMSNorm(h, shape.rms_eps, device, norm_out_fp32)
        self.post_attention_layernorm = RMSNorm(h, shape.rms_eps, device, norm_out_fp32)
        with torch.device("meta"):   # plain nn.Linear skeleton; HF's replace_with_bnb_linear swaps these
            self.q_proj, self.k_proj, self.v_proj, self.o_proj = (nn.Linear(h, h, bias=False) for _ in range(4))
            self.gate_proj, self.up_proj = nn.Linear(h, i, bias=False), nn.Linear(h, i, bias=False)
            self.down_proj = nn.Linear(i, h, bias=False)

    def forward(self, x, cos, sin):
        b, s, h = x.shape
        y = self.input_layernorm(x)
        fused = USE_FUSED_OPS and x.is_cuda and fused_ops.available()
        q, k, v = lora_group((self.q_proj, self.k_proj, self.v_proj), y)
        if q.dtype != torch.bfloat16:   # fp32 flow: attention runs in bf16 (autocast in the reference)
            q, k, v = q.to(torch.bfloat16), k.to(torch.bfloat16), v.to(torch.bfloat16)
        q, k = q.view(b, s, self.heads, self.head_dim), k.view(b, s, self.heads, self.head_dim)
        if fused:
            q, k = fused_ops.rope_qk(q, k, cos, sin)
        else:
            q, k = _apply_rope(q, cos, sin), _apply_rope(k, cos, sin)
        q, k = q.transpose(1, 2), k.transpose(1, 2)
        v = v.view(b, s, self.heads, self.head_dim).transpose(1, 2)
        a = CausalAttention.apply(q, k, v) if _cudnn is not None else F.scaled_dot_product_attention(q, k, v, is_causal=True)
        attn = self.o_proj(a.transpose(1, 2).reshape(b, s, h))
        pn = self.post_attention_layernorm
        if fused and not pn.out_fp32 and x.dtype == torch.bfloat16 and attn.dtype == torch.bfloat16 and h <= 8192 and h % 8 == 0:
            x, y = fused_ops.add_rmsnorm(x, attn, pn.weight, pn.eps)   # residual add + norm in one pass (and in backward)
        else:
            x = x + attn
            y = pn(x)
        g, u = lora_group((self.gate_proj, self.up_proj), y)
        if g.dtype != torch.bfloat16:
            g, u = g.to(torch.bfloat16), u.to(torch.bfloat16)
        if fused:
            return x + self.down_proj(fused_ops.swiglu(g, u))
        return x + self.down_proj(F.silu(g) * u)


def find_all_linear_names(model, bits=4):
    """qlora.py:248-259 restated: the leaf names of every quantized linear, minus lm_head."""
    cls = bnb.nn.Linear4bit if bits == 4 else (bnb.nn.Linear8bitLt if bits == 8 else torch.nn.Linear)
    names = set()
    for name, module in model.named_modules():
        if isinstance(module, cls):
            parts = name.split(".")
            names.add(parts[0] if len(parts) == 1 else parts[-1])
    names.discard("lm_head")  # needed for 16-bit
    return sorted(names)


def quantize_with_hf(model: nn.Module, double_quant: bool = True):
    """The reference's construction path (qlora.py:310-330 -> transformers): BitsAndBytesConfig -> replace_with_bnb_linear."""
    from transformers import BitsAndBytesConfig
    from transformers.integrations.bitsandbytes import replace_with_bnb_linear

    cfg = BitsAndBytesConfig(load_in_4bit=True, bnb_4bit_quant_type="nf4", bnb_4bit_use_double_quant=double_quant,
                             bnb_4bit_compute_dtype=torch.bfloat16)
    return replace_with_bnb_linear(model, modules_to_not_convert=["lm_head"], quantization_config=cfg), cfg


class LlamaQLoRA(nn.Module):
    def __init__(self, shape: LlamaShape, device, lora_r=64, lora_alpha=16, lora_dropout=0.0, seed=0,
                 double_quant=True, grad_checkpointing=True, quantized=True, norm_out_fp32=False):
        super().__init__()
        self.shape = shape
        self.grad_checkpointing = grad_checkpointing
        self.lora_dropout = float(lora_dropout)
        gen = torch.Generator(device=device).manual_seed(seed)
        # step counter the seeded dropout masks are derived from; bump it once per optimizer micro-step
        self.dropout_seed = torch.zeros((), dtype=torch.int64, device=device)

        self.embed_tokens = nn.Embedding(shape.vocab, shape.hidden, device=device, dtype=torch.bfloat16)
        self.embed_tokens.weight.requires_grad_(False)
        self.layers = nn.ModuleList([DecoderLayer(shape, device, norm_out_fp32) for _ in range(shape.layers)])
        self.norm = RMSNorm(shape.hidden, shape.rms_eps, device)
        self.lm_head = nn.Linear(shape.hidden, shape.vocab, bias=False, device=device, dtype=torch.bfloat16)
        self.lm_head.weight.requires_grad_(False)
        nn.init.normal_(self.embed_tokens.weight, std=0.02)
        nn.init.normal_(self.lm_head.weight, std=0.02)
        self._rope_cache = {}
        # data parallel: called with i when the backward of decoder layer i has been enqueued (harness/dp.py starts the
        # allreduce of the gradient buckets that layer completes)
        self.layer_backward_done = None

        if quantized:
            quantize_with_hf(self, double_quant)   # nn.Linear (meta) -> bnb.nn.Linear4bit (meta), lm_head kept
        # materialise + (for the quantized arm) quantize every projection, layer by layer
        leaf_names = ("q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj")
        for layer in self.layers:
            for name in leaf_names:
                mod = getattr(layer, name)
                w = torch.empty(mod.out_features, mod.in_features, device=device, dtype=torch.bfloat16).normal_(0.0, 0.02, generator=gen)
                if quantized:
                    assert isinstance(mod, bnb.nn.Linear4bit), type(mod)
                    old = mod.weight
                    # HF's Bnb4bitQuantize.convert: re-create the parameter with the kwargs of the meta one, then move
                    # it to the device — the move quantizes (K1 + K2)
                    mod.weight = bnb.nn.Params4bit(w, requires_grad=False, **old.__dict__).to(device)
                else:  # plain bf16 nn.Linear: the un-quantized cuBLAS ceiling arm
                    mod.weight = nn.Parameter(w, requires_grad=False)
                del w
        if lora_r > 0:
            targets = find_all_linear_names(self) if quantized else list(leaf_names)
            assert sorted(targets) == sorted(leaf_names), targets
            for layer in self.layers:
                for name in targets:
                    setattr(layer, name, LoRALinear4bit(getattr(layer, name), lora_r, lora_alpha, lora_dropout, device, self.dropout_seed))
                # adapters that are used together live side by side: lora_A of q/k/v (gate/up) are row blocks of ONE buffer, so
                # the grouped launch's batched projection x . [A_q; A_k; A_v]^T needs no concatenation (same values, same init)
                for grp in (("q_proj", "k_proj", "v_proj"), ("gate_proj", "up_proj")):
                    mods = [getattr(layer, n) for n in grp]
                    buf = torch.cat([m.lora_A.weight.detach() for m in mods], 0).contiguous()
                    for j, m in enumerate(mods):
                        m.lora_A.weight = nn.Parameter(buf[j * lora_r:(j + 1) * lora_r])

    _A_ORDER = {"q_proj": 0, "k_proj": 1, "v_proj": 2, "gate_proj": 3, "up_proj": 4}

    def _trainable_named(self):
        """Trainable (name, parameter) pairs, layer by layer; inside a layer the lora_A of q/k/v and of gate/up come first and
        adjacent — a flat gradient buffer laid out in this order gives the grouped dA GEMM ONE contiguous destination."""
        def key(item):
            name = item[0]
            parts = name.split(".")
            layer = int(parts[1]) if parts[0] == "layers" else 1 << 30
            lin = parts[2] if len(parts) > 2 else ""
            first = 0 if ("lora_A" in name and lin in self._A_ORDER) else 1
            return (layer, first, self._A_ORDER.get(lin, 9) if first == 0 else 0)
        named = [(n, p) for n, p in self.named_parameters() if p.requires_grad]
        return sorted(named, key=key)   # stable: the remaining parameters keep their module order

    def trainable_parameters(self):
        return [p for _, p in self._trainable_named()]

    def trainable_parameter_layers(self):
        """Decoder-layer index of every trainable parameter, in `trainable_parameters()` order."""
        return [int(n.split(".")[1]) for n, _ in self._trainable_named()]

    def forward(self, input_ids, labels):
        b, s = input_ids.shape
        key = (s, input_ids.device)
        if key not in self._rope_cache:
            self._rope_cache[key] = _rope_tables(s, self.shape.hidden // self.shape.heads, self.shape.rope_theta, input_ids.device)
        cos, sin = self._rope_cache[key]
        x = self.embed_tokens(input_ids)
        # like peft's enable_input_require_grads: checkpointed layers need an input that requires grad
        if self.grad_checkpointing and self.training:
            x = x.requires_grad_(True)
        # the seeded dropout is a pure function of (dropout_seed, call site): recompute-safe without RNG state;
        # torch's nn.Dropout (fused ops unavailable) needs the checkpoint to restore the RNG state
        seeded = USE_FUSED_OPS and x.is_cuda and fused_ops.available()
        preserve = self.lora_dropout > 0 and not seeded
        for idx, layer in enumerate(self.layers):
            if self.layer_backward_done is not None and x.requires_grad:
                x.register_hook(lambda g, i=idx: self.layer_backward_done(i))   # grad wrt layer i's input: layer i is done
            if self.grad_checkpointing and self.training:
                x = checkpoint(layer, x, cos, sin, use_reentrant=False, preserve_rng_state=preserve)
            else:
                x = layer(x, cos, sin)
        logits = self.lm_head(self.norm(x))
        # HF causal-LM loss: shift, ignore_index -100, fp32
        return F.cross_entropy(logits[:, :-1].reshape(-1, logits.shape[-1]).float(), labels[:, 1:].reshape(-1), ignore_index=-100)


def count_linear4bit_flops(shape: LlamaShape, tokens: int) -> float:
    """2*M*N*K over every Linear4bit of one forward pass."""
    per_layer = 4 * shape.hidden * shape.hidden + 3 * shape.hidden * shape.inter
    return 2.0 * tokens * per_layer * shape.layers


def synthetic_batch(shape: LlamaShape, seq: int, seed: int, pin: bool = False):
    """OASST-shaped synthetic sample: random token ids, first 16 positions (the 'source') masked with -100
    (scripts/finetune_llama2_guanaco_7b.sh: source_max_len 16; qlora.py:481-484)."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, shape.vocab, (1, seq), generator=g, dtype=torch.int64)
    labels = ids.clone()
    labels[:, :16] = -100
    if pin:
        ids, labels = ids.pin_memory(), labels.pin_memory()
    return ids, labels

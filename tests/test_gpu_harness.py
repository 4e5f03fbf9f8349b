"""GPU tests of the bench harness (caller-side scaffolding): fused RoPE / SwiGLU kernels vs their torch formulations,
and one tiny Llama-QLoRA training step (fused kernel + fused LoRA step + checkpointing) vs the all-unfused variant."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def H():
    assert torch.cuda.is_available()
    import harness.llama_qlora as H
    from harness import fused_ops

    fused_ops.build()
    assert fused_ops.available()
    return H


def test_rope_and_swiglu_match_torch(H):
    from harness import fused_ops

    torch.manual_seed(0)
    b, s, h, d = 2, 64, 4, 128
    cos, sin = H._rope_tables(s, d, 10000.0, "cuda")
    q = torch.randn(b, s, h, d, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    k = torch.randn(b, s, h, d, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    gq, gk = torch.randn_like(q), torch.randn_like(k)
    qo, ko = fused_ops.rope_qk(q, k, cos, sin)
    (qo * gq).sum().backward(retain_graph=True)
    (ko * gk).sum().backward()
    got = [qo.detach().float(), ko.detach().float(), q.grad.float(), k.grad.float()]
    q2, k2 = q.detach().clone().requires_grad_(True), k.detach().clone().requires_grad_(True)
    qr, kr = H._apply_rope(q2, cos, sin), H._apply_rope(k2, cos, sin)
    (qr * gq).sum().backward()
    (kr * gk).sum().backward()
    ref = [qr.detach().float(), kr.detach().float(), q2.grad.float(), k2.grad.float()]
    for a, r in zip(got, ref):
        assert (a - r).abs().max().item() <= 0.04 and ((a - r).norm() / r.norm()).item() < 5e-3
    g = torch.randn(4, 100, 704, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    u = torch.randn(4, 100, 704, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    dy = torch.randn_like(g)
    out = fused_ops.swiglu(g, u)
    out.backward(dy)
    g2, u2 = g.detach().clone().requires_grad_(True), u.detach().clone().requires_grad_(True)
    ref_out = torch.nn.functional.silu(g2) * u2
    ref_out.backward(dy)
    assert torch.equal(out, ref_out)   # forward reproduces torch's two roundings exactly
    for a, r in ((g.grad, g2.grad), (u.grad, u2.grad)):
        assert ((a.float() - r.float()).norm() / r.float().norm()).item() < 1e-2


@pytest.mark.parametrize("d", [512, 704, 4096, 8192, 16384])   # register-resident row kernel up to 8192, two-pass above
def test_rmsnorm_matches_torch(H, d):
    from harness import fused_ops

    torch.manual_seed(0)
    x = (torch.randn(3, 100, d, device="cuda") * 2).to(torch.bfloat16).requires_grad_(True)
    w = (1 + 0.1 * torch.randn(d, device="cuda")).float()
    gy = torch.randn_like(x)
    y = fused_ops.rmsnorm(x, w, 1e-5)
    y.backward(gy)
    x2 = x.detach().float().requires_grad_(True)
    y2 = torch.nn.functional.rms_norm(x2, (d,), w, 1e-5)
    y2.backward(gy.float())
    assert ((y.float() - y2).norm() / y2.norm()).item() < 3e-3
    assert ((x.grad.float() - x2.grad).norm() / x2.grad.norm()).item() < 5e-3


def _tiny_step(H, fused, group, dropout=0.0, norm_out_fp32=False, seed_bump=1):
    shape = H.SHAPES["tiny"]
    ids, labels = H.synthetic_batch(shape, 256, seed=0)
    ids, labels = ids.cuda(), labels.cuda()
    H.GROUP_LINEARS = group
    torch.manual_seed(0)  # lora_A / embeddings / lm_head are initialised from the global RNG
    model = H.LlamaQLoRA(shape, torch.device("cuda"), lora_r=16, seed=7, lora_dropout=dropout, norm_out_fp32=norm_out_fp32).train()
    torch.manual_seed(1)
    for idx, m in enumerate(mm for mm in model.modules() if isinstance(mm, H.LoRALinear4bit)):
        m.fused = fused
        m.salt = idx             # the same call-site ids in every model built by these tests
        torch.nn.init.normal_(m.lora_B.weight, std=0.05)  # non-zero B so the LoRA path carries signal
    model.dropout_seed.add_(seed_bump)
    loss = model(ids, labels)
    loss.backward()
    H.GROUP_LINEARS = True
    return loss.item(), torch.cat([p.grad.float().flatten() for p in model.trainable_parameters()]), model


def test_tiny_model_step_fused_vs_unfused(H):
    """One tiny Llama-QLoRA training step built through HF's replace_with_bnb_linear: fused NF4 GEMM + fused LoRA step +
    grouped q/k/v / gate/up launches + caller-side fusions vs the all-unfused variant."""
    res = []
    for fused, group in ((True, True), (True, False), (False, False)):
        H.USE_FUSED_OPS = fused
        res.append(_tiny_step(H, fused, group)[:2])
    H.USE_FUSED_OPS = True
    losses = [r[0] for r in res]
    assert all(torch.isfinite(torch.tensor(losses)))
    for i in (0, 1):
        assert abs(losses[i] - losses[2]) < 2e-2 * abs(losses[2])
        cos = torch.nn.functional.cosine_similarity(res[i][1], res[2][1], dim=0).item()
        assert cos > 0.99, (i, cos)
    # grouped vs per-linear launches of the same fused kernels: near-identical gradients
    assert torch.nn.functional.cosine_similarity(res[0][1], res[1][1], dim=0).item() > 0.9995


def test_tiny_model_lora_dropout_fused_matches_unfused_same_mask(H):
    """--lora_dropout 0.1 (the recipe's setting): the seeded mask is a function of (seed tensor, call site, index), so the
    fused-grouped model, the fused per-linear model and the unfused (peft-form) model all see the SAME masks; the checkpoint
    recompute regenerates them.  A different seed gives different gradients."""
    base_loss, base_grad, _ = _tiny_step(H, False, False, dropout=0.1)
    for fused, group in ((True, True), (True, False)):
        loss, grad, _ = _tiny_step(H, fused, group, dropout=0.1)
        assert abs(loss - base_loss) < 2e-2 * abs(base_loss)
        assert torch.nn.functional.cosine_similarity(grad, base_grad, dim=0).item() > 0.99
    loss2, grad2, _ = _tiny_step(H, True, True, dropout=0.1, seed_bump=2)
    assert torch.nn.functional.cosine_similarity(grad2, base_grad, dim=0).item() < 0.9999
    l0, g0, _ = _tiny_step(H, True, True, dropout=0.0)
    assert torch.nn.functional.cosine_similarity(g0, base_grad, dim=0).item() < 0.9999   # dropout really changes the step


def test_seeded_dropout_statistics_and_determinism(H):
    from harness import fused_ops

    x = torch.ones(1 << 20, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    seed = torch.tensor(5, device="cuda", dtype=torch.int64)
    y = fused_ops.seeded_dropout(x, 0.1, seed, 3)
    keep = (y != 0).float().mean().item()
    assert abs(keep - 0.9) < 3e-3 and torch.allclose(y[y != 0].float(), torch.tensor(1 / 0.9).to(torch.bfloat16).float())
    assert torch.equal(fused_ops.seeded_dropout(x, 0.1, seed, 3), y)            # same (seed, salt): same mask
    assert not torch.equal(fused_ops.seeded_dropout(x, 0.1, seed, 4), y)        # another call site
    assert not torch.equal(fused_ops.seeded_dropout(x, 0.1, seed + 1, 3), y)    # another step
    y.backward(torch.ones_like(y))
    assert torch.equal(x.grad, y.detach())                                      # backward applies the same mask and scale


def test_tiny_model_fp32_norm_flow(H):
    """`norm_out_fp32=True`: the reference's dtype flow (fp32 norm outputs -> Linear4bit sees fp32, returns fp32).  Same
    values as the bf16-emitting norms up to the norm's own rounding, fused vs unfused agree."""
    l_f, g_f, _ = _tiny_step(H, True, True, norm_out_fp32=True)
    l_u, g_u, _ = _tiny_step(H, False, False, norm_out_fp32=True)
    l_b, g_b, _ = _tiny_step(H, True, True, norm_out_fp32=False)
    assert abs(l_f - l_u) < 2e-2 * abs(l_u) and abs(l_f - l_b) < 2e-2 * abs(l_b)
    assert torch.nn.functional.cosine_similarity(g_f, g_u, dim=0).item() > 0.99
    assert torch.nn.functional.cosine_similarity(g_f, g_b, dim=0).item() > 0.99


@pytest.mark.parametrize("d", [512, 4096, 8192])
def test_add_rmsnorm_matches_unfused(H, d):
    """Residual add + RMSNorm in one kernel (forward and backward) vs `x + delta` followed by the stand-alone norm op."""
    from harness import fused_ops

    torch.manual_seed(0)
    x = (torch.randn(2, 70, d, device="cuda") * 2).to(torch.bfloat16).requires_grad_(True)
    dl = torch.randn(2, 70, d, device="cuda").to(torch.bfloat16).requires_grad_(True)
    w = (1 + 0.1 * torch.randn(d, device="cuda")).float()
    g_s, g_y = torch.randn_like(x), torch.randn_like(x)
    s, y = fused_ops.add_rmsnorm(x, dl, w, 1e-5)
    torch.autograd.backward([s, y], [g_s, g_y])
    x2, d2 = x.detach().clone().requires_grad_(True), dl.detach().clone().requires_grad_(True)
    s2 = x2 + d2
    y2 = fused_ops.rmsnorm(s2, w, 1e-5)
    torch.autograd.backward([s2, y2], [g_s, g_y])
    assert torch.equal(s, s2) and torch.equal(y, y2)
    for a, b in ((x.grad, x2.grad), (dl.grad, d2.grad)):
        assert ((a.float() - b.float()).norm() / b.float().norm()).item() < 4e-3   # one rounding instead of two


def test_causal_attention_matches_sdpa_and_repeats(H):
    """The bench model's attention at the Llama-2-7B shape (seq 2048 = 16 key blocks of the backward, 32 heads of 128): the
    forward is F.scaled_dot_product_attention's result bit for bit, the gradients agree with its backward up to the order
    of the dQ sums, and a second backward gives the same bits."""
    if H._cudnn is None:
        pytest.skip("nvidia-cudnn-frontend is not installed")
    g = torch.Generator(device="cuda").manual_seed(0)
    b, s, h, d = 1, 2048, 32, 128
    qkv = [torch.randn(b, s, h, d, device="cuda", dtype=torch.bfloat16, generator=g) for _ in range(3)]
    go = torch.randn(b, s, h, d, device="cuda", dtype=torch.bfloat16, generator=g).transpose(1, 2)

    def run(fn):
        q, k, v = (t.clone().requires_grad_(True) for t in qkv)
        o = fn(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2))   # [b, h, s, d] views, as DecoderLayer passes them
        o.backward(go)
        return [o.detach(), q.grad, k.grad, v.grad]

    got = run(H.CausalAttention.apply)
    ref = run(lambda q, k, v: torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=True))
    assert torch.equal(got[0], ref[0])
    for a, r in zip(got[1:], ref[1:]):
        assert ((a.float() - r.float()).norm() / r.float().norm()).item() < 1e-3
    again = run(H.CausalAttention.apply)
    assert all(torch.equal(a, b) for a, b in zip(got, again))

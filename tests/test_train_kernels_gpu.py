"""GPU parity of the training kernels (stage-2 step of train_denoiser.py) against torch.autograd in fp32.

Each kernel's inputs are bf16; the reference evaluates the same op in fp32 on the bf16-rounded inputs and
differentiates it with autograd.  Tolerances: one bf16 rounding of the result for activation gradients
(rel-L2 <= 6e-3; attention 1.2e-2: P and dS are rounded to bf16 before their MMAs, as in every flash backward),
1e-3 for fp32 weight gradients / reductions.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-20)).item()


def _g(seed=0):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(*shape, g, scale=1.0):
    return (torch.randn(*shape, device="cuda", generator=g) * scale).bfloat16()


# ------------------------------------------------------------------ GEMM dgrad / wgrad
# ((B, M, N, K), the kernel gemm_dgrad picks on a 148-SM B200); test_kernel_dispatch_gpu.py checks the labels
DGRAD_CASES = [
    ((1, 128, 128, 64), "gemm1cta128"),        # one tile, one k-block
    ((1, 200, 136, 72), "gemm1cta128"),        # ragged everything
    ((2, 300, 256, 512), "gemm1cta128"),       # batched rows
    ((1, 2336, 3072, 3072), "gemm2cta256"),    # to_out dgrad at 512^2
    ((1, 2336, 3072, 9216), "gemm2cta256"),    # QKV dgrad, long K
    ((2, 1024, 1024, 4096), "gemm1cta128"),    # batched rows: 32 pair tiles, below the pair kernel's 74
    ((1, 4736, 512, 256), "gemm1cta128"),      # 38 pair tiles; the 256-wide 1-CTA kernel is unreachable
    ((2, 1024, 3072, 3072), "gemm2cta256"),    # pair kernel with batch
]


@pytest.mark.parametrize("B,M,N,K", [shape for shape, _ in DGRAD_CASES])
def test_gemm_dgrad(B, M, N, K):
    from gpt_image_edit_b200 import train_ops as T
    from test_kernel_dispatch_gpu import _require_variant, _run_on_variant

    variant = (dict(DGRAD_CASES)[(B, M, N, K)], 1)
    _require_variant("dgrad", B, M, N, K, T.EPI_STORE, variant)
    g = _g(1)
    dy = _randn(B, M, K, g=g)
    w = _randn(K, N, g=g, scale=0.05)          # nn.Linear weight [out = K, in = N]
    dx = _run_on_variant(lambda: T.linear_dgrad(dy, w), variant)
    ref = dy.float() @ w.float()
    assert dx.shape == (B, M, N)
    assert _rel(dx, ref) < 4e-3


def test_gemm_dgrad_pitched_views_and_epilogues():
    from gpt_image_edit_b200 import train_ops as T

    g = _g(2)
    S_txt, S_img, K, N = 96, 400, 256, 512
    big = _randn(2, S_txt + S_img, 3 * K, g=g)
    dy = big[:, S_txt:, K:2 * K]                       # image rows, middle column block
    w = _randn(K, N, g=g, scale=0.05)
    u = _randn(2, S_img, N, g=g)
    base = dy.float() @ w.float()
    out = T.linear_dgrad(dy, w, epilogue=T.EPI_DGELU, aux=u)
    uf = u.float().requires_grad_(True)
    torch.nn.functional.gelu(uf, approximate="tanh").backward(base.bfloat16().float())
    assert _rel(out, uf.grad) < 6e-3
    out = T.linear_dgrad(dy, w, epilogue=T.EPI_DSILU, aux=u)
    uf = u.float().requires_grad_(True)
    torch.nn.functional.silu(uf).backward(base.bfloat16().float())
    assert _rel(out, uf.grad) < 6e-3
    acc = _randn(2, S_img, N, g=g)
    out = T.linear_dgrad(dy, w, epilogue=T.EPI_RESID, aux=acc)
    assert _rel(out, acc.float() + base) < 4e-3


# ((B, rows, M, N), the kernel gemm_wgrad picks on a 148-SM B200)
WGRAD_CASES = [
    ((1, 64, 128, 128), "gemm1cta128"),
    ((1, 100, 136, 200), "gemm1cta128"),       # ragged: token tail inside a 64-row box, M/N tails
    ((3, 150, 256, 384), "gemm1cta128"),       # contraction over three batch items with a ragged tail each
    ((1, 2336, 3072, 3072), "gemm2cta256"),    # to_out wgrad at 512^2
    ((2, 1000, 1024, 4608), "gemm1cta128"),    # batch 2: 72 pair tiles, below the pair kernel's 74
    ((1, 288, 12288, 3584), "gemm2cta256"),    # MLP2 first linear
    ((2, 1000, 2048, 3072), "gemm2cta256"),    # pair kernel, contraction over two batch items
]


@pytest.mark.parametrize("B,rows,M,N", [shape for shape, _ in WGRAD_CASES])
def test_gemm_wgrad(B, rows, M, N):
    from gpt_image_edit_b200 import train_ops as T
    from test_kernel_dispatch_gpu import EPI_F32, _require_variant, _run_on_variant

    variant = (dict(WGRAD_CASES)[(B, rows, M, N)], 2)
    _require_variant("wgrad", B, M, N, rows, EPI_F32, variant)
    g = _g(3)
    dy = _randn(B, rows, M, g=g)
    x = _randn(B, rows, N, g=g)
    dw = _run_on_variant(lambda: T.linear_wgrad(dy, x), variant)
    ref = torch.einsum("brm,brn->mn", dy.float(), x.float())
    assert dw.dtype == torch.float32 and dw.shape == (M, N)
    assert _rel(dw, ref) < 1e-3
    dw2 = T.linear_wgrad(dy, x, out=dw.clone(), accumulate=True)
    assert _rel(dw2, 2 * ref) < 1e-3


def test_gemm_wgrad_row_slices_of_joint_buffer():
    from gpt_image_edit_b200 import train_ops as T

    g = _g(4)
    S_txt, S_img, d = 40, 300, 256
    dybuf = _randn(2, S_txt + S_img, 3 * d, g=g)
    xbuf = _randn(2, S_txt + S_img, d, g=g)
    dy, x = dybuf[:, S_txt:, :], xbuf[:, S_txt:, :]
    dw = T.linear_wgrad(dy, x)
    ref = torch.einsum("brm,brn->mn", dy.float(), x.float())
    assert _rel(dw, ref) < 1e-3


# ------------------------------------------------------------------ attention forward with LSE + backward
def _attn_ref(q, k, v, do):
    qf, kf, vf = (t.float().requires_grad_(True) for t in (q, k, v))
    B, S, H, D = q.shape
    s = torch.einsum("bqhd,bkhd->bhqk", qf, kf) / math.sqrt(D)
    p = s.softmax(-1)
    o = torch.einsum("bhqk,bkhd->bqhd", p, vf).reshape(B, S, H * D)
    o.backward(do.float())
    lse2 = torch.logsumexp(s, dim=-1) * math.log2(math.e)
    return o.detach(), lse2.detach(), qf.grad, kf.grad, vf.grad


@pytest.mark.parametrize("B,S,H", [
    (1, 128, 1),     # one block
    (1, 256, 2),
    (2, 200, 2),     # ragged tail
    (1, 1000, 3),    # pair forward kernel (>= 512 rows), ragged
    (1, 2336, 2),    # S of the 512^2 training config
])
def test_attention_lse_and_backward(B, S, H):
    from gpt_image_edit_b200 import train_ops as T

    g = _g(5)
    qkv = _randn(B, S, 3, H, 128, g=g)
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]       # strided views of one fused buffer
    do = _randn(B, S, H * 128, g=g)
    o, lse = T.attention_fwd_lse(q, k, v)
    o_ref, lse_ref, dq_ref, dk_ref, dv_ref = _attn_ref(q, k, v, do)
    assert _rel(o, o_ref) < 8e-3
    assert (lse[:, :, :S] - lse_ref).abs().max().item() < 2e-3
    dq, dk, dv = T.attention_bwd(q, k, v, o, do, lse)
    assert _rel(dv, dv_ref) < 1.2e-2, f"dv {_rel(dv, dv_ref)}"
    assert _rel(dk, dk_ref) < 1.2e-2, f"dk {_rel(dk, dk_ref)}"
    assert _rel(dq, dq_ref) < 1.2e-2, f"dq {_rel(dq, dq_ref)}"
    # no atomics anywhere: bit-reproducible
    dq2, dk2, dv2 = T.attention_bwd(q, k, v, o, do, lse)
    assert torch.equal(dq, dq2) and torch.equal(dk, dk2) and torch.equal(dv, dv2)


def test_attention_backward_peaked_rows():
    """heavy-tailed scores: a few keys dominate each row (lse far from the uniform case)."""
    from gpt_image_edit_b200 import train_ops as T

    g = _g(6)
    B, S, H = 1, 384, 2
    q = _randn(B, S, H, 128, g=g, scale=3.0)
    k = _randn(B, S, H, 128, g=g, scale=3.0)
    v = _randn(B, S, H, 128, g=g)
    do = _randn(B, S, H * 128, g=g)
    o, lse = T.attention_fwd_lse(q, k, v)
    o_ref, lse_ref, dq_ref, dk_ref, dv_ref = _attn_ref(q, k, v, do)
    assert _rel(o, o_ref) < 1e-2
    dq, dk, dv = T.attention_bwd(q, k, v, o, do, lse)
    assert _rel(dv, dv_ref) < 1.5e-2 and _rel(dk, dk_ref) < 2e-2 and _rel(dq, dq_ref) < 2e-2


# ------------------------------------------------------------------ row kernels
def test_gate_resid_and_backward():
    from gpt_image_edit_b200 import train_ops as T

    g = _g(7)
    B, S_txt, S_img, D = 2, 40, 150, 512
    S = S_txt + S_img
    x, y, dout = _randn(B, S, D, g=g), _randn(B, S, D, g=g), _randn(B, S, D, g=g)
    mod = _randn(B, 4 * D, g=g)
    gate_t, gate_i = mod[:, :D], mod[:, 2 * D:3 * D]            # pitched views of a modulation row
    out = T.gate_resid(x, y, gate_t, gate_b=gate_i, split_row=S_txt)
    gfull = torch.cat([gate_t.float()[:, None].expand(B, S_txt, D), gate_i.float()[:, None].expand(B, S_img, D)], 1)
    assert _rel(out, x.float() + gfull * y.float()) < 4e-3
    dy, dgate = T.gate_bwd(dout, y=y, gate=gate_t, gate_b=gate_i, split_row=S_txt, part_row0=S_txt)
    assert _rel(dy, gfull * dout.float()) < 4e-3
    assert _rel(dgate, (dout.float() * y.float())[:, S_txt:].sum(1)) < 1e-4
    _, colsum = T.gate_bwd(dout, want_dy=False)
    assert _rel(colsum, dout.float().sum(1)) < 1e-4


def test_ln_modulate_backward():
    from gpt_image_edit_b200 import ops, train_ops as T

    g = _g(8)
    B, S_txt, S_img, D = 2, 24, 100, 768
    S = S_txt + S_img
    x = _randn(B, S, D, g=g, scale=2.0) + 0.5
    x = x.bfloat16()
    dy, dres = _randn(B, S, D, g=g), _randn(B, S, D, g=g)
    mod = _randn(B, 4 * D, g=g, scale=0.3)
    sc_t, sh_t, sc_i, sh_i = mod[:, :D], mod[:, D:2 * D], mod[:, 2 * D:3 * D], mod[:, 3 * D:]
    xf = x.float().requires_grad_(True)
    sc = torch.cat([sc_t.float()[:, None].expand(B, S_txt, D), sc_i.float()[:, None].expand(B, S_img, D)], 1).clone().requires_grad_(True)
    sh = torch.zeros_like(sc).requires_grad_(True)
    yref = torch.nn.functional.layer_norm(xf, (D,), eps=1e-6) * (1 + sc) + sh
    yref.backward(dy.float())
    out, dscale, dshift = T.ln_modulate_bwd(x, dy, sc_t, scale_b=sc_i, split_row=S_txt, part_row0=S_txt, dres=dres)
    assert _rel(out, dres.float() + xf.grad) < 6e-3
    assert _rel(dscale, sc.grad[:, S_txt:].sum(1)) < 5e-3      # xhat is rounded to bf16 as in the forward
    assert _rel(dshift, sh.grad[:, S_txt:].sum(1)) < 1e-4
    # forward / backward consistency with the forward kernel itself
    y = ops.ln_modulate(x, sc_t, sh_t, split_row=S_txt, scale_b=sc_i, shift_b=sh_i)
    assert torch.isfinite(y.float()).all()
    out2, _, _ = T.ln_modulate_bwd(x, dy, sc_t, scale_b=sc_i, split_row=S_txt, want_mod_grads=False)
    assert _rel(out2, xf.grad) < 6e-3


def _rope_tables(S, g):
    ang = torch.rand(S, 64, device="cuda", generator=g) * 6.28
    cos = torch.cos(ang).repeat_interleave(2, dim=1).contiguous()
    sin = torch.sin(ang).repeat_interleave(2, dim=1).contiguous()
    return cos, sin


def _norm_rope_ref(x, w, cos, sin, eps=1e-6):
    # x [B,S,H,128] fp32, w [128], cos/sin [S,128]
    r = torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + eps)
    y = x * r * w
    y2 = y.reshape(*y.shape[:-1], 64, 2)
    rot = torch.stack([-y2[..., 1], y2[..., 0]], -1).reshape(y.shape)
    return y * cos[None, :, None, :] + rot * sin[None, :, None, :]


def test_rmsnorm_rope_out_of_place_and_backward():
    from gpt_image_edit_b200 import ops, train_ops as T

    g = _g(9)
    B, S_txt, S_img, H = 2, 16, 70, 3
    S, d = S_txt + S_img, H * 128
    qkv_pre = _randn(B, S, 3 * d, g=g)
    wq, wk, wqa, wka = (( torch.rand(128, device="cuda", generator=g) + 0.5).bfloat16() for _ in range(4))
    cos, sin = _rope_tables(S, g)
    out = T.rmsnorm_rope(qkv_pre, H, wq, wk, cos, sin, wq_added=wqa, wk_added=wka, n_added=S_txt)
    inplace = qkv_pre.clone()
    ops.rmsnorm_rope_(inplace, H, wq, wk, cos, sin, wq_added=wqa, wk_added=wka, n_added=S_txt)
    assert torch.equal(out[:, :, :2 * d], inplace[:, :, :2 * d])      # same kernel arithmetic as the inference path

    dqkv = _randn(B, S, 3 * d, g=g)
    xq = qkv_pre[:, :, :d].float().reshape(B, S, H, 128).requires_grad_(True)
    xk = qkv_pre[:, :, d:2 * d].float().reshape(B, S, H, 128).requires_grad_(True)
    ws = [t.float().requires_grad_(True) for t in (wqa, wka, wq, wk)]

    def apply(x, wa, wb):
        return torch.cat([_norm_rope_ref(x[:, :S_txt], wa, cos[:S_txt], sin[:S_txt]),
                          _norm_rope_ref(x[:, S_txt:], wb, cos[S_txt:], sin[S_txt:])], 1)

    oq, ok = apply(xq, ws[0], ws[2]), apply(xk, ws[1], ws[3])
    (oq * dqkv[:, :, :d].float().reshape(B, S, H, 128)).sum().backward()
    (ok * dqkv[:, :, d:2 * d].float().reshape(B, S, H, 128)).sum().backward()
    dv_before = dqkv[:, :, 2 * d:].clone()
    wg = T.rmsnorm_rope_bwd_(dqkv, qkv_pre, H, wq, wk, cos, sin, wq_added=wqa, wk_added=wka, n_added=S_txt)
    assert _rel(dqkv[:, :, :d], xq.grad.reshape(B, S, d)) < 6e-3
    assert _rel(dqkv[:, :, d:2 * d], xk.grad.reshape(B, S, d)) < 6e-3
    assert torch.equal(dqkv[:, :, 2 * d:], dv_before)
    for i in range(4):
        assert _rel(wg[i], ws[i].grad) < 5e-3, i


def test_gelu_outer_mse():
    from gpt_image_edit_b200 import train_ops as T

    g = _g(10)
    x = _randn(300, 1024, g=g, scale=2.0)
    assert _rel(T.gelu(x), torch.nn.functional.gelu(x.float(), approximate="tanh")) < 4e-3
    dmod = torch.randn(3, 768, device="cuda", generator=g)
    act = _randn(3, 256, g=g)
    dw = T.outer_acc(dmod, act)
    assert _rel(dw, dmod.t() @ act.float()) < 1e-5
    dw2 = T.outer_acc(dmod, act, out=dw.clone(), accumulate=True)
    assert _rel(dw2, 2 * (dmod.t() @ act.float())) < 1e-5
    pred = _randn(2, 1024, 64, g=g)
    target = torch.randn(2, 1024, 64, device="cuda", generator=g)
    loss, dpred = T.mse_loss(pred, target)
    pf = pred.float().requires_grad_(True)
    ref = ((pf - target) ** 2).mean()
    ref.backward()
    assert abs(loss.item() - ref.item()) < 1e-4 * ref.item()
    assert _rel(dpred, pf.grad) < 4e-3


def test_adamw_matches_torch_and_clip():
    from gpt_image_edit_b200 import train_ops as T

    g = _g(11)
    n = 100_003
    p = torch.randn(n, device="cuda", generator=g)
    ref_p = torch.nn.Parameter(p.clone())
    opt = torch.optim.AdamW([ref_p], lr=1e-3, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.05)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    p16 = torch.empty(n, device="cuda", dtype=torch.bfloat16)
    for step in range(1, 4):
        grad = torch.randn(n, device="cuda", generator=g) * 3
        ss = T.grad_sumsq(grad)
        assert abs(ss.item() - grad.double().pow(2).sum().item()) < 1e-4 * ss.item()
        coef, norm = T.clip_coef(ss, 1.0)
        ref_p.grad = grad.clone()
        total = torch.nn.utils.clip_grad_norm_([ref_p], 1.0)
        assert abs(norm.item() - total.item()) < 1e-3 * total.item()
        opt.step()
        T.adamw_step_(p, m, v, grad, p16=p16, lr=1e-3, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.05, step=step, gscale=coef)
        assert _rel(p, ref_p.data) < 1e-5
        assert torch.equal(p16, p.bfloat16())
    x = torch.randn(4097, device="cuda", generator=g).bfloat16()
    assert torch.equal(T.cast(T.cast(x, torch.float32), torch.bfloat16), x)

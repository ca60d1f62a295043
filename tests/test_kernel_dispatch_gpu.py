"""Each GEMM kernel variant with the epilogues the model runs on it, and attention at its edge shapes.

`b2f_gemm_bf16`, `b2f_gemm_qkv_norm_rope`, `b2f_gemm_dgrad` and `b2f_gemm_wgrad` each pick one of several kernels
from the problem shape (gemm.cu: `gemm_bf16_impl`, `gemm_dgrad`, `gemm_wgrad`).  Every kernel has its own epilogue
addressing and its own batch / row / gate / second-output indexing, so each variant is tested with each epilogue at
the layout the model uses: A, out and resid are row slices of wider [B, S_all, .] buffers, GATE_RESID runs in place
with the gate a column slice of the [B, 6d] modulation tensor, and everything around the output window holds a
sentinel that must survive.  `_gemm_variant` restates the host dispatch rules; `_run_on_variant` reads the kernel
that actually ran from the profiler tags, so a case cannot pass on a different kernel than the one it is meant for.

References are fp32 (`x.float() @ w.float().T` on the bf16 inputs) with the bf16 rounding points of the epilogue
comments in include/b2f.h.  Limits: rel-L2 <= 4e-3 (6e-3 after an activation) over the whole output, and for every
128-row x 64-column block max|out - ref| <= 2 bf16 ulp of that block's max|ref|, which catches one wrong tile or one
wrong gate row that a global norm would average away.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

# epilogue codes (include/b2f.h)
EPI_BIAS, EPI_GELU_TANH, EPI_SILU, EPI_GATE_RESID, EPI_RESID, EPI_GELU_ERF = 0, 1, 2, 3, 4, 5
EPI_QKV, EPI_QUICK_GELU, EPI_DGELU, EPI_DSILU, EPI_F32 = 6, 7, 8, 9, 10

SENTINEL = -7.5  # exact in bf16; never produced by the cases below
B200_SMS = 148


def _cdiv(a, b):
    return -(-a // b)


def _gemm_variant(kind, B, M, N, K, epi, num_sms):
    """(profiler tag prefix, MODE) of the kernel the library launches with its default settings.

    kind "fwd": b2f_gemm_bf16 / b2f_gemm_qkv_norm_rope (epi EPI_QKV) for out[B, M, N] = A[B, M, K] . W[N, K]^T;
    "dgrad": b2f_gemm_dgrad for dX[B, M, N] = dY[B, M, K] . W[K, N];
    "wgrad": b2f_gemm_wgrad for dW[M, N] = sum over B x K tokens (the batch does not enter the rule)."""
    half = num_sms // 2
    mode = {"fwd": 0, "dgrad": 1, "wgrad": 2}[kind]
    m_tiles = _cdiv(M, 256) * (1 if kind == "wgrad" else B)
    if N >= 256 and m_tiles * _cdiv(N, 256) >= half:
        if kind == "fwd" and epi != EPI_QKV and N % 192 == 0:
            waves256 = _cdiv(m_tiles * _cdiv(N, 256), half)
            waves192 = _cdiv(m_tiles * _cdiv(N, 192), half)
            if waves192 * 192 * 100 < waves256 * 256 * 95:
                return ("gemm2cta192", 0)
        return ("gemm2cta256", mode)
    m128 = _cdiv(M, 128) * (1 if kind == "wgrad" else B)
    use256 = N >= 256 and m128 * _cdiv(N, 256) >= num_sms
    return ("gemm1cta256" if use256 else "gemm1cta128", mode)


def _num_sms():
    from gpt_image_edit_b200 import _lib

    n, major, minor, smem = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
    _lib.check(_lib.lib.b2f_device_info(C.byref(n), C.byref(major), C.byref(minor), C.byref(smem)), "b2f_device_info")
    return n.value


def _require_variant(kind, B, M, N, K, epi, intended):
    """Skip a case whose intended kernel (chosen for a 148-SM B200) is not the one this device would run."""
    assert _gemm_variant(kind, B, M, N, K, epi, B200_SMS) == intended
    sms = _num_sms()
    got = _gemm_variant(kind, B, M, N, K, epi, sms)
    if got != intended:
        pytest.skip(f"{sms} SMs route this shape to {got}, not the intended {intended}")


def _run_on_variant(fn, intended):
    """fn() with the GEMM profiler on; asserts that it made exactly one GEMM launch, on the `intended` kernel."""
    from gpt_image_edit_b200 import _lib

    _lib.prof_shapes()   # drain whatever an earlier test left (shapes first: collect recycles the events)
    _lib.prof_collect()
    _lib.prof_enable(True)
    try:
        result = fn()
        shapes = _lib.prof_shapes()
    finally:
        _lib.prof_enable(False)
        _lib.prof_collect()
    ran = [(tuple(tag.split()[:2]), n) for tag, n, _, _ in shapes]
    assert ran == [((intended[0], f"m{intended[1]}"), 1)], f"expected one launch of {intended}, profiler saw {shapes}"
    return result


# ------------------------------------------------------------------ references and limits
def _bf(t):
    return t.bfloat16().float()


def _rel_l2(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-20)).item()


def _check_close(out, ref, rel_lim, what):
    """Global rel-L2 <= rel_lim, and per 128x64 block max|out - ref| <= 2 bf16 ulp of the block's max|ref|."""
    o, r = out.float(), ref.float()
    err = _rel_l2(o, r)
    assert err <= rel_lim, f"{what}: rel-L2 {err:.3e} > {rel_lim:.0e}"
    B, M, N = o.shape
    pad = (0, (-N) % 64, 0, (-M) % 128)
    d = F.pad((o - r).abs(), pad).view(B, -1, 128, (N + pad[1]) // 64, 64).amax(dim=(2, 4))
    a = F.pad(r.abs(), pad).view(B, -1, 128, (N + pad[1]) // 64, 64).amax(dim=(2, 4))
    _, e = torch.frexp(a)                               # a = m 2^e, m in [0.5, 1): ulp(a) = 2^(e - 8)
    lim = torch.ldexp(torch.full_like(a, 2.0), e - 8)
    bad = (d > lim).nonzero()
    if len(bad):
        b, i, j = bad[0].tolist()
        raise AssertionError(f"{what}: {len(bad)} of {d.numel()} 128x64 blocks exceed 2 ulp; first: batch {b} rows "
                             f"{128 * i}.. cols {64 * j}..: max err {d[b, i, j].item():.4g}, limit {lim[b, i, j].item():.4g} "
                             f"(block max|ref| {a[b, i, j].item():.4g})")


def _epi_ref(acc, epi, bias, resid=None, gate=None):
    """fp32 result of a forward epilogue on the fp32 accumulator, rounding to bf16 where the kernel does."""
    x = acc + bias.float() if bias is not None else acc
    if epi == EPI_BIAS:
        return x
    x = _bf(x)
    if epi == EPI_GELU_TANH:
        return F.gelu(x, approximate="tanh")
    if epi == EPI_GELU_ERF:
        return F.gelu(x)
    if epi == EPI_SILU:
        return F.silu(x)
    if epi == EPI_QUICK_GELU:
        return x * _bf(torch.sigmoid(_bf(1.702 * x)))
    if epi == EPI_RESID:
        return resid.float() + x
    if epi == EPI_GATE_RESID:
        return resid.float() + _bf(gate.float()[:, None, :] * x)
    raise ValueError(epi)


def _outside_untouched(buf, index, what):
    chk = buf.clone()
    chk[index] = SENTINEL
    n = (chk != SENTINEL).sum().item()
    assert n == 0, f"{what}: {n} elements outside the output window were written"


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(*shape, g, scale=1.0):
    return (torch.randn(*shape, device="cuda", generator=g) * scale).bfloat16()


def _row_slice(g, B, S_all, r0, M, K, scale=1.0):
    """[B, M, K] view at row r0 of a [B, S_all, K + 64] buffer whose other rows and columns are NaN: a kernel that
    reads outside its operand's rows or columns turns its output into NaN."""
    buf = torch.full((B, S_all, K + 64), float("nan"), device="cuda", dtype=torch.bfloat16)
    buf[:, r0:r0 + M, :K] = _randn(B, M, K, g=g, scale=scale)
    return buf[:, r0:r0 + M, :K]


@pytest.fixture(autouse=True, scope="module")
def _fp32_references():
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False    # the references are true fp32 products
    yield
    torch.backends.cuda.matmul.allow_tf32 = prev


# ------------------------------------------------------------------ the dispatch rules
# forward cases: (id, B, S_all, row0, M, N, K, intended variant) -- variants for a 148-SM B200
FWD_SHAPES = [
    ("1cta128", 2, 420, 40, 300, 392, 200, ("gemm1cta128", 0)),
    # last pair tile: rows 768..1023, the second CTA (896..1023) partly beyond M; N and K tails (3080 = 12 * 256 + 8)
    ("pair256_tails", 2, 1130, 96, 1000, 3080, 3080, ("gemm2cta256", 0)),
    # last pair tile: rows 1024..1279, the second CTA (1152..) entirely beyond M = 1100
    ("pair256_cta1_idle", 2, 1230, 96, 1100, 3080, 3080, ("gemm2cta256", 0)),
    ("pair192_to_out_c1024", 1, 8736, 544, 8192, 3072, 3072, ("gemm2cta192", 0)),   # image rows of the joint buffer
    ("pair192_ragged", 2, 4130, 96, 4000, 3072, 3080, ("gemm2cta192", 0)),
]
FWD_EPILOGUES = [
    ("bias", EPI_BIAS, True), ("nobias", EPI_BIAS, False), ("gelu_tanh", EPI_GELU_TANH, True),
    ("gelu_erf", EPI_GELU_ERF, True), ("silu", EPI_SILU, True), ("quick_gelu", EPI_QUICK_GELU, True),
    ("resid", EPI_RESID, True), ("gate_resid", EPI_GATE_RESID, True),
]
# fused QKV + RMSNorm + RoPE with a second output block: (id, B, S_all, row0 = rope_row0, M, d, K, n_extra, variant)
QKV_SHAPES = [
    ("pair256", 2, 1128, 96, 1000, 1536, 1536, 4 * 1536, ("gemm2cta256", 0)),
    ("1cta128", 1, 256, 24, 200, 256, 256, 1024, ("gemm1cta128", 0)),
]
# dgrad epilogues on the CTA-pair kernel: (B, S_all, row0, M, N, K)
DGRAD_SHAPE = (2, 1128, 96, 1000, 3072, 12288)
DGRAD_VARIANT = ("gemm2cta256", 1)


def test_dispatch_rules_cpu():
    """The tables of this file and of the dgrad / wgrad tests name the kernel each shape runs on a B200, and the
    256-wide 1-CTA kernel is unreachable: wherever its rule would fire, the pair kernel's has fired first."""
    for _, B, _, _, M, N, K, intended in FWD_SHAPES:
        for _, epi, _ in FWD_EPILOGUES:
            assert _gemm_variant("fwd", B, M, N, K, epi, B200_SMS) == intended, (B, M, N, K, epi)
    for _, B, _, _, M, d, K, n_extra, intended in QKV_SHAPES:
        assert _gemm_variant("fwd", B, M, 3 * d + n_extra, K, EPI_QKV, B200_SMS) == intended
    B, _, _, M, N, K = DGRAD_SHAPE
    assert _gemm_variant("dgrad", B, M, N, K, EPI_DGELU, B200_SMS) == DGRAD_VARIANT

    import test_train_kernels_gpu as T

    for (B, M, N, K), intended in T.DGRAD_CASES:
        assert _gemm_variant("dgrad", B, M, N, K, EPI_BIAS, B200_SMS) == (intended, 1), (B, M, N, K)
    for (B, rows, M, N), intended in T.WGRAD_CASES:
        assert _gemm_variant("wgrad", B, M, N, rows, EPI_F32, B200_SMS) == (intended, 2), (B, rows, M, N)

    for sms in (132, 148, 160):
        for B in (1, 2, 3, 4, 8):
            for M in range(64, 9000, 184):
                for N in (256, 384, 512, 1024, 1536, 2048, 3072, 4608, 6144, 12288):
                    for kind in ("fwd", "dgrad", "wgrad"):
                        assert _gemm_variant(kind, B, M, N, 256, EPI_BIAS, sms)[0] != "gemm1cta256", (kind, B, M, N, sms)


# ------------------------------------------------------------------ forward GEMM: variant x epilogue
@pytest.fixture(scope="module", params=FWD_SHAPES, ids=[s[0] for s in FWD_SHAPES])
def fwd_case(request):
    name, B, S_all, r0, M, N, K, intended = request.param
    g = _gen(sum(request.param[1:7]))
    x = _row_slice(g, B, S_all, r0, M, K)
    w = _randn(N, K, g=g, scale=K ** -0.5)
    bias = _randn(N, g=g, scale=0.5)
    resid = _randn(B, M, N, g=g)
    mod = _randn(B, 6 * N, g=g)                      # AdaLN modulation rows; the gate is chunk 2
    acc = x.float() @ w.float().t()
    return dict(B=B, S_all=S_all, r0=r0, M=M, N=N, K=K, intended=intended, x=x, w=w, bias=bias, resid=resid,
                gate=mod[:, 2 * N:3 * N], acc=acc)


@pytest.mark.gpu
@pytest.mark.parametrize("epi_name,epi,with_bias", FWD_EPILOGUES, ids=[e[0] for e in FWD_EPILOGUES])
def test_gemm_variant_epilogue(fwd_case, epi_name, epi, with_bias):
    from gpt_image_edit_b200 import ops

    c = fwd_case
    B, S_all, r0, M, N, K = (c[k] for k in ("B", "S_all", "r0", "M", "N", "K"))
    _require_variant("fwd", B, M, N, K, epi, c["intended"])
    bias = c["bias"] if with_bias else None
    window = (slice(None), slice(r0, r0 + M), slice(64, 64 + N))

    def run():
        buf = torch.full((B, S_all, N + 128), SENTINEL, device="cuda", dtype=torch.bfloat16)
        out = buf[window]
        kw = {}
        if epi == EPI_GATE_RESID:                    # x = x + gate * proj(...), in place
            out.copy_(c["resid"])
            kw = dict(resid=out, gate=c["gate"])
        elif epi == EPI_RESID:
            kw = dict(resid=c["resid"])
        _run_on_variant(lambda: ops.linear(c["x"], c["w"], bias, epilogue=epi, out=out, **kw), c["intended"])
        return buf

    buf = run()
    resid = c["resid"] if epi in (EPI_RESID, EPI_GATE_RESID) else None
    ref = _epi_ref(c["acc"], epi, bias, resid, c["gate"])
    _check_close(buf[window], ref, 4e-3 if epi in (EPI_BIAS, EPI_RESID) else 6e-3, f"{c['intended'][0]} {epi_name}")
    _outside_untouched(buf, window, epi_name)
    if c["intended"][0].startswith("gemm2cta"):
        assert torch.equal(run(), buf), "two runs of the pair kernel differ"


# ------------------------------------------------------------------ fused QKV + norm + RoPE with a second output
def _rope_tables(S):
    inv = 10000.0 ** (-torch.arange(64, device="cuda", dtype=torch.float64) / 64)
    ang = (torch.arange(S, device="cuda", dtype=torch.float64)[:, None] * inv).repeat_interleave(2, dim=1)
    return ang.cos().float().contiguous(), ang.sin().float().contiguous()


def _norm_rope_ref(x, w, cos, sin, eps=1e-6):
    """fp32 chain of per-head RMSNorm + RoPE from x = bf16(acc + b): y = bf16(x rsqrt(mean x^2 + eps)); z = bf16(y w);
    out = z cos + rot(z) sin with interleaved pairs.  x [B, M, H*128] (bf16 values), cos/sin [M, 128]."""
    B, M, n = x.shape
    x = x.view(B, M, n // 128, 128)
    y = _bf(x * torch.rsqrt(x.square().mean(-1, keepdim=True) + eps))
    z = _bf(y * w.float())
    rot = torch.stack((-z[..., 1::2], z[..., 0::2]), dim=-1).flatten(-2)
    return (z * cos[:, None] + rot * sin[:, None]).view(B, M, n)


@pytest.mark.gpu
@pytest.mark.parametrize("case", QKV_SHAPES, ids=[s[0] for s in QKV_SHAPES])
def test_qkv_norm_rope_second_output(case):
    """The single-stream block's [to_q; to_k; to_v; proj_mlp] launch: Q/K normed and rotated, V plain, and the GELU'd
    MLP block written into columns [d, 5d) of the [attn | mlp] buffer."""
    from gpt_image_edit_b200 import ops

    _, B, S_all, r0, M, d, K, n_extra, intended = case
    H, N = d // 128, 3 * d + n_extra
    _require_variant("fwd", B, M, N, K, EPI_QKV, intended)
    g = _gen(d + M)
    x = _row_slice(g, B, S_all, r0, M, K)
    w = _randn(N, K, g=g, scale=K ** -0.5)
    bias = _randn(N, g=g, scale=0.5)
    wq, wk = ((1 + 0.1 * torch.randn(128, device="cuda", generator=g)).bfloat16() for _ in range(2))
    cos, sin = _rope_tables(S_all)
    qkv_buf = torch.full((B, S_all, 3 * d + 64), SENTINEL, device="cuda", dtype=torch.bfloat16)
    cat = torch.full((B, S_all, 5 * d + 128), SENTINEL, device="cuda", dtype=torch.bfloat16)
    q_win = (slice(None), slice(r0, r0 + M), slice(0, 3 * d))
    e_win = (slice(None), slice(r0, r0 + M), slice(d, 5 * d))
    qkv, extra = qkv_buf[q_win], cat[e_win]
    _run_on_variant(lambda: ops.linear_qkv_norm_rope(x, w, bias, wq, wk, cos, sin, rope_row0=r0, out=qkv,
                                                     out_extra=extra, epi_extra=ops.EPI_GELU_TANH), intended)
    _outside_untouched(qkv_buf, q_win, "qkv buffer")
    _outside_untouched(cat, e_win, "cat buffer columns [0, d) and [5d, .)")

    # the unfused path: GEMM, then the standalone rmsnorm_rope kernel; the MLP block through its own GEMM
    lin = ops.linear(x, w[:3 * d], bias[:3 * d])
    ref = ops.rmsnorm_rope_(lin.clone(), H, wq, wk, cos[r0:].contiguous(), sin[r0:].contiguous())
    mism = (qkv[..., :2 * d] != ref[..., :2 * d]).float().mean().item()
    assert mism <= 1e-3, f"Q/K: {mism:.4%} of the elements differ from the unfused path"
    assert torch.equal(qkv[..., 2 * d:], ref[..., 2 * d:]), "V differs from the unfused GEMM"
    assert torch.equal(extra, ops.linear(x, w[3 * d:], bias[3 * d:], epilogue=ops.EPI_GELU_TANH)), \
        "second output block differs from the unfused GELU GEMM"

    # the fp32 chain.  Q/K: three roundings (x, y, z) precede the rotation, so a 1-ulp difference of x = bf16(acc + b)
    # between the kernel's and torch's summation order can grow past 2 ulp of the output (2.2 ulp seen in one block of
    # the pair case); the per-block limit therefore starts the chain at the GEMM's own x (the V columns and the plain
    # GEMM cases check that x against fp32), and rel-L2 covers the whole chain from the fp32 accumulator.
    acc = x.float() @ w.float().t()
    rc, rs = cos[r0:r0 + M], sin[r0:r0 + M]
    for name, h0, wn in (("Q", 0, wq), ("K", d, wk)):
        full = _norm_rope_ref(_bf(acc[..., h0:h0 + d] + bias[h0:h0 + d].float()), wn, rc, rs)
        err = _rel_l2(qkv[..., h0:h0 + d], full)
        assert err <= 6e-3, f"{name}: rel-L2 {err:.3e} against the fp32 chain"
        _check_close(qkv[..., h0:h0 + d], _norm_rope_ref(lin[..., h0:h0 + d].float(), wn, rc, rs), 6e-3, name)
    _check_close(qkv[..., 2 * d:], _epi_ref(acc[..., 2 * d:3 * d], EPI_BIAS, bias[2 * d:3 * d]), 4e-3, "V")
    _check_close(extra, _epi_ref(acc[..., 3 * d:], EPI_GELU_TANH, bias[3 * d:]), 6e-3, "MLP block")


# ------------------------------------------------------------------ dgrad epilogues on the pair kernel
@pytest.mark.gpu
@pytest.mark.parametrize("epi", [EPI_DGELU, EPI_DSILU, EPI_RESID], ids=["dgelu", "dsilu", "resid"])
def test_dgrad_epilogue_pair_kernel(epi):
    from gpt_image_edit_b200 import train_ops as T

    B, S_all, r0, M, N, K = DGRAD_SHAPE
    _require_variant("dgrad", B, M, N, K, epi, DGRAD_VARIANT)
    g = _gen(epi)
    dy = _row_slice(g, B, S_all, r0, M, K)
    w = _randn(K, N, g=g, scale=K ** -0.5)            # nn.Linear weight [out = K, in = N]
    aux = _randn(B, M, N, g=g)                        # saved pre-activation, or the gradient to add to
    window = (slice(None), slice(r0, r0 + M), slice(64, 64 + N))

    def run():
        buf = torch.full((B, S_all, N + 128), SENTINEL, device="cuda", dtype=torch.bfloat16)
        _run_on_variant(lambda: T.linear_dgrad(dy, w, epilogue=epi, aux=aux, out=buf[window]), DGRAD_VARIANT)
        return buf

    buf = run()
    base = _bf(dy.float() @ w.float())
    if epi == EPI_RESID:
        ref = aux.float() + base
    else:
        u = aux.float().requires_grad_(True)
        act = (lambda t: F.gelu(t, approximate="tanh")) if epi == EPI_DGELU else F.silu
        act(u).backward(base)
        ref = u.grad
    _check_close(buf[window], ref, 4e-3 if epi == EPI_RESID else 6e-3, f"dgrad epi {epi}")
    _outside_untouched(buf, window, f"dgrad epi {epi}")
    assert torch.equal(run(), buf), "two runs of the pair kernel differ"


# ------------------------------------------------------------------ attention edges
def _attn_ref(q, k, v, causal=False, scale=None, bias=None):
    """fp32 softmax attention on the bf16 inputs, one head at a time.  q [B,Sq,H,dh], k/v [B,Skv,Hkv,dh],
    bias [H,Sq,Skv] -> [B,Sq,H,dh]."""
    B, Sq, H, dh = q.shape
    Skv, Hkv = k.shape[1], k.shape[2]
    scale = 1 / math.sqrt(dh) if scale is None else scale
    out = torch.empty(B, Sq, H, dh, device=q.device)
    for h in range(H):
        hk = h // (H // Hkv)
        s = q[:, :, h].float() @ k[:, :, hk].float().transpose(-1, -2) * scale
        if bias is not None:
            s = s + bias[h].float()
        if causal:
            mask = torch.ones(Sq, Skv, device=q.device, dtype=torch.bool).tril()
            s = s.masked_fill(~mask, float("-inf"))
        out[:, :, h] = torch.softmax(s, dim=-1) @ v[:, :, hk].float()
    return out


def _heads(g, B, S, H, scale=1.0, dv=128):
    """[B, S, H, 128] view with batch stride S * ld into a buffer with NaN rows after it and NaN columns beside it;
    head dims >= dv are zero (heads zero-padded into the 128-wide slot)."""
    ld = H * 128 + 64
    buf = torch.full((B * S + 64, ld), float("nan"), device="cuda", dtype=torch.bfloat16)
    t = buf.as_strided((B, S, H, 128), (S * ld, ld, 128, 1))
    t.zero_()
    t[..., :dv] = _randn(B, S, H, dv, g=g, scale=scale)
    return t


def _out_window(B, Sq, H):
    ld = H * 128 + 128
    buf = torch.full((B * Sq + 2, ld), SENTINEL, device="cuda", dtype=torch.bfloat16)
    window = (slice(1, 1 + B * Sq), slice(64, 64 + H * 128))
    return buf, window, buf[window].as_strided((B, Sq, H * 128), (Sq * ld, ld, 1))


def _check_attention(buf, window, out, ref, dv=128):
    B, Sq, H, _ = ref.shape
    o = out.float().unflatten(-1, (H, 128))
    assert torch.isfinite(o).all(), "non-finite output"
    if dv < 128:
        assert (o[..., dv:] == 0).all(), "output columns of the zero-padded V are not zero"
    o, r = o[..., :dv], ref[..., :dv]
    row = (o - r).norm(dim=-1) / r.norm(dim=-1)
    worst = row.argmax().item()
    assert row.max().item() <= 2e-2, (f"per-row rel-L2 {row.max().item():.3e} at (batch, row, head) "
                                      f"{tuple(torch.unravel_index(torch.tensor(worst), row.shape))}")
    err = _rel_l2(o, r)
    assert err <= 8e-3, f"rel-L2 {err:.3e}"
    _outside_untouched(buf, window, "attention output buffer")


@pytest.mark.gpu
@pytest.mark.parametrize("lo", [0, 37])
@pytest.mark.parametrize("skv", [1, 2, 127, 128, 129, 1025])
def test_attention_decode_from_kv_cache(skv, lo):
    """Qwen2.5-VL decode step: one query token of sequence b against K/V rows [lo, past] of its KV cache."""
    from gpt_image_edit_b200 import ops

    Bc, Lmax, H, Hkv, b = 2, 2048, 28, 4, 1
    past = lo + skv - 1
    g = _gen(skv * 100 + lo)
    cache = torch.full((2, Bc, Lmax, Hkv, 128), float("nan"), device="cuda", dtype=torch.bfloat16)
    cache[:, :, :past + 1] = _randn(2, Bc, past + 1, Hkv, 128, g=g)
    q = _randn(Bc, 1, H, 128, g=g)
    k, v = cache[0, b:b + 1, lo:past + 1], cache[1, b:b + 1, lo:past + 1]
    buf, window, out = _out_window(1, 1, H)
    ops.attention(q[b:b + 1], k, v, out=out)
    _check_attention(buf, window, out, _attn_ref(q[b:b + 1], k, v))


@pytest.mark.gpu
@pytest.mark.parametrize("skv", [40, 513])
@pytest.mark.parametrize("sq", [511, 512, 513, 1025])
def test_attention_pair_threshold(sq, skv):
    """Sq = 511 runs the single-CTA kernel, Sq >= 512 the CTA-pair kernel; Skv = 40 is less than one KV block."""
    from gpt_image_edit_b200 import ops

    B, H, Hkv = 2, 4, 2
    g = _gen(sq * 1000 + skv)
    q, k, v = _heads(g, B, sq, H), _heads(g, B, skv, Hkv), _heads(g, B, skv, Hkv)
    buf, window, out = _out_window(B, sq, H)
    ops.attention(q, k, v, out=out)
    _check_attention(buf, window, out, _attn_ref(q, k, v))


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 2, 127, 129, 257, 1000])
def test_attention_causal_tails(S):
    from gpt_image_edit_b200 import ops

    B, H, Hkv = 2, 4, 2
    g = _gen(S)
    q, k, v = _heads(g, B, S, H), _heads(g, B, S, Hkv), _heads(g, B, S, Hkv)
    buf, window, out = _out_window(B, S, H)
    ops.attention(q, k, v, out=out, causal=True)
    _check_attention(buf, window, out, _attn_ref(q, k, v, causal=True))


@pytest.mark.gpu
@pytest.mark.parametrize("pitched", [False, True])
def test_attention_t5_bias(pitched):
    """T5 encoder self-attention: no score scale, relative position bias, head_dim 64 zero-padded to 128."""
    from gpt_image_edit_b200 import ops
    from gpt_image_edit_b200.text_encoders import t5_relative_position_bucket

    B, L, H = 2, 512, 4
    g = _gen(512 + pitched)
    q, k, v = (_heads(g, B, L, H, scale=0.45, dv=64) for _ in range(3))
    table = ((torch.rand(32, H, device="cuda", generator=g) * 2 - 1) * 8).bfloat16()
    bias = table[t5_relative_position_bucket(L).cuda()].permute(2, 0, 1).contiguous()     # [H, L, L]
    if pitched:
        wide = torch.full((H, L + 3, L + 24), float("nan"), device="cuda", dtype=torch.bfloat16)
        wide[:, :L, :L] = bias
        bias = wide[:, :L, :L]
        assert bias.stride(0) > L * L
    buf, window, out = _out_window(B, L, H)
    ops.attention(q, k, v, out=out, scale=1.0, bias=bias)
    _check_attention(buf, window, out, _attn_ref(q, k, v, scale=1.0, bias=bias), dv=64)


@pytest.mark.gpu
def test_attention_explicit_scale():
    """Qwen2.5-VL vision tower: head_dim 80 zero-padded to 128, scale 80^-0.5 (not 128^-0.5)."""
    from gpt_image_edit_b200 import ops

    B, S, H = 2, 300, 4
    g = _gen(80)
    q, k, v = (_heads(g, B, S, H, dv=80) for _ in range(3))
    buf, window, out = _out_window(B, S, H)
    ops.attention(q, k, v, out=out, scale=80 ** -0.5)
    _check_attention(buf, window, out, _attn_ref(q, k, v, scale=80 ** -0.5), dv=80)


@pytest.mark.gpu
def test_attention_causal_needs_square():
    from gpt_image_edit_b200 import ops
    from gpt_image_edit_b200._lib import B2FError

    g = _gen(7)
    q, k, v = _heads(g, 1, 256, 2), _heads(g, 1, 300, 2), _heads(g, 1, 300, 2)
    buf, window, out = _out_window(1, 256, 2)
    with pytest.raises(B2FError):
        ops.attention(q, k, v, out=out, causal=True)
    torch.cuda.synchronize()
    assert (buf == SENTINEL).all(), "a rejected call wrote its output"

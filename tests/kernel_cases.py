"""Per-kernel numerics cases: each function runs one C-ABI kernel on the GPU and returns
(error, tolerance, description) against a plain PyTorch fp32 or float64 reference of the same op
computed from the SAME fp16-rounded inputs.  Shared by tests/test_kernels_gpu.py and scripts/gpu_diag.py."""
import math

import torch
import torch.nn.functional as F

from magicdance_b200 import ops

DEV = "cuda"


def rel(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a - b).norm() / (b.norm() + 1e-30))


def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def case_gemm(m, n, k, bias=False, residual=False, splits=1, seed=0):
    a = _rand(m, k, seed=seed).half()
    w = _rand(n, k, seed=seed + 1, scale=k ** -0.5).half()
    b = _rand(n, seed=seed + 2).float() if bias else None
    r = _rand(m, n, seed=seed + 3).half() if residual else None
    out = ops.gemm(a, w, bias=b, residual=r, splits=splits)
    ref = a.float() @ w.float().t()
    if bias:
        ref = ref + b
    if residual:
        ref = ref + r.float()
    return rel(out.float(), ref), 2e-3, f"gemm m={m} n={n} k={k} bias={bias} res={residual} splits={splits}"


def case_tuned(tune, fn, *args):
    """Runs another case under `ops.tuning(**tune)` — the library's launch heuristics (mdb_set_tuning) — so that a
    kernel variant that the heuristics reserve for large grids is exercised on a small problem.
    tune: tuple of (name, value) pairs, e.g. (("pair_min_tiles", 1),)."""
    with ops.tuning(**dict(tune)):
        err, tol, desc = fn(*args)
        torch.cuda.synchronize()
    return err, tol, " ".join(f"{k}={v}" for k, v in tune) + ": " + desc


PAIR = (("pair_min_tiles", 1),)     # persistent CTA-pair GEMM (gemm_pair_kernel) whatever the grid size
NOPAIR = (("pair_min_tiles", 1 << 30),)  # single-CTA tiles on a large grid
ATT2Q = (("attn40_2q_min_ctas", 0),)     # d=40 attention on the two-Q-tile kernel at two CTAs per SM


def case_gemm_ln(m, n, k, offset=0.5, seed=0):
    """LayerNorm folded into the GEMM (ops.gemm(ln_u=...), engine.fold_layernorm) against LayerNorm -> Linear in fp32;
    offset: row mean of the activations (the correction rstd (acc - mean u) must not cancel)."""
    from magicdance_b200.engine import fold_layernorm
    x = (_rand(m, k, seed=seed) * 1.3 + offset).half()
    w = _rand(n, k, seed=seed + 1, scale=k ** -0.5)
    gamma = 1 + 0.1 * _rand(k, seed=seed + 2)
    beta = 0.1 * _rand(k, seed=seed + 3)
    b = 0.1 * _rand(n, seed=seed + 4)
    w_ln, u, v = fold_layernorm(w, gamma, beta, b, DEV)
    out = ops.gemm(x, w_ln, bias=v, ln_u=u, ln_eps=1e-5)
    ref = F.layer_norm(x.double(), (k,), gamma.double(), beta.double(), 1e-5) @ w.double().t() + b.double()
    return rel(out.float(), ref), 3e-3, f"gemm with folded LayerNorm m={m} n={n} k={k} offset={offset}"


def case_gemm_batch_bias(batch, hw, n, k, seed=0):
    m = batch * hw
    a = _rand(m, k, seed=seed).half()
    w = _rand(n, k, seed=seed + 1, scale=k ** -0.5).half()
    ball = _rand(batch, n + 64, seed=seed + 2).float()
    bias = ball[:, 32:32 + n]
    out = ops.gemm(a, w, bias=bias, bias_batch_stride=ball.stride(0), rows_per_batch=hw)
    ref = (a.float() @ w.float().t()).reshape(batch, hw, n) + bias[:, None, :]
    return rel(out.float(), ref.reshape(m, n)), 2e-3, f"gemm per-batch bias B={batch} hw={hw} n={n} k={k}"


def case_gemm_dual(m, n, k1, k2, seed=0):
    a1 = _rand(m, k1, seed=seed).half()
    a2 = _rand(m, k2, seed=seed + 5).half()
    w = _rand(n, k1 + k2, seed=seed + 1, scale=(k1 + k2) ** -0.5).half()
    out = ops.gemm(a1, w, a2=a2)
    ref = torch.cat([a1, a2], 1).float() @ w.float().t()
    return rel(out.float(), ref), 2e-3, f"gemm dual-source m={m} n={n} k={k1}+{k2}"


def case_gemm_strided_out(m, n, k, seed=0):
    """D written into a column slice of a wider, zero-initialised buffer (text V^T layout)."""
    a = _rand(m, k, seed=seed).half()
    w = _rand(n, k, seed=seed + 1, scale=k ** -0.5).half()
    ld = (n + 7) // 8 * 8
    buf = torch.zeros(m, 2 * ld, dtype=torch.float16, device=DEV)
    ops.gemm(a, w, out=buf[:, ld:ld + n])
    ref = a.float() @ w.float().t()
    untouched = float(buf[:, :ld].abs().max()) + (float(buf[:, ld + n:].abs().max()) if ld > n else 0.0)
    return rel(buf[:, ld:ld + n].float(), ref) + untouched, 2e-3, f"gemm strided out m={m} n={n} k={k}"


def case_geglu(m, c, seed=0):
    from magicdance_b200.engine import pack_geglu
    x = _rand(m, c, seed=seed).half()
    w = _rand(8 * c, c, seed=seed + 1, scale=c ** -0.5)
    b = _rand(8 * c, seed=seed + 2, scale=0.1)
    wp, bp = pack_geglu(w, b, DEV)
    out = ops.gemm(x, wp, bias=bp, epilogue=ops.EPI_GEGLU)
    y = x.float() @ w.half().float().t() + b
    v, g = y.chunk(2, dim=-1)
    ref = v * F.gelu(g)
    return rel(out.float(), ref), 3e-3, f"geglu m={m} c={c}"


def case_conv(batch, h, w, cin, cout, bias=True, residual=False, splits=1, seed=0):
    x = _rand(batch, cin, h, w, seed=seed).half()
    wt = _rand(cout, cin, 3, 3, seed=seed + 1, scale=(9 * cin) ** -0.5).half()
    b = _rand(cout, seed=seed + 2).float() if bias else None
    from magicdance_b200.engine import pack_conv3x3
    xn = x.permute(0, 2, 3, 1).contiguous().reshape(batch * h * w, cin)
    r = _rand(batch * h * w, cout, seed=seed + 3).half() if residual else None
    out = ops.gemm(xn, pack_conv3x3(wt, DEV), bias=b, residual=r, conv=(batch, h, w, cin), splits=splits)
    ref = F.conv2d(x.float(), wt.float(), b, padding=1).permute(0, 2, 3, 1).reshape(batch * h * w, cout)
    if residual:
        ref = ref + r.float()
    return rel(out.float(), ref), 2e-3, f"conv3x3 igemm B={batch} {h}x{w} {cin}->{cout} splits={splits}"


def case_conv_s2(batch, h, w, cin, cout, seed=0):
    """3x3 stride-2 pad-1 conv (Downsample.op, openaimodel.py:175) as implicit GEMM: TMA element strides of 2"""
    x = _rand(batch * h * w, cin, seed=seed).half()
    wt = _rand(cout, 3, 3, cin, seed=seed + 1, scale=(9 * cin) ** -0.5).half()
    b = _rand(cout, seed=seed + 2).float()
    out = ops.gemm(x, wt.reshape(cout, 9 * cin), bias=b, conv=(batch, h, w, cin), conv_stride=2)
    xr = x.float().reshape(batch, h, w, cin).permute(0, 3, 1, 2)
    ref = F.conv2d(xr, wt.float().permute(0, 3, 1, 2), b, stride=2, padding=1).permute(0, 2, 3, 1).reshape(-1, cout)
    return rel(out.float(), ref), 2e-3, f"conv 3x3 stride 2 (implicit GEMM) B={batch} {h}x{w} {cin}->{cout}"


def case_conv_direct(batch, h, w, cin, cout, stride, silu, residual=False, seed=0):
    x = _rand(batch, cin, h, w, seed=seed).half()
    wt = _rand(cout, cin, 3, 3, seed=seed + 1, scale=(9 * cin) ** -0.5).half()
    b = _rand(cout, seed=seed + 2).float()
    from magicdance_b200.engine import pack_conv3x3
    xn = x.permute(0, 2, 3, 1).contiguous().reshape(batch * h * w, cin)
    ho, wo = (h - 1) // stride + 1, (w - 1) // stride + 1
    r = _rand(batch * ho * wo, cout, seed=seed + 3).half() if residual else None
    out = ops.conv3x3_direct(xn, pack_conv3x3(wt, DEV), b, batch=batch, h=h, w=w, cin=cin, cout=cout, stride=stride,
                             silu=silu, residual=r)
    ref = F.conv2d(x.float(), wt.float(), b, padding=1, stride=stride)
    if silu:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 3, 1).reshape(batch * ho * wo, cout)
    if residual:
        ref = ref + r.float()
    return rel(out.float(), ref), 2e-3, f"conv3x3 direct B={batch} {h}x{w} {cin}->{cout} s={stride} silu={silu}"


def case_down(batch, h, w, c, seed=0):
    x = _rand(batch, c, h, w, seed=seed).half()
    wt = _rand(c, c, 3, 3, seed=seed + 1, scale=(9 * c) ** -0.5).half()
    b = _rand(c, seed=seed + 2).float()
    from magicdance_b200.engine import pack_conv3x3
    xn = x.permute(0, 2, 3, 1).contiguous().reshape(batch * h * w, c)
    col = ops.im2col3x3(xn, batch=batch, h=h, w=w, c=c, stride=2)
    out = ops.gemm(col, pack_conv3x3(wt, DEV), bias=b)
    ref = F.conv2d(x.float(), wt.float(), b, padding=1, stride=2).permute(0, 2, 3, 1).reshape(-1, c)
    return rel(out.float(), ref), 2e-3, f"downsample im2col+gemm B={batch} {h}x{w} c={c}"


def case_conv_im2col(batch, h, w, cin, cout, seed=0):
    """general-size 3x3 conv: explicit im2col (stride 1) + GEMM, for latents that do not tile into TMA boxes"""
    x = _rand(batch, cin, h, w, seed=seed).half()
    wt = _rand(cout, cin, 3, 3, seed=seed + 1, scale=(9 * cin) ** -0.5).half()
    b = _rand(cout, seed=seed + 2).float()
    from magicdance_b200.engine import pack_conv3x3
    xn = x.permute(0, 2, 3, 1).contiguous().reshape(batch * h * w, cin)
    col = ops.im2col3x3(xn, batch=batch, h=h, w=w, c=cin, stride=1)
    out = ops.gemm(col, pack_conv3x3(wt, DEV), bias=b)
    ref = F.conv2d(x.float(), wt.float(), b, padding=1).permute(0, 2, 3, 1).reshape(-1, cout)
    return rel(out.float(), ref), 2e-3, f"conv3x3 im2col+gemm B={batch} {h}x{w} {cin}->{cout}"


def case_upsample(batch, h, w, c, seed=0):
    x = _rand(batch, c, h, w, seed=seed).half()
    xn = x.permute(0, 2, 3, 1).contiguous().reshape(batch * h * w, c)
    out = ops.upsample2x(xn, batch=batch, h=h, w=w, c=c)
    ref = F.interpolate(x.float(), scale_factor=2, mode="nearest").permute(0, 2, 3, 1).reshape(-1, c)
    return rel(out.float(), ref), 0.0, f"upsample2x B={batch} {h}x{w} c={c}"


def case_groupnorm(batch, hw, c1, c2, eps, silu, mode=None, offset=0.3, seed=0):
    """mode: 0 auto, 1 two kernels (stats + last-CTA fold -> apply), 2 single-launch cluster kernel.
    offset: mean of the activations — a large value against a spread of ~1 is the catastrophic-cancellation case of
    E[x^2] - mean^2 that the pivot-shifted sums avoid.  Also checks run-to-run bit-equality (no atomics)."""
    x1 = (_rand(batch * hw, c1, seed=seed) * 1.5 + offset).half()
    x2 = (_rand(batch * hw, c2, seed=seed + 1) - 0.2 + offset).half() if c2 else None
    c = c1 + c2
    g = (1 + 0.1 * _rand(c, seed=seed + 2)).float()
    b = (0.1 * _rand(c, seed=seed + 3)).float()
    out = ops.groupnorm(x1, g, b, batch=batch, hw=hw, eps=eps, silu=silu, x2=x2, mode=mode)
    again = ops.groupnorm(x1, g, b, batch=batch, hw=hw, eps=eps, silu=silu, x2=x2, mode=mode)
    xc = x1 if x2 is None else torch.cat([x1, x2], 1)
    xr = xc.double().reshape(batch, hw, c).permute(0, 2, 1)
    ref = F.group_norm(xr, 32, g.double(), b.double(), eps)
    if silu:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 1).reshape(batch * hw, c)
    err = rel(out.float(), ref)
    if not torch.equal(out, again):
        err = float("inf")  # non-deterministic
    return err, 2e-3, f"groupnorm B={batch} hw={hw} c={c1}+{c2} silu={silu} mode={mode} offset={offset}"


def case_layernorm(rows, c, seed=0):
    x = (_rand(rows, c, seed=seed) * 2 + 0.5).half()
    g = (1 + 0.1 * _rand(c, seed=seed + 2)).float()
    b = (0.1 * _rand(c, seed=seed + 3)).float()
    out = ops.layernorm(x, g, b)
    ref = F.layer_norm(x.float(), (c,), g, b, 1e-5)
    return rel(out.float(), ref), 1.5e-3, f"layernorm rows={rows} c={c}"


ATT_BKV = 64       # keys per tile of every attention kernel (csrc/attention.cu, BKV)
ATT_LAZY_LOG2 = 8  # the running max moves only when a tile's max exceeds it by more than this (log2 units)
V_PAD_FILL = 3e4   # V^T columns [n, ldv) of a padded layout: large and finite, so a masked key with P != 0 shows


def _vt_padded(v, batches, n, ldv):
    """V [batches*n, c] -> V^T [c, batches*ldv]; padding columns hold +-V_PAD_FILL (the kernel must give them P = 0)"""
    c = v.shape[1]
    vt = torch.full((c, batches, ldv), V_PAD_FILL, dtype=torch.float16, device=v.device)
    vt[1::2] = -V_PAD_FILL
    vt[:, :, :n] = v.reshape(batches, n, c).permute(2, 0, 1)
    return vt.reshape(c, batches * ldv)


def attention_keys(b, k0, v0, n0, kv0_batches, k1=None, v1=None, n1=0, kv1_batches=1, bank_batches=0):
    """keys / values that batch element b attends to, in the kernels' tile order (source 0, then source 1)"""
    s0 = slice(b * n0, (b + 1) * n0) if kv0_batches > 1 else slice(0, n0)
    kk, vv = [k0[s0]], [v0[s0]]
    if n1 and b < bank_batches:
        s1 = slice(b * n1, (b + 1) * n1) if kv1_batches > 1 else slice(0, n1)
        kk.append(k1[s1])
        vv.append(v1[s1])
    return torch.cat(kk, 0), torch.cat(vv, 0)


def attention_ref(q, heads, d, batch, nq, **kv):
    """float64 softmax(q k^T / sqrt(d)) v per batch element from the same fp16 operands; kv: attention_keys' keywords"""
    refs = []
    for b in range(batch):
        kk, vv = attention_keys(b, **kv)
        qq = q[b * nq:(b + 1) * nq].double().reshape(nq, heads, d).transpose(0, 1)
        kk = kk.double().reshape(-1, heads, d).transpose(0, 1)
        vv = vv.double().reshape(-1, heads, d).transpose(0, 1)
        s = (qq @ kk.transpose(1, 2)) * d ** -0.5
        refs.append((s.softmax(-1) @ vv).transpose(0, 1).reshape(nq, heads * d))
    return torch.cat(refs, 0)


def case_attention(batch, heads, d, nq, n0, n1=0, kv1_batches=1, bank_batches=None, ldv_pad=False, mode="", seed=0):
    """mode: '+'-joined layout options of the hot path —
    qk_fused   Q and K0 are the two column halves of one [B*N, 2c] projection (self-attention, engine.py attn1);
    shared_kv  one key/value set for the whole batch (kv0_batches = 1: the text context, engine.py attn2);
    wide_out   the output is a column slice of a wider buffer (ldo > heads*d); its other columns stay untouched."""
    modes = set(filter(None, mode.split("+")))
    assert modes <= {"qk_fused", "shared_kv", "wide_out"}, modes
    c = heads * d
    kvb = 1 if "shared_kv" in modes else batch
    if "qk_fused" in modes:
        assert n0 == nq and kvb == batch
        qk = _rand(batch * nq, 2 * c, seed=seed).half()
        q, k0 = qk[:, :c], qk[:, c:]
    else:
        q = _rand(batch * nq, c, seed=seed).half()
        k0 = _rand(kvb * n0, c, seed=seed + 1).half()
    v0 = _rand(kvb * n0, c, seed=seed + 2).half()
    ldv = (n0 + 7) // 8 * 8 if ldv_pad else n0
    vt0 = _vt_padded(v0, kvb, n0, ldv)
    kw, kv = {}, dict(k0=k0, v0=v0, n0=n0, kv0_batches=kvb)
    bb = batch if bank_batches is None else bank_batches
    if n1:
        k1 = _rand(kv1_batches * n1, c, seed=seed + 3).half()
        v1 = _rand(kv1_batches * n1, c, seed=seed + 4).half()
        kw = dict(k1=k1, vt1=v1.t().contiguous(), n1=n1, kv1_batches=kv1_batches, bank_batches=bb)
        kv.update(k1=k1, v1=v1, n1=n1, kv1_batches=kv1_batches, bank_batches=bb)
    out, gap = None, 16
    if "wide_out" in modes:
        buf = torch.full((batch * nq, c + 3 * gap), 7.0, dtype=torch.float16, device=DEV)
        out = buf[:, gap:gap + c]
    res = ops.attention(q, k0, vt0, n0, heads=heads, d=d, batch=batch, nq=nq, out=out, kv0_batches=kvb,
                        ldv0_batch=ldv, **kw)
    err = rel(res.float(), attention_ref(q, heads, d, batch, nq, **kv))
    if out is not None and not (torch.all(buf[:, :gap] == 7.0) and torch.all(buf[:, gap + c:] == 7.0)):
        err = float("inf")  # wrote outside its column slice
    return err, 3e-3, (f"attention B={batch} h={heads} d={d} nq={nq} n0={n0} n1={n1} "
                       f"kv1b={kv1_batches} bank_b={bb} ldv={ldv} {mode}")


# ---- attention logits that drive the online-softmax rescale path ---------------------------------------------------
# With randn Q and K the logits are ~N(0, 1): after tile 0 no tile's max ever beats the running max by
# ATT_LAZY_LOG2, so the O / l rescale and the re-emission of P (attn2/attn3's second pass) never run.  Here every
# logit is placed: per head a unit direction u, q_i = a_i s u + r_i, k_j = t_j s u + r_j with the noise r
# orthogonal to u and s^2 = sqrt(d) / log2(e), so the logit of row i and key j is a_i t_j + r_i.r_j / sqrt(d) in
# log2 units (the noise is ~0.36 log2 units).  a_i (0 or 1) picks the peaky rows, t_j (log2 units) is the key profile.
# tests/test_kernel_cases_cpu.py replays the kernels' per-row bookkeeping on these inputs and checks that each
# pattern reaches the branch it claims.
PEAKY_PATTERNS = ("rise", "slow_rise", "mixed_rows", "fall", "bank_peak", "ragged_peak")


def _tile_ramp(j):
    """-2 .. 0 across each 64-key tile: the softmax weight of a tile is spread over its keys, its max at the end"""
    return -2.0 * (1.0 - (j % ATT_BKV).double() / (ATT_BKV - 1))


def peaky_profiles(pattern, batch, nq, n0, n1):
    """row amplitudes a [batch, nq] and key profiles t0 [batch, n0] (source 0), t1 [n1] (source 1, one bank)"""
    a = torch.ones(batch, nq, dtype=torch.float64)
    j0 = torch.arange(n0)
    tile0 = (j0 // ATT_BKV).double()
    t1 = torch.zeros(n1, dtype=torch.float64)
    if pattern in ("rise", "mixed_rows"):
        # steps of 12 and 18 alternately: a rescale on every tile; the optimistic P of an 18-step (2^18) overflows fp16
        steps = torch.tensor([12.0 if i % 2 == 0 else 18.0 for i in range(int(tile0.max()) + 1)])
        level = torch.cat([torch.zeros(1), steps.cumsum(0)[:-1]]).double()[j0 // ATT_BKV]
        t0 = level + _tile_ramp(j0)
        if pattern == "mixed_rows":
            # in every 128-row Q tile: warp 1 rises, warp 2 stays flat, warps 0 and 3 rise on odd rows only —
            # lanes of one warp and warps of one CTA disagree on the rescale vote
            r = torch.arange(nq) % 128
            w = r // 32
            a[:] = torch.where(w == 1, 1.0, torch.where(w == 2, 0.0, (r % 2).double()))
    elif pattern == "slow_rise":
        # +5.5 per tile: every other tile is accepted against the old max (P up to ~2^6), the next one rescales
        t0 = 5.5 * tile0 + _tile_ramp(j0)
    elif pattern == "fall":
        # max in tile 0; later tiles 30 .. ~150 log2 units below it (-32: room for the noise): P underflows to 0
        # (ex2.approx.ftz, ex2_poly's clamp at -125)
        t0 = torch.where(tile0 == 0, 0.0, -32.0 - 15.0 * (tile0 - 1)) + _tile_ramp(j0)
    elif pattern == "bank_peak":
        # source 0 flat, the peak in the bank: the rescale happens at the source boundary
        t0 = _tile_ramp(j0)
        j1 = torch.arange(n1)
        t1 = 12.0 * (j1 // ATT_BKV + 1).double() + _tile_ramp(j1)
    elif pattern == "ragged_peak":
        # the peak in the last, partly valid tile (masked exponentials)
        assert n0 % ATT_BKV
        t0 = torch.where(tile0 == tile0.max(), 12.0, 0.0) + _tile_ramp(j0)
    else:
        raise ValueError(pattern)
    t0 = t0.expand(batch, n0).clone()
    if pattern == "ragged_peak":
        # the last K tile of batch b runs on into the first keys of batch b+1: give those the largest logits of the
        # whole tensor, so that a key past n0 that is not masked dominates batch b's output
        t0[1:, :ATT_BKV - n0 % ATT_BKV] = 40.0
    return a, t0, t1


def attention_peaky_inputs(batch, heads, d, nq, n0, n1, pattern, bank_batches, seed=0, device=None):
    """fp16 operands of one peaky attention case (K/V per batch element for source 0, one shared bank for source 1)"""
    device = DEV if device is None else device
    g = torch.Generator(device="cpu").manual_seed(seed)
    c = heads * d
    a, t0, t1 = peaky_profiles(pattern, batch, nq, n0, n1)
    u = torch.randn(heads, d, generator=g, dtype=torch.float64)
    u = u / u.norm(dim=1, keepdim=True)
    s = (d ** 0.5 / math.log2(math.e)) ** 0.5

    def build(amp):  # amp [rows] -> [rows, heads*d]: amp s u + noise orthogonal to u, per head
        r = 0.5 * torch.randn(amp.shape[0], heads, d, generator=g, dtype=torch.float64)
        r = r - (r * u).sum(-1, keepdim=True) * u
        return (amp[:, None, None] * s * u + r).reshape(-1, c).half().to(device)

    q = build(a.reshape(-1))
    k0 = build(t0.reshape(-1))
    v0 = torch.randn(batch * n0, c, generator=g).half().to(device)
    k1 = build(t1) if n1 else None
    v1 = torch.randn(n1, c, generator=g).half().to(device) if n1 else None
    kv = dict(k0=k0, v0=v0, n0=n0, kv0_batches=batch, k1=k1, v1=v1, n1=n1, kv1_batches=1,
              bank_batches=bank_batches if n1 else 0)
    return q, kv


def case_attention_peaky(batch, heads, d, nq, n0, n1, pattern, bank_batches=None, seed=0):
    bb = batch if bank_batches is None else bank_batches
    q, kv = attention_peaky_inputs(batch, heads, d, nq, n0, n1, pattern, bb, seed=seed)
    ldv = (n0 + 7) // 8 * 8
    kw = {}
    if n1:
        kw = dict(k1=kv["k1"], vt1=kv["v1"].t().contiguous(), n1=n1, kv1_batches=1, bank_batches=bb)
    out = ops.attention(q, kv["k0"], _vt_padded(kv["v0"], batch, n0, ldv), n0, heads=heads, d=d, batch=batch, nq=nq,
                        ldv0_batch=ldv, **kw)
    ref = attention_ref(q, heads, d, batch, nq, **kv)
    return rel(out.float(), ref), 3e-3, (f"attention {pattern} B={batch} h={heads} d={d} nq={nq} n0={n0} n1={n1} "
                                          f"bank_b={bb}")


def case_time_path(batch, t_count=0, seed=0):
    """t_count: 0 = one timestep per row, else t_count timesteps repeated over the rows (row b uses t[b % t_count])"""
    base = [981, 441, 1, 999, 500, 21, 7, 123]
    nt = t_count or batch
    t = torch.tensor([(base[i % 8] + 13 * (i // 8)) % 1000 for i in range(nt)], dtype=torch.long, device=DEV)
    emb = ops.timestep_embedding(t, 320, rows=batch)
    half = 160
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32, device=DEV) / half)
    args = t[torch.arange(batch, device=DEV) % nt, None].float() * freqs[None]
    ref = torch.cat([torch.cos(args), torch.sin(args)], -1)
    e1 = float((emb - ref).abs().max())
    w = _rand(1280, 320, seed=seed, scale=320 ** -0.5).half()
    b = _rand(1280, seed=seed + 1).float()
    out = ops.skinny_linear(ref, w, b, silu_in=True, silu_out=True)
    r2 = F.silu(F.silu(ref) @ w.float().t() + b)
    return max(e1, rel(out, r2)), 1e-4, f"timestep embedding + skinny linear B={batch} timesteps={nt}"


def case_layout(batch, c, h, w, copies=1, seed=0):
    """copies > 1: the NHWC result repeats the batch (the cond | uncond pair); bit-exact"""
    x = _rand(batch, c, h, w, seed=seed)
    y = ops.nchw_f32_to_nhwc_f16(x, copies=copies)
    ref = x.half().permute(0, 2, 3, 1).reshape(-1, c).repeat(copies, 1)
    e1 = float((y.float() - ref.float()).abs().max()) if y.shape == ref.shape else float("inf")
    z = ops.nhwc_f16_to_nchw_f32(y[:batch * h * w], batch=batch, c=c, h=h, w=w)
    e2 = float((z - x.half().float()).abs().max())
    return e1 + e2, 0.0, f"layout converts B={batch} c={c} {h}x{w} copies={copies}"


def case_add(batch, n, bcast, seed=0):
    a = _rand(batch, n, seed=seed).half()
    b = _rand(1 if bcast else batch, n, seed=seed + 1).half()
    out = ops.add(a, b, batch=batch, b_batches=1 if bcast else batch)
    ref = (a.float() + b.float()).half()
    return float((out.float() - ref.float()).abs().max()), 0.0, f"add B={batch} n={n} bcast={bcast}"


def case_cfg_ddim(sigma=0.0, update_x=False, seed=0):
    """sigma > 0: the stochastic DDIM step (noise added); update_x: x is overwritten with x_prev in place, and
    pred_x0 must still come from the old x"""
    x, ec, eu, noise = (_rand(2, 4, 64, 64, seed=seed + i) for i in range(4))
    x_old = x.clone()
    a_t, a_prev, scale = 0.0047, 0.0058, 7.0
    coef = torch.tensor([scale, math.sqrt(a_t), math.sqrt(a_prev), math.sqrt(1 - a_prev - sigma ** 2), sigma,
                         math.sqrt(1 - a_t)], dtype=torch.float32, device=DEV)
    xp, p0 = ops.cfg_ddim_update(x, ec, eu, coef, noise=noise if sigma > 0 else None, update_x=update_x)
    xo, ec, eu, noise = (t.double() for t in (x_old, ec, eu, noise))
    e = eu + scale * (ec - eu)
    rp0 = (xo - math.sqrt(1 - a_t) * e) / math.sqrt(a_t)
    rxp = math.sqrt(a_prev) * rp0 + math.sqrt(1 - a_prev - sigma ** 2) * e + sigma * noise * (sigma > 0)
    err = max(rel(xp, rxp), rel(p0, rp0))
    if not torch.equal(x, xp if update_x else x_old):
        err = float("inf")  # x must hold x_prev exactly (update_x) or be left alone
    return err, 1e-5, f"cfg + ddim update sigma={sigma} update_x={update_x}"


def case_softmax_rows(rows, cols, ld, scale=1.0, seed=0):
    """in-place row softmax (VAE attention) against float64; row 0 peaky, row 1 constant; the pitch gap
    [cols, ld) must stay untouched"""
    x = (_rand(rows, ld, seed=seed) * 3).half()
    x[0, :cols] = -4.0
    x[0, cols // 3] = 30.0
    x[1, :cols] = 2.5
    before = x.clone()
    ref = (x[:, :cols].double() * scale).softmax(-1)
    ops.softmax_rows(x[:, :cols], scale=scale)
    err = rel(x[:, :cols].float(), ref)
    if not torch.equal(x[:, cols:], before[:, cols:]):
        err = float("inf")
    return err, 1e-3, f"softmax rows={rows} cols={cols} ld={ld} scale={scale}"


def case_im2col_br(batch, h, w, c, seed=0):
    """im2col for the VAE encoder's Downsample: pad (0, 1, 0, 1), 3x3 window, stride 2; bit-exact"""
    x = _rand(batch, c, h, w, seed=seed).half()
    xn = x.permute(0, 2, 3, 1).contiguous().reshape(batch * h * w, c)
    col = ops.im2col3x3(xn, batch=batch, h=h, w=w, c=c, stride=2, pad="br")
    u = F.unfold(F.pad(x.float(), (0, 1, 0, 1)), 3, stride=2)  # [B, c*9, L], column order (channel, ky, kx)
    ref = u.reshape(batch, c, 9, -1).permute(0, 3, 2, 1).reshape(-1, 9 * c)
    err = float((col.float() - ref).abs().max()) if col.shape == ref.shape else float("inf")
    return err, 0.0, f"im2col 3x3 stride 2 pad (0,1,0,1) B={batch} {h}x{w} c={c}"


ALL_CASES = [
    (case_layout, (2, 4, 64, 64)),
    (case_layout, (1, 3, 256, 256)),
    (case_add, (2, 4096 * 320, False)),
    (case_add, (2, 64 * 1280, True)),
    (case_upsample, (2, 8, 8, 1280)),
    (case_time_path, (2,)),
    (case_time_path, (37,)),  # more rows than one skinny-linear launch holds (16)
    (case_cfg_ddim, ()),
    (case_layernorm, (4096, 320)),
    (case_layernorm, (300, 640)),
    (case_layernorm, (64, 1280)),
    (case_groupnorm, (2, 4096, 320, 0, 1e-5, True)),                 # auto: cluster of 4, 5 words per pixel
    (case_groupnorm, (1, 1024, 640, 320, 1e-5, True)),               # concat: groups straddle the two sources
    (case_groupnorm, (2, 64, 1280, 1280, 1e-5, True)),               # 8x8 level: one CTA per group
    (case_groupnorm, (2, 256, 1280, 0, 1e-6, False)),
    (case_groupnorm, (1, 16, 1280, 640, 1e-5, True)),
    (case_groupnorm, (2, 4096, 640, 320, 1e-5, True)),               # 960 channels at 64x64: the largest slice
    (case_groupnorm, (4, 1000, 320, 0, 1e-5, True)),                 # pixel count not a multiple of anything
    (case_groupnorm, (2, 4096, 320, 0, 1e-5, True, None, 40.0)),     # mean 40, spread 1.5: pivot-shifted variance
    (case_groupnorm, (16, 4096, 320, 0, 1e-5, True)),                # eight frames (cond+uncond), 10-channel groups: two kernels
    (case_groupnorm, (16, 1024, 1280, 640, 1e-5, True)),             # wide groups: the cluster kernel at every batch size
    (case_groupnorm, (25, 256, 1280, 0, 1e-6, False)),               # bank build: 25 timesteps
    (case_groupnorm, (16, 64, 1280, 1280, 1e-5, True)),
    (case_groupnorm, (16, 1024, 1280, 640, 1e-5, True, 1)),          # the same on the two-kernel path
    (case_groupnorm, (25, 256, 1280, 0, 1e-6, False, 1)),
    (case_groupnorm, (2, 4096, 320, 0, 1e-5, True, 1)),              # two-kernel path forced on small batches
    (case_groupnorm, (1, 1024, 640, 320, 1e-5, True, 1)),
    (case_groupnorm, (1, 16, 1280, 640, 1e-5, True, 1)),
    (case_groupnorm, (3, 1000, 320, 0, 1e-5, True, 1)),
    (case_groupnorm, (2, 4096, 128, 0, 1e-6, True, 1)),              # VAE: 4 channels per group
    (case_groupnorm, (8, 4096, 320, 0, 1e-5, True, 1, 40.0)),        # large mean on the two-kernel path
    (case_groupnorm, (16, 1024, 640, 0, 1e-5, True, 2)),             # cluster path forced on a large batch
    (case_groupnorm, (2, 16384, 128, 0, 1e-6, True, 2)),             # VAE widths on the cluster path
    (case_gemm, (128, 128, 64)),
    (case_gemm, (128, 160, 128)),
    (case_gemm, (4096, 320, 320, True, True)),
    (case_gemm, (1000, 640, 1280, True, False)),
    (case_gemm, (64, 1280, 2560, True, True)),
    (case_gemm, (77, 1280, 768)),
    (case_gemm, (320, 4096, 320)),
    (case_gemm, (64, 1280, 2560, True, True, 8)),
    (case_gemm, (256, 1280, 11520, True, False, 12)),
    (case_gemm, (256, 1280, 1280, True, True, 4)),
    (case_gemm, (1024, 640, 640, True, True, 2)),
    (case_gemm, (2048, 320, 1280, True, True, 2)),
    (case_gemm, (100, 1280, 2560, True, True, 8)),
    (case_gemm, (512, 1280, 5120, True, True, 0)),     # automatic: 160-wide tiles, 4 splits in a cluster
    (case_gemm, (512, 1280, 1280, True, True, 0)),     # automatic: 80-wide tiles, no split (short K)
    (case_gemm, (128, 1280, 2560, True, True, 0)),
    (case_gemm_ln, (8192, 320, 320)),                  # norm2 -> attn2.to_q at 64x64 (cond | uncond of one frame)
    (case_gemm_ln, (2048, 640, 640)),
    (case_gemm_ln, (512, 1280, 1280)),                 # 80-wide tiles: 16 CTAs recompute the same row statistics
    (case_gemm_ln, (100, 1280, 1280)),                 # ragged M
    (case_gemm_ln, (1024, 640, 640, 20.0)),            # row mean 20 against a spread of 1.3
    (case_gemm_batch_bias, (2, 1024, 640, 320)),
    (case_gemm_dual, (1024, 640, 640, 320)),
    (case_gemm_strided_out, (320, 77, 768)),
    (case_geglu, (4096, 320)),
    (case_geglu, (64, 1280)),
    (case_conv, (1, 64, 64, 320, 320)),
    (case_conv, (2, 32, 32, 640, 640, True, True)),
    (case_conv, (2, 16, 16, 1280, 1280)),
    (case_conv, (3, 8, 8, 1280, 1280, True, True)),
    (case_conv, (2, 4, 4, 1280, 1280)),
    (case_conv, (1, 8, 8, 2560, 1280, True, False, 8)),
    (case_conv, (2, 16, 16, 1280, 1280, True, True, 4)),
    (case_conv, (2, 32, 32, 640, 640, True, True, 2)),
    (case_conv, (1, 8, 256, 128, 128, True, True)),        # rows wider than the 128-pixel tile (VAE levels): x0 != 0
    (case_conv, (1, 4, 512, 128, 64, True, False)),
    (case_tuned, (PAIR, case_conv, 2, 6, 256, 64, 128, True, True)),
    (case_conv, (2, 16, 16, 1280, 1280, True, True, 0)),   # automatic: long K -> 160-wide tiles, 4 splits
    (case_conv, (2, 8, 8, 2560, 1280, True, True, 0)),     # automatic: 8 splits
    (case_conv, (1, 16, 16, 1280, 1280, True, False, 0)),  # ControlNet at one frame: M = 256
    # ---- persistent CTA-pair GEMM forced onto small and odd problems ----
    (case_tuned, (PAIR, case_gemm, 512, 256, 128)),                       # 256-wide tile, 2 pairs, one K pass of 2 chunks
    (case_tuned, (PAIR, case_gemm, 384, 320, 320, True, True)),           # odd M tiles: last pair half empty; bias+residual
    (case_tuned, (PAIR, case_gemm, 1000, 640, 1280, True, False)),        # ragged M (TMA store clips rows)
    (case_tuned, (PAIR, case_gemm, 300, 384, 192, True, True)),           # 128-wide tiles
    (case_tuned, (PAIR, case_gemm, 4096, 320, 2880, True, True)),         # long K: ring wraps; 320-wide tile = full N
    (case_tuned, (PAIR, case_gemm, 65536, 320, 320, True, True)),         # 512 tiles over 74 pairs: 7 rounds, both buffers
    (case_tuned, (PAIR, case_gemm, 4096, 1280, 640, True, True)),         # 256-wide tiles, 5 N tiles (K too short for 320)
    (case_tuned, (PAIR, case_gemm, 4096, 1280, 1280, True, True)),        # 320-wide tiles (2 x 160 MMAs, one accumulator)
    (case_tuned, (PAIR, case_gemm, 1000, 640, 2560, True, True)),         # 320-wide, ragged M, 2 N tiles
    (case_tuned, (PAIR, case_gemm, 520, 200, 128, True, True)),           # N = 200: last chunk 8 columns wide, 2nd half empty
    (case_tuned, (PAIR, case_gemm_batch_bias, 2, 1024, 640, 320)),
    (case_tuned, (PAIR, case_gemm_dual, 1024, 640, 640, 320)),
    (case_tuned, (PAIR, case_gemm_strided_out, 320, 80, 768)),            # output row pitch > N
    (case_tuned, (PAIR, case_geglu, 512, 320)),
    (case_tuned, (PAIR, case_geglu, 4096, 320)),
    (case_tuned, (PAIR, case_conv, 1, 64, 64, 320, 320)),
    (case_tuned, (PAIR, case_conv, 8, 64, 64, 320, 320, True, True)),     # full-width conv tile: 128 pairs over 74 clusters
    (case_tuned, (PAIR, case_conv, 2, 32, 32, 640, 640, True, True)),
    (case_tuned, (PAIR, case_conv, 3, 8, 8, 1280, 1280, True, True)),     # 192 rows: second CTA of the pair half out of range
    (case_tuned, (PAIR, case_conv, 16, 16, 16, 1280, 1280)),
    # ---- the same large shapes on the single-CTA tiles (what the heuristics would not pick) ----
    (case_tuned, (NOPAIR, case_gemm, 65536, 320, 320, True, True)),
    (case_tuned, (NOPAIR, case_conv, 8, 64, 64, 320, 320, True, True)),
    (case_conv_direct, (1, 64, 64, 4, 320, 1, False, True)),
    (case_conv_direct, (2, 64, 64, 320, 4, 1, False)),
    (case_conv_direct, (1, 256, 256, 3, 16, 1, True)),
    (case_conv_direct, (1, 128, 128, 16, 32, 2, True)),
    (case_conv_direct, (1, 64, 64, 96, 256, 2, True)),
    (case_conv_s2, (2, 64, 64, 320, 320)),        # the three Downsample convs of one frame (cond | uncond)
    (case_conv_s2, (2, 32, 32, 640, 640)),
    (case_conv_s2, (2, 16, 16, 1280, 1280)),       # 8x8 output: two images per 128-row tile
    (case_conv_s2, (1, 16, 16, 1280, 1280)),       # ControlNet at one frame: half a tile
    (case_tuned, (PAIR, case_conv_s2, 16, 64, 64, 320, 320)),   # eight frames: the pair kernel
    (case_down, (2, 32, 32, 640)),
    (case_down, (1, 24, 16, 640)),
    (case_conv_im2col, (1, 12, 8, 1280, 1280)),
    (case_conv_im2col, (2, 6, 10, 640, 320)),
    (case_attention, (1, 8, 40, 4096, 4096)),
    (case_attention, (2, 8, 40, 1024, 1024, 1024, 2)),
    (case_attention, (2, 8, 40, 1024, 1024, 1024, 1, 1)),
    (case_attention, (2, 8, 40, 1024, 77, 0, 1, None, True)),
    (case_attention, (2, 8, 80, 256, 256, 256, 1)),
    (case_attention, (1, 8, 40, 384, 384, 128, 1)),
    (case_attention, (2, 8, 80, 200, 200, 0, 1)),
    (case_attention, (1, 8, 160, 320, 320, 64, 1)),
    (case_attention, (2, 8, 80, 1024, 77, 0, 1, None, True)),
    (case_attention, (2, 8, 160, 64, 64, 64, 2)),
    (case_attention, (1, 8, 160, 16, 16, 16, 1)),
    (case_attention, (2, 8, 160, 256, 77, 0, 1, None, True)),
    # ---- d=40 on the two-Q-tile kernel at two CTAs per SM (what large grids get) ----
    (case_tuned, (ATT2Q, case_attention, 1, 8, 40, 4096, 4096)),
    (case_tuned, (ATT2Q, case_attention, 2, 8, 40, 1024, 1024, 1024, 2)),
    (case_tuned, (ATT2Q, case_attention, 2, 8, 40, 1024, 1024, 1024, 1, 1)),
    (case_tuned, (ATT2Q, case_attention, 2, 8, 40, 1024, 77, 0, 1, None, True)),
    (case_tuned, (ATT2Q, case_attention, 1, 8, 40, 384, 384, 128, 1)),
    (case_attention, (16, 8, 40, 2048, 2048, 2048, 1, 8)),   # 2048 CTAs: the heuristics pick the two-Q-tile kernel
    # ---- d=80 on the two-Q-tile kernel (one CTA, eight softmax warps per SM) ----
    (case_tuned, (ATT2Q, case_attention, 2, 8, 80, 256, 256, 256, 1)),
    (case_tuned, (ATT2Q, case_attention, 2, 8, 80, 200, 200, 0, 1)),          # ragged: the second Q tile is partly empty
    (case_tuned, (ATT2Q, case_attention, 2, 8, 80, 1024, 77, 0, 1, None, True)),
    (case_tuned, (ATT2Q, case_attention, 1, 8, 80, 384, 384, 128, 1)),        # odd number of Q tiles
    (case_attention, (16, 8, 80, 1024, 1024, 1024, 1, 8)),   # 1024 CTAs: picked by the heuristics
    # ---- hot-path layouts: fused Q|K projection, one text context for the batch, output slice of a wider buffer ----
    (case_attention, (2, 8, 40, 1024, 1024, 0, 1, None, False, "qk_fused")),
    (case_attention, (2, 8, 80, 256, 256, 0, 1, None, False, "qk_fused+wide_out")),
    (case_attention, (2, 8, 160, 64, 64, 0, 1, None, False, "qk_fused")),
    (case_tuned, (ATT2Q, case_attention, 2, 8, 40, 1024, 1024, 0, 1, None, False, "qk_fused+wide_out")),
    (case_tuned, (ATT2Q, case_attention, 2, 8, 80, 384, 384, 0, 1, None, False, "qk_fused")),
    (case_attention, (2, 8, 40, 1024, 77, 0, 1, None, True, "shared_kv")),
    (case_attention, (2, 8, 80, 256, 77, 0, 1, None, True, "shared_kv+wide_out")),
    (case_attention, (2, 8, 160, 256, 77, 0, 1, None, True, "shared_kv")),
    (case_tuned, (ATT2Q, case_attention, 2, 8, 40, 1024, 77, 0, 1, None, True, "shared_kv")),
    (case_tuned, (ATT2Q, case_attention, 2, 8, 80, 256, 77, 0, 1, None, True, "shared_kv")),
    (case_attention, (2, 8, 160, 256, 200, 64, 1, 1, False, "wide_out")),
    (case_layout, (2, 4, 64, 64, 2)),
    (case_layout, (1, 4, 24, 40, 2)),
    (case_time_path, (16, 8)),                 # cond | uncond: rows 8..15 repeat the eight timesteps
    (case_time_path, (6, 1)),                  # one timestep for the whole batch
    (case_cfg_ddim, (0.05,)),                  # stochastic step: sigma * noise
    (case_cfg_ddim, (0.0, True)),              # x advances in place
    (case_cfg_ddim, (0.05, True)),
    (case_softmax_rows, (64, 8, 8)),
    (case_softmax_rows, (16, 4096, 4096)),
    (case_softmax_rows, (32, 1000, 1000)),     # not a multiple of 256 threads x 8
    (case_softmax_rows, (8, 2056, 2112)),      # row pitch > cols
    (case_softmax_rows, (16, 4096, 4160, 0.125)),
    (case_im2col_br, (2, 9, 7, 64)),
    (case_im2col_br, (1, 8, 8, 128)),
    (case_im2col_br, (1, 32, 30, 128)),
]

# ---- online-softmax rescale path: every peaky pattern on every attention kernel ----
# (pattern, n0, n1, bank_batches); all with B=2, 2 heads, 256 queries (two Q tiles)
PEAKY_SHAPES = [("rise", 640, 0, None), ("slow_rise", 768, 0, None), ("mixed_rows", 512, 0, None),
                ("fall", 640, 0, None), ("bank_peak", 256, 128, 1), ("ragged_peak", 77, 0, None),
                ("ragged_peak", 200, 0, None)]
PEAKY_KERNELS = [(None, 160), (None, 40), (None, 80), (ATT2Q, 40), (ATT2Q, 80)]  # attn_tc, attn3 x2, attn2 x2
for _tune, _d in PEAKY_KERNELS:
    for _pat, _n0, _n1, _bb in PEAKY_SHAPES:
        _args = (2, 2, _d, 256, _n0, _n1, _pat, _bb)
        ALL_CASES.append((case_attention_peaky, _args) if _tune is None else
                         (case_tuned, (_tune, case_attention_peaky) + _args))

"""Both attention kernels against a float64 statement of softmax(Q K^T / 8) V, with probes that pin every key column, query
row, frame and head.

attention_tc_kernel (arp_attention, every block but the last) and cls_attention_kernel (arp_cls_attention, the class-token
row of the pruned last block) are fed chosen inputs and compared with a float64 reference computed from exactly the 16-bit
Q, K and V the kernels read, over the L real keys of each (frame, head).

Probes (each for L = 197 and 50, through both kernels):
  pointer        every query row attends to one key by a weight margin of e^32; the target is a cyclic shift that differs
                 per frame and head and covers every key column from tile-0 rows, spread rows and rows 192..196. Q, K and V
                 are small integers: every logit is exact and every output row must equal its target's V row bit for bit.
  row maximum    the pointer codes on top of a random background: a maximum that misses the spike column overflows fp16.
  leak           frames alternate between two orthogonal Q / K subspaces; frame b's queries score frame b+1's first rows (its
                 pad keys) at +512, and the last frame's real logits are all <= -100, so a zero-filled pad key would win.
  uniform        Q = 0: the output is the mean of the L real V rows (divisor L, not the padded NK).
  dynamic range  row maxima from -1000 to +1000 in raw logits, rows whose weights span the 2^-29 flush limit.
  persistent     random inputs at B in {1, 12, 13, 25, 50, 1024}: one item per CTA up to 83.
  plus position / order independence, sentinel rows around the outputs and a cross-check of the two kernels.

CPU: the probe inputs are exact in both operand formats, the pointer targets cover every column from every row group, and
the float64 reference under each plausible wrong semantics moves the answer by >= 100x the probe's bar.
GPU (-m gpu): every probe against its bar; every measured error is printed next to its bar."""
import ctypes as C
import math

import pytest
import torch

W, H, DH = 768, 12, 64
U32 = 2.0 ** -24                    # fp32 unit roundoff
LOG2E = 1.0 / math.log(2.0)
SCALE_LOG2E = 0.125 * LOG2E
FP16, BF16 = torch.float16, torch.bfloat16
# P is TRUNCATED to the operand format (pack_bf16_trunc): relative error in [0, u) with u = 2^-(stored mantissa bits)
U_TRUNC = {FP16: 2.0 ** -10, BF16: 2.0 ** -7}
MANT = {FP16: 10, BF16: 7}
EMIN = {FP16: -14, BF16: -126}
# weights flushed to zero (ex2.approx.ftz below 2^-126): the fp16 build pre-scales the row maximum to 2^15 * 2^-112 = 2^-97,
# so anything below 2^-29 of the maximum flushes; one binade of slack for the ex2.approx error at the boundary
FLUSH_LOG2 = {FP16: -28.0, BF16: -125.0}


def _report(name, err, bar):
    print(f"attention_reference {name}: max err {err:.3e}  bar {bar:.3e}")


def nk(L):
    return (L + 15) // 16 * 16


# ------------------------------------------------------------------------------------------------
# float64 reference
# ------------------------------------------------------------------------------------------------
def heads_view(qkv, B, L):
    """qkv [B*L, 3W] -> q, k, v [B, H, L, DH] float64"""
    x = qkv.double().view(B, L, 3, H, DH).permute(2, 0, 3, 1, 4)
    return x[0], x[1], x[2]


def with_pad(x, L):
    """[B, H, L, DH] -> [B, H, NK, DH] as the tensor core reads the keys: the pad rows of frame b are frame b+1's first
    NK - L rows, the last frame's are the TMA's zero fill"""
    nxt = torch.zeros_like(x[:, :, :nk(L) - L])
    nxt[:-1] = x[1:, :, :nk(L) - L]
    return torch.cat([x, nxt], 2)


def ulp16(x, dt):
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** (EMIN[dt] - MANT[dt]))))
    return torch.exp2(e.clamp_min(EMIN[dt]) - MANT[dt])


def _softmax_chunk(q, k, v, dt, kernel):
    """O and its error terms for q [b, h, Lq, DH] against the real keys k, v [b, h, L, DH] (float64).

    Returns (O, bar, var, sys): per output element the bound |O_kernel - O| <= bar, and for the mean signed error over a
    probe the variance of the zero-mean part (var) and the bound on the systematic part (sys).

    Tensor-core kernel (kernel="tc"), with w the normalised true weights and A_k = |V_k - O| per head dimension:
      * P is truncated to 16 bits, p~_k = p_k (1 - t_k), t_k in [0, u): normalised by the tensor core's own sum of the
        p~ (the ones block), O~ - O = -sum_k w_k (t_k - t_bar) A_k-signed / (1 - t_bar), so |.| <= u / (1 - u) sum_k w_k A_k.
        Its mean over a probe is zero when V is independent of the weights; its variance <= u^2 / 12 sum_k w_k^2 A_k^2.
      * S is an fp32 sum of 64 exact products: |dS_k| <= 64 u32 sum_d |q_d k_d| (raw), a relative weight error dS_k / 8.
      * the exp2 argument s * scale - (m * scale + offset) is formed in fp32 (two roundings of operands up to
        |s| scale + |m| scale + 97) and ex2.approx adds ~2^-22: ln2 * 2 u32 (|s| c + 2 |m| c + 97 + |x|) + 2^-21 relative.
      * weights below the flush limit (2^-29 of the row maximum in the fp16 build) are lost whole: sum over them w_k A_k.
      * P V and the row sum are fp32 sums of NK exact products: NK u32 (sum_k w_k |V_k| + |O|); rcp.approx and the scale
        2 u32 |O|.
      * the output is rounded once to 16 bits: 1/2 ulp(O), variance ulp^2 / 12 (round to nearest).
    Class-token kernel (kernel="cls"): fp32 scores (the same dS_k), an fp32 softmax with the true maximum (__expf: 2 u32 |z|
    + 2^-21 relative, z = (s - m) / 8), fp32 sums over L keys (L u32 (sum w|V| + |O|)), an IEEE division and a multiply
    (2 u32 |O|), one rounding to 16 bits — no truncated P."""
    s = q @ k.transpose(-1, -2)                                           # raw logits
    m = s.amax(-1, keepdim=True)
    z = (s - m) / 8.0                                                     # natural log of the relative weight
    w = torch.exp(z)
    w = w / w.sum(-1, keepdim=True)
    o = w @ v
    a = (v.unsqueeze(-3) - o.unsqueeze(-2)).abs()                         # [b, h, Lq, L, DH]
    ds = 64 * U32 * (q.abs() @ k.abs().transpose(-1, -2)) / 8.0
    L = k.shape[-2]
    if kernel == "tc":
        u = U_TRUNC[dt]
        x = z * LOG2E
        dl = ds + math.log(2.0) * 2 * U32 * (s.abs() * SCALE_LOG2E + 2 * m.abs() * SCALE_LOG2E + 97 + x.abs()) + 2.0 ** -21
        dl = dl + (x < FLUSH_LOG2[dt]).double()                           # flushed: the whole weight is lost
        trunc = u / (1 - u) * (w.unsqueeze(-1) * a).sum(-2)
        sys_ = (((w * dl).unsqueeze(-1)) * a).sum(-2) + nk(L) * U32 * (w @ v.abs() + o.abs()) + 2 * U32 * o.abs()
        var = u * u / 12 * ((w * w).unsqueeze(-1) * a * a).sum(-2)
        pre = trunc + sys_
    else:
        dl = ds + 2 * U32 * z.abs() + 2.0 ** -21
        sys_ = (((w * dl).unsqueeze(-1)) * a).sum(-2) + L * U32 * (w @ v.abs() + o.abs()) + 2 * U32 * o.abs()
        var = torch.zeros_like(o)
        pre = sys_
    ulp = ulp16(o.abs() + pre, dt)
    return o, pre + ulp / 2, var + ulp * ulp / 12, sys_


def reference(q, k, v, dt, kernel, max_elems=1 << 25):
    """softmax(q k^T / 8) v over the real keys, float64, chunked over frames: (O, bar, var, sys) as [B, H, Lq, DH]"""
    per_frame = q.shape[1] * q.shape[2] * k.shape[2] * DH
    step = max(1, max_elems // per_frame)
    parts = [_softmax_chunk(q[i:i + step], k[i:i + step], v[i:i + step], dt, kernel) for i in range(0, q.shape[0], step)]
    return tuple(torch.cat([p[j] for p in parts]) for j in range(4))


def to_rows(x):
    """[B, H, Lq, DH] -> [B*Lq, W] in the kernels' output layout"""
    B, _, Lq, _ = x.shape
    return x.permute(0, 2, 1, 3).reshape(B * Lq, W)


def weights_16bit(s, m_used, dt):
    """the weights the tensor-core kernel forms from raw logits s with row maximum m_used, relative to that maximum:
    y = (s - m) c, exp2(y) — inf where the 16-bit value overflows (fp16: 2^(y + 15) >= 2^16; bf16: the fp32 exp2 >= 2^128),
    0 where ex2.approx.ftz flushes (fp16: 2^(y - 97) < 2^-126; bf16: 2^y < 2^-126)"""
    y = (s - m_used) * SCALE_LOG2E
    lo, hi = (-29.0, 1.0) if dt == FP16 else (-126.0, 128.0)
    p = torch.exp2(y.clamp(lo, hi))
    p[y >= hi] = math.inf
    p[y < lo] = 0.0
    return p


def wrong_answer(qkv, B, L, kind, dt):
    """the float64 answer of the tensor-core kernel under a wrong semantics, [B*L, W]:
    pad            the NK - L pad keys take part (frame b+1's first rows, the last frame's zero fill)
    neighbour      frame b+1's first rows take part (every frame but the last)
    zero_fill      the last frame's zero-filled pad keys take part
    divisor_nk     the row sum runs over all NK keys, P V over the real ones
    frame, head    V of the next frame / head
    max_miss       the row maximum misses the row's largest column (16-bit weights: fp16 overflow)
    no_max         no maximum subtracted (16-bit weights: overflow / underflow)"""
    q, k, v = heads_view(qkv, B, L)
    kp, vp = with_pad(k, L), with_pad(v, L)
    n_real = torch.full((B,), L)
    if kind in ("pad", "neighbour"):
        n_real[:-1] = nk(L)
    if kind in ("pad", "zero_fill"):
        n_real[-1] = nk(L)
    if kind == "frame":
        v = v.roll(-1, 0)
    if kind == "head":
        v = v.roll(-1, 1)
    out = torch.empty(B, H, L, DH, dtype=torch.float64)
    for b in range(B):
        n = int(n_real[b])
        kb, vb = kp[b, :, :n], vp[b, :, :n]
        if n == L:
            vb = v[b]
        s = q[b] @ kb.transpose(-1, -2)
        if kind in ("max_miss", "no_max"):
            if kind == "max_miss":
                second = s.clone()
                second.scatter_(-1, s.argmax(-1, keepdim=True), -math.inf)
                m_used = second.amax(-1, keepdim=True)
            else:
                m_used = torch.zeros_like(s[..., :1])
            p = weights_16bit(s, m_used, dt)
            out[b] = (p @ vb) / p.sum(-1, keepdim=True)
            continue
        p = torch.exp((s - s.amax(-1, keepdim=True)) / 8)
        den = p.sum(-1, keepdim=True)
        if kind == "divisor_nk":
            sp = q[b] @ kp[b].transpose(-1, -2)
            den = torch.exp((sp - s.amax(-1, keepdim=True)) / 8).sum(-1, keepdim=True)
        out[b] = (p @ vb) / den
    return to_rows(out)


# ------------------------------------------------------------------------------------------------
# probes (float64 CPU tensors [B*L, 3W] whose every value is exact in fp16 and in bf16)
# ------------------------------------------------------------------------------------------------
def exact16(x):
    """x rounded to 8 significant bits (bf16), magnitudes below 2^-12 set to zero: exact in both formats"""
    y = x.to(BF16).double()
    return torch.where(y.abs() < 2.0 ** -12, torch.zeros_like(y), y)


def pack(q, k, v):
    """q, k, v [B, H, L, DH] -> qkv [B*L, 3W]"""
    B, _, L, _ = q.shape
    return torch.stack([q, k, v]).permute(1, 3, 0, 2, 4).reshape(B * L, 3 * W).contiguous()


def targets(B, L):
    """pointer target of (frame, head, row): a cyclic shift by 7 (b H + h), prime to 197 and to 50"""
    r = torch.arange(L)
    shift = 7 * torch.arange(B * H).view(B, H, 1)
    return (r.view(1, 1, L) + shift) % L


def pointer_probe(B, L, beta=256.0, background=0.0, seed=0):
    """key j's code is e_(j % 14) + e_(14 + j // 14) (j < NK <= 208: dims 0..28); a query is beta times its target's
    code: logits 2 beta on the target, beta on the keys that share one index, 0 elsewhere (a weight margin of
    e^(beta / 8) = e^32). V entries are odd integers (never 0) that name the frame (dim 1), the head (dim 2) and the key
    (dim 0; dims 3.. a hash of all three), |V| <= 255: exact in bf16. A zero V_t would not do: the e^-32 weights
    of the other keys would then be all of a bf16 output. background > 0 adds N(0, background^2) noise in the
    free dims 29..63 of Q and K."""
    j = torch.arange(nk(L))
    codes = torch.zeros(nk(L), DH, dtype=torch.float64)
    codes[j, j % 14] = 1.0
    codes[j, 14 + j // 14] = 1.0
    t = targets(B, L)
    q = beta * codes[t]
    k = codes[:L].expand(B, H, L, DH).clone()
    b_ = torch.arange(B).view(B, 1, 1, 1)
    h_ = torch.arange(H).view(1, H, 1, 1)
    j_ = torch.arange(L).view(1, 1, L, 1)
    d_ = torch.arange(DH).view(1, 1, 1, DH)
    v = (2 * ((b_ * 7919 + h_ * 104729 + j_ * 1299709 + d_ * 15485863) % 64) - 63).double().expand(B, H, L, DH).clone()
    v[..., 0] = (2 * j_[..., 0] + 1 - 256).double()
    v[..., 1] = (2 * (b_[..., 0] % 100) + 1 - 100).double()
    v[..., 2] = (2 * h_[..., 0] + 1).double()
    if background:
        g = torch.Generator().manual_seed(seed)
        q[..., 29:] = exact16(background * torch.randn(B, H, L, DH - 29, generator=g, dtype=torch.float64))
        k[..., 29:] = exact16(background * torch.randn(B, H, L, DH - 29, generator=g, dtype=torch.float64))
    return pack(q, k, v), t


def pointer_answer(qkv, B, L, t):
    """[B*L, W]: row r of (frame b, head h) is V[b, h, t[b, h, r]]"""
    _, _, v = heads_view(qkv, B, L)
    return to_rows(torch.gather(v, 2, t.to(v.device).unsqueeze(-1).expand(B, H, L, DH)))


def leak_probe(B, L, seed=0):
    """frame b lives in dims 32 (b % 2) .. +31: dims +0..+28 random (sd 1.4: logits of sd ~10 raw), dim +29 the lure —
    q = 8 on every row of frame b, and k = 64 on frame b+1's first NK - L rows (frame b's pad keys: +512 if they leak in;
    frame b+1's own queries live in the other subspace and never see it) — and dim +30 pushes every real logit of the LAST
    frame down by 256 (q = -16, k = 16), so that its zero-filled pad keys (logit 0) would win. V = 0.5 + N(0, 1)."""
    g = torch.Generator().manual_seed(seed)
    q = torch.zeros(B, H, L, DH, dtype=torch.float64)
    k = torch.zeros_like(q)
    for b in range(B):
        o = 32 * (b % 2)
        q[b, :, :, o:o + 29] = exact16(1.4 * torch.randn(H, L, 29, generator=g, dtype=torch.float64))
        k[b, :, :, o:o + 29] = exact16(1.4 * torch.randn(H, L, 29, generator=g, dtype=torch.float64))
        q[b, :, :, o + 29] = 8.0
        if b + 1 < B:
            k[b + 1, :, :nk(L) - L, o + 29] = 64.0
    q[B - 1, :, :, 32 * ((B - 1) % 2) + 30] = -16.0
    k[B - 1, :, :, 32 * ((B - 1) % 2) + 30] = 16.0
    v = exact16(0.5 + torch.randn(B, H, L, DH, generator=g, dtype=torch.float64))
    return pack(q, k, v)


def uniform_probe(B, L, seed=0):
    """Q = 0: every logit is 0, every weight exactly 1 (2^15 in the fp16 build): the output is the mean of the L real V
    rows. K random, V = 1 + N(0, 1) (a non-zero mean, so that a wrong divisor moves the mean of the output)"""
    g = torch.Generator().manual_seed(seed)
    k = exact16(torch.randn(B, H, L, DH, generator=g, dtype=torch.float64))
    v = exact16(1.0 + torch.randn(B, H, L, DH, generator=g, dtype=torch.float64))
    return pack(torch.zeros_like(k), k, v)


def dynamic_range_probe(B, L, seed=0):
    """dim 63: k = 8 on every key and q = offset / 8 with row offsets spread over -1000..+1000 (multiples of 8, exact):
    every logit of a row is shifted by the same offset, so the weights do not change but the maximum the kernel subtracts
    runs over +-1000. dims 0..62: q ~ alpha N(0, 1) with alpha log-spaced over 0.25..8 per row, k ~ N(0, 1): logit spreads
    of sd 2..63 raw — the widest rows' weights span far more than the 2^-29 flush limit. V = 0.5 + N(0, 1)."""
    g = torch.Generator().manual_seed(seed)
    n = B * H * L
    alpha = torch.logspace(math.log10(0.25), math.log10(8.0), n, dtype=torch.float64)[torch.randperm(n, generator=g)]
    q = exact16(alpha.view(B, H, L, 1) * torch.randn(B, H, L, DH, generator=g, dtype=torch.float64))
    k = exact16(torch.randn(B, H, L, DH, generator=g, dtype=torch.float64))
    offs = torch.linspace(-1000.0, 1000.0, n, dtype=torch.float64)[torch.randperm(n, generator=g)]
    q[..., 63] = torch.round(offs / 8.0).view(B, H, L)                    # logit offset 8 q: multiples of 8 up to +-1000
    k[..., 63] = 8.0
    v = exact16(0.5 + torch.randn(B, H, L, DH, generator=g, dtype=torch.float64))
    return pack(q, k, v)


def random_qkv(B, L, seed, device="cpu"):
    """realistic inputs: Q, K ~ 1.5 N(0, 1) (logits of sd 18 raw), V ~ 0.5 + 1.5 N(0, 1), rounded to bf16 (exact in both)"""
    g = torch.Generator(device=device).manual_seed(seed)
    x = 1.5 * torch.randn(B * L, 3 * W, generator=g, device=device)
    x[:, 2 * W:] += 0.5
    y = x.to(BF16).float()
    return torch.where(y.abs() < 2.0 ** -12, torch.zeros_like(y), y)


PROBES = {
    "pointer": lambda B, L: pointer_probe(B, L)[0],
    "row_maximum": lambda B, L: pointer_probe(B, L, background=1.0, seed=1)[0],
    "leak": lambda B, L: leak_probe(B, L, seed=2),
    "uniform": lambda B, L: uniform_probe(B, L, seed=3),
    "dynamic_range": lambda B, L: dynamic_range_probe(B, L, seed=4),
}
# the wrong semantics each probe is built to expose, per operand format (a maximum that misses a column only changes the
# answer where the missed weight overflows, i.e. in the fp16 build; in bf16 the normalisation hides it)
DECISIVE = {
    "pointer": {FP16: ["neighbour", "frame", "head", "max_miss"], BF16: ["neighbour", "frame", "head"]},
    "row_maximum": {FP16: ["max_miss", "frame", "head"], BF16: ["frame", "head"]},
    "leak": {FP16: ["neighbour", "zero_fill", "pad"], BF16: ["neighbour", "zero_fill", "pad"]},
    "uniform": {FP16: ["divisor_nk", "pad"], BF16: ["divisor_nk", "pad"]},
    "dynamic_range": {FP16: ["no_max", "frame", "head"], BF16: ["no_max", "frame", "head"]},
}


# ------------------------------------------------------------------------------------------------
# CPU: the probes are exact and decisive
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [197, 50])
@pytest.mark.parametrize("probe", sorted(PROBES))
def test_probe_inputs_are_exact_in_both_formats(probe, L):
    qkv = PROBES[probe](3, L)
    for dt in (FP16, BF16):
        assert torch.equal(qkv.to(dt).double(), qkv), (probe, dt)
    if probe == "pointer":
        q, k, v = heads_view(qkv, 3, L)
        s = q @ k.transpose(-1, -2)
        assert torch.equal(s, torch.round(s)) and s.abs().max() <= 512     # integer logits: exact in fp32 accumulation
        assert (v != 0).all()


@pytest.mark.parametrize("L", [197, 50])
def test_pointer_targets_cover_every_column_from_every_row_group(L):
    """B = 17 (the GPU probe's size): every key column is some row's target from query tile 0 (rows < 128), from the
    spread rows of tile 1 (128..191) and from rows 192..196 (L = 197); for L = 50 from rows 0..47 and from rows 48, 49.
    The class-token kernel sees row 0's targets only: 204 items cover every column as well."""
    t = targets(17, L)
    groups = [(0, 128), (128, 192), (192, 197)] if L == 197 else [(0, 48), (48, 50)]
    for lo, hi in groups:
        assert set(t[:, :, lo:hi].flatten().tolist()) == set(range(L)), (lo, hi)
    assert set(t[:, :, 0].flatten().tolist()) == set(range(L))
    for b in range(17):                                                   # a permutation of the keys per (frame, head)
        for h in range(H):
            assert sorted(t[b, h].tolist()) == list(range(L))


@pytest.mark.parametrize("L", [197, 50])
def test_leak_probe_geometry(L):
    """the last frame's real logits are all <= -100 (a zero-filled pad key, logit 0, would win by e^12.5), and frame b's
    pad keys score +512 above the real keys' ~N(0, 10^2)"""
    B = 3
    qkv = leak_probe(B, L, seed=2)
    q, k, _ = heads_view(qkv, B, L)
    s_last = q[-1] @ k[-1].transpose(-1, -2)
    assert s_last.max() <= -100
    kp = with_pad(k, L)
    s_pad = q[0] @ kp[0, :, L:].transpose(-1, -2)
    s_real = q[0] @ k[0].transpose(-1, -2)
    assert s_pad.min() >= s_real.max() + 300


@pytest.mark.parametrize("L", [197, 50])
@pytest.mark.parametrize("probe", sorted(PROBES))
def test_wrong_semantics_move_the_answer_far_past_the_bar(probe, L):
    """The tensor-core kernel's float64 answer under each wrong semantics the probe targets moves the output by >= 100x
    the probe's per-element bar somewhere, or its mean by >= 100x the mean bar, or makes it non-finite (fp16 overflow).
    The pointer and row-maximum probes are also decisive against a one-column miss: every row's own target is missed."""
    B = 3
    qkv = PROBES[probe](B, L)
    q, k, v = heads_view(qkv, B, L)
    for dt in (FP16, BF16):
        o, bar, var, sys_ = (to_rows(x) for x in reference(q, k, v, dt, "tc"))
        mean_bar = 6 * math.sqrt(var.sum().item()) / o.numel() + sys_.mean().item()
        for kind in DECISIVE[probe][dt]:
            got = wrong_answer(qkv, B, L, kind, dt)
            if not torch.isfinite(got).all():
                continue
            d = got - o
            elem = (d.abs() / bar).max().item()
            mean = abs(d.mean().item()) / mean_bar
            print(f"attention_reference decisive {probe} L={L} {dt} {kind}: x{elem:.3g} per element, x{mean:.3g} mean")
            assert max(elem, mean) >= 100, (probe, L, dt, kind, elem, mean)


def test_the_reference_is_the_textbook_softmax():
    """the chunked float64 reference equals a plain softmax over the real keys (and the bar collapses to the output
    rounding for exact pointer rows)"""
    qkv = random_qkv(2, 50, seed=5).double()
    q, k, v = heads_view(qkv, 2, 50)
    o = reference(q, k, v, FP16, "tc", max_elems=1)[0]
    want = torch.softmax(q @ k.transpose(-1, -2) * 0.125, -1) @ v
    assert (o - want).abs().max() < 1e-12
    qkv, t = pointer_probe(2, 50)
    q, k, v = heads_view(qkv, 2, 50)
    o = to_rows(reference(q, k, v, FP16, "tc")[0])
    assert (o - pointer_answer(qkv, 2, 50, t)).abs().max() < 1e-9


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def capi():
    from arp_b200 import capi as m
    from arp_b200.build import build
    build()
    return m


@pytest.fixture(scope="module")
def eng(capi):
    e = capi.Engine(device=0, patch=16, in_h=64, in_w=64, max_batch=16)
    yield e
    e.close()


def cls_q(qkv, B, L):
    """the class-token rows' Q third: [B, W]"""
    return qkv.view(B, L, 3 * W)[:, 0, :W].contiguous()


def check(tag, got, o, bar, var, sys_):
    """every element within its bar, the mean signed error within 6 deviations of its zero-mean part plus the systematic
    bound; both printed next to their bars"""
    got = got.double()
    assert torch.isfinite(got).all(), tag
    d = got - o
    ratio = (d.abs() / bar).max().item()
    mean_bar = 6 * math.sqrt(var.sum().item()) / d.numel() + sys_.mean().item()
    _report(f"{tag} per-element (err / bar)", ratio, 1.0)
    _report(f"{tag} mean signed", abs(d.mean().item()), mean_bar)
    assert ratio <= 1.0, (tag, ratio)
    assert abs(d.mean().item()) <= mean_bar, (tag, d.mean().item(), mean_bar)


def run_both(capi, eng, tag, qkv, B, L):
    """attention over all rows and class-token attention of row 0, each against its float64 reference and bars"""
    dt = capi.operand_dtype()
    x = qkv.to("cuda", dt)
    q, k, v = heads_view(x, B, L)
    ref = [to_rows(r) for r in reference(q, k, v, dt, "tc")]
    out = eng.attention(x, B, L)
    check(f"{tag} attention L={L} {dt}", out, *ref)
    ref_c = [to_rows(r) for r in reference(q[:, :, :1], k, v, dt, "cls")]
    out_c = eng.cls_attention(cls_q(x, B, L), x, B, L)
    check(f"{tag} cls_attention L={L} {dt}", out_c, *ref_c)
    return x, out, out_c


POINTER_B = 17


@pytest.mark.gpu
@pytest.mark.parametrize("L", [197, 50])
def test_pointer_rows_are_their_target_v_rows_bit_for_bit(capi, eng, L):
    qkv, t = pointer_probe(POINTER_B, L)
    x, out, out_c = run_both(capi, eng, "pointer", qkv, POINTER_B, L)
    want = pointer_answer(x, POINTER_B, L, t).to(x.dtype)
    bad = (out != want).any(1).nonzero().flatten()
    assert bad.numel() == 0, f"{bad.numel()} rows differ, first rows {bad[:8].tolist()}"
    assert torch.equal(out_c, want.view(POINTER_B, L, W)[:, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("L", [197, 50])
def test_row_maximum_spike_in_every_column(capi, eng, L):
    qkv, t = pointer_probe(POINTER_B, L, background=1.0, seed=1)
    x, out, out_c = run_both(capi, eng, "row_maximum", qkv, POINTER_B, L)
    want = pointer_answer(x, POINTER_B, L, t).to(x.dtype)
    assert torch.equal(out, want), (out != want).any(1).nonzero().flatten()[:8].tolist()
    assert torch.equal(out_c, want.view(POINTER_B, L, W)[:, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("L", [197, 50])
def test_no_neighbour_or_zero_fill_key_leaks_in(capi, eng, L):
    run_both(capi, eng, "leak", leak_probe(9, L, seed=2), 9, L)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [197, 50])
def test_uniform_rows_are_the_mean_of_the_real_v_rows(capi, eng, L):
    run_both(capi, eng, "uniform", uniform_probe(9, L, seed=3), 9, L)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [197, 50])
def test_dynamic_range_of_the_row_maxima(capi, eng, L):
    run_both(capi, eng, "dynamic_range", dynamic_range_probe(9, L, seed=4), 9, L)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 12, 13, 25, 50, 1024])
@pytest.mark.parametrize("L", [197, 50])
def test_persistent_loop_random_inputs(capi, eng, L, B):
    """B * 12 items over min(B * 12, 148) CTAs: one per CTA (B <= 12), a few with both buffer parities, 83 per CTA"""
    run_both(capi, eng, f"persistent B={B}", random_qkv(B, L, seed=100 + B, device="cuda"), B, L)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [197, 50])
def test_every_slot_and_every_call_gives_the_same_bits(capi, eng, L):
    """one frame's qkv in all 1024 slots: every item gives identical bits (the last frame's pad keys are zero fill, every
    other frame's are a neighbour's rows — both masked); two calls on one handle (the launch order reverses) agree"""
    B = 1024
    x = random_qkv(1, L, seed=7, device="cuda").to(capi.operand_dtype()).repeat(B, 1)
    a, b = eng.attention(x, B, L), eng.attention(x, B, L)
    assert torch.equal(a, b)
    a = a.view(B, L, W)
    assert torch.equal(a, a[:1].expand(B, L, W)), (a != a[:1]).any(2).any(1).nonzero().flatten()[:8].tolist()
    q = cls_q(x, B, L)
    c1, c2 = eng.cls_attention(q, x, B, L), eng.cls_attention(q, x, B, L)
    assert torch.equal(c1, c2) and torch.equal(c1, c1[:1].expand(B, W))


SENTINEL_ROWS = 40


def _guarded(rows, dt):
    buf = torch.empty(rows + 2 * SENTINEL_ROWS, W, device="cuda", dtype=dt)
    buf.view(torch.int16).fill_(0x5A5A)
    return buf, buf.clone()


def _sentinels_intact(buf, ref, rows):
    g = SENTINEL_ROWS
    return torch.equal(buf[:g], ref[:g]) and torch.equal(buf[g + rows:], ref[g + rows:])


@pytest.mark.gpu
@pytest.mark.parametrize("L", [197, 50])
def test_outputs_stay_inside_their_rows(capi, eng, L):
    """sentinel rows before and after the B*L output rows of arp_attention and the B rows of arp_cls_attention (B*12 = 60
    items: the last block of 8 warps is half empty)"""
    dt = capi.operand_dtype()
    B = 5
    x = random_qkv(B, L, seed=8, device="cuda").to(dt)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    buf, ref = _guarded(B * L, dt)
    eng._check(eng._lib.arp_attention(eng._h, C.c_void_p(x.data_ptr()), C.c_void_p(buf[SENTINEL_ROWS:].data_ptr()), B, L,
                                      st))
    torch.cuda.synchronize()
    assert _sentinels_intact(buf, ref, B * L)
    assert torch.equal(buf[SENTINEL_ROWS:SENTINEL_ROWS + B * L], eng.attention(x, B, L))
    q = cls_q(x, B, L)
    buf, ref = _guarded(B, dt)
    eng._check(eng._lib.arp_cls_attention(eng._h, C.c_void_p(q.data_ptr()), C.c_void_p(x.data_ptr()),
                                          C.c_void_p(buf[SENTINEL_ROWS:].data_ptr()), B, L, st))
    torch.cuda.synchronize()
    assert _sentinels_intact(buf, ref, B)
    assert torch.equal(buf[SENTINEL_ROWS:SENTINEL_ROWS + B], eng.cls_attention(q, x, B, L))


@pytest.mark.gpu
@pytest.mark.parametrize("L", [197, 50])
def test_class_token_row_of_both_kernels(capi, eng, L):
    """the same qkv through both kernels: row 0 of attention and the class-token attention each within their own bar of
    the float64 answer, hence within the sum of the bars of each other"""
    B = 25
    x, out, out_c = run_both(capi, eng, "cross-check", random_qkv(B, L, seed=9, device="cuda"), B, L)
    dt = capi.operand_dtype()
    q, k, v = heads_view(x, B, L)
    _, bar, _, _ = reference(q[:, :, :1], k, v, dt, "tc")
    _, bar_c, _, _ = reference(q[:, :, :1], k, v, dt, "cls")
    row0 = out.view(B, L, W)[:, 0].double()
    assert ((row0 - out_c.double()).abs() <= to_rows(bar) + to_rows(bar_c)).all()


@pytest.mark.gpu
def test_cls_attention_refuses_bad_arguments(capi, eng):
    x = random_qkv(2, 197, seed=10, device="cuda").to(capi.operand_dtype())
    q = cls_q(x, 2, 197)
    for L in (196, 208, 0):
        with pytest.raises(capi.ArpError) as e:
            eng.cls_attention(q, x, 2, L)
        assert e.value.code == capi.ARP_ERR_INVALID
    out = torch.empty(2, W, device="cuda", dtype=x.dtype)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for ptrs in ((None, x, out), (q, None, out), (q, x, None)):
        args = [None if p is None else C.c_void_p(p.data_ptr()) for p in ptrs]
        assert eng._lib.arp_cls_attention(eng._h, *args, 2, 197, st) == capi.ARP_ERR_INVALID

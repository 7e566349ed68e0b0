"""The reward heads and the adapter tail against a float64 statement of each stage, with the adapter branch carrying weight.

The default adapter checkpoint gates the AdapterMLP at sigma(4) = 0.982 with zero biases, so the MLP supplies under 2 % of
the feature and a wiring error in the adapter tail (a missing ReLU, a dropped bias) moves a cosine by less than the
end-to-end golden bars. Here each stage is fed chosen inputs through the entry points that start at it (tower records:
Engine.label_tower; stored embeddings: Engine.label_embeddings) and compared with a float64 restatement of that stage
alone, with a "live" checkpoint: gate sigma(0) or sigma(-1.5), non-zero adapter biases, a non-identity ln_post.

CPU: the float64 reference reproduces the oracle (AdapterOracle.compute_reward / compute_reward_goal, both normalisations,
and port.compute_reward_clip / compute_reward_clip_goal) from the oracle's own class-token taps, for the default and the
live checkpoint; text_tower.adapter_text_embedding equals AdapterOracle.encode_text with a live text branch.
GPU (-m gpu): the 16-bit adapter tail against the reference rounded at the 16-bit path's rounding points, the fp32 tail
against the plain reference; the instruction side (groups, first / mean, feature norms 1e-3..1e3, cosines near +-1, 0,
+-0.2, per-scale norms over 6 orders of magnitude); the goal distances (sign, exact 0 at the goal, 1-frame episodes,
near-goal frames); ln_post + proj of clip_head_kernel from the tower record's last tap.

Bars are derived from each stage's arithmetic (comments at each); every measured error is printed next to its bar."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

S, E = 13, 512                     # adapter scales, CLIP embedding width
D, DMID, DIN, W = S * E, 12 * E, 12 * 768, 768
U32 = 2.0 ** -24                   # fp32 unit roundoff
SCALE = 1.0 / 0.07                 # exp(logit_scale) of a random-init CLIP


def _report(name, err, bar):
    print(f"heads_reference {name}: max err {err:.3e}  bar {bar:.3e}")


def _unit_roundoff(dtype):
    return {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}[dtype]


# ------------------------------------------------------------------------------------------------
# float64 reference
# ------------------------------------------------------------------------------------------------
def clip_feature_ref(x_cls, ln_g, ln_b, proj):
    """clip head before normalisation: ln_post(class-token row) @ proj, float64"""
    x = x_cls.double()
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return ((x - mu) / torch.sqrt(var + 1e-5) * ln_g.double() + ln_b.double()) @ proj.double()


def adapter_tail_ref(taps, f, sd, round_to=None):
    """(gated feature a, mlp output, gate s), float64. taps [n, 12*768], f [n, 512] the un-normalised CLIP feature.
    round_to = the operand dtype: round where the 16-bit tail rounds (the taps as tower_unpack_kernel packs them,
    inter_w, featf -> featb, fc1_w, the 16-bit hid2, fc2_w); accumulation stays float64."""
    dev = taps.device
    r = (lambda t: t.to(dev).to(round_to).double()) if round_to is not None else (lambda t: t.to(dev).double())
    g = lambda k: sd[k].to(dev).double()  # noqa: E731
    inter = r(taps) @ r(sd["image_intermediate_linear.weight"]).T
    feat = torch.cat([inter, f.to(dev).double()], -1)
    h = torch.relu(r(feat) @ r(sd["image_adapter.layers.0.weight"]).T + g("image_adapter.layers.0.bias"))
    mlp = r(h) @ r(sd["image_adapter.layers.3.weight"]).T + g("image_adapter.layers.3.bias")
    s = torch.sigmoid(g("image_residual_weight").reshape(()))
    return s * feat + (1 - s) * mlp, mlp, float(s)


def cosines_ref(a, text, ensemble=False):
    """[n, n_text] cosines of the un-normalised features a with the text rows as given (unit over the whole row, or per
    512-wide scale for the ensemble, which averages the 13 per-scale cosines)"""
    a, t = a.double(), text.to(a.device).double()
    if ensemble:
        n = a.shape[0]
        an = F.normalize(a.view(n, -1, E), dim=-1).reshape(n, -1)
        return an @ t.T / (a.shape[1] // E)
    return F.normalize(a, dim=-1) @ t.T


def group_rewards_ref(cos, off, reduce, scale):
    """group-major rewards [G, n]: group g = text rows [off[g], off[g+1]), row 0 of the group or the mean"""
    rows = [cos[:, off[g]] if reduce == "first" else cos[:, off[g]:off[g + 1]].mean(1) for g in range(len(off) - 1)]
    return scale * torch.stack(rows)


def goal_ref(feat, ep_off, sign, normalize):
    """sign * ||f_t - f_goal(t)||, goal = the episode's last frame; features L2-normalised first for the adapter variant"""
    x = feat.double()
    if normalize:
        x = F.normalize(x, dim=-1)
    goal = torch.empty(x.shape[0], dtype=torch.long)
    for e in range(len(ep_off) - 1):
        goal[int(ep_off[e]):int(ep_off[e + 1])] = int(ep_off[e + 1]) - 1
    return sign * (x - x[goal.to(x.device)]).norm(dim=-1)


# ------------------------------------------------------------------------------------------------
# the live checkpoint
# ------------------------------------------------------------------------------------------------
def live(sd, res_w, seed=0):
    """sd with the adapter branch carrying weight: gate sigma(res_w), adapter biases drawn like PyTorch's Linear default
    (U(+-1/sqrt(fan_in))), ln_post / ln_final weight 1 + 0.3 N(0,1) and bias 0.1 N(0,1). Image and text sides."""
    out = dict(sd)
    dev = next(iter(sd.values())).device
    g = torch.Generator(device=dev).manual_seed(4242 + seed)
    for side in ("image", "text"):
        w0, w3 = sd[f"{side}_adapter.layers.0.weight"], sd[f"{side}_adapter.layers.3.weight"]
        for k, w in (("0", w0), ("3", w3)):
            bound = w.shape[1] ** -0.5
            out[f"{side}_adapter.layers.{k}.bias"] = (torch.rand(w.shape[0], generator=g, device=dev) * 2 - 1) * bound
        out[f"{side}_residual_weight"] = torch.tensor(float(res_w), device=dev)
    for ln in ("clip_model.visual.ln_post", "clip_model.ln_final"):
        if ln + ".weight" in sd:
            n = sd[ln + ".weight"].shape[0]
            out[ln + ".weight"] = 1 + 0.3 * torch.randn(n, generator=g, device=dev)
            out[ln + ".bias"] = 0.1 * torch.randn(n, generator=g, device=dev)
    return out


# ------------------------------------------------------------------------------------------------
# CPU: the reference is the oracle
# ------------------------------------------------------------------------------------------------
TEXTS = ["navigate a maze to collect the yellow cheese.", "the goal is to collect the coin.",
         "His voice echoed through the empty hallway."]
# the oracle runs in fp32: a cosine of unit vectors over D <= 6656 terms after fp32 GEMMs of K <= 13312 terms carries
# about sqrt(K) * u32 = 7e-6 relative error per feature element, which projects onto a text as ~7e-6 / sqrt(D) per
# standard deviation; 1e-6 on the cosine is > 10 such deviations, and the default checkpoint's smallest mutant
# (a dropped fc2 bias) moves it by 6.5e-6
BAR_ORACLE_COS = 1e-6


@pytest.fixture(scope="module")
def g6():
    from _util import load_golden, rebuild_inputs
    meta, _ = load_golden("g6_clipft_b16_64")
    data, _clip_sd, adapter_sd = rebuild_inputs(meta)
    return meta, np.ascontiguousarray(data["ob"][:5, -1]), adapter_sd


def _oracle_taps(ad):
    return torch.cat([ad.acts[f"visual.transformer.resblocks.{l}"].permute(1, 0, 2)[:, 0, :].float() for l in range(12)],
                     -1)


@pytest.mark.parametrize("res_w", [None, 0.0, -1.5])
def test_adapter_reference_reproduces_the_oracle(g6, res_w):
    from oracle import port
    meta, ims, sd = g6
    sd = sd if res_w is None else live(sd, res_w)
    ad = port.AdapterOracle(sd, meta["arch"])
    vis = {k[len("clip_model.visual."):]: v for k, v in sd.items() if k.startswith("clip_model.visual.")}
    tokens = port.clip_shim.tokenize(TEXTS)
    for ensemble in (False, True):
        for reduce in ("first", "mean"):
            want = ad.compute_reward(ims, TEXTS, ensemble=ensemble, reduce=reduce)
            taps = _oracle_taps(ad)                      # the image forward of that call
            f = clip_feature_ref(taps[:, 11 * W:], vis["ln_post.weight"], vis["ln_post.bias"], vis["proj"])
            a, _, _ = adapter_tail_ref(taps, f, sd)
            t = ad.encode_text(tokens, "per_scale" if ensemble else "all").reshape(len(TEXTS), -1)
            got = group_rewards_ref(cosines_ref(a, t, ensemble), [0, len(TEXTS)], reduce, float(ad.logit_scale.exp()))[0]
            err = (got - torch.from_numpy(want).double()).abs().max().item() / float(ad.logit_scale.exp())
            assert err <= BAR_ORACLE_COS, (res_w, ensemble, reduce, err)
    want = ad.compute_reward_goal(ims)
    taps = _oracle_taps(ad)
    f = clip_feature_ref(taps[:, 11 * W:], vis["ln_post.weight"], vis["ln_post.bias"], vis["proj"])
    got = goal_ref(adapter_tail_ref(taps, f, sd)[0], [0, len(ims)], +1.0, normalize=True).numpy()
    assert got[-1] == 0 and np.all(want >= 0)
    assert np.abs(got - want).max() <= 2 * BAR_ORACLE_COS * math.sqrt(D), (res_w, got, want)


@pytest.mark.parametrize("live_ln", [False, True])
def test_clip_reference_reproduces_the_port(live_ln):
    from _util import load_golden, rebuild_inputs
    from oracle import port
    meta, _ = load_golden("g1_clip_b32_64")
    data, clip_sd, _ = rebuild_inputs(meta)
    if live_ln:
        g = torch.Generator().manual_seed(7)
        clip_sd = dict(clip_sd, **{"visual.ln_post.weight": 1 + 0.3 * torch.randn(W, generator=g),
                                   "visual.ln_post.bias": 0.1 * torch.randn(W, generator=g)})
    model = port.clip_shim.build(meta["arch"], meta["seed"])
    model.load_state_dict(clip_sd)
    model = model.float().eval()
    seen = {}
    model.visual.transformer.resblocks[11].register_forward_hook(lambda m, i, o: seen.__setitem__("x", o.detach()))
    ims = np.ascontiguousarray(data["ob"][:4, -1])
    with torch.no_grad():
        t = F.normalize(model.encode_text(port.clip_shim.tokenize(TEXTS)).double(), dim=-1)
    scale = float(model.logit_scale.detach().exp())
    for reduce in ("first", "mean"):
        want = port.compute_reward_clip(model, ims, TEXTS, reduce=reduce)
        f = clip_feature_ref(seen["x"].permute(1, 0, 2)[:, 0, :], clip_sd["visual.ln_post.weight"],
                             clip_sd["visual.ln_post.bias"], clip_sd["visual.proj"])
        got = group_rewards_ref(cosines_ref(f, t), [0, len(TEXTS)], reduce, scale)[0].numpy()
        assert np.abs(got - want).max() / scale <= BAR_ORACLE_COS, (reduce, got, want)
    want = port.compute_reward_clip_goal(model, ims)
    f = clip_feature_ref(seen["x"].permute(1, 0, 2)[:, 0, :], clip_sd["visual.ln_post.weight"],
                         clip_sd["visual.ln_post.bias"], clip_sd["visual.proj"])
    got = goal_ref(f, [0, len(ims)], -1.0, normalize=False).numpy()
    assert got[-1] == 0 and np.all(want <= 0)
    # fp32 features of norm |f| over 512 terms: sqrt(E) * u32 * |f| per distance, 10x
    assert np.abs(got - want).max() <= 10 * math.sqrt(E) * U32 * f.norm(dim=-1).max().item(), (got, want)


@pytest.mark.parametrize("normalize", ["all", "per_scale"])
def test_text_adapter_embedding_equals_the_oracle_with_a_live_text_branch(g6, normalize):
    from arp_b200.text_tower import adapter_text_embedding
    from oracle import port
    meta, _, sd = g6
    sd = live(sd, -1.5)
    ad = port.AdapterOracle(sd, meta["arch"])
    tokens = port.clip_shim.tokenize(TEXTS)
    want = ad.encode_text(tokens, normalize).reshape(len(TEXTS), -1).double()
    got, scale = adapter_text_embedding(sd, tokens, "cpu", ensemble=normalize == "per_scale")
    assert scale == pytest.approx(float(ad.logit_scale.exp()))
    # two fp32 restatements of the same unit rows: each element within a few sqrt(K) * u32 of the other, K <= 13312
    err = (got.double() - want).abs().max().item()
    assert err <= 10 * math.sqrt(2 * D) * U32, err
    # ... and the live branch matters: the default gate's text embedding is far from it
    base = ad.encode_text(tokens, normalize)
    ad.sd["text_residual_weight"] = torch.tensor(4.0)
    assert (ad.encode_text(tokens, normalize) - base).abs().max() > 1e3 * err


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
def adapter_sd_gpu():
    """the default image adapter (no CLIP tensors: the tower-record entry points do not read them)"""
    from arp_b200.weights import random_adapter_state_dict
    return random_adapter_state_dict("ViT-B/16", seed=21, device="cuda", clip_sd={})


def _engine(capi, head, reduce="first", precision="16bit", max_batch=128):
    return capi.Engine(device=0, patch=16, in_h=64, in_w=64, preprocess=capi.PRE_BILINEAR, head=head,
                       reduce=capi.REDUCE_MEAN if reduce == "mean" else capi.REDUCE_FIRST, max_batch=max_batch,
                       precision=capi.precision_enum(precision))


def _records(T, seed):
    """synthetic tower records: taps like residual-stream class-token rows (N(0,1), one outlier channel of +-20 per
    block, within fp16 range), an O(1) CLIP feature"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    taps = torch.randn(T, 12, W, generator=g, device="cuda")
    taps[:, :, 77] = 20 * torch.sign(torch.randn(T, 12, generator=g, device="cuda"))
    f = torch.randn(T, E, generator=g, device="cuda")
    return torch.cat([taps.reshape(T, DIN), f], -1).contiguous()


def _unit_texts(n, ensemble, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    t = torch.randn(n, D, generator=g, device="cuda", dtype=torch.float64)
    t = F.normalize(t.view(n, S, E), dim=-1).reshape(n, D) if ensemble else F.normalize(t, dim=-1)
    return t.float()


def _tail_sigma(mlp, a, s, u, ensemble):
    """one standard deviation of a cosine's error when every element of the mlp output carries an independent relative
    error of rms u: projected on a unit text independent of those errors, the gated feature's relative error u *
    (1-s) * |mlp| / |a| spreads over D directions (per scale for the ensemble, which averages 13 such cosines)"""
    if ensemble:
        n = a.shape[0]
        r = (mlp.view(n, S, E).norm(dim=-1) / a.view(n, S, E).norm(dim=-1)) ** 2
        return ((1 - s) * u * torch.sqrt(r.sum(-1) / E) / S).max().item()
    return ((1 - s) * u * mlp.norm(dim=-1) / a.norm(dim=-1)).max().item() / math.sqrt(D)


TOWER_T = 301                      # not a multiple of HEAD_FR = 4; crosses two max_batch = 128 chunk boundaries
TOWER_HEADS = ["HEAD_ADAPTER", "HEAD_ADAPTER_ENSEMBLE"]


@pytest.mark.gpu
@pytest.mark.parametrize("res_w", [0.0, -1.5])
@pytest.mark.parametrize("precision", ["16bit", "fp32resid", "fp32"])
@pytest.mark.parametrize("head", TOWER_HEADS)
def test_adapter_tail_from_tower_records(capi, adapter_sd_gpu, head, precision, res_w):
    ensemble = head == "HEAD_ADAPTER_ENSEMBLE"
    sd = live(adapter_sd_gpu, res_w, seed=1)
    rec = _records(TOWER_T, seed=3)
    texts = _unit_texts(16, ensemble, seed=5)
    off = torch.tensor([0, 40, 41, 170, TOWER_T], dtype=torch.int64)
    op = capi.operand_dtype()
    round_to = None if precision == "fp32" else op
    a, mlp, s = adapter_tail_ref(rec[:, :DIN], rec[:, DIN:], sd, round_to)
    cos = cosines_ref(a, texts, ensemble)
    # Bars. The 16-bit tail against the reference rounded at the same points: the kernel differs only by its fp32
    # accumulation order (sqrt(K) * u32 <= 7e-6 relative for K <= 13312) and by the one-ulp flips that error causes at the
    # ~sqrt(K) * u32 / u16 of the 16-bit rounding points that sit that close to a midpoint (1 % of featb in fp16); through
    # fc1 they flip part of hid2, at most all of it: a relative error of at most u16 rms on the mlp output. A cosine then
    # moves by ~_tail_sigma(u16) per standard deviation; the bar is 6 of them over the <= 4816 (frame, text) pairs. The
    # mean over the 301 frames of a text's error shrinks by sqrt(301) for such independent errors but not for a wiring
    # error, which shifts every frame the same way (a dropped bias): its bar is 6 deviations of that mean.
    # The fp32 tail against the plain reference: fp32 accumulation only, sqrt(2D) * u32 relative on every element of a.
    if round_to is not None:
        sig = _tail_sigma(mlp, a, s, _unit_roundoff(op), ensemble)
    else:
        sig = math.sqrt(2 * D) * U32 / math.sqrt(E if ensemble else D)
    bar, bar_mean = 6 * sig, 6 * sig / math.sqrt(TOWER_T)
    e = _engine(capi, getattr(capi, head), "first", precision)
    e.load_state_dict({k: v for k, v in sd.items() if k.startswith(("image_intermediate_linear.", "image_adapter.",
                                                                     "image_residual_weight"))})
    e.set_text_groups([texts[i:i + 1] for i in range(16)], SCALE)          # every (frame, text) cosine as a reward row
    got = e.label_tower(rec, off, 4)[0].double() / SCALE                   # [16, T]
    err = (got - cos.T).abs()
    tag = f"tail {head} {precision} res_w={res_w}"
    _report(tag, err.max().item(), bar)
    _report(tag + " frame-mean", (got - cos.T).mean(1).abs().max().item(), bar_mean)
    if round_to is not None:
        plain = cosines_ref(adapter_tail_ref(rec[:, :DIN], rec[:, DIN:], sd)[0], texts, ensemble)
        print(f"heads_reference {tag}: against the plain float64 reference (not asserted): "
              f"{(got - plain.T).abs().max().item():.3e}")
    assert err.max().item() <= bar
    assert (got - cos.T).mean(1).abs().max().item() <= bar_mean
    # ragged groups, mean over each
    sizes = [1, 2, 3, 4, 6]
    goff = np.concatenate([[0], np.cumsum(sizes)])
    e.close()
    e = _engine(capi, getattr(capi, head), "mean", precision)
    e.load_state_dict({k: v for k, v in sd.items() if k.startswith(("image_intermediate_linear.", "image_adapter.",
                                                                     "image_residual_weight"))})
    e.set_text_groups([texts[goff[g]:goff[g + 1]] for g in range(len(sizes))], SCALE)
    got = e.label_tower(rec, off, 4)[0].double()
    want = group_rewards_ref(cos, goff, "mean", SCALE)
    err = ((got - want) / SCALE).abs().max().item()
    _report(tag + " ragged mean", err, bar)
    assert err <= bar
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["16bit", "fp32resid", "fp32"])
def test_adapter_goal_from_tower_records(capi, adapter_sd_gpu, precision):
    sd = live(adapter_sd_gpu, 0.0, seed=2)
    rec = _records(TOWER_T, seed=4)
    rec[149] = rec[150]                      # a frame whose record equals its goal's: distance 0 in any arithmetic
    off = torch.tensor([0, 1, 60, 61, 62, 151, 152, 250, TOWER_T], dtype=torch.int64)   # 1-frame episodes
    op = capi.operand_dtype()
    round_to = None if precision == "fp32" else op
    a, mlp, s = adapter_tail_ref(rec[:, :DIN], rec[:, DIN:], sd, round_to)
    want = goal_ref(a, off.tolist(), +1.0, normalize=True)
    # |d(a_t) - d(a_g)| <= |da_t|/|a_t| + |da_g|/|a_g| for unit-normalised features: twice the whole-vector relative
    # error (not one projection of it) — u16 * (1-s) |mlp| / |a| on the 16-bit tail, sqrt(2D) * u32 on the fp32 one
    if round_to is not None:
        bar = 2 * (1 - s) * _unit_roundoff(op) * (mlp.norm(dim=-1) / a.norm(dim=-1)).max().item()
    else:
        bar = 2 * math.sqrt(2 * D) * U32
    e = _engine(capi, capi.HEAD_ADAPTER_GOAL, precision=precision)
    e.load_state_dict({k: v for k, v in sd.items() if k.startswith(("image_intermediate_linear.", "image_adapter.",
                                                                     "image_residual_weight"))})
    got = e.label_tower(rec, off, 4)[0].double()
    last = off[1:] - 1
    assert torch.all(got[last.cuda()] == 0) and got[149] == 0
    assert torch.all(got >= 0)                                             # +1: the adapter variant's sign
    err = (got - want).abs().max().item()
    _report(f"goal HEAD_ADAPTER_GOAL {precision}", err, bar)
    assert err <= bar
    e.close()


GROUP_SIZES = [1, 16, 2, 8, 3, 1, 4, 5, 2, 6, 1, 3, 4, 2, 5, 1]          # 64 texts in 16 ragged groups
EMB_T = 203
COS_TARGETS = [1.0, -1.0, 0.0, 0.2, -0.2, 0.99999, -0.99999]


def _frames_at_cosines(texts, T, ensemble, seed, scale_norms):
    """features of norms 1e-3..1e3 (log-spaced), frame b at cosine COS_TARGETS[b % 7] to text b % 64 (per scale for the
    ensemble, whose 13 scales' norms also spread over 6 orders of magnitude)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    n_text, dim = texts.shape
    blocks = S if ensemble else 1
    t = texts.double().view(n_text, blocks, dim // blocks)
    out = torch.empty(T, blocks, dim // blocks, dtype=torch.float64, device="cuda")
    for b in range(T):
        tb = t[b % n_text]
        c = COS_TARGETS[b % len(COS_TARGETS)]
        n = torch.randn(blocks, dim // blocks, generator=g, device="cuda", dtype=torch.float64)
        n = F.normalize(n - (n * tb).sum(-1, keepdim=True) * tb, dim=-1)
        out[b] = c * tb + math.sqrt(max(0.0, 1 - c * c)) * n
    norms = torch.logspace(-3, 3, T, dtype=torch.float64, device="cuda")[torch.randperm(T, generator=g, device="cuda")]
    out = out * norms.view(T, 1, 1)
    if scale_norms:
        out = out * torch.logspace(-3, 3, S, dtype=torch.float64, device="cuda").view(1, S, 1)
    return out.reshape(T, dim).float()


@pytest.mark.gpu
@pytest.mark.parametrize("reduce", ["first", "mean"])
@pytest.mark.parametrize("head", ["HEAD_CLIP", "HEAD_ADAPTER", "HEAD_ADAPTER_ENSEMBLE"])
def test_instruction_side_from_stored_embeddings(capi, head, reduce):
    ensemble = head == "HEAD_ADAPTER_ENSEMBLE"
    dim = E if head == "HEAD_CLIP" else D
    g = torch.Generator(device="cuda").manual_seed(9)
    t = torch.randn(64, dim, generator=g, device="cuda", dtype=torch.float64)
    texts = (F.normalize(t.view(64, S, E), dim=-1).reshape(64, D) if ensemble else F.normalize(t, dim=-1)).float()
    emb = _frames_at_cosines(texts, EMB_T, ensemble, seed=10, scale_norms=ensemble)
    off = np.concatenate([[0], np.cumsum(GROUP_SIZES)])
    e = _engine(capi, getattr(capi, head), reduce)
    e.set_text_groups([texts[off[k]:off[k + 1]] for k in range(len(GROUP_SIZES))], SCALE)
    got = e.label_embeddings(emb, torch.tensor([0, EMB_T]), 4)[0].double()
    want = group_rewards_ref(cosines_ref(emb, texts, ensemble), off, reduce, SCALE)
    # inputs are exact fp32 values: the kernel's only error is fp32 arithmetic — a norm and a dot product over L = 512
    # (clip, and each scale of the ensemble) or 6656 terms, sqrt(L) * u32 relative per standard deviation; a cosine's
    # error is at most 2 such relative errors (dot and norm) times |cos| <= 1, plus the unit rows' own fp32 rounding
    # (u32 per element, sqrt(L) * u32 over the row). Bar: 6 deviations, i.e. 6 * 3 * sqrt(L) * u32.
    bar = 18 * math.sqrt(E if head != "HEAD_ADAPTER" else D) * U32
    err = ((got - want) / SCALE).abs().max().item()
    _report(f"embeddings {head} {reduce}", err, bar)
    assert err <= bar
    e.close()


@pytest.mark.gpu
def test_clip_goal_from_stored_embeddings(capi):
    T = 64
    g = torch.Generator(device="cuda").manual_seed(12)
    emb = torch.randn(T, E, generator=g, device="cuda") * torch.logspace(-2, 2, T, device="cuda").view(T, 1)
    off = [0, 1, 20, 21, 40, 63, T]                                        # 1-frame episodes
    # frames a tiny step from their goal: the distance cancels in fp32 (|a - g| << |a|)
    for t_, rel in ((18, 1e-3), (17, 1e-6), (38, 1e-4), (61, 1e-5)):
        goal = next(off[k + 1] - 1 for k in range(len(off) - 1) if off[k] <= t_ < off[k + 1])
        emb[t_] = emb[goal] + rel * emb[goal].norm() * F.normalize(torch.randn(E, generator=g, device="cuda"), dim=0)
    e = _engine(capi, capi.HEAD_CLIP_GOAL)
    got = e.label_embeddings(emb, torch.tensor(off), 4)[0].double()
    want = goal_ref(emb, off, -1.0, normalize=False)
    for k in range(1, len(off)):
        assert got[off[k] - 1] == 0
    assert torch.all(got <= 0)                                             # -1: clip_goal_conditioned's sign
    # each a_k - g_k of fp32 inputs is rounded once (u32 relative to the difference itself, whatever the cancellation),
    # then squared and summed over 512 terms: sqrt(E) * u32 relative per deviation; the bar is 6 of them, relative
    rel = ((got - want).abs() / want.abs().clamp_min(1e-30)).max().item()
    _report("goal HEAD_CLIP_GOAL relative", rel, 6 * math.sqrt(E) * U32 + 2 * U32)
    assert rel <= 6 * math.sqrt(E) * U32 + 2 * U32
    e.close()


@pytest.mark.gpu
def test_ln_post_and_proj_of_the_clip_head(capi):
    """tap 11 of the tower record is the class-token row clip_head_kernel reads (fp32 path) or its operand-rounded copy
    (16-bit paths); the record's last 512 columns are ln_post(row) @ proj. The only test here that runs the ViT."""
    from arp_b200.weights import random_adapter_state_dict, random_clip_state_dict
    clip_sd = random_clip_state_dict("ViT-B/16", seed=2, device="cuda", with_text=False)
    sd = live(random_adapter_state_dict("ViT-B/16", seed=2, device="cuda", clip_sd=clip_sd), 0.0, seed=3)
    ln_g, ln_b, proj = (sd[f"clip_model.visual.{k}"] for k in ("ln_post.weight", "ln_post.bias", "proj"))
    ob = np.random.default_rng(0).integers(0, 256, (16, 64, 64, 3), dtype=np.uint8)
    op = capi.operand_dtype()
    for precision in ("fp32", "16bit", "fp32resid"):
        e = _engine(capi, capi.HEAD_ADAPTER, precision=precision, max_batch=16)
        assert not e.load_state_dict(sd)
        rec = torch.from_numpy(e.embed_tower_host(ob)).cuda()
        e.close()
        x = rec[:, 11 * W:12 * W].double()
        want = clip_feature_ref(x, ln_g, ln_b, proj)
        got = rec[:, DIN:].double()
        xc = x - x.mean(-1, keepdim=True)
        rstd = 1 / torch.sqrt((xc ** 2).mean(-1, keepdim=True) + 1e-5)
        y = xc * rstd                                                     # normalised row, before the affine
        # fp32: the LayerNorm statistics and the 768-term projection, sqrt(W) * u32 relative per deviation of
        # sum_i |y_i g_i P_ij| + |b_i P_ij|; bar 6 deviations plus the statistics' own rounding (another sqrt(W) * u32)
        mag = ((y * ln_g.double()).abs() + ln_b.double().abs()) @ proj.double().abs()
        bar = 12 * math.sqrt(W) * U32 * mag
        if precision != "fp32":
            # the row the head read is x + dx, dx_i independent round-to-nearest errors, uniform in +-u16 |x_i|
            # (variance (u16 x_i)^2 / 3). To first order the feature moves by J^T dx with the LayerNorm + proj Jacobian
            # J = rstd (I - 11^T/W - y y^T/W) diag(g) P; the bar is 6 standard deviations of that sum.
            eye = torch.eye(W, dtype=torch.float64, device="cuda")
            m = eye - 1.0 / W - y.unsqueeze(2) * y.unsqueeze(1) / W          # [n, W, W], symmetric
            jac = rstd.unsqueeze(2) * m @ (ln_g.double().view(W, 1) * proj.double())
            var = torch.einsum("bij,bi->bj", jac ** 2, (_unit_roundoff(op) * x) ** 2 / 3)
            bar = bar + 6 * torch.sqrt(var)
        err = (got - want).abs()
        _report(f"ln_post+proj {precision}", (err / bar).max().item(), 1.0)
        assert torch.all(err <= bar), (precision, (err / bar).max().item())

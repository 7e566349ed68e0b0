"""Adapter fine-tuning forward (SURVEY.md §8(f)4): drop-in for finetune_module/clip_multiscale_adapter.py's
`CLIPMultiscaleAdapter` as a TRAINABLE module (`forward(batch)` = VIP-I + inverse-dynamics losses, :179-252).

Split along the reference's own gradient boundary. CLIP is frozen (finetune.py:147-148), the forward hooks detach
what they capture (finetune_module/utils.py:6-11) and the images carry no gradient, so everything CLIP computes is
a pure forward: the class-token row of every vision block plus `encode_image`. That half runs in the native
library (`arp_encode_taps_chw`: the same tcgen05 GEMM / attention / LayerNorm kernels as the labeler, fed with the
caller-preprocessed fp32 image batch). The half that carries gradients — the intermediate linears, the two gated
AdapterMLPs, the inverse-dynamics MLP, the residual gates and `lambda_id` — stays in PyTorch autograd with the
reference's parameter names, so `state_dict()` / `load_state_dict()` exchange checkpoints with the reference
(finetune.py:164, label_reward.py:174-176) and `finetune.py`'s training loop runs on it unchanged.

One deliberate difference: the reference runs the frozen tower once per image role (3 or 4 `encode_image` calls per
step, :207-215); here all roles go through it as ONE batch (no cross-sample op exists in eval/frozen CLIP, Q6).

There is no CPU fallback for the frozen tower: `encode_image` needs the sm_100a library and a B200.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F
from torch import nn

from . import capi, text_tower
from .weights import ARCH

_MEAN = (0.48145466, 0.4578275, 0.40821073)
_STD = (0.26862954, 0.26130258, 0.27577711)


class AdapterMLP(nn.Module):
    """finetune_module/layers.py:6-60 with the arguments the adapter uses (ReLU, Identity norm, orthogonal weights,
    zero biases): `layers` = Sequential(Linear, Identity, ReLU, [Linear, Identity, ReLU]*, Linear)."""

    def __init__(self, input_dim=512, hidden_dim=1024, output_dim=1024, num_layers=2):
        super().__init__()
        mods = [nn.Linear(input_dim, hidden_dim), nn.Identity(), nn.ReLU()]
        for _ in range(num_layers - 2):
            mods += [nn.Linear(hidden_dim, hidden_dim), nn.Identity(), nn.ReLU()]
        mods.append(nn.Linear(hidden_dim, output_dim))
        gain = nn.init.calculate_gain("relu")
        for m in mods:
            if isinstance(m, nn.Linear):
                nn.init.orthogonal_(m.weight, gain=gain)
                nn.init.zeros_(m.bias)
        self.layers = nn.Sequential(*mods)

    def forward(self, x):
        return self.layers(x)


class FrozenClip(nn.Module):
    """Stands where `self.clip_model` stands in the reference: holds CLIP's state_dict (saved / loaded under
    `clip_model.`), has no `nn.Parameter`s (so `for p in model.clip_model.parameters(): p.requires_grad = False`
    is a no-op and the optimizer never sees CLIP), and evaluates the vision tower through the native library."""

    def __init__(self, state_dict: dict, arch: str = "ViT-B/16", max_batch: int = 256, precision: str = "16bit"):
        prec = capi.precision_enum(precision)
        super().__init__()
        self.arch = arch
        self.patch, self.vision_width, self.vision_layers, self.embed_dim, self.text_width, self.text_layers = ARCH[arch][:6]
        self._sd = {k: v.detach().clone() for k, v in state_dict.items() if torch.is_tensor(v)}
        self._max_batch, self._precision = int(max_batch), prec
        self._engine = None
        self._engine_stale = True
        self._text_cache: dict = {}

    # -- what the reference reads off clip_model (clip_multiscale_adapter.py:59-61,102) -------------------------
    @property
    def logit_scale(self) -> torch.Tensor:
        return self._sd["logit_scale"]

    # -- nn.Module plumbing: CLIP's tensors travel with .to()/.state_dict()/.load_state_dict() ------------------
    def _apply(self, fn, recurse=True):
        super()._apply(fn)
        self._sd = {k: fn(v) for k, v in self._sd.items()}
        self._engine_stale = True
        self._text_cache.clear()
        return self

    def _save_to_state_dict(self, destination, prefix, keep_vars):
        for k, v in self._sd.items():
            destination[prefix + k] = v if keep_vars else v.detach()

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        seen = set()
        for k, v in state_dict.items():
            if not k.startswith(prefix):
                continue
            name = k[len(prefix):]
            if name in self._sd:
                if tuple(v.shape) != tuple(self._sd[name].shape):
                    error_msgs.append(f"size mismatch for {k}: {tuple(v.shape)} vs {tuple(self._sd[name].shape)}")
                    continue
                self._sd[name] = v.detach().to(self._sd[name].device, self._sd[name].dtype).clone()
                seen.add(name)
            elif strict:
                unexpected_keys.append(k)
        if strict:
            missing_keys.extend(prefix + n for n in self._sd if n not in seen)
        if seen:
            self._engine_stale = True
            self._text_cache.clear()

    # -- frozen forward passes ----------------------------------------------------------------------------------
    def _get_engine(self, device: torch.device):
        if device.type != "cuda":
            raise RuntimeError("the frozen CLIP tower runs in libarp_b200.so on a B200: move the module and its "
                               "inputs to a CUDA device (there is no CPU fallback)")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        if self._engine is None or self._engine.cfg.device != idx:
            self._engine = capi.Engine(device=idx, patch=self.patch, in_h=224, in_w=224, preprocess=capi.PRE_BILINEAR,
                                       head=capi.HEAD_CLIP, max_batch=self._max_batch, layers=self.vision_layers,
                                       width=self.vision_width, heads=self.vision_width // 64,
                                       embed_dim=self.embed_dim, precision=self._precision)
            self._engine_stale = True
        if self._engine_stale:
            missing = self._engine.load_state_dict({k: v for k, v in self._sd.items() if k.startswith("visual.")})
            if missing:
                raise RuntimeError(f"CLIP state_dict lacks vision-tower tensors: {missing[:4]} ...")
            self._engine_stale = False
        return self._engine

    @torch.no_grad()
    def image_taps(self, image: torch.Tensor):
        """image fp32 [T,3,224,224] -> (class-token row of every vision block [T, layers*width], encode_image [T, embed])."""
        return self._get_engine(image.device).encode_taps(image)

    @torch.no_grad()
    def encode_image(self, image: torch.Tensor) -> torch.Tensor:
        return self.image_taps(image)[1]

    @torch.no_grad()
    def text_taps(self, tokens: torch.Tensor):
        """tokens int [n,77] -> (EOT row of every text block [n, layers*width], encode_text [n, embed]). The instruction
        set of a run is tiny and repeats every step, so results are cached per token row."""
        dev = self._sd["logit_scale"].device
        rows = [tuple(int(t) for t in r) for r in tokens.detach().cpu().tolist()]
        todo = [r for r in dict.fromkeys(rows) if r not in self._text_cache]
        if todo:
            feat, taps = text_tower.encode_text(self._sd, torch.tensor(todo, dtype=torch.long), dev)
            taps = torch.cat(taps, dim=-1)
            for i, r in enumerate(todo):
                self._text_cache[r] = (taps[i], feat[i])
            while len(self._text_cache) > 4096:
                self._text_cache.pop(next(iter(self._text_cache)))
        return (torch.stack([self._text_cache[r][0] for r in rows]), torch.stack([self._text_cache[r][1] for r in rows]))


class CLIPMultiscaleAdapter(nn.Module):
    """Same constructor arguments, attribute names, parameter names and `forward(batch)` contract as
    finetune_module/clip_multiscale_adapter.py:39-252. Extra keyword-only arguments:
      clip_state_dict  CLIP weights (openai/CLIP `state_dict` keys); the reference downloads them in `load_clip` (:118-119),
                       here they come from the caller or from `model_path` (a torch.save'd state_dict)
      augmentation     callable applied to the resized 0..255 image batch when train=True (the reference's kornia
                       ColorJitter, :24-36; kornia is the caller's dependency, default identity)
    """

    def __init__(self, model_path: str = None, input_dim: int = 512, hidden_dim: int = 1024, output_dim: int = 512,
                 action_dim: int = 15, num_layers: int = 2, device: torch.device = None,
                 use_discrete_action: bool = False, use_vip_loss: bool = False, use_id_loss: bool = False,
                 lambda_id: float = 0.1, goal_conditioned: bool = False, *, clip_state_dict: dict = None,
                 arch: str = "ViT-B/16", augmentation=None, max_batch: int = 256, precision: str = "16bit",
                 init: str = "orthogonal"):
        super().__init__()
        self.model_path = model_path
        if clip_state_dict is None:
            if not model_path:
                raise ValueError("no network here: pass clip_state_dict= or model_path= (a saved CLIP state_dict)")
            from .weights import load_checkpoint
            clip_state_dict = load_checkpoint(model_path)
        self.clip_model = FrozenClip(clip_state_dict, arch=arch, max_batch=max_batch, precision=precision)
        self.num_clip_layers = self.clip_model.text_layers                    # :59 (text tower depth; 12 = vision depth too)
        self.visual_dim = self.clip_model.vision_width
        self.text_dim = self.clip_model.text_width
        # The reference ALWAYS jitters training images: kornia ColorJitter(0.1, 0.2, 0.2, 0.03, same_on_batch=True, p=0.75)
        # (clip_multiscale_adapter.py:24-36, :128-129). Same default here when kornia is importable; otherwise identity,
        # and preprocess(train=True) warns once so that a fine-tuning run does not silently lose its augmentation.
        self._augmentation_missing = False
        if augmentation is None:
            try:
                from kornia.augmentation import ColorJitter  # type: ignore
                augmentation = nn.Sequential(ColorJitter(0.1, 0.2, 0.2, 0.03, same_on_batch=True, p=0.75))
            except Exception:  # noqa: BLE001 — kornia is the caller's dependency (not in this image)
                augmentation, self._augmentation_missing = (lambda x: x), True
        self.augmentation = augmentation
        self.device = device
        self.use_vip_loss, self.use_id_loss = use_vip_loss, use_id_loss
        L = self.num_clip_layers
        orth = nn.init.orthogonal_
        if init != "orthogonal":      # 13312x6656 orthogonal init is an O(n^3) QR; a checkpoint load overwrites it anyway
            nn.init.orthogonal_ = lambda w, gain=1.0: nn.init.normal_(w, std=gain / math.sqrt(w.shape[1]))
        try:
            self.image_intermediate_linear = nn.Linear(self.visual_dim * L, self.text_dim * L, bias=False)
            self.text_intermediate_linear = nn.Linear(self.text_dim * L, self.text_dim * L, bias=False)
            self.image_adapter = AdapterMLP(input_dim * (L + 1), hidden_dim * (L + 1), output_dim * (L + 1), num_layers)
            self.text_adapter = AdapterMLP(input_dim * (L + 1), hidden_dim * (L + 1), output_dim * (L + 1), num_layers)
            self.inverse_layer = AdapterMLP(4 * output_dim * (L + 1), hidden_dim, action_dim, num_layers)
        finally:
            nn.init.orthogonal_ = orth
        self.image_residual_weight = nn.Parameter(torch.tensor(4.0))
        self.text_residual_weight = nn.Parameter(torch.tensor(4.0))
        self.use_discrete_action = use_discrete_action
        self.loss_fn = nn.CrossEntropyLoss() if use_discrete_action else nn.MSELoss()
        self.lambda_id = nn.Parameter(torch.ones([]) * math.log(1 / 0.07))      # :111 (the float argument is unused there too)
        self.gamma = 0.98
        self.goal_conditioned = goal_conditioned
        if device is not None:
            self.to(device)

    @property
    def logit_scale(self) -> torch.Tensor:       # :102 — CLIP's value, detached, not a parameter (Q5)
        return self.clip_model.logit_scale.detach()

    # :121-133
    def preprocess(self, x: torch.Tensor, train: bool = False) -> torch.Tensor:
        B, H, W, C = x.shape
        assert C == 3
        x = x.permute(0, 3, 1, 2).float()
        if H != 224 and W != 224:                  # pinned torchvision 0.12: bilinear, align_corners=False, no antialias
            x = F.interpolate(x, size=(224, 224), mode="bilinear", align_corners=False, antialias=False)
        if train:
            if self._augmentation_missing:
                import warnings
                warnings.warn("CLIPMultiscaleAdapter.preprocess(train=True): kornia is not importable, so the reference's "
                              "ColorJitter augmentation is NOT applied; pass augmentation= explicitly (identity: "
                              "augmentation=lambda x: x)", RuntimeWarning, stacklevel=2)
                self._augmentation_missing = False
            with torch.no_grad():
                x = self.augmentation(x)
        x = x / 255.0
        mean = torch.tensor(_MEAN, device=x.device, dtype=x.dtype).view(1, 3, 1, 1)
        std = torch.tensor(_STD, device=x.device, dtype=x.dtype).view(1, 3, 1, 1)
        return ((x - mean) / std).contiguous()

    # the half with gradients: :144-151 / :167-176
    def adapt_image(self, taps: torch.Tensor, feat: torch.Tensor) -> torch.Tensor:
        f = torch.cat([self.image_intermediate_linear(taps), feat], dim=-1)
        res = torch.sigmoid(self.image_residual_weight)
        return F.normalize(res * f + (1.0 - res) * self.image_adapter(f), dim=-1)

    def adapt_text(self, taps: torch.Tensor, feat: torch.Tensor) -> torch.Tensor:
        f = torch.cat([self.text_intermediate_linear(taps), feat], dim=-1)
        res = torch.sigmoid(self.text_residual_weight)
        return F.normalize(res * f + (1.0 - res) * self.text_adapter(f), dim=-1)

    def encode_image(self, image: torch.Tensor) -> torch.Tensor:     # :135-151
        taps, feat = self.clip_model.image_taps(image)
        return self.adapt_image(taps, feat)

    def encode_text(self, text: torch.Tensor) -> torch.Tensor:       # :153-177
        shape = text.shape
        if len(shape) == 3:
            text = text.reshape(-1, shape[-1])
            # the reference indexes the hooks' output with arange(batch_size) over batch_size*num_text rows (:165) and
            # fails to broadcast unless num_text == 1; rows are independent, so every row gets its own EOT here
        taps, feat = self.clip_model.text_taps(text)
        adapted = self.adapt_text(taps, feat)
        if len(shape) == 3:
            adapted = adapted.reshape(shape[0], shape[1], -1).mean(dim=1)
        return adapted

    def loss_from_features(self, adapted_images, adapted_text, r: torch.Tensor, action: torch.Tensor) -> torch.Tensor:
        """:217-250 for one image key. adapted_images = (a0, a1, a2[, a3]) unit-norm [B, D]; adapted_text [B, D] or None."""
        a0, a1, a2 = adapted_images[:3]
        if self.goal_conditioned:
            a3 = adapted_images[3]
            s0, s1, s2 = (-torch.linalg.norm(a3 - a, dim=-1) for a in (a0, a1, a2))
            other = a3
        else:
            scale = self.logit_scale.exp().to(a0.device)
            s0, s1, s2 = (scale * (a * adapted_text).sum(dim=-1) for a in (a0, a1, a2))   # diag(a @ t.T)
            other = adapted_text
        r = r - 1
        vip_loss = (1 - self.gamma) * -s0.mean() + torch.log(1e-8 + torch.mean(torch.exp(-(r + self.gamma * s2 - s1))))
        total = 0.0
        if self.use_vip_loss:
            total = total + vip_loss
        if self.use_id_loss:
            concat = torch.cat([a1, other, a2, other], dim=-1)
            total = total + self.lambda_id * self.loss_fn(self.inverse_layer(concat), action)
        return total

    def forward(self, batch: dict) -> torch.Tensor:                  # :179-252
        roles = ("image0", "image1", "image2") + (("image3",) if self.goal_conditioned else ())
        total = 0.0
        adapted_text = None
        for image_key in batch["image1"].keys():
            B = batch["image1"][image_key].shape[0]
            # image3 goes through preprocess in the reference too (:199-203) but is only encoded when goal-conditioned
            imgs = self.preprocess(torch.cat([batch[r][image_key] for r in roles], dim=0), train=True)
            adapted = torch.split(self.encode_image(imgs), B)          # ONE pass of the frozen tower for all roles
            if not self.goal_conditioned and adapted_text is None:
                adapted_text = self.encode_text(batch["instruct"])
            total = total + self.loss_from_features(adapted, adapted_text, batch["r"], batch["action"])
        if not torch.is_tensor(total):
            raise ValueError("neither use_vip_loss nor use_id_loss is set: the reference fails on `0.0.mean()` (:252)")
        return total.mean()

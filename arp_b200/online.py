"""Drop-in for the reference's ONLINE reward, `arp_dt/envs/vl_reward.py` (SURVEY.md §8(f)1): the per-step
CLIP reward a rollout uses to decrement the return-to-go token (envs/rollout_procgen.py:133-150).

Same function names and argument meaning as the reference:

    get_torch_clip_reward(clip_model, obs, pos_text, use_crop=False)                    vl_reward.py:11-23
    get_torch_clip_goal_conditioned_reward(clip_model, obs, goal_image, use_crop)       vl_reward.py:26-41
    get_torch_clip_adapter_reward(clip_model, obs, pos_text, use_crop)                  vl_reward.py:44-59
    get_torch_clip_adapter_goal_conditioned_reward(clip_model, obs, goal_image, ...)    vl_reward.py:62-77

where `clip_model` is an OnlineClip (it stands in for the reference's `(model, preprocess)` tuple built at
main_procgen.py:569-587). Each call is ONE CUDA-graph launch of the native pipeline at batch 1
(arp_online_reward, include/arp_b200.h): decode (Pillow-exact bicubic) -> ViT -> head, with the instruction
embedding cached instead of re-tokenised and re-encoded at every environment step.
`get_vip_reward` (vl_reward.py:80-97) scores with a VIP ResNet, not CLIP, and is out of scope.

No CPU fallback: constructing an OnlineClip without the native library and a B200 raises.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import capi
from .label_reward import _resolve_clip_weights, center_crop
from .text_tower import adapter_text_embedding, clip_text_embedding
from .tokenizer import resolve as resolve_tokenizer
from .weights import load_checkpoint


class OnlineClip:
    """CLIP (vl_type "clip", "clip_goal_conditioned") or the fine-tuned multiscale adapter ("clip_ft",
    "clip_ft_goal_conditioned") for single-frame scoring. Engines are created per frame size (a centre crop
    changes the resize tables) and text embeddings are cached per instruction."""

    def __init__(self, vl_type: str = "clip", *, vl_checkpoint=None, clip_state_dict=None, arch: str = "ViT-B/16",
                 device: int | None = None, max_batch: int = 2, precision: str = "16bit", tokenizer=None):
        self._precision = capi.precision_enum(precision)
        if vl_type not in ("clip", "clip_goal_conditioned", "clip_ft", "clip_ft_goal_conditioned"):
            raise ValueError(vl_type)                                         # rollout_procgen.py:145
        self.vl_type, self.arch = vl_type, arch
        self.adapter = vl_type.startswith("clip_ft")
        self.goal = vl_type.endswith("goal_conditioned")
        self.device_index = int(os.environ.get("LOCAL_RANK", "0")) if device is None else device
        self.max_batch = max_batch
        self._tokenize = resolve_tokenizer(tokenizer)   # refuses the stand-in unless opted in (tokenizer.py)
        if self.adapter:
            assert vl_checkpoint, "You have to specifiy vl_checkpoint."     # main_procgen.py:585
            sd = load_checkpoint(vl_checkpoint) if not isinstance(vl_checkpoint, dict) else vl_checkpoint
            if not any(k.startswith("clip_model.") for k in sd):
                base = _resolve_clip_weights(clip_state_dict, arch)
                sd = {**{"clip_model." + k: v for k, v in base.items()}, **sd}
        else:
            sd = _resolve_clip_weights(clip_state_dict, arch)
        self.sd = sd
        self._engines: dict[tuple[int, int], capi.Engine] = {}
        self._text_cache: dict[tuple, tuple] = {}
        self._engine_text: dict[tuple[int, int], tuple] = {}

    # -- plumbing -----------------------------------------------------------------------------------
    def _head(self) -> int:
        if self.adapter:
            return capi.HEAD_ADAPTER_GOAL if self.goal else capi.HEAD_ADAPTER
        return capi.HEAD_CLIP_GOAL if self.goal else capi.HEAD_CLIP

    def _engine(self, h: int, w: int) -> capi.Engine:
        e = self._engines.get((h, w))
        if e is None:
            # clip.load's preprocess for every vl_type (main_procgen.py:570,572): PIL bicubic, not the adapter's bilinear
            e = capi.Engine(device=self.device_index, patch=32 if self.arch.endswith("/32") else 16, in_h=h, in_w=w,
                            preprocess=capi.PRE_PIL_BICUBIC, head=self._head(), max_batch=self.max_batch,
                            precision=self._precision)
            missing = e.load_state_dict(self.sd, strict=False)
            if missing:
                raise RuntimeError(f"checkpoint lacks {len(missing)} tensors, e.g. {missing[:3]}")
            self._engines[(h, w)] = e
        return e

    def _with_text(self, e: capi.Engine, key_hw, pos_text):
        texts = tuple(pos_text) if isinstance(pos_text, (list, tuple)) else (pos_text,)
        if self._engine_text.get(key_hw) != texts:
            if texts not in self._text_cache:
                tokens = self._tokenize(list(texts))
                self._text_cache[texts] = (adapter_text_embedding(self.sd, tokens, e.device, ensemble=False)
                                           if self.adapter else clip_text_embedding(self.sd, tokens, e.device))
            emb, scale = self._text_cache[texts]
            e.set_text(emb, scale)
            self._engine_text[key_hw] = texts
        return e

    def logits(self, obs: np.ndarray, pos_text) -> np.ndarray:
        """[n_text] logits of one frame against the instruction(s)."""
        obs = np.asarray(obs)
        key = obs.shape[:2]
        e = self._with_text(self._engine(*key), key, pos_text)
        return e.online_reward(obs, want_logits=True)["logits"][0]

    def features(self, frames: np.ndarray) -> np.ndarray:
        """encode_image of [n,H,W,3] frames (CLIP: un-normalised; adapter: normalised), float32 [n, dim]."""
        frames = np.asarray(frames)
        e = self._engine(*frames.shape[1:3])
        if not self.goal and self._engine_text.get(frames.shape[1:3]) is None:
            raise RuntimeError("text heads need an instruction before features can be read")
        return e.online_reward(frames, want_features=True)["features"]

    def close(self):
        for e in self._engines.values():
            e.close()
        self._engines.clear()


def _crop_obs(obs: np.ndarray) -> np.ndarray:
    return center_crop(obs[None, ...], (obs.shape[0] // 2, obs.shape[0] // 2))[0]   # vl_reward.py:13-14


def _text_reward(clip_model: OnlineClip, obs, pos_text, use_crop):
    obs = np.asarray(obs)
    if use_crop:
        obs = _crop_obs(obs)
    lg = clip_model.logits(np.ascontiguousarray(obs), pos_text)
    # logits_per_text is [n_text, 1]: list -> mean over texts, str -> row 0 (vl_reward.py:19-23); float32 [1]
    r = lg.mean(axis=0, keepdims=True) if isinstance(pos_text, list) else lg[:1]
    return r.astype(np.float32)


def _goal_reward(clip_model: OnlineClip, obs, goal_image, use_crop):
    obs, goal_image = np.asarray(obs), np.asarray(goal_image)
    if use_crop:
        obs = _crop_obs(obs)
        # reference quirk kept: the goal is cropped with the ALREADY CROPPED obs' size (vl_reward.py:29-30)
        goal_image = center_crop(goal_image[None, ...], (obs.shape[0] // 2, obs.shape[0] // 2))[0]
    if obs.shape == goal_image.shape:
        f = clip_model.features(np.stack([obs, goal_image]))
        fo, fg = f[0], f[1]
    else:
        fo = clip_model.features(np.ascontiguousarray(obs)[None])[0]
        fg = clip_model.features(np.ascontiguousarray(goal_image)[None])[0]
    d = torch.from_numpy(fo) - torch.from_numpy(fg)
    return -1 * torch.norm(d).item()                                                 # float, like .item()


def get_torch_clip_reward(clip_model: OnlineClip, obs, pos_text, use_crop=False):
    return _text_reward(clip_model, obs, pos_text, use_crop)


def get_torch_clip_goal_conditioned_reward(clip_model: OnlineClip, obs, goal_image, use_crop=False):
    return _goal_reward(clip_model, obs, goal_image, use_crop)


def get_torch_clip_adapter_reward(clip_model: OnlineClip, obs, pos_text, use_crop=False):
    return _text_reward(clip_model, obs, pos_text, use_crop)


def get_torch_clip_adapter_goal_conditioned_reward(clip_model: OnlineClip, obs, goal_image, use_crop=False):
    return _goal_reward(clip_model, obs, goal_image, use_crop)


def update_rtg(rtg, clip_reward, scale, reward_min=0.0, use_normalize=False):
    """rollout_procgen.py:147-150 — `rtg[key] -= clip_reward / scale` (or the min-shifted form)."""
    if use_normalize:
        return rtg - (clip_reward - reward_min) / scale
    return rtg - clip_reward / scale

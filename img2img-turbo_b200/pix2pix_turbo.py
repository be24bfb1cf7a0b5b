"""Drop-in mirror of /root/reference/src/pix2pix_turbo.py (Pix2Pix_Turbo, TwinConv) over libi2it.

Same constructor kwargs, attributes and .forward() signature as the reference, so
src/inference_paired.py and the gradio apps call it unchanged (put this directory first on sys.path;
see INTEGRATION.md).  The four diffusers calls of the reference forward
(vae.encode / unet / sched.step / vae.decode, pix2pix_turbo.py:198-203 and :204-218) are ONE call into the
C ABI (i2it_forward); LoRA, TwinConv, gamma and the time embedding are folded at load (i2it_finalize_weights).
Does not import diffusers / peft / xformers.
"""
from __future__ import annotations

import copy
import os
import sys
import warnings
from types import SimpleNamespace
from typing import Optional

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import i2it  # noqa: E402
import weights as W  # noqa: E402
import _host  # noqa: E402
from _host import NetHandle, TurboBase, load_sd_turbo_base  # noqa: E402
from model import download_url  # noqa: E402

CKPT_URLS = {
    "edge_to_image": "https://www.cs.cmu.edu/~img2img-turbo/models/edge_to_image_loras.pkl",
    "sketch_to_image_stochastic": "https://www.cs.cmu.edu/~img2img-turbo/models/sketch_to_image_stochastic_lora.pkl",
}


class TwinConv(torch.nn.Module):
    """x -> conv_pre(x)*(1-r) + conv_cur(x)*r   (reference pix2pix_turbo.py:16-26).

    In this implementation the blend is folded into ONE conv weight at load, W = (1-r) W_pre + r W_cur
    (i2it_finalize_weights); this module only carries the two parameter sets and `r`, and its forward is the
    literal reference formula for host-side checks."""

    def __init__(self, convin_pretrained, convin_curr):
        super().__init__()
        self.conv_in_pretrained = copy.deepcopy(convin_pretrained)
        self.conv_in_curr = copy.deepcopy(convin_curr)
        self.r = None

    def forward(self, x):
        x1 = self.conv_in_pretrained(x).detach()
        x2 = self.conv_in_curr(x)
        return x1 * (1 - self.r) + x2 * (self.r)


class Pix2Pix_Turbo(TurboBase):
    MODEL_KIND = i2it.PIX2PIX

    def __init__(self, pretrained_name=None, pretrained_path=None, ckpt_folder="checkpoints", lora_rank_unet=8,
                 lora_rank_vae=4, *, cfg=None, seed=0, lora_b_std=0.02, perturb_norm=False, text_stack=None,
                 use_cuda_graph=True, keep_stages=False, twin=False):
        super().__init__()
        self._init_common(cfg, None, text_stack, use_cuda_graph, keep_stages)
        # twin=True: random-init model WITH a TwinConv conv_in (two distinct weight sets) — the synthetic stand-in for the
        # sketch_to_image_stochastic checkpoint (BASELINE config #4)
        twin = bool(twin) or pretrained_name == "sketch_to_image_stochastic"
        ckpt = None
        if pretrained_name in CKPT_URLS:
            os.makedirs(ckpt_folder, exist_ok=True)
            outf = os.path.join(ckpt_folder, os.path.basename(CKPT_URLS[pretrained_name]))
            download_url(CKPT_URLS[pretrained_name], outf)
            ckpt = torch.load(outf, map_location="cpu")
        elif pretrained_path:
            ckpt = torch.load(pretrained_path, map_location="cpu")
        elif pretrained_name:
            raise ValueError(f"unknown pretrained_name {pretrained_name!r}")
        else:
            print("Initializing model with random weights")            # reference pix2pix_turbo.py:132
        if ckpt is not None:
            lora_rank_unet, lora_rank_vae = ckpt["rank_unet"], ckpt["rank_vae"]
            twin = twin or any("conv_in_pretrained" in k for k in ckpt["state_dict_unet"])
        # base weights: seeded random init in the diffusers layout (offline), overlaid by a local SD-Turbo snapshot if any
        self._sd = W.make_state_dict("pix2pix", self._cfg, seed=seed, twin=twin, lora_rank_unet=lora_rank_unet,
                                     lora_rank_vae=lora_rank_vae, lora_b_std=lora_b_std, perturb_norm=perturb_norm)
        have_base = load_sd_turbo_base(self._sd, ["unet", "vae"]) if self._cfg is W.SD_TURBO else False
        if ckpt is not None:
            if not have_base:
                warnings.warn("SD-Turbo base weights are not available offline: checkpoint LoRA/skip tensors are applied on "
                              "top of a seeded random base (set $I2IT_SD_TURBO_DIR to a local snapshot for real outputs)")
            self._apply_checkpoint(ckpt)
        self.lora_rank_unet, self.lora_rank_vae = lora_rank_unet, lora_rank_vae
        self.target_modules_vae = (ckpt or {}).get("vae_lora_target_modules", list(W.TARGETS_VAE))
        self.target_modules_unet = (ckpt or {}).get("unet_lora_target_modules", list(W.TARGETS_UNET))
        # peft LoraConfig default lora_alpha = 8 (reference passes only r) -> scale 8/r
        self._adapter_scales = {"default": 8.0 / lora_rank_unet, "vae_skip": 8.0 / lora_rank_vae}
        self.unet, self.vae = NetHandle(self, "unet."), NetHandle(self, "vae.")
        self.unet.conv_in = SimpleNamespace(r=None) if twin else SimpleNamespace()
        self.vae.decoder = SimpleNamespace(gamma=1, ignore_skip=False)
        self.vae.config = SimpleNamespace(scaling_factor=self._cfg["scaling_factor"])
        self._twin = twin
        self._lora_w_unet = 1.0      # runtime adapter weights; the reference never resets them after a stochastic call
        self._lora_w_vae = 1.0

    # ---- checkpoint format of save_model (reference pix2pix_turbo.py:221-229, read at :66-78) ----
    def _apply_checkpoint(self, ckpt):
        """The reference creates adapters ONLY for the checkpoint's target modules (LoraConfig(target_modules=sd[...]),
        pix2pix_turbo.py:66-78) and then overlays the checkpoint tensors.  So: drop every adapter of the seeded base, overlay,
        and check that each layer the checkpoint's target lists name got its LoRA pair."""
        for k in [k for k in self._sd if ".lora_A." in k or ".lora_B." in k]:
            del self._sd[k]
        for part, prefix in (("state_dict_unet", "unet."), ("state_dict_vae", "vae.")):
            for k, v in ckpt[part].items():
                self._sd[prefix + k.replace(".base_layer.", ".")] = v.detach().float().cpu()
        for prefix, targets, adapter in (("unet.", ckpt.get("unet_lora_target_modules"), "default"),
                                         ("vae.", ckpt.get("vae_lora_target_modules"), "vae_skip")):
            if not targets:
                continue
            layers = {k[:-len(".weight")] for k in self._sd if k.startswith(prefix) and k.endswith(".weight") and ".lora_" not in k
                      and self._sd[k].dim() in (2, 4)}
            missing = [l for l in sorted(layers) if W._suffix_match(l[len(prefix):], list(targets))
                       and f"{l}.lora_A.{adapter}.weight" not in self._sd]
            if missing:
                warnings.warn(f"checkpoint lists {len(missing)} {prefix[:-1]} LoRA target layers without LoRA tensors (e.g. "
                              f"{missing[0]}): they run without an adapter (the reference would initialise lora_B = 0, a no-op)")

    @staticmethod
    def _peft_keys(sd):
        """State dict in peft's spelling: the base weight/bias of every LoRA-wrapped layer is `X.base_layer.weight`
        (what the reference's strict load_state_dict expects, pix2pix_turbo.py:66-78,111-125)."""
        wrapped = {k.split(".lora_A.")[0] for k in sd if ".lora_A." in k}
        out = {}
        for k, v in sd.items():
            stem, _, leaf = k.rpartition(".")
            out[f"{stem}.base_layer.{leaf}" if (stem in wrapped and leaf in ("weight", "bias")) else k] = v
        return out

    def save_model(self, outf):
        sd = {"unet_lora_target_modules": self.target_modules_unet, "vae_lora_target_modules": self.target_modules_vae,
              "rank_unet": self.lora_rank_unet, "rank_vae": self.lora_rank_vae,
              "state_dict_unet": {k: v for k, v in self._peft_keys(self.unet.state_dict()).items() if "lora" in k or "conv_in" in k},
              "state_dict_vae": {k: v for k, v in self._peft_keys(self.vae.state_dict()).items() if "lora" in k or "skip" in k}}
        torch.save(sd, outf)

    def set_eval(self):
        self.unet.eval()
        self.vae.eval()

    def set_train(self):
        raise NotImplementedError("training/backward is outside this build's scope (inference hot path only)")

    def _set_adapter_weights(self, prefix, names, weights):
        w = 1.0 if weights is None else float(weights[0] if isinstance(weights, (list, tuple)) else weights)
        if prefix == "unet.":
            self._lora_w_unet = w
        else:
            self._lora_w_vae = w

    @classmethod
    def from_pretrained(cls, pretrained_name=None, **kw):
        """Convenience alias (the reference has only the constructor)."""
        return cls(pretrained_name=pretrained_name, **kw)

    def forward(self, c_t, prompt=None, prompt_tokens=None, deterministic=True, r=1.0, noise_map=None, *, eps=None):
        # either the prompt or the prompt_tokens should be provided  (reference :188)
        assert (prompt is None) != (prompt_tokens is None), "Either prompt or prompt_tokens should be provided"
        dt = self.compute_dtype
        in_dtype = c_t.dtype
        caption_enc = self._encode_text(prompt, prompt_tokens)
        B, _, H, Wd = c_t.shape
        x = self._prep(c_t, dt)
        if eps is None:
            # latent_dist.sample(): randn from the global RNG on the device, in the activation dtype (SURVEY fact 5)
            eps = torch.randn((B, 4, H // 8, Wd // 8), device=_host.DEVICE, dtype=dt)
            torch.randn((B, 4, H // 8, Wd // 8), device=_host.DEVICE, dtype=dt)   # DDPM variance noise: drawn, x1e-10, discarded
        eps = self._prep(eps, dt)
        if caption_enc.shape[0] not in (1, B):
            raise ValueError("prompt batch must be 1 or match the image batch")
        if deterministic:
            if self._twin:
                raise TypeError("deterministic forward on a TwinConv model: conv_in.r is None (as in the reference)")
            eng = self._finalize(self._lora_w_unet, self._lora_w_vae, float(self.vae.decoder.gamma), -1.0)
            out = self._staged_forward(eng, x, caption_enc, eps)
        else:
            if noise_map is None:
                raise ValueError("noise_map is required when deterministic=False")
            # unet.set_adapters(["default"],[r]); set_weights_and_activate_adapters(vae,["vae_skip"],[r]);
            # conv_in.r = r; decoder.gamma = r   (reference :206-217)
            self._lora_w_unet = self._lora_w_vae = float(r)
            self.vae.decoder.gamma = r
            eng = self._finalize(r, r, r, r if self._twin else -1.0)
            nm = self._prep(noise_map.expand(B, -1, -1, -1) if noise_map.shape[0] != B else noise_map, dt)
            out = self._staged_forward(eng, x, caption_enc, eps, noise=nm, r=float(r))
            if self._twin:
                self.unet.conv_in.r = None
        return out if in_dtype == dt else out.to(in_dtype)

    def forward_u8(self, images_u8, prompt=None, prompt_tokens=None, deterministic=True, r=1.0, noise_map=None, *, eps=None,
                   sketch=False):
        """uint8 HWC boundary (SURVEY 8f #3): `images_u8` [B,H,W,3] uint8 (host or device) -> [B,H,W,3] uint8 CUDA tensor.
        Fuses F.to_tensor (edge/canny images, inference_paired.py:50) or the sketch threshold (:56-57) on the way in and
        ToPILImage()(out*0.5+0.5) (:72) on the way out; everything between is the same i2it_forward."""
        assert (prompt is None) != (prompt_tokens is None), "Either prompt or prompt_tokens should be provided"
        dt = self.compute_dtype
        caption_enc = self._encode_text(prompt, prompt_tokens)
        x = images_u8.to(device=_host.DEVICE, non_blocking=True).contiguous()
        B, H, Wd, _ = x.shape
        if eps is None:
            eps = torch.randn((B, 4, H // 8, Wd // 8), device=_host.DEVICE, dtype=dt)
            torch.randn((B, 4, H // 8, Wd // 8), device=_host.DEVICE, dtype=dt)
        eps = self._prep(eps, dt)
        mode = i2it.IN_SKETCH if sketch else i2it.IN_UNIT
        if deterministic:
            if self._twin:
                raise TypeError("deterministic forward on a TwinConv model: conv_in.r is None (as in the reference)")
            eng = self._finalize(self._lora_w_unet, self._lora_w_vae, float(self.vae.decoder.gamma), -1.0)
            return self._staged_forward(eng, x, caption_enc, eps, u8_mode=mode)
        if noise_map is None:
            raise ValueError("noise_map is required when deterministic=False")
        self._lora_w_unet = self._lora_w_vae = float(r)
        self.vae.decoder.gamma = r
        eng = self._finalize(r, r, r, r if self._twin else -1.0)
        nm = self._prep(noise_map.expand(B, -1, -1, -1) if noise_map.shape[0] != B else noise_map, dt)
        out = self._staged_forward(eng, x, caption_enc, eps, noise=nm, r=float(r), u8_mode=mode)
        if self._twin:
            self.unet.conv_in.r = None
        return out

    def canny_u8(self, images_u8, low_threshold=100, high_threshold=200):
        """Edge maps of photos on the device, bit for bit what the reference CLI feeds the model
        (canny_from_pil, src/image_prep.py:6-12; default thresholds of src/inference_paired.py:18-19):
        `images_u8` [B,H,W,3] (or [H,W,3]) uint8 RGB, host or device -> [B,H,W,3] uint8 CUDA tensor in {0, 255}.
        Photo to image: `forward_u8(canny_u8(photo), prompt)`; the inverted map the CLI saves is `255 - edges`."""
        x = torch.as_tensor(images_u8)
        if x.dim() == 3:
            x = x.unsqueeze(0)
        x = x.to(device=_host.DEVICE, non_blocking=True).contiguous()
        return self._get_engine().canny_u8(x, low_threshold, high_threshold)

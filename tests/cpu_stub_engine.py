"""TEST DOUBLE of i2it.Engine that computes on the CPU — test infrastructure, never imported by the product.

Purpose: run the reference's inference CLIs (src/inference_paired.py, inference_unpaired.py: live when recording, replayed from
tests/golden/ in the suite) on any host against the repo's drop-in modules (pix2pix_turbo / cyclegan_turbo / model), to prove
the import contract and the call sequence of SURVEY.md section 8b end to end: constructor kwargs, .set_eval()/.eval()/.half(),
.unet.enable_xformers_memory_efficient_attention(), forward signatures, dtype/shape of what comes back.

The stub implements the i2it.Engine methods the wrappers call and computes with the CPU ORACLE (tests may import oracle/), so the
images the CLIs write are the oracle's.  `install()` swaps it in and makes `.cuda()` a no-op; both are process-local monkeypatches
done by tests/run_reference_cli.py only."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "oracle"), os.path.join(ROOT, "img2img-turbo_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

CALLS = []          # (method, summary) log the tests inspect


class StubEngine:
    def __init__(self, dtype=torch.bfloat16, model_kind=0, cfg=None, device=None, keep_stages=False, use_cuda_graph=True, **kw):
        import weights as W
        self.dtype, self.kind, self.cfg = dtype, model_kind, cfg or W.SD_TURBO
        self.cross_dim = self.cfg["cross_dim"]
        self.sd, self.scales, self.final, self.text = {}, {}, None, None
        CALLS.append(("create", str(dtype)))

    def load_state_dict(self, sd):
        self.sd.update({k: v.detach().float().cpu() for k, v in sd.items() if not k.startswith("text_encoder.")})

    def set_adapter_scale(self, name, s):
        self.scales[name] = s

    def finalize(self, lw_unet=1.0, lw_vae=1.0, gamma=1.0, twin_r=-1.0):
        self.final = (lw_unet, lw_vae, gamma, twin_r)
        self.text = None
        CALLS.append(("finalize", self.final))

    def set_text(self, text):
        self.text = text.detach().float().cpu()
        CALLS.append(("set_text", tuple(text.shape)))

    def close(self):
        pass

    def _run(self, x, text, eps, noise, r, direction):
        import oracle as O
        text = self.text if text is None else text.float().cpu()
        lw_unet, lw_vae, gamma, twin_r = self.final
        with torch.no_grad():
            if self.kind == 1:
                return O.cyclegan_forward(self.sd, x, text, eps, "a2b" if direction == 0 else "b2a", self.cfg)
            if noise is not None:
                return O.pix2pix_forward(self.sd, x, text, eps, self.cfg, deterministic=False, r=r, noise_map=noise)
            return O.pix2pix_forward(self.sd, x, text, eps, self.cfg, lora_weight=lw_unet, decoder_gamma=gamma)

    def forward(self, x, text_emb, eps, noise_map=None, r=1.0, direction=0, out=None, out_latent=None):
        CALLS.append(("forward", tuple(x.shape), str(x.dtype), noise_map is not None, r, direction))
        y = self._run(x.float().cpu(), text_emb, eps.float().cpu(), None if noise_map is None else noise_map.float().cpu(), r,
                      direction).to(self.dtype)
        if out is not None:
            out.copy_(y)
            return out
        return y


def install():
    import _host
    import i2it
    i2it.Engine = StubEngine
    _host.DEVICE = "cpu"
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self

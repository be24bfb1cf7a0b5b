"""ctypes binding of libi2it.so (the C ABI declared in include/i2it.h).

PyTorch is plumbing here: it owns device memory and streams; every FLOP of the image path runs inside
libi2it's sm_100a kernels.  There is NO fallback: if the library is missing or the device is not a
B200, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libi2it.so")

F16, BF16, F32 = 0, 1, 2
PIX2PIX, CYCLEGAN = 0, 1
A2B, B2A = 0, 1
ACT_NONE, ACT_CLAMP1, ACT_GEGLU = 0, 1, 2
IN_UNIT, IN_NORMALIZE, IN_SKETCH = 0, 1, 2      # uint8 input transforms of i2it_forward_u8

_TORCH2DT = {torch.float16: F16, torch.bfloat16: BF16, torch.float32: F32}
_DT2TORCH = {F16: torch.float16, BF16: torch.bfloat16}

# every symbol include/i2it.h declares (tests check the library exports all of them)
SYMBOLS = [
    "i2it_default_config", "i2it_create", "i2it_destroy", "i2it_last_error", "i2it_set_weight",
    "i2it_set_adapter_scale", "i2it_finalize_weights", "i2it_workspace_bytes", "i2it_forward",
    "i2it_set_text", "i2it_encode_text", "i2it_forward_u8", "i2it_prep_launch_count", "i2it_debug_fast_div", "i2it_launch_count", "i2it_profile", "i2it_read_stage", "i2it_op_conv2d", "i2it_op_group_norm", "i2it_op_layer_norm",
    "i2it_op_attention", "i2it_op_upsample2x", "i2it_canny_u8",
]


class Config(C.Structure):
    _fields_ = [
        ("dtype", C.c_int), ("model_kind", C.c_int), ("device", C.c_int),
        ("unet_channels", C.c_int * 4), ("unet_heads", C.c_int * 4),
        ("cross_dim", C.c_int), ("temb_dim", C.c_int), ("vae_channels", C.c_int * 4),
        ("scaling_factor", C.c_float), ("keep_stages", C.c_int), ("use_cuda_graph", C.c_int),
        ("text_heads", C.c_int), ("text_act", C.c_int),
    ]


_lib = None


def load_library(path: Optional[str] = None):
    """dlopen libi2it.so and declare prototypes.  Fails loudly when the extension is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or os.environ.get("I2IT_LIB", LIB_PATH)
    if not os.path.exists(path):
        raise RuntimeError(
            f"libi2it.so not found at {path}: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C img2img-turbo_b200/csrc`).  There is no CPU/PyTorch fallback for the image path.")
    lib = C.CDLL(path)
    vp, ci, cf = C.c_void_p, C.c_int, C.c_float
    lib.i2it_default_config.argtypes = [C.POINTER(Config)]
    lib.i2it_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    lib.i2it_destroy.argtypes = [vp]
    lib.i2it_destroy.restype = None
    lib.i2it_last_error.argtypes = [vp]
    lib.i2it_last_error.restype = C.c_char_p
    lib.i2it_set_weight.argtypes = [vp, C.c_char_p, vp, C.POINTER(C.c_int64), ci, ci, ci]
    lib.i2it_set_adapter_scale.argtypes = [vp, C.c_char_p, cf]
    lib.i2it_finalize_weights.argtypes = [vp, cf, cf, cf, cf]
    lib.i2it_workspace_bytes.argtypes = [vp, ci, ci, ci, C.POINTER(C.c_size_t)]
    lib.i2it_forward.argtypes = [vp, vp, vp, ci, vp, vp, cf, vp, vp, ci, ci, ci, ci, vp]
    lib.i2it_set_text.argtypes = [vp, vp, ci, vp]
    lib.i2it_encode_text.argtypes = [vp, vp, ci, vp, vp]
    lib.i2it_forward_u8.argtypes = [vp, vp, ci, vp, ci, vp, vp, cf, vp, vp, ci, ci, ci, ci, vp]
    lib.i2it_canny_u8.argtypes = [vp, vp, ci, ci, ci, cf, cf, vp, vp]
    lib.i2it_prep_launch_count.argtypes = [vp, C.POINTER(ci)]
    lib.i2it_debug_fast_div.argtypes = [C.c_longlong, ci, ci]
    lib.i2it_debug_fast_div.restype = C.c_longlong
    lib.i2it_launch_count.argtypes = [vp, ci, ci, ci, ci, C.POINTER(ci)]
    lib.i2it_profile.argtypes = [vp, ci, C.c_char_p, C.c_size_t, vp]
    lib.i2it_read_stage.argtypes = [vp, C.c_char_p, vp, C.c_size_t, C.POINTER(ci)]
    lib.i2it_op_conv2d.argtypes = [vp, vp, ci, ci, ci, ci, ci, vp, vp, ci, ci, ci, ci, vp, ci, ci, vp, ci, ci, vp]
    lib.i2it_op_group_norm.argtypes = [vp, vp, ci, ci, ci, ci, vp, vp, cf, ci, vp, ci, vp]
    lib.i2it_op_layer_norm.argtypes = [vp, vp, ci, ci, ci, vp, vp, cf, vp, ci, vp]
    lib.i2it_op_attention.argtypes = [vp, vp, ci, vp, ci, vp, ci, ci, ci, ci, ci, ci, ci, vp, ci, vp]
    lib.i2it_op_upsample2x.argtypes = [vp, vp, ci, ci, ci, ci, vp, vp]
    for name in SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("i2it_destroy", "i2it_last_error"):
            fn.restype = ci
    _lib = lib
    return lib


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Engine:
    """One engine per (device, stream).  Thin, typed wrapper over the C handle."""

    def __init__(self, dtype: torch.dtype = torch.bfloat16, model_kind: int = PIX2PIX, cfg: Optional[dict] = None,
                 device: Optional[int] = None, keep_stages: bool = False, use_cuda_graph: bool = True,
                 text_heads: int = 0, text_act: str = "gelu"):
        if not torch.cuda.is_available():
            raise RuntimeError("libi2it needs a CUDA device (B200 / sm_100a); no CPU fallback exists")
        self.lib = load_library()
        self.dtype = dtype
        c = Config()
        self.lib.i2it_default_config(C.byref(c))
        c.dtype = _TORCH2DT[dtype]
        c.model_kind = model_kind
        c.device = torch.cuda.current_device() if device is None else device
        c.keep_stages = int(keep_stages)
        c.use_cuda_graph = int(use_cuda_graph)
        c.text_heads = int(text_heads)                       # 0: hidden / 64
        c.text_act = 1 if text_act == "quick_gelu" else 0
        if cfg is not None:
            for i in range(4):
                c.unet_channels[i] = cfg["unet_channels"][i]
                c.unet_heads[i] = cfg["unet_heads"][i]
                c.vae_channels[i] = cfg["vae_channels"][i]
            c.cross_dim = cfg["cross_dim"]
            c.temb_dim = cfg["temb_dim"]
            c.scaling_factor = cfg["scaling_factor"]
        self.cross_dim = c.cross_dim
        self.device = c.device
        self._h = C.c_void_p(0)
        rc = self.lib.i2it_create(C.byref(c), C.byref(self._h))
        if rc != 0:
            raise RuntimeError("i2it_create failed: " + self.lib.i2it_last_error(C.c_void_p(0)).decode())

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise RuntimeError(f"{what} failed: " + self.lib.i2it_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.i2it_destroy(self._h)
            self._h = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights -------------------------------------------------------------------------------
    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        for k, v in sd.items():
            t = v.detach()
            if t.dtype not in _TORCH2DT:
                t = t.float()
            t = t.contiguous()
            shape = (C.c_int64 * t.dim())(*t.shape)
            self._check(self.lib.i2it_set_weight(self._h, k.encode(), _ptr(t), shape, t.dim(), _TORCH2DT[t.dtype],
                                                 int(t.is_cuda)), f"i2it_set_weight({k})")

    def set_adapter_scale(self, adapter: str, alpha_over_r: float):
        self._check(self.lib.i2it_set_adapter_scale(self._h, adapter.encode(), alpha_over_r), "i2it_set_adapter_scale")

    def finalize(self, lora_weight_unet: float = 1.0, lora_weight_vae: float = 1.0, skip_gamma: float = 1.0,
                 twin_r: float = -1.0):
        self._text_batch = None          # cached text projections die with the folded weights
        self._check(self.lib.i2it_finalize_weights(self._h, lora_weight_unet, lora_weight_vae, skip_gamma, twin_r),
                    "i2it_finalize_weights")

    # ---- the hot path ----------------------------------------------------------------------------
    def set_text(self, text_emb: torch.Tensor):
        """Cache the cross-attention K / V^T of a prompt embedding [1|B,77,cross]; later forwards pass text_emb=None."""
        if not (text_emb.is_cuda and text_emb.is_contiguous() and text_emb.dtype == self.dtype):
            raise ValueError("libi2it operands must be contiguous CUDA tensors in the engine dtype")
        if text_emb.dim() != 3 or text_emb.shape[1:] != (77, self.cross_dim):
            raise ValueError(f"text_emb must be [1|B,77,{self.cross_dim}]")
        self._check(self.lib.i2it_set_text(self._h, _ptr(text_emb), text_emb.shape[0], _stream()), "i2it_set_text")
        self._text_batch = text_emb.shape[0]

    def encode_text(self, tokens: torch.Tensor, hidden: int) -> torch.Tensor:
        """CLIP text tower on the engine: tokens [B,77] (any integer dtype) -> last_hidden_state [B,77,hidden] in the engine dtype.
        Needs the `text_encoder.*` tensors in the loaded state dict."""
        ids = tokens.to(device="cuda", dtype=torch.int32).contiguous()
        out = torch.empty(ids.shape[0], ids.shape[1], hidden, device="cuda", dtype=self.dtype)
        self._check(self.lib.i2it_encode_text(self._h, _ptr(ids), ids.shape[0], _ptr(out), _stream()), "i2it_encode_text")
        return out

    def _check_operands(self, B, H, W, text_emb, eps, others):
        for t in (text_emb, eps) + tuple(others):
            if t is not None:
                if not (t.is_cuda and t.is_contiguous() and t.dtype == self.dtype):
                    raise ValueError("libi2it operands must be contiguous CUDA tensors in the engine dtype")
        if text_emb is not None:
            if text_emb.shape[1:] != (77, self.cross_dim) or text_emb.shape[0] not in (1, B):
                raise ValueError(f"text_emb must be [1|B,77,{self.cross_dim}]")
            tb = text_emb.shape[0]
        else:
            tb = getattr(self, "_text_batch", None)
            if tb is None:
                raise ValueError("text_emb=None needs a previous set_text()")
        if eps.shape != (B, 4, H // 8, W // 8):
            raise ValueError("eps must be [B,4,H/8,W/8]")
        return tb

    def forward(self, x: torch.Tensor, text_emb: Optional[torch.Tensor], eps: torch.Tensor,
                noise_map: Optional[torch.Tensor] = None, r: float = 1.0, direction: int = A2B,
                out: Optional[torch.Tensor] = None, out_latent: Optional[torch.Tensor] = None) -> torch.Tensor:
        B, Cc, H, W = x.shape
        assert Cc == 3, "image must be [B,3,H,W]"
        tb = self._check_operands(B, H, W, text_emb, eps, (x, noise_map, out, out_latent))
        if out is None:
            out = torch.empty_like(x)
        self._check(self.lib.i2it_forward(self._h, _ptr(x), _ptr(text_emb), tb, _ptr(eps), _ptr(noise_map),
                                          float(r), _ptr(out), _ptr(out_latent), B, H, W, direction, _stream()),
                    "i2it_forward")
        return out

    def forward_u8(self, x_u8: torch.Tensor, in_mode: int, text_emb: Optional[torch.Tensor], eps: torch.Tensor,
                   noise_map: Optional[torch.Tensor] = None, r: float = 1.0, direction: int = A2B,
                   out: Optional[torch.Tensor] = None, out_latent: Optional[torch.Tensor] = None) -> torch.Tensor:
        """uint8 HWC boundary: x_u8 [B,H,W,3] uint8 CUDA -> [B,H,W,3] uint8 CUDA (pre/post-processing fused on device)."""
        B, H, W, Cc = x_u8.shape
        assert Cc == 3 and x_u8.dtype == torch.uint8 and x_u8.is_cuda and x_u8.is_contiguous(), "image must be uint8 CUDA [B,H,W,3]"
        tb = self._check_operands(B, H, W, text_emb, eps, (noise_map, out_latent))
        if out is None:
            out = torch.empty_like(x_u8)
        assert out.dtype == torch.uint8 and out.is_cuda and out.is_contiguous() and out.shape == x_u8.shape
        self._check(self.lib.i2it_forward_u8(self._h, _ptr(x_u8), int(in_mode), _ptr(text_emb), tb, _ptr(eps), _ptr(noise_map),
                                             float(r), _ptr(out), _ptr(out_latent), B, H, W, direction, _stream()),
                    "i2it_forward_u8")
        return out

    def canny_u8(self, x_u8: torch.Tensor, low: float, high: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """cv2.Canny(img, low, high) of every image, bit for bit, replicated to three channels: x_u8 [B,H,W,3] uint8 CUDA (RGB)
        -> [B,H,W,3] uint8 CUDA in {0, 255}, ready for forward_u8(..., IN_UNIT, ...)."""
        if not (x_u8.dtype == torch.uint8 and x_u8.is_cuda and x_u8.is_contiguous() and x_u8.dim() == 4 and x_u8.shape[3] == 3):
            raise ValueError("canny_u8: image must be a contiguous uint8 CUDA tensor [B,H,W,3]")
        if out is None:
            out = torch.empty_like(x_u8)
        if not (out.dtype == torch.uint8 and out.is_cuda and out.is_contiguous() and out.shape == x_u8.shape):
            raise ValueError("canny_u8: out must be a contiguous uint8 CUDA tensor shaped like the image")
        B, H, W, _ = x_u8.shape
        self._check(self.lib.i2it_canny_u8(self._h, _ptr(x_u8), B, H, W, float(low), float(high), _ptr(out), _stream()),
                    "i2it_canny_u8")
        return out

    def prep_launch_count(self) -> int:
        n = C.c_int(0)
        self._check(self.lib.i2it_prep_launch_count(self._h, C.byref(n)), "i2it_prep_launch_count")
        return n.value

    def launch_count(self, B: int, H: int, W: int, direction: int = A2B) -> int:
        n = C.c_int(0)
        self._check(self.lib.i2it_launch_count(self._h, B, H, W, direction, C.byref(n)), "i2it_launch_count")
        return n.value

    def profile(self, reps: int = 3):
        """Per-launch timings of the last forward's plan: list of dicts (kind, ms, flops, bytes, shape)."""
        import json
        cap = 1 << 22
        buf = C.create_string_buffer(cap)
        self._check(self.lib.i2it_profile(self._h, reps, buf, cap, _stream()), "i2it_profile")
        return json.loads(buf.value.decode())

    def workspace_bytes(self, B: int, H: int, W: int) -> int:
        n = C.c_size_t(0)
        self._check(self.lib.i2it_workspace_bytes(self._h, B, H, W, C.byref(n)), "i2it_workspace_bytes")
        return n.value

    def read_stage(self, name: str, max_elems: int = 1 << 26, image: Optional[int] = None) -> torch.Tensor:
        """fp32 NCHW copy of a named stage of the last forward (keep_stages engines); image=i reads one image of the batch."""
        if image is not None:
            name = f"{name}@{int(image)}"
        dims = (C.c_int * 4)()
        buf = torch.empty(max_elems, dtype=torch.float32, device="cuda")
        self._check(self.lib.i2it_read_stage(self._h, name.encode(), _ptr(buf), max_elems, dims), f"i2it_read_stage({name})")
        n, c, h, w = list(dims)
        return buf[: n * c * h * w].view(n, c, h, w).clone()

    # ---- diagnostic single ops (NHWC tensors in the engine dtype; weights fp32 CUDA) -----------------
    def op_conv2d(self, x_nhwc, w, bias=None, stride=1, asym_pad=False, residual=None, act=ACT_NONE, out_fp32=False):
        N, H, W, Cin = x_nhwc.shape
        Cout, _, k, _ = w.shape
        oc = Cout // 2 if act == ACT_GEGLU else Cout
        out = torch.empty(N, H // stride, W // stride, oc, device="cuda", dtype=torch.float32 if out_fp32 else self.dtype)
        w = w.float().contiguous()
        b = bias.float().contiguous() if bias is not None else None
        self._check(self.lib.i2it_op_conv2d(self._h, _ptr(x_nhwc), N, H, W, Cin, x_nhwc.stride(2), _ptr(w), _ptr(b), Cout, k,
                                            stride, int(asym_pad), _ptr(residual),
                                            residual.stride(2) if residual is not None else 0, act, _ptr(out), oc,
                                            int(out_fp32), _stream()), "i2it_op_conv2d")
        return out

    def op_group_norm(self, x_nhwc, gamma, beta, eps, silu):
        N, H, W, Cc = x_nhwc.shape
        out = torch.empty_like(x_nhwc)
        self._check(self.lib.i2it_op_group_norm(self._h, _ptr(x_nhwc), N, H * W, Cc, x_nhwc.stride(2), _ptr(gamma.float()),
                                                _ptr(beta.float()), eps, int(silu), _ptr(out), Cc, _stream()),
                    "i2it_op_group_norm")
        return out

    def op_layer_norm(self, x, gamma, beta, eps=1e-5):
        rows, Cc = x.shape
        out = torch.empty_like(x)
        self._check(self.lib.i2it_op_layer_norm(self._h, _ptr(x), rows, Cc, x.stride(0), _ptr(gamma.float()), _ptr(beta.float()),
                                                eps, _ptr(out), Cc, _stream()), "i2it_op_layer_norm")
        return out

    def op_attention(self, q, k, vt, heads):
        B, Nq, Cc = q.shape
        kvb, Nk, _ = k.shape
        out = torch.empty_like(q)
        self._check(self.lib.i2it_op_attention(self._h, _ptr(q), q.stride(1), _ptr(k), k.stride(1), _ptr(vt), vt.stride(1), B, Nq,
                                               Nk, heads, Cc // heads, kvb, _ptr(out), Cc, _stream()), "i2it_op_attention")
        return out

    def op_upsample2x(self, x_nhwc):
        N, H, W, Cc = x_nhwc.shape
        out = torch.empty(N, 2 * H, 2 * W, Cc, device="cuda", dtype=self.dtype)
        self._check(self.lib.i2it_op_upsample2x(self._h, _ptr(x_nhwc), N, H, W, Cc, _ptr(out), _stream()), "i2it_op_upsample2x")
        return out

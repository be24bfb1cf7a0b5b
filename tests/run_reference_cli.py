"""The reference's inference CLIs (src/inference_paired.py, src/inference_unpaired.py) driving the drop-in modules: recorded
once from the unmodified scripts, replayed by tests/test_reference_cli.py without the reference tree.

    python tests/run_reference_cli.py record <reference checkout>/src     # rewrites tests/golden/reference_cli_*.pt
    python tests/run_reference_cli.py replay <case> <out.pt>

record: builds the seeded checkpoint of each case, then runs the UNMODIFIED script (runpy, its own argv) with img2img-turbo_b200/
first on sys.path, so its `from pix2pix_turbo import Pix2Pix_Turbo` resolves to this repo, and the reference's src/ after it
(image_prep / my_utils stay the reference's).  The model class the script imports is wrapped in a recorder that saves the
constructor arguments, every call the script makes on the model (arguments, the global RNG state before the call: the forward
draws its posterior noise from it, and the tensor it returns) and the calls the engine received.
replay: constructs the model from the recorded arguments, makes the same calls in the same RNG state and saves what comes back.

Both modes run the CPU test double of the engine (tests/cpu_stub_engine.py, which computes with the CPU oracle) on every host,
so a replay reproduces the recording up to float summation order."""
import importlib
import json
import os
import runpy
import sys
import tempfile
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "img2img-turbo_b200"), os.path.join(ROOT, "tests")]
GOLD = os.path.join(ROOT, "tests", "golden")

import torch  # noqa: E402

import cpu_stub_engine  # noqa: E402
from _host import NetHandle  # noqa: E402

MODEL = "{model}"        # stands for the checkpoint path in recorded arguments
CASES = {
    "inference_paired": {
        "module": "pix2pix_turbo", "cls": "Pix2Pix_Turbo", "image": (70, 66, 1),      # cropped to 64x64 by the script
        "argv": ["--input_image", "{image}", "--prompt", "a test prompt", "--model_path", MODEL, "--output_dir", "{out}",
                 "--use_fp16"]},
    "inference_unpaired": {
        "module": "cyclegan_turbo", "cls": "CycleGAN_Turbo", "image": (128, 64, 2),
        "argv": ["--input_image", "{image}", "--prompt", "driving in the night", "--model_path", MODEL, "--direction", "a2b",
                 "--output_dir", "{out}", "--image_prep", "no_resize", "--use_fp16"]},
}


def golden_path(case):
    return os.path.join(GOLD, f"reference_cli_{case}.pt")


class _Tok:
    model_max_length = 77


def make_checkpoint(case, d):
    """The seeded reduced-width (W.TINY) checkpoint the case's script loads, in the format it expects."""
    import weights as W
    path = os.path.join(d, "model.pkl")
    if case == "inference_paired":
        from pix2pix_turbo import Pix2Pix_Turbo
        Pix2Pix_Turbo(cfg=W.TINY, text_stack=(_Tok(), None), seed=3).save_model(path)      # save_model() pickle
        return path
    from cyclegan_turbo import CycleGAN_Turbo
    m = CycleGAN_Turbo(cfg=W.TINY, text_stack=(_Tok(), None), synthetic_caption="c", synthetic_direction="a2b", seed=4)

    def part(adapter):
        return {k[len("unet."):].replace(f".{adapter}.weight", ".weight"): v for k, v in m._sd.items()
                if k.startswith("unet.") and f".{adapter}." in k}
    # the checkpoint format written by train_cyclegan_turbo.py:293-307 (the real files carry the full VAE state dicts; the
    # trained tensors — LoRA pairs and skip convs — are enough here)
    torch.save({"rank_unet": 8, "rank_vae": 4, "l_target_modules_encoder": [], "l_target_modules_decoder": [],
                "l_modules_others": [], "vae_lora_target_modules": [], "sd_encoder": part("default_encoder"),
                "sd_decoder": part("default_decoder"), "sd_other": part("default_others"),
                "sd_vae_enc": {k: v for k, v in m._sd.items() if k.startswith(("vae.encoder", "vae_b2a.encoder")) and "lora" in k},
                "sd_vae_dec": {k: v for k, v in m._sd.items()
                               if k.startswith(("vae.decoder", "vae_b2a.decoder")) and ("lora" in k or "skip" in k)}}, path)
    return path


def _result(r, target):
    if r is target:
        return "self"
    if isinstance(r, torch.Tensor):
        return r.detach().clone()
    assert r is None, f"unexpected return value {type(r)}"
    return None


class Recorder:
    """Stands in for the model object (and its .unet / .vae handles) the script holds: forwards every call and logs it."""

    def __init__(self, target, log, prefix=""):
        object.__setattr__(self, "_target", target)
        object.__setattr__(self, "_log", log)
        object.__setattr__(self, "_prefix", prefix)

    def __getattr__(self, name):
        v = getattr(self._target, name)
        if callable(v):
            return lambda *a, **k: self._call(self._prefix + name, v, a, k)
        if isinstance(v, (SimpleNamespace, NetHandle)):
            return Recorder(v, self._log, self._prefix + name + ".")
        return v

    def __setattr__(self, name, value):
        raise AttributeError(f"attribute writes are not recorded ({self._prefix}{name})")

    def __call__(self, *a, **k):
        return self._call(self._prefix + "__call__", self._target, a, k)

    def _call(self, path, fn, a, k):
        entry = {"call": path, "args": list(a), "kwargs": dict(k), "rng": torch.get_rng_state()}
        r = fn(*a, **k)
        entry["result"] = _result(r, self._target)
        self._log.append(entry)
        return self if r is self._target else r


def record(ref_src):
    from PIL import Image
    cpu_stub_engine.install()
    sys.path.insert(sys.path.index(os.path.join(ROOT, "img2img-turbo_b200")) + 1, os.path.abspath(ref_src))
    for case, spec in CASES.items():
        mod = importlib.import_module(spec["module"])
        cls = getattr(mod, spec["cls"])
        log = []
        cpu_stub_engine.CALLS.clear()

        def construct(*a, **k):
            log.append({"call": "__init__", "args": list(a), "kwargs": dict(k), "rng": torch.get_rng_state(), "result": None})
            return Recorder(cls(*a, **k), log)
        with tempfile.TemporaryDirectory() as d:
            model = make_checkpoint(case, d)
            w, h, seed = spec["image"]
            g = torch.Generator().manual_seed(seed)
            Image.fromarray((torch.rand(h, w, 3, generator=g) * 255).to(torch.uint8).numpy()).save(os.path.join(d, "in.png"))
            subst = {"{image}": os.path.join(d, "in.png"), MODEL: model, "{out}": os.path.join(d, "out")}
            script = os.path.join(ref_src, case + ".py")
            sys.argv = [script] + [subst.get(a, a) for a in spec["argv"]]
            setattr(mod, spec["cls"], construct)
            try:
                runpy.run_path(script, run_name="__main__")
            finally:
                setattr(mod, spec["cls"], cls)
            out_img = Image.open(os.path.join(d, "out", "in.png"))
            unsub = {v: k for k, v in subst.items()}
            for e in log:
                e["args"] = [unsub.get(a, a) if isinstance(a, str) else a for a in e["args"]]
                e["kwargs"] = {k: unsub.get(v, v) if isinstance(v, str) else v for k, v in e["kwargs"].items()}
        assert log and log[0]["call"] == "__init__", f"{case}: the script did not construct {spec['cls']} from this repo"
        gold = {"script": f"src/{case}.py", "argv": spec["argv"],
                "module": os.path.relpath(mod.__file__, ROOT), "calls": log,
                "engine_calls": [list(map(str, c)) for c in cpu_stub_engine.CALLS],
                "output_image": [out_img.size[0], out_img.size[1], out_img.mode]}
        torch.save(gold, golden_path(case))
        print(case, [e["call"] for e in log], os.path.getsize(golden_path(case)), "bytes")


def replay(case, out):
    cpu_stub_engine.install()
    spec = CASES[case]
    gold = torch.load(golden_path(case))
    cls = getattr(importlib.import_module(spec["module"]), spec["cls"])
    results = []
    with tempfile.TemporaryDirectory() as d:
        model = make_checkpoint(case, d)
        sub = lambda v: model if v == MODEL else v                                   # noqa: E731
        m = None
        for c in gold["calls"]:
            args, kwargs = [sub(a) for a in c["args"]], {k: sub(v) for k, v in c["kwargs"].items()}
            torch.set_rng_state(c["rng"])
            if c["call"] == "__init__":
                m = cls(*args, **kwargs)
                results.append(None)
                continue
            *path, name = c["call"].split(".")
            obj = m
            for p in path:
                obj = getattr(obj, p)
            r = (obj if name == "__call__" else getattr(obj, name))(*args, **kwargs)
            results.append(_result(r, obj))
    torch.save({"results": results, "engine_calls": [list(map(str, c)) for c in cpu_stub_engine.CALLS]}, out)
    print("REPLAY " + json.dumps([c["call"] for c in gold["calls"]]))


if __name__ == "__main__":
    mode = sys.argv[1]
    if mode == "record":
        record(sys.argv[2])
    elif mode == "replay":
        replay(sys.argv[2], sys.argv[3])
    else:
        raise SystemExit(f"unknown mode {mode!r}: record <reference src dir> | replay <case> <out.pt>")

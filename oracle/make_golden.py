"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from
/root/reference, which only exists in the build container) on synthetic state dicts from
video_depth_anything_b200.synth, and pin oracle/vda_oracle.py against it.

    python oracle/make_golden.py            # writes tests/golden/*.npz + MANIFEST.json

Environment shims (SURVEY.md App. F): an `easydict` stub (hard import at dpt_temporal.py:19);
the model class is taken from /root/reference/metric_depth (upstream constructor,
metric_depth/video_depth_anything/video_depth.py:35-56) and the top-level driver
`infer_video_depth` (video_depth.py:166-254, affine alignment) is bound onto it from the
top-level file's source without importing its broken torch.hub constructor.
"""
from __future__ import annotations

import importlib.util
import json
import os
import sys
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = "/root/reference"
GOLD = os.path.join(ROOT, "tests", "golden")


def import_reference():
    ed = types.ModuleType("easydict")

    class EasyDict(dict):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.__dict__ = self

    ed.EasyDict = EasyDict
    sys.modules["easydict"] = ed
    sys.path.insert(0, os.path.join(REF, "metric_depth"))
    from video_depth_anything.video_depth import VideoDepthAnything as MetricVDA  # noqa
    import video_depth_anything.video_depth as metric_mod

    # Top-level driver: same package, but its video_depth.py differs (affine alignment + broken ctor).
    # Load that single file as a sibling module of the metric package so relative imports resolve,
    # with `utils.util` taken from the top-level tree (identical to metric_depth/utils/util.py).
    spec_u = importlib.util.spec_from_file_location("utils.util", os.path.join(REF, "utils", "util.py"))
    um = importlib.util.module_from_spec(spec_u)
    spec_u.loader.exec_module(um)
    pkg = types.ModuleType("utils")
    pkg.util = um
    sys.modules.setdefault("utils", pkg)
    sys.modules.setdefault("utils.util", um)
    spec = importlib.util.spec_from_file_location(
        "video_depth_anything.video_depth_top", os.path.join(REF, "video_depth_anything", "video_depth.py"))
    top = importlib.util.module_from_spec(spec)
    top.__package__ = "video_depth_anything"
    spec.loader.exec_module(top)
    return MetricVDA, metric_mod, top


def ivd_frames() -> np.ndarray:
    """The uint8 [50, 60, 80, 3] input video of the infer_video_depth golden cases, regenerated from its seed (the .npz
    files store the reference's depths only): smooth-ish frames so the cubic resize is exercised on non-noise data too."""
    rng = np.random.default_rng(0)
    base = rng.integers(0, 256, (50, 15, 20, 3), dtype=np.uint8)
    frames = np.repeat(np.repeat(base, 4, axis=1), 4, axis=2)
    return (frames.astype(np.int32) + rng.integers(-20, 20, frames.shape)).clip(0, 255).astype(np.uint8)


def build_ref(MetricVDA, enc, sd):
    from video_depth_anything_b200.synth import MODEL_CONFIGS
    m = MetricVDA(**MODEL_CONFIGS[enc]).eval()
    missing = m.load_state_dict(sd, strict=True)   # proves the key/shape contract (App. C)
    return m


def main():
    from video_depth_anything_b200.synth import MODEL_CONFIGS, synth_state_dict
    from oracle import vda_oracle as O

    torch.set_num_threads(os.cpu_count())
    MetricVDA, metric_mod, top = import_reference()
    os.makedirs(GOLD, exist_ok=True)
    manifest = {"generator": "oracle/make_golden.py", "torch": torch.__version__, "cases": {}}

    fwd_cases = [
        # name, encoder, seed, x shape, x seed, depth store stride, tap token stride (keeps every file under 1 MB)
        ("fwd_vits_T8_56x70", "vits", 0, (1, 8, 3, 56, 70), 1234, 1, 8),
        ("fwd_vits_T32_42x42", "vits", 1, (1, 32, 3, 42, 42), 1235, 1, 8),
        ("fwd_vitl_T4_28x42", "vitl", 0, (1, 4, 3, 28, 42), 1236, 1, 8),
        ("fwd_vits_T2_518x518", "vits", 0, (1, 2, 3, 518, 518), 1237, 2, 64),
    ]
    models = {}
    for name, enc, seed, shape, xseed, stride, tap_stride in fwd_cases:
        sd = synth_state_dict(**MODEL_CONFIGS[enc], seed=seed)
        ref = build_ref(MetricVDA, enc, sd)
        models[(enc, seed)] = (sd, ref)
        x = torch.randn(shape, generator=torch.Generator().manual_seed(xseed))
        t0 = time.time()
        with torch.no_grad():
            d_ref = ref(x)
            perm = torch.randperm(shape[1], generator=torch.Generator().manual_seed(7))
            d_perm = ref(x[:, perm])
        t_ref = time.time() - t0
        stages = {}
        d_or = O.forward(sd, x, enc, stages)
        diff = (d_or - d_ref).abs().max().item()
        rel = O.rel_err(d_or, d_ref)
        # temporal sensitivity (SURVEY §0 trap 7): permuting frames must change the output
        inv = torch.argsort(perm)
        sens = O.rel_err(d_perm[:, inv], d_ref)
        frac_pos = (d_ref > 0).float().mean().item()
        print(f"{name}: oracle-vs-ref max abs {diff:.3e} rel(max,p999,mean) {rel}; "
              f"perm-sensitivity {sens}; frac>0 {frac_pos:.4f}; depth mean {d_ref.mean():.4f} "
              f"std {d_ref.std():.4f}; ref time {t_ref:.1f}s")
        assert diff < 5e-5, name
        assert frac_pos > 0.99, name
        taps = {f"tap{i}": stages[f"tap{i}"][:, ::tap_stride].numpy().astype(np.float32) for i in range(4)}
        np.savez_compressed(os.path.join(GOLD, name + ".npz"),
                            depth=d_ref.numpy()[..., ::stride, ::stride].astype(np.float32), **taps)
        manifest["cases"][name] = dict(kind="forward", encoder=enc, seed=seed, x_shape=list(shape), x_seed=xseed,
                                       stride=stride, tap_stride=tap_stride,
                                       oracle_vs_ref_max_abs=diff, oracle_vs_ref_rel=rel,
                                       perm_sensitivity=sens, frac_positive=frac_pos)

    # ---- infer_video_depth: top-level (affine) and metric (identity) drivers ----
    sd, ref = models[("vits", 0)]
    frames = ivd_frames()
    for name, mod, mode in (("ivd_affine_vits_50x60x80", top, "affine"),
                            ("ivd_identity_vits_50x60x80", metric_mod, "identity")):
        fn = mod.VideoDepthAnything.infer_video_depth
        t0 = time.time()
        d_ref, _ = fn(ref, frames.copy(), 24, input_size=56, device="cpu", fp32=True)
        t_ref = time.time() - t0
        d_or = O.infer_video_depth(sd, frames, "vits", input_size=56, mode=mode)
        diff = float(np.abs(d_or - d_ref).max())
        print(f"{name}: oracle-vs-ref max abs {diff:.3e}; out {d_ref.shape} mean {d_ref.mean():.4f}; ref {t_ref:.1f}s")
        assert diff < 5e-5, name
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), depth=d_ref.astype(np.float32))
        manifest["cases"][name] = dict(kind="infer_video_depth", encoder="vits", seed=0, mode=mode, input_size=56,
                                       n_frames=50, oracle_vs_ref_max_abs=diff)

    # ---- window index closed form vs literal replay ----
    for n in (1, 5, 22, 23, 32, 33, 50, 100, 131, 2048):
        assert O.window_source_indices(n) == O.window_source_indices_literal(n), n
    manifest["window_index_closed_form_checked_for"] = [1, 5, 22, 23, 32, 33, 50, 100, 131, 2048]

    with open(os.path.join(GOLD, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    print("wrote", GOLD)


if __name__ == "__main__":
    main()

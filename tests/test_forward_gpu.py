"""GPU parity of VideoDepthAnything.forward / infer_video_depth (through the C ABI) against
  (a) the reference's own outputs committed under tests/golden/ and
  (b) the oracle restatement on the same seeded inputs,
with the tolerance of BASELINE.json's north_star: per-pixel relative depth error <= 1e-2, measured as
|d - ref| / max(|ref|, 1e-3 max|ref|) (SURVEY.md §8d)."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from e2e_checks import GOLD, build_model, golden_case, stage_report  # noqa: E402
from oracle import vda_oracle as O  # noqa: E402
from oracle.make_golden import ivd_frames  # noqa: E402

TOL = 1e-2           # north_star: per-pixel relative depth error, every advertised dtype, on the MAX (no percentile escape)
TOL_VALIDATION = 1e-3   # north_star: fp32-accumulate validation mode (`fp32=True`)


def _check(dtype, mx, p999, mean, what):
    msg = f"{what} {dtype}: rel err max {mx:.3e} p99.9 {p999:.3e} mean {mean:.3e}"
    print(msg)
    assert mx <= TOL, msg
MAN = json.load(open(os.path.join(GOLD, "MANIFEST.json")))["cases"]
FWD = [k for k, v in MAN.items() if v["kind"] == "forward"]
IVD = [k for k, v in MAN.items() if v["kind"] == "infer_video_depth"]


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("name", FWD)
def test_forward_vs_reference_golden(name, dtype):
    (mx, p999, mean), d = golden_case(name, dtype)
    assert (d > 0).float().mean() > 0.99
    _check(dtype, mx, p999, mean, name)


@pytest.mark.parametrize("name", IVD)
def test_infer_video_depth_vs_reference_golden(name):
    c = MAN[name]
    g = np.load(os.path.join(GOLD, name + ".npz"))
    m, _ = build_model(c["encoder"], c["seed"], torch.float16)
    m.metric = c["mode"] == "identity"
    out, fps = m.infer_video_depth(ivd_frames(), 24, input_size=c["input_size"], device="cuda")
    assert fps == 24 and out.shape == g["depth"].shape and out.dtype == np.float32
    mx, p999, mean = O.rel_err(torch.from_numpy(out), torch.from_numpy(g["depth"]))
    assert mx <= TOL, f"{name}: rel err max {mx:.3e} p99.9 {p999:.3e} mean {mean:.3e}"


def test_forward_frame_permutation_sensitivity():
    """The temporal path is live: permuting input frames changes outputs by far more than the tolerance."""
    m, _ = build_model("vits", 0, torch.bfloat16)
    x = torch.randn(1, 8, 3, 56, 70, generator=torch.Generator().manual_seed(1234)).cuda()
    perm = torch.randperm(8, generator=torch.Generator().manual_seed(7))
    d = m.forward(x)
    dp = m.forward(x[:, perm.cuda()])
    mx, _, _ = O.rel_err(dp[:, torch.argsort(perm).cuda()].cpu(), d.cpu())
    assert mx > 3e-2


def test_forward_is_deterministic_and_pure():
    m, _ = build_model("vits", 0, torch.bfloat16)
    x = torch.randn(1, 4, 3, 42, 56, generator=torch.Generator().manual_seed(3)).cuda()
    x0 = x.clone()
    a = m.forward(x)
    b = m.forward(x)
    assert torch.equal(a, b) and torch.equal(x, x0) and a.dtype == torch.float32 and (a >= 0).all()


def test_forward_rejects_bad_shapes():
    m, _ = build_model("vits", 0, torch.bfloat16)
    with pytest.raises(AssertionError):
        m.forward(torch.zeros(1, 2, 3, 50, 56).cuda())


def test_stagewise_vs_oracle_vits():
    fin, rows, d, ref = stage_report("vits", 0, (1, 8, 3, 56, 70), 1234, torch.float16)
    worst = max(r[1] for r in rows)
    assert fin[0] <= TOL and worst < 2e-2, (fin, rows)


@pytest.mark.parametrize("enc,dtype,tol", [("vitl", torch.bfloat16, TOL), ("vitl", torch.float16, TOL),
                                           ("vits", torch.bfloat16, TOL)], ids=["vitl-bf16", "vitl-fp16", "vits-bf16"])
def test_full_size_window_vs_oracle(enc, dtype, tol):
    """BASELINE.json configs[0]/[1]: one 1x32x518x518 window, oracle evaluated in fp32 on the same GPU
    (TF32 off) as the checker."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    fin, rows, d, ref = stage_report(enc, 0, (1, 32, 3, 518, 518), 1234, dtype, oracle_device="cuda")
    assert (ref > 0).float().mean() > 0.99
    _check(dtype, *fin, f"{enc} 1x32x518x518")


@pytest.mark.parametrize("enc", ["vitl", "vits"])
def test_validation_mode_full_size_window(enc):
    """north_star's validation bar: <= 1e-3 per pixel against the fp32 reference in an fp32-accumulate mode.  `fp32=True`
    (reference video_depth.py:203-205: autocast off) selects the validation engine -- fp16 activations, hi | lo fp16
    weight pairs, fp32 accumulation / residuals / statistics -- from a model whose own dtype is bf16."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    m, sd = build_model(enc, 0, torch.bfloat16)
    x = torch.randn(1, 32, 3, 518, 518, generator=torch.Generator().manual_seed(1234))
    d = m.forward(x.cuda(), fp32=True).float().cpu()
    ref = O.forward({k: v.cuda() for k, v in sd.items()}, x.cuda(), enc).float().cpu()
    mx, p999, mean = O.rel_err(d, ref)
    print(f"{enc} 1x32x518x518 validation mode: rel err max {mx:.3e} p99.9 {p999:.3e} mean {mean:.3e}")
    assert mx <= TOL_VALIDATION, (mx, p999, mean)
    fast = m.forward(x.cuda()).float().cpu()                 # the fast path is a different engine, same weights
    assert O.rel_err(fast, ref)[0] <= TOL


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_metric_config_518x924_vs_oracle(dtype):
    """BASELINE.json configs[3] geometry (1280x720 video -> 518x924 network input, 2443 tokens per frame, bicubic
    pos-embed, non-square maps everywhere) on a short clip, against the fp32 oracle run on the GPU."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    fin, rows, d, ref = stage_report("vitl", 0, (1, 4, 3, 518, 924), 1234, dtype, oracle_device="cuda")
    assert (ref > 0).float().mean() > 0.99
    _check(dtype, *fin, "vitl 1x4x518x924")


def test_batch_of_clips_equals_single_clips():
    """BASELINE.json configs[4]: independent clips in one batch give the per-clip results bit-for-bit."""
    m, _ = build_model("vits", 0, torch.bfloat16)
    x = torch.randn(2, 8, 3, 56, 70, generator=torch.Generator().manual_seed(11)).cuda()
    both = m.forward(x)
    assert torch.equal(both[0], m.forward(x[:1])[0]) and torch.equal(both[1], m.forward(x[1:])[0])


def test_sharded_driver_single_process_equals_plain():
    """parallel.infer_video_depth_sharded without a process group is exactly infer_video_depth (N>1 logic is covered
    on CPU with gloo in tests/test_parallel_cpu.py; tests/multi_gpu_check.py runs it under torchrun on N GPUs)."""
    from video_depth_anything_b200.parallel import infer_video_depth_sharded
    name = IVD[0]
    c = MAN[name]
    m, _ = build_model(c["encoder"], c["seed"], torch.float16)
    m.metric = c["mode"] == "identity"
    frames = ivd_frames()
    a, _ = m.infer_video_depth(frames, 24, input_size=c["input_size"], device="cuda")
    b, _ = infer_video_depth_sharded(m, frames, 24, input_size=c["input_size"])
    assert np.array_equal(a, b)


@pytest.mark.parametrize("n,h0,w0,size", [(70, 56, 70, 56), (33, 60, 80, 98), (5, 42, 42, 42)],
                         ids=["70f-same-size", "33f-resized", "5f-padded"])
def test_feature_reuse_is_bit_identical(n, h0, w0, size):
    """SURVEY.md §8(f)-2: encoding each source frame once and reusing its tap features across overlapping windows
    gives exactly the frames of the plain per-window path (kernels are batch-invariant), on multi-window videos,
    resized inputs and a video shorter than one window (padded with its last frame)."""
    m, _ = build_model("vits", 0, torch.bfloat16)
    frames = np.random.default_rng(n).integers(0, 256, (n, h0, w0, 3), dtype=np.uint8)
    a, _ = m.infer_video_depth(frames, 24, input_size=size, device="cuda", reuse_features=True)
    b, _ = m.infer_video_depth(frames, 24, input_size=size, device="cuda", reuse_features=False)
    assert a.shape == (n, h0, w0) and np.isfinite(a).all()
    assert np.array_equal(a, b)


def test_infer_video_depth_vs_oracle_resized_multiwindow():
    """Device preprocessing (INTER_CUBIC resize + normalise), feature reuse, output resize and alignment together
    against the oracle's infer_video_depth (cv2 preprocessing, per-window forward) on a 2-window resized video."""
    from video_depth_anything_b200.synth import MODEL_CONFIGS, synth_state_dict
    m, _ = build_model("vits", 0, torch.float16)
    sd = synth_state_dict(**MODEL_CONFIGS["vits"], seed=0)
    frames = np.random.default_rng(5).integers(0, 256, (40, 45, 64, 3), dtype=np.uint8)
    out, _ = m.infer_video_depth(frames, 24, input_size=56, device="cuda")
    ref = O.infer_video_depth(sd, frames, "vits", input_size=56)
    mx, p999, mean = O.rel_err(torch.from_numpy(out), torch.from_numpy(ref))
    assert mx <= TOL, f"rel err max {mx:.3e} p99.9 {p999:.3e} mean {mean:.3e}"


@pytest.mark.parametrize("reuse", [True, False], ids=["feature-reuse", "per-window"])
def test_bounded_device_buffers_are_bit_identical_to_unbounded(reuse, monkeypatch):
    """The long-video driver keeps only a ring of uploaded uint8 frames (4 x 64 + frame 0) and a ring of aligned frames
    (4 x 22) on the device; a 330-frame video (15 windows: both rings wrap several times) must come out bit-identical to
    the same call with the rings switched off, and every frame must have been written."""
    from video_depth_anything_b200 import video_depth as vd
    m, _ = build_model("vits", 0, torch.bfloat16)
    n, h0, w0 = 330, 45, 64
    frames = np.random.default_rng(3).integers(0, 256, (n, h0, w0, 3), dtype=np.uint8)
    a, _ = m.infer_video_depth(frames, 24, input_size=56, device="cuda", reuse_features=reuse)
    up_ring = []
    real_init = vd.FrameUploader.__init__

    def spy(self, *args, **kw):
        real_init(self, *args, **kw)
        up_ring.append(self.ring)
    monkeypatch.setattr(vd.FrameUploader, "__init__", spy)
    a2, _ = m.infer_video_depth(frames, 24, input_size=56, device="cuda", reuse_features=reuse)
    assert up_ring == [True]
    monkeypatch.setattr(vd.FrameUploader, "RING_CHUNKS", 1 << 20)
    monkeypatch.setattr(vd.WindowAligner, "RING_SEGS", 1 << 20)
    b, _ = m.infer_video_depth(frames, 24, input_size=56, device="cuda", reuse_features=reuse)
    assert up_ring == [True, False]
    assert a.shape == (n, h0, w0) and np.isfinite(a).all() and (a > 0).any(axis=(1, 2)).all()
    assert np.array_equal(a, a2) and np.array_equal(a, b)

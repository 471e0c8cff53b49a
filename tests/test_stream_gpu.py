"""GPU: streaming inference (VideoDepthAnything.stream / DepthStream, vda_attention_temporal_step) against the oracle's
definition of it (stream_oracle.stream_depths), plus determinism, isolation and bounded per-step cost."""
import gc

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import stream_oracle as SO  # noqa: E402
from e2e_checks import build_model  # noqa: E402
from oracle import vda_oracle as O  # noqa: E402
from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, ops, synth_state_dict  # noqa: E402
from video_depth_anything_b200.windows import get_resize_hw  # noqa: E402

TOL = 1e-2
TOL_VALIDATION = 1e-3


# ---------------------------------------------------------------------------------------------- kernel
def _step_reference(qkv, cache, pe, n, slots, heads=8):
    """fp32 restatement of vda_attention_temporal_step on the same 16-bit inputs."""
    hw, C3 = qkv.shape
    C, dh = C3 // 3, C3 // 3 // heads
    q = qkv[:, :C].float() + pe[n, :C]
    ks = [cache[s, :, :C].float() + pe[p, C:2 * C] for p, s in enumerate(slots)] + [qkv[:, C:2 * C].float() + pe[n, C:2 * C]]
    vs = [cache[s, :, C:].float() + pe[p, 2 * C:] for p, s in enumerate(slots)] + [qkv[:, 2 * C:].float() + pe[n, 2 * C:]]
    k = torch.stack(ks, 1).reshape(hw, n + 1, heads, dh)
    v = torch.stack(vs, 1).reshape(hw, n + 1, heads, dh)
    s = torch.einsum("phd,pjhd->phj", q.reshape(hw, heads, dh), k) * dh ** -0.5
    return torch.einsum("phj,pjhd->phd", s.softmax(-1), v).reshape(hw, C)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("dh", [8, 24, 32, 48, 128])
def test_step_kernel_vs_fp32(dtype, dh):
    g = torch.Generator(device="cuda").manual_seed(dh)
    C, hw, slots = 8 * dh, 37, 32
    tol = 1e-2 if dtype == torch.bfloat16 else 2e-3
    for n in (0, 1, 17, 31):
        for scale in (1.0, 12.0):                           # 12: scores of magnitude ~1e2..1e3 (softmax saturates)
            qkv = (torch.randn(hw, 3 * C, device="cuda", generator=g) * scale).to(dtype)
            cache = (torch.randn(slots, hw, 2 * C, device="cuda", generator=g) * scale).to(dtype)
            pe = torch.randn(32, 3 * C, device="cuda", generator=g)
            perm = torch.randperm(slots, device="cuda", generator=g).tolist()
            write, ctx_slots = perm[0], perm[1:1 + n]       # out of order; the write slot is not read
            ctx = torch.tensor([n, write] + ctx_slots, dtype=torch.int32, device="cuda")
            before = cache.clone()
            out = torch.empty(hw, C, dtype=dtype, device="cuda")
            ops.attention_temporal_step(qkv, cache, pe, ctx, out)
            ref = _step_reference(qkv, before, pe, n, ctx_slots)
            err = (out.float() - ref).abs().max().item()
            assert err <= tol * ref.abs().max().item(), (n, scale, err)
            assert torch.equal(cache[write], qkv[:, C:]), "k'|v' of the current frame must land in the write slot as is"
            keep = [s for s in range(slots) if s != write]
            assert torch.equal(cache[keep], before[keep])


def test_step_kernel_rejects_bad_arguments():
    from video_depth_anything_b200._lib import VdaError
    qkv = torch.zeros(10, 3 * 20, dtype=torch.bfloat16, device="cuda")           # head dim 20/8: not a multiple of 8
    cache = torch.zeros(4, 10, 40, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(VdaError):
        ops.attention_temporal_step(qkv, cache, torch.zeros(32, 60, device="cuda"), torch.zeros(2, dtype=torch.int32,
                                    device="cuda"), torch.empty(10, 20, dtype=torch.bfloat16, device="cuda"))


# ---------------------------------------------------------------------------------------------- end to end
def _frames(n, h, w, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (n, h, w, 3), dtype=np.uint8)


def _oracle(sd, frames, enc, size):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return torch.from_numpy(SO.stream_depths({k: v.cuda() for k, v in sd.items()}, frames, enc, input_size=size))


def _push_all(stream, frames):
    return torch.from_numpy(np.stack([stream.push(f) for f in frames]))


@pytest.fixture(scope="module")
def vits_case():
    sd = synth_state_dict(**MODEL_CONFIGS["vits"], seed=0)
    frames = _frames(42, 50, 70)                   # network input 56x84, resized back to 50x70; the context slides from t = 32
    return sd, frames, _oracle(sd, frames, "vits", 56)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_stream_vits_vs_oracle(vits_case, dtype):
    sd, frames, ref = vits_case
    m, _ = build_model("vits", 0, dtype)
    got = _push_all(m.stream(input_size=56), frames)
    errs = [O.rel_err(got[t], ref[t])[0] for t in range(len(frames))]
    print(f"vits stream {dtype}: worst frame rel err {max(errs):.3e}")
    assert max(errs) <= TOL, errs
    assert (got >= 0).all()


def test_stream_vits_validation_mode_vs_oracle(vits_case):
    sd, frames, ref = vits_case
    m, _ = build_model("vits", 0, torch.bfloat16)
    got = _push_all(m.stream(input_size=56, fp32=True), frames)
    errs = [O.rel_err(got[t], ref[t])[0] for t in range(len(frames))]
    print(f"vits stream fp32=True: worst frame rel err {max(errs):.3e}")
    assert max(errs) <= TOL_VALIDATION, errs


def test_stream_vitl_518_vs_oracle():
    m, sd = build_model("vitl", 0, torch.bfloat16)
    frames = _frames(34, 518, 518, seed=1)
    got = _push_all(m.stream(), frames)
    ref = _oracle(sd, frames, "vitl", 518)
    errs = [O.rel_err(got[t], ref[t])[0] for t in range(len(frames))]
    print(f"vitl 518x518 stream bf16: worst frame rel err {max(errs):.3e}")
    assert max(errs) <= TOL, errs


def test_stream_step0_equals_forward():
    m, _ = build_model("vits", 0, torch.bfloat16)
    frame = _frames(1, 56, 84, seed=2)[0]
    assert get_resize_hw(56, 84, 56) == (56, 84)
    got = torch.from_numpy(m.stream(input_size=56).push(frame))
    fdev = torch.from_numpy(frame).cuda()[None]
    x = ops.preprocess_frames(fdev, torch.zeros(1, dtype=torch.int32, device="cuda"), 56, 84)
    ref = m.forward(x[None])[0, 0].cpu()
    assert O.rel_err(got, ref)[0] <= TOL


def test_infer_video_depth_one_is_a_stream():
    m, _ = build_model("vits", 0, torch.bfloat16)
    frames = _frames(5, 50, 70, seed=3)
    a = _push_all(m.stream(input_size=56), frames)
    b = torch.from_numpy(np.stack([m.infer_video_depth_one(f, input_size=56) for f in frames]))
    assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------- determinism, isolation
def test_streams_are_deterministic_and_independent():
    m, _ = build_model("vits", 0, torch.bfloat16)
    fa, fb = _frames(36, 50, 70, seed=4), _frames(36, 50, 70, seed=5)
    x = torch.randn(1, 8, 3, 56, 84, generator=torch.Generator().manual_seed(6)).cuda()
    w0 = m.forward(x).cpu()
    alone_a = _push_all(m.stream(input_size=56), fa)
    assert torch.equal(alone_a, _push_all(m.stream(input_size=56), fa))
    alone_b = _push_all(m.stream(input_size=56), fb)
    sa, sb = m.stream(input_size=56), m.stream(input_size=56)
    inter_a, inter_b = [], []
    for a, b in zip(fa, fb):
        inter_a.append(sa.push(a))
        inter_b.append(sb.push(b))
    assert torch.equal(alone_a, torch.from_numpy(np.stack(inter_a)))
    assert torch.equal(alone_b, torch.from_numpy(np.stack(inter_b)))
    assert torch.equal(w0, m.forward(x).cpu()), "streaming must not change the windowed forward"


# ---------------------------------------------------------------------------------------------- bounded cost
def test_step_cost_is_bounded():
    m, _ = build_model("vits", 0, torch.bfloat16)
    frames = _frames(121, 50, 70, seed=7)
    st = m.stream(input_size=56)
    launches, mem = {}, {}
    for t, f in enumerate(frames):
        n0 = ops.LAUNCHES
        st.push(f)
        launches[t] = ops.LAUNCHES - n0
        if t in (60, 120):
            gc.collect()                                  # objects of earlier tests may be freed at any point of the loop
            mem[t] = torch.cuda.memory_allocated()
    assert launches[1] == launches[60] == launches[120] > 0
    assert mem[60] == mem[120]
    # one eager step under the profiler: every GEMM works on one frame's rows, no windowed temporal attention runs
    ops.PROFILE = []
    try:
        st.push(frames[0])
        torch.cuda.synchronize()
        prof = list(ops.PROFILE)
    finally:
        ops.PROFILE = None
    hp, wp = 56 // 14, 84 // 14
    rows = [info["M"] for name, info, _, _ in prof if name == "gemm"]
    assert rows and max(rows) <= 64 * hp * wp            # the largest per-frame map: output_conv1 at 8hp x 8wp
    names = [name for name, *_ in prof]
    assert names.count("attention_temporal_step") == 8 and "attention_temporal" not in names


# ---------------------------------------------------------------------------------------------- errors
def test_stream_raises_after_new_weights_and_on_bad_frames():
    m, sd = build_model("vits", 0, torch.bfloat16)
    st = m.stream(input_size=56)
    f = _frames(2, 50, 70, seed=8)
    st.push(f[0])
    with pytest.raises(ValueError):
        st.push(_frames(1, 60, 70)[0])                    # another size mid-stream
    with pytest.raises(ValueError):
        st.push(f[1].astype(np.float32))
    with pytest.raises(ValueError):
        st.push(f[1][..., :2])
    m.load_state_dict(sd)
    with pytest.raises(RuntimeError):
        st.push(f[1])
    m.stream(input_size=56).push(f[1])                    # a new stream works
    with pytest.raises(RuntimeError):
        m.infer_video_depth_one(f[0], device="cpu")
    with pytest.raises(RuntimeError):
        VideoDepthAnything(**MODEL_CONFIGS["vits"]).stream()

"""CPU: the streaming context / cache-slot plan (windows.stream_context) and the streaming oracle
(tests/stream_oracle.py): stream_depths against its causal windowed forward, whose non-causal form equals oracle.forward
(pinned to the reference by test_oracle_golden.py)."""
import numpy as np
import pytest
import torch

import stream_oracle as SO
from oracle import vda_oracle as O
from video_depth_anything_b200.synth import MODEL_CONFIGS, synth_state_dict
from video_depth_anything_b200.windows import STREAM_CONTEXT, stream_context


def test_stream_context_plan_300_steps():
    L = STREAM_CONTEXT
    assert L == 31
    held = {}                                       # simulated device cache: slot -> frame it holds
    used = set()
    for t in range(300):
        ids, slots, write = stream_context(t, L)
        assert len(ids) == min(t, L)
        assert ids == SO.stream_context_ids(t, L)
        if t:
            assert ids[0] == 0 and slots[0] == 0
        assert all(a < b for a, b in zip(ids, ids[1:]))
        assert all(j < t for j in ids)
        for j, s in zip(ids, slots):
            assert held[s] == j, (t, j, s)          # every read finds the frame it claims
        assert write not in slots                   # the slot written this step is not read this step
        held[write] = t
        used.add(write)
    assert len(used) <= L + 1 and max(used) <= L


def test_stream_context_rejects_bad_step():
    with pytest.raises(ValueError):
        stream_context(-1)


@pytest.fixture(scope="module")
def vits():
    sd = synth_state_dict(**MODEL_CONFIGS["vits"], seed=0)
    frames = np.random.default_rng(5).integers(0, 256, (12, 42, 56, 3), dtype=np.uint8)
    return sd, frames


def test_stream_depths_equal_causal_forward(vits):
    """No context slides for t <= 31, so streaming frames 0..11 is the causal windowed forward of those 12 frames."""
    sd, frames = vits
    got = torch.from_numpy(SO.stream_depths(sd, frames, "vits", input_size=42))
    x = torch.stack([torch.from_numpy(O.preprocess_frame(f, 42)) for f in frames])[None]
    ref = SO.forward(sd, x, "vits", causal=True)[0]
    assert got.shape == ref.shape == (12, 42, 56)
    for t in range(12):
        assert O.rel_err(got[t], ref[t])[0] <= 1e-5, t


def test_stream_step0_equals_single_frame_forward(vits):
    sd, frames = vits
    got = torch.from_numpy(SO.stream_depths(sd, frames[:1], "vits", input_size=42))
    ref = O.forward(sd, torch.from_numpy(O.preprocess_frame(frames[0], 42))[None, None], "vits")[0]
    assert O.rel_err(got, ref)[0] <= 1e-5



def test_restated_head_equals_oracle_forward(vits):
    """Without the mask, the streaming oracle's forward is oracle.forward; with it, frame 0 changes."""
    sd, frames = vits
    x = torch.stack([torch.from_numpy(O.preprocess_frame(f, 42)) for f in frames[:6]])[None]
    ref = O.forward(sd, x, "vits")
    assert O.rel_err(SO.forward(sd, x, "vits", causal=False), ref)[0] <= 1e-5
    assert O.rel_err(SO.forward(sd, x, "vits", causal=True)[0, 0], ref[0, 0])[0] > 1e-4

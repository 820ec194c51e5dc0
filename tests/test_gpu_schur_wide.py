"""GPU parity on windows with more frames than cfg-5: the Schur complement's tile-local Y reaches its widest
row stride, and from 24 keyframes on the chunk accumulator no longer fits shared memory and k_schur
accumulates in the global partial instead."""
import dataclasses

import pytest

from okvis_b200 import synthetic
from test_gpu_solver import compare

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(okb):
    c = okb.Context(0, 2)
    yield c
    c.close()


@pytest.mark.parametrize("n_frames", [24, 28])
def test_four_camera_wide_window(ctx, oracle, n_frames):
    cfg = dataclasses.replace(synthetic.CONFIGS[5], n_frames=n_frames, n_landmarks=600)
    compare(ctx, oracle, synthetic.make_window(5, 0, cfg=cfg), max_iterations=6)

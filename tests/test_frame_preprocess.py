"""ImagePreprocessor (composite on white, crop to the foreground box, pad to a square) — SURVEY 8(f) rank 3, second half.

CPU: the numpy restatement (oracle/preprocess_oracle.py) against the outputs of the reference's OWN
`ImagePreprocessor.process_images` (actionmesh/preprocessing/image_processor.py) on the same seeded frames, stored by
oracle/gen_golden.py in tests/golden/frame_preprocess.npz.
GPU (-m gpu): B200FramePreprocessor's uint8 output `array_equal` to the restatement, shared and independent cropping,
non-square frames, the invalid-alpha error."""
import os

import numpy as np
import pytest

from oracle import preprocess_oracle, synth


@pytest.mark.parametrize("independent", [False, True])
def test_restatement_matches_the_reference_module(golden_dir, independent):
    gold = np.load(os.path.join(golden_dir, "frame_preprocess.npz"))
    frames = synth.make_rgba_frames()
    ref = [gold[f"independent{int(independent)}_frame{i}"] for i in range(len(frames))]
    ours = preprocess_oracle.frame_preprocess(frames, independent, 0.1)
    assert len(ref) == len(ours)
    for a, b in zip(ref, ours):
        assert np.array_equal(np.asarray(a), b)
    bad = frames[0].copy()
    bad[..., 3] = 255
    with pytest.raises(ValueError):
        preprocess_oracle.frame_preprocess([bad])


@pytest.mark.gpu
@pytest.mark.parametrize("independent", [False, True])
def test_gpu_frame_preprocessing_is_bit_exact(amb_lib, independent):
    from PIL import Image

    from actionmesh_b200.preprocess import B200FramePreprocessor

    for H, W in ((96, 128), (130, 70)):
        frames = synth.make_rgba_frames(H=H, W=W, seed=H)
        want = preprocess_oracle.frame_preprocess(frames, independent, 0.1)
        proc = B200FramePreprocessor(independent_cropping=independent, padding_ratio=0.1)
        got = proc.process_images([Image.fromarray(f, "RGBA") for f in frames])
        assert len(got) == len(want)
        for a, b in zip(got, want):
            assert np.array_equal(np.asarray(a), b)
    bad = synth.make_rgba_frames(n=1)[0]
    bad[..., 3] = 255
    with pytest.raises(ValueError):
        B200FramePreprocessor().process_images([Image.fromarray(bad, "RGBA")])

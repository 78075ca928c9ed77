"""CPU: the PRODUCT's host-side mirrors (pyannote_audio_b200.inference / signal / pipeline / core) against the vectors
produced by executing the reference's own files (tests/golden/make_golden_pipeline.py, make_golden_apply.py).  These
are the pieces of the drop-in surface that run on the host; the device kernels are compared with the oracle in the
`-m gpu` tests, and the oracle with the same vectors in test_oracle_*_golden.py."""
import os

import numpy as np
import pytest

from pyannote_audio_b200.core import SlidingWindow, SlidingWindowFeature
from pyannote_audio_b200.inference import Inference
from pyannote_audio_b200.pipeline import binarize_frames
from pyannote_audio_b200.signal import Binarize

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FRAMES = SlidingWindow(start=0.0, duration=0.0619375, step=0.016875)
CHUNKS = SlidingWindow(start=0.0, duration=10.0, step=1.0)


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_pipeline_vectors.npz"))


@pytest.fixture(scope="module")
def ref_apply():
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_apply_vectors.npz"))


def test_inference_aggregate_and_trim_match_reference(ref):
    scores = ref["agg_scores"]
    for name, kw in (("plain", dict()), ("hamming", dict(hamming=True)), ("warm", dict(warm_up=(1.0, 1.5), hamming=True)),
                     ("skip", dict(skip_average=True, missing=0.0)), ("missing0", dict(missing=0.0))):
        got = Inference.aggregate(SlidingWindowFeature(scores.copy(), CHUNKS), FRAMES, **kw)
        np.testing.assert_array_equal(got.data, ref[f"agg_{name}"], err_msg=name)
        sw = got.sliding_window
        assert (sw.start, sw.duration, sw.step) == tuple(ref[f"agg_{name}_sw"])
    tr = Inference.trim(SlidingWindowFeature(scores.copy(), CHUNKS), warm_up=(0.1, 0.05))
    assert tuple(tr.data.shape) == tuple(ref["trim_data_shape"])
    sw = tr.sliding_window
    np.testing.assert_allclose([sw.start, sw.duration, sw.step], ref["trim_sw"], rtol=0, atol=1e-15)


def test_binarize_frames_matches_reference_to_annotation(ref):
    for name in ("full", "cap1"):
        disc = ref[f"rec_{name}"]
        sw = SlidingWindow(*[float(v) for v in ref[f"rec_{name}_sw"][[1, 2, 0]]])       # (duration, step, start)
        ann, rows = binarize_frames(disc, sw)
        want = ref[f"ann_{name}"]
        got = [(s.start, s.end, lab) for s, _, lab in ann.itertracks(yield_label=True)]
        assert len(got) == len(want)
        np.testing.assert_array_equal(np.array([[a, b] for a, b, _ in got]), want[:, :2])
        assert [int(lab) for _, _, lab in got] == [int(v) for v in want[:, 2]]


def test_signal_binarize_matches_reference(ref, ref_apply):
    scores = SlidingWindowFeature(ref["binz_scores"], FRAMES)
    ann = Binarize(onset=0.6, offset=0.4)(scores)
    got = np.array([(s.start, s.end, float(lab)) for s, _, lab in ann.itertracks(yield_label=True)]).reshape(-1, 3)
    np.testing.assert_array_equal(got, ref["binz_rows"])
    # VoiceActivityDetection's binarisation of the aggregated speech scores, with and without min_duration_on
    for name in ("vad", "vad_short"):
        sw = SlidingWindow(*[float(v) for v in ref_apply[f"{name}_scores_sw"][[1, 2, 0]]])
        for sub, mon in (("", 0.0), ("_on", 0.25)):
            ann = Binarize(onset=0.5, offset=0.5, min_duration_on=mon)(SlidingWindowFeature(ref_apply[f"{name}_scores"], sw))
            got = np.array([(s.start, s.end) for s, _ in ann.itertracks()]).reshape(-1, 2)
            np.testing.assert_array_equal(got, ref_apply[f"{name}{sub}_rows"])


def test_audio_matches_reference_io(ref):
    """Audio.__call__ / crop / downmix_and_resample on in-memory waveforms against the reference's core/io.py executed
    by path (downmix, channel selection, 44.1 -> 16 kHz and 16 -> 8 kHz resampling, crops inside / padded)."""
    import torch

    from pyannote_audio_b200.audio import Audio
    from pyannote_audio_b200.core import Segment

    g = torch.Generator().manual_seed(5)                 # the generator's stereo input, drawn from the same seed
    stereo = torch.rand(2, 24000, generator=g) * 2 - 1
    assert np.array_equal(stereo[:, :64].numpy(), ref["io_stereo_head"])
    assert stereo.double().sum().item() == float(ref["io_stereo_sum"])
    hi = torch.from_numpy(ref["io_hi"])
    a16 = Audio(sample_rate=16000, mono="downmix")
    w, sr = a16({"waveform": stereo, "sample_rate": 16000})
    assert sr == 16000 and np.array_equal(w.numpy(), ref["io_downmix"])
    w, _ = a16({"waveform": stereo, "sample_rate": 16000, "channel": 1})
    assert np.array_equal(w.numpy(), ref["io_channel1"])
    w, sr = a16({"waveform": hi, "sample_rate": 44100})
    assert sr == int(ref["io_resampled_sr"]) == 16000 and np.array_equal(w.numpy(), ref["io_resampled"])
    w, sr = Audio(sample_rate=8000, mono="downmix")({"waveform": stereo, "sample_rate": 16000})
    assert sr == 8000 and np.array_equal(w.numpy(), ref["io_half_rate"])
    for name, (a, b), mode in (("in", (0.2, 0.7), "raise"), ("pad_end", (1.2, 2.0), "pad"), ("pad_start", (-0.25, 0.5), "pad")):
        w, _ = a16.crop({"waveform": stereo, "sample_rate": 16000}, Segment(a, b), mode=mode)
        assert np.array_equal(w.numpy(), ref[f"io_crop_{name}"]), name


def test_diarize_output_serialize_matches_reference(ref_apply):
    """DiarizeOutput.serialize (speaker_diarization.py:78-124) on the reference's own output of the synthetic file."""
    import json

    from pyannote_audio_b200.core import Annotation
    from pyannote_audio_b200.pipeline import DiarizeOutput

    def annotation(rows):
        labels = np.array([f"SPEAKER_{int(k):02d}" for k in rows[:, 2]], dtype=object)
        return Annotation.from_rows(rows[:, 0], rows[:, 1], labels, uri="golden")

    for name in ("std", "xo"):
        out = DiarizeOutput(annotation(ref_apply[f"{name}_diar"]), annotation(ref_apply[f"{name}_excl"]),
                            ref_apply[f"{name}_speaker_embeddings"])
        assert out.serialize() == json.loads(str(ref_apply[f"{name}_serialized"]))
        assert out.speaker_diarization.labels() == list(ref_apply[f"{name}_labels"])

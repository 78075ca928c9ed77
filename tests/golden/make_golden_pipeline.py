"""Generates tests/golden/reference_pipeline_vectors.npz by EXECUTING the reference's own pipeline-level source files
where they lie under /root/reference -- run once in the build container:

    PYTHONPATH=. python tests/golden/make_golden_pipeline.py

tests/golden/make_golden.py pins the five leaf modules that import cleanly.  The files pinned here
(core/inference.py, core/plda.py, utils/signal.py, pipelines/utils/diarization.py, pipelines/clustering.py,
pipelines/speaker_diarization.py) import packages that are absent from this image (lightning, pyannote.core,
pyannote.pipeline, pyannote.metrics, torchcodec, ...).  They are loaded by path with
  * inert stub modules for everything the functions under test never touch, and
  * a stand-in for `pyannote.core` (Segment / SlidingWindow / SlidingWindowFeature / Annotation below: the public
    behaviour of pyannote.core 6 as documented, restated -- the one piece that stays unpinned),
and the functions are then called verbatim: Inference.aggregate / trim, SpeakerDiarizationMixin.speaker_count /
to_diarization / to_annotation / set_num_speakers, Binarize, BaseClustering.filter_embeddings / constrained_argmax /
assign_embeddings, AgglomerativeClustering.cluster / __call__, VBxClustering.__call__, PLDA, SpeakerDiarization.reconstruct.
Inputs and outputs go to the .npz; tests/test_oracle_golden.py checks the oracle restatement against them.
Nothing here is needed (or available) at test time on the GPU box.
"""
import importlib.util
import numbers
import os
import sys
import tempfile
import types

import numpy as np

REF = os.environ.get("PYANNOTE_REFERENCE", "/root/reference")
SPA = os.path.join(REF, "src", "pyannote", "audio")


# ---------------------------------------------------------------------------------------------------------------
# stand-in for pyannote.core (only what the functions under test use)
# ---------------------------------------------------------------------------------------------------------------
class Segment:
    def __init__(self, start=0.0, end=0.0):
        self.start, self.end = start, end

    @property
    def duration(self):
        return self.end - self.start if self else 0.0

    @property
    def middle(self):
        return 0.5 * (self.start + self.end)

    def __bool__(self):
        return bool((self.end - self.start) > 1e-6)

    def __and__(self, other):
        return Segment(max(self.start, other.start), min(self.end, other.end))

    def __iter__(self):
        yield self.start
        yield self.end


class SlidingWindow:
    def __init__(self, duration=0.030, step=0.010, start=0.000, end=None):
        self.duration, self.step, self.start, self.end = duration, step, start, end

    def closest_frame(self, t):
        return int(np.rint((t - self.start - 0.5 * self.duration) / self.step))

    def __getitem__(self, i):
        start = self.start + i * self.step
        if self.end is not None and start >= self.end:
            return None
        return Segment(start=start, end=start + self.duration)

    def range_to_segment(self, i0, n):
        start = self.start + (i0 - 0.5) * self.step + 0.5 * self.duration
        duration = n * self.step
        end = start + duration
        if i0 == 0:
            start = self.start
        return Segment(start, end)

    def crop(self, focus, mode="loose", fixed=None, return_ranges=False):
        assert mode == "loose" and fixed is None and isinstance(focus, Segment)
        i = int(np.ceil((focus.start - self.duration - self.start) / self.step))
        j = int(np.floor((focus.end - self.start) / self.step))
        return [[i, j + 1]] if return_ranges else np.array(range(i, j + 1), dtype=np.int64)


class SlidingWindowFeature(np.lib.mixins.NDArrayOperatorsMixin):
    def __init__(self, data, sliding_window, labels=None):
        self.sliding_window, self.data, self.labels = sliding_window, data, labels
        self._i = -1

    def __len__(self):
        return self.data.shape[0]

    @property
    def extent(self):
        return self.sliding_window.range_to_segment(0, len(self))

    def __getitem__(self, i):
        return self.data[i]

    def __iter__(self):
        self._i = -1
        return self

    def __next__(self):
        self._i += 1
        try:
            return self.sliding_window[self._i], self.data[self._i]
        except IndexError:
            raise StopIteration()

    def crop(self, focus, mode="loose", fixed=None, return_data=True):
        ranges = self.sliding_window.crop(focus, mode=mode, fixed=fixed, return_ranges=True)
        n_samples = self.data.shape[0]
        clipped = []
        for start, end in ranges:
            if end < 0 or start >= n_samples:
                continue
            clipped += [[max(start, 0), min(end, n_samples)]]
        if clipped:
            data = np.vstack([self.data[start:end, :] for start, end in clipped])
        else:
            data = np.empty((0,) + self.data.shape[1:])
        if return_data:
            return data
        sw = SlidingWindow(start=self.sliding_window[clipped[0][0]].start, duration=self.sliding_window.duration,
                           step=self.sliding_window.step)
        return SlidingWindowFeature(data, sw, labels=self.labels)

    _HANDLED_TYPES = (np.ndarray, numbers.Number)

    def __array__(self, dtype=None, copy=None):
        return self.data

    def __array_ufunc__(self, ufunc, method, *inputs, **kwargs):
        out = kwargs.get("out", ())
        for x in inputs + out:
            if not isinstance(x, self._HANDLED_TYPES + (SlidingWindowFeature,)):
                return NotImplemented
        inputs = tuple(x.data if isinstance(x, SlidingWindowFeature) else x for x in inputs)
        if out:
            kwargs["out"] = tuple(x.data if isinstance(x, SlidingWindowFeature) else x for x in out)
        data = getattr(ufunc, method)(*inputs, **kwargs)
        if type(data) is tuple:
            return tuple(type(self)(x, self.sliding_window) for x in data)
        if method == "at":
            return None
        return type(self)(data, self.sliding_window)


class Annotation:
    """(segment, track) -> label, iterated in (start, end, track) order; empty segments are not stored."""

    def __init__(self, uri=None, modality=None):
        self.uri, self._tracks = uri, {}

    def __setitem__(self, key, label):
        segment, track = key
        if not segment:
            return
        self._tracks[(segment.start, segment.end, track)] = label

    def __delitem__(self, key):
        segment, track = key
        del self._tracks[(segment.start, segment.end, track)]

    def itertracks(self, yield_label=False):
        for (s, e, t) in sorted(self._tracks, key=lambda k: (k[0], k[1], str(k[2]))):
            yield (Segment(s, e), t, self._tracks[(s, e, t)]) if yield_label else (Segment(s, e), t)

    def labels(self):
        return sorted(set(self._tracks.values()), key=str)

    def rename_labels(self, mapping=None, generator="string", copy=True):
        renamed = Annotation(uri=self.uri)
        renamed._tracks = {key: mapping.get(label, label) for key, label in self._tracks.items()}
        return renamed

    def __bool__(self):
        return len(self._tracks) > 0


class Timeline:
    pass


def string_generator():
    import itertools
    import string

    r = 1
    while True:
        for c in itertools.product(string.ascii_uppercase, repeat=r):
            yield "".join(c)
        r += 1


def pairwise(iterable):
    import itertools

    a, b = itertools.tee(iterable)
    next(b, None)
    return zip(a, b)


# ---------------------------------------------------------------------------------------------------------------
# loading the reference files by path
# ---------------------------------------------------------------------------------------------------------------
class _Anything:
    """Inert class: any construction / call / attribute works (base classes, decorators' arguments, parameters)."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return self

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Anything()


class _Stub(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        cls = type(name, (_Anything,), {})
        setattr(self, name, cls)
        return cls


def stub(name):
    if name not in sys.modules:
        m = _Stub(name)
        m.__path__ = []
        sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent:
        setattr(stub(parent), child, sys.modules[name])
    return sys.modules[name]


def load(modname, relpath):
    spec = importlib.util.spec_from_file_location(modname, os.path.join(SPA, relpath))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[modname] = mod
    parent, _, child = modname.rpartition(".")
    setattr(stub(parent), child, mod)
    spec.loader.exec_module(mod)
    return mod


def load_reference():
    for n in ["lightning", "lightning.pytorch", "lightning.pytorch.utilities", "lightning.pytorch.utilities.memory",
              "pyannote", "pyannote.audio", "pyannote.audio.core", "pyannote.audio.core.io", "pyannote.audio.core.model",
              "pyannote.audio.core.task", "pyannote.audio.core.pipeline", "pyannote.audio.utils",
              "pyannote.audio.utils.multi_task", "pyannote.audio.utils.reproducibility", "pyannote.audio.utils.hf_hub",
              "pyannote.audio.utils.permutation", "pyannote.audio.pipelines", "pyannote.audio.pipelines.utils",
              "pyannote.audio.pipelines.speaker_verification", "pyannote.audio.pipelines.utils.getter",
              "pyannote.core", "pyannote.core.utils", "pyannote.core.utils.types", "pyannote.core.utils.generators",
              "pyannote.metrics", "pyannote.metrics.diarization", "pyannote.pipeline", "pyannote.pipeline.parameter"]:
        stub(n)
    core = sys.modules["pyannote.core"]
    core.Segment, core.SlidingWindow, core.SlidingWindowFeature = Segment, SlidingWindow, SlidingWindowFeature
    core.Annotation, core.Timeline = Annotation, Timeline
    gen = sys.modules["pyannote.core.utils.generators"]
    gen.string_generator, gen.pairwise = string_generator, pairwise

    class Pipeline:                                      # pyannote.pipeline.Pipeline: plain attribute storage is enough
        def __init__(self, *a, **k):
            pass

    sys.modules["pyannote.pipeline"].Pipeline = Pipeline
    import enum

    class Resolution(enum.Enum):                         # pyannote.audio.core.task.Resolution
        FRAME = 1
        CHUNK = 2

    sys.modules["pyannote.audio.core.task"].Resolution = Resolution
    ref = {}
    ref["powerset"] = load("pyannote.audio.utils.powerset", "utils/powerset.py")
    ref["vbx"] = load("pyannote.audio.utils.vbx", "utils/vbx.py")
    ref["plda"] = load("pyannote.audio.core.plda", "core/plda.py")
    ref["multi_task"] = load("pyannote.audio.utils.multi_task", "utils/multi_task.py")
    ref["inference"] = load("pyannote.audio.core.inference", "core/inference.py")
    sys.modules["pyannote.audio"].Inference = ref["inference"].Inference
    ref["signal"] = load("pyannote.audio.utils.signal", "utils/signal.py")
    ref["diarization"] = load("pyannote.audio.pipelines.utils.diarization", "pipelines/utils/diarization.py")
    pu = sys.modules["pyannote.audio.pipelines.utils"]
    pu.SpeakerDiarizationMixin = ref["diarization"].SpeakerDiarizationMixin
    ref["clustering"] = load("pyannote.audio.pipelines.clustering", "pipelines/clustering.py")
    ref["speaker_diarization"] = load("pyannote.audio.pipelines.speaker_diarization", "pipelines/speaker_diarization.py")
    return ref


FRAMES = dict(duration=0.0619375, step=0.016875)           # PyanNet receptive field (tests/golden: rf_* vectors)
CHUNKS = dict(duration=10.0, step=1.0)


def main():
    ref = load_reference()
    Inference = ref["inference"].Inference
    Mixin = ref["diarization"].SpeakerDiarizationMixin
    out = {}
    rng = np.random.default_rng(2024)
    frames = SlidingWindow(start=0.0, **FRAMES)
    chunks = SlidingWindow(start=0.0, **CHUNKS)
    C, F, K = 7, 589, 3

    # ---- Inference.aggregate / trim (core/inference.py:498-690) ---------------------------------------------------
    scores = rng.uniform(0.0, 1.0, (C, F, K)).astype(np.float32)
    scores[2, :, 1] = np.nan                                  # a class missing in one chunk
    scores[5, 100:300, :] = np.nan
    out["agg_scores"] = scores
    for name, kw in (("plain", dict()), ("hamming", dict(hamming=True)),
                     ("warm", dict(warm_up=(1.0, 1.5), hamming=True)),          # seconds (aggregate's own unit)
                     ("skip", dict(skip_average=True, missing=0.0)), ("missing0", dict(missing=0.0))):
        res = Inference.aggregate(SlidingWindowFeature(scores.copy(), chunks), frames, **kw)
        out[f"agg_{name}"] = res.data
        out[f"agg_{name}_sw"] = np.array([res.sliding_window.start, res.sliding_window.duration, res.sliding_window.step])
    tr = Inference.trim(SlidingWindowFeature(scores.copy(), chunks), warm_up=(0.1, 0.05))
    out["trim_data_shape"] = np.array(tr.data.shape)
    out["trim_sw"] = np.array([tr.sliding_window.start, tr.sliding_window.duration, tr.sliding_window.step])

    # ---- speaker_count / to_diarization / reconstruct / to_annotation ----------------------------------------------
    # binarized segmentations with speech turns (runs), as the powerset conversion would produce
    C2 = 12
    binar = np.zeros((C2, F, K), dtype=np.float32)
    for c in range(C2):
        for k in range(K):
            t = 0
            state = rng.uniform() < 0.5
            while t < F:
                run = int(rng.integers(20, 160))
                if state:
                    binar[c, t:t + run, k] = 1.0
                state = not state
                t += run
    binar[7] = 0.0                                           # a silent chunk
    out["bin_seg"] = binar.astype(np.uint8)
    for name, wu in (("w0", (0.0, 0.0)), ("w1", (0.1, 0.1))):
        cnt = Mixin.speaker_count(SlidingWindowFeature(binar.copy(), chunks), frames, warm_up=wu)
        out[f"count_{name}"] = cnt.data
        out[f"count_{name}_sw"] = np.array([cnt.sliding_window.start, cnt.sliding_window.duration, cnt.sliding_window.step])
    count = Mixin.speaker_count(SlidingWindowFeature(binar.copy(), chunks), frames, warm_up=(0.0, 0.0))
    hard = rng.integers(0, 4, (C2, K)).astype(np.int8)
    hard[binar.sum(axis=1) == 0] = -2                        # inactive speakers (speaker_diarization.py:720)
    hard[3, 1] = hard[3, 0]                                   # two local speakers in one cluster
    out["rec_hard"] = hard
    SD = ref["speaker_diarization"].SpeakerDiarization

    class _Self:
        to_diarization = staticmethod(Mixin.to_diarization)

    for name, cmax in (("full", None), ("cap1", 1)):
        cnt = SlidingWindowFeature(count.data.copy(), count.sliding_window)
        if cmax is not None:
            cnt.data = np.minimum(cnt.data, cmax).astype(np.int8)            # speaker_diarization.py:735,744
        disc = SD.reconstruct(_Self(), SlidingWindowFeature(binar.copy(), chunks), hard, cnt)
        out[f"rec_{name}"] = disc.data
        out[f"rec_{name}_sw"] = np.array([disc.sliding_window.start, disc.sliding_window.duration, disc.sliding_window.step])
        ann = Mixin.to_annotation(disc, min_duration_on=0.0, min_duration_off=0.0)
        rows = [(seg.start, seg.end, float(lab)) for seg, _, lab in ann.itertracks(yield_label=True)]
        out[f"ann_{name}"] = np.array(rows, dtype=np.float64).reshape(-1, 3)
    # Binarize with hysteresis on float scores (utils/signal.py:254-318), no padding / no min durations
    tt = np.arange(600)[:, None]
    fl = 0.5 + 0.42 * np.sin(2 * np.pi * tt / np.array([[83.0, 47.0]]) + np.array([[0.3, 1.1]])) \
        + 0.09 * rng.standard_normal((600, 2))            # crosses both thresholds, with chatter in between
    out["binz_scores"] = fl
    b = ref["signal"].Binarize(onset=0.6, offset=0.4)
    ann = b(SlidingWindowFeature(fl, frames))
    out["binz_rows"] = np.array([(seg.start, seg.end, float(lab)) for seg, _, lab in ann.itertracks(yield_label=True)],
                                dtype=np.float64).reshape(-1, 3)
    out["set_num_speakers"] = np.array([[np.nan if v is None else float(v) for v in Mixin.set_num_speakers(*a)]
                                        for a in ((None, None, None), (3, None, None), (None, 2, 5), (None, 4, 4))])

    # ---- clustering (pipelines/clustering.py) ----------------------------------------------------------------------
    from pyannote_audio_b200 import synthetic as syn

    plda_arrays = syn.make_plda(2)
    with tempfile.TemporaryDirectory() as td:
        np.savez(os.path.join(td, "xvec_transform.npz"), mean1=plda_arrays["mean1"], mean2=plda_arrays["mean2"],
                 lda=plda_arrays["lda"])
        np.savez(os.path.join(td, "plda.npz"), mu=plda_arrays["mu"], tr=plda_arrays["tr"], psi=plda_arrays["psi"])
        plda = ref["plda"].PLDA(os.path.join(td, "xvec_transform.npz"), os.path.join(td, "plda.npz"))
    # 3 speakers x 2 sessions each: centroid linkage at 0.6 finds the 6 sessions, VBx merges them into 3 speakers
    Cc = 100
    rng = np.random.default_rng(7)
    seg = np.zeros((Cc, F, K), dtype=np.float32)
    for c in range(Cc):
        for k in range(K):
            if rng.uniform() < 0.75:
                a = int(rng.integers(0, 400))
                seg[c, a:a + int(rng.integers(40, 189)), k] = 1.0
    seg[11] = 0.0
    spk = rng.standard_normal((3, 256))
    sessions = spk[:, None, :] + 0.6 * rng.standard_normal((3, 2, 256))
    which, sess = rng.integers(0, 3, (Cc, K)), rng.integers(0, 2, (Cc, K))
    emb = (sessions[which, sess] + 0.3 * rng.standard_normal((Cc, K, 256))).astype(np.float32)
    emb[5, 2] = np.nan                                        # an embedding the extractor could not compute
    out["cl_seg"], out["cl_emb"] = seg.astype(np.uint8), emb      # float32 values; the pipeline hands float64 arrays over
    emb = emb.astype(np.float64)
    segs = SlidingWindowFeature(seg.copy(), chunks)
    cl = ref["clustering"]
    vbx = cl.VBxClustering(plda)
    vbx.threshold, vbx.Fa, vbx.Fb = 0.6, 0.07, 0.8
    tr_, ci, si = vbx.filter_embeddings(emb.copy(), segmentations=segs)
    out["cl_filter_chunk"], out["cl_filter_speaker"] = ci, si
    for name, kw in (("auto", dict(num_clusters=None, min_clusters=1, max_clusters=np.inf)),
                     ("forced2", dict(num_clusters=2, min_clusters=2, max_clusters=2)),
                     ("max2", dict(num_clusters=None, min_clusters=1, max_clusters=2)),
                     ("min5", dict(num_clusters=None, min_clusters=5, max_clusters=np.inf))):
        h, s_, c_ = vbx(emb.copy(), segmentations=SlidingWindowFeature(seg.copy(), chunks), **kw)
        out[f"vbx_{name}_hard"], out[f"vbx_{name}_soft"], out[f"vbx_{name}_centroids"] = h, s_, c_
    # float32 embeddings, as get_embeddings hands them over (speaker_diarization.py:461-478): the row normalisation
    # before the linkage then happens in float32
    h, s_, c_ = vbx(out["cl_emb"].copy(), segmentations=SlidingWindowFeature(seg.copy(), chunks), num_clusters=None,
                    min_clusters=1, max_clusters=np.inf)
    out["vbx_f32_hard"], out["vbx_f32_soft"], out["vbx_f32_centroids"] = h, s_, c_
    soft = rng.standard_normal((9, 3, 5))
    soft[4, 1, 2] = np.nan
    out["carg_soft"] = soft
    out["carg_hard"] = vbx.constrained_argmax(soft.copy())
    ahc = cl.AgglomerativeClustering(metric="cosine")
    ahc.threshold, ahc.method, ahc.min_cluster_size = 0.7, "centroid", 4
    for name, kw in (("auto", dict(num_clusters=None, min_clusters=None, max_clusters=None)),
                     ("forced3", dict(num_clusters=3)), ("min5", dict(min_clusters=5, max_clusters=20))):
        h, s_, c_ = ahc(emb.copy(), segmentations=SlidingWindowFeature(seg.copy(), chunks), **kw)
        out[f"ahc_{name}_hard"], out[f"ahc_{name}_soft"], out[f"ahc_{name}_centroids"] = h, s_, c_
    # ---- Audio (core/io.py): in-memory waveforms through __call__ / crop / downmix_and_resample ---------------------
    import torch

    io_mod = load("pyannote.audio.core.io", "core/io.py")
    g = torch.Generator().manual_seed(5)
    stereo = torch.rand(2, 24000, generator=g) * 2 - 1
    hi = torch.rand(1, 22050, generator=g) * 2 - 1                    # 0.5 s at 44.1 kHz
    # the test draws the same stereo input from the seed (stored, it would push the file over 1 MB); its first samples
    # and its sum are kept to show that it does
    out["io_stereo_head"], out["io_stereo_sum"] = stereo[:, :64].numpy(), np.array(stereo.double().sum().item())
    out["io_hi"] = hi.numpy()
    A = io_mod.Audio
    w, sr = A(sample_rate=16000, mono="downmix")({"waveform": stereo, "sample_rate": 16000})
    out["io_downmix"] = w.numpy()
    w, sr = A(sample_rate=16000, mono="downmix")({"waveform": stereo, "sample_rate": 16000, "channel": 1})
    out["io_channel1"] = w.numpy()
    w, sr = A(sample_rate=16000, mono="downmix")({"waveform": hi, "sample_rate": 44100})
    out["io_resampled"], out["io_resampled_sr"] = w.numpy(), np.array(sr)
    w, sr = A(sample_rate=8000, mono="downmix")({"waveform": stereo, "sample_rate": 16000})
    out["io_half_rate"] = w.numpy()
    for name, (a, b), mode in (("in", (0.2, 0.7), "raise"), ("pad_end", (1.2, 2.0), "pad"), ("pad_start", (-0.25, 0.5), "pad")):
        w, sr = A(sample_rate=16000, mono="downmix").crop({"waveform": stereo, "sample_rate": 16000}, Segment(a, b), mode=mode)
        out[f"io_crop_{name}"] = w.numpy()
    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_pipeline_vectors.npz")
    np.savez_compressed(dst, **out)
    print(f"wrote {dst}: {len(out)} arrays, {os.path.getsize(dst) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()

"""CPU: pins the oracle restatement against (a) vectors produced by the reference's own source files
(tests/golden/reference_vectors.npz, generator tests/golden/make_golden.py) and (b) the literal known-answer
vectors of the reference's own tests (cited per test)."""
import numpy as np
import torch

from oracle import nets, pipeline as P
from pyannote_audio_b200 import synthetic as syn


def test_stats_pool_matches_reference_module(golden):
    x = torch.from_numpy(golden["sp_x"])
    np.testing.assert_allclose(nets.stats_pool(x).numpy(), golden["sp_y_none"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(nets.stats_pool(x, torch.from_numpy(golden["sp_w2"])).numpy(), golden["sp_y_w2"],
                               rtol=0, atol=1e-6)
    np.testing.assert_allclose(nets.stats_pool(x, torch.from_numpy(golden["sp_w3"])).numpy(), golden["sp_y_w3"],
                               rtol=0, atol=1e-6)


def _r4(t):
    return torch.round(t, decimals=4)


def test_stats_pool_known_answers():
    # /root/reference/tests/test_stats_pool.py:28-63, 111-131
    x = torch.Tensor([[[2.0, 4.0], [2.0, 4.0]], [[1.0, 1.0], [1.0, 1.0]]])
    assert torch.equal(_r4(nets.stats_pool(x)), torch.Tensor([[3.0, 3.0, 1.4142, 1.4142], [1.0, 1.0, 0.0, 0.0]]))
    w = torch.Tensor([[0.5, 0.01], [0.2, 0.1]])
    assert torch.equal(_r4(nets.stats_pool(x, w)),
                       torch.Tensor([[2.0392, 2.0392, 1.4142, 1.4142], [1.0, 1.0, 0.0, 0.0]]))
    w0 = torch.zeros(2, 2)
    assert torch.equal(_r4(nets.stats_pool(x, w0)), torch.zeros(2, 4))


def test_powerset_matches_reference_module(golden):
    m = nets.powerset_mapping(3, 2)
    assert np.array_equal(m.numpy(), golden["ps_mapping"])
    ml = nets.powerset_to_multilabel(torch.from_numpy(golden["ps_logits"]), m)
    assert np.array_equal(ml.numpy(), golden["ps_multilabel"])


def test_powerset_roundtrip():
    # /root/reference/tests/utils/test_powerset.py:29-51 (3 classes, max 2): multilabel -> powerset -> multilabel
    m = nets.powerset_mapping(3, 2)
    for k in range(7):
        onehot = torch.zeros(1, 1, 7)
        onehot[0, 0, k] = 1.0
        assert torch.equal(nets.powerset_to_multilabel(torch.log(onehot + 1e-9), m)[0, 0], m[k])


def test_receptive_field_matches_reference_module(golden):
    K, S, Pd, D = nets.SINCNET_K, nets.SINCNET_S, nets.SINCNET_P, nets.SINCNET_D
    got = [nets.multi_conv_num_frames(n, K, S, Pd, D) for n in (160000, 32000, 80000, 991, 1261)]
    assert got == list(golden["rf_num_frames"])
    assert [nets.multi_conv_receptive_field_size(n, K, S, Pd, D) for n in (1, 2, 589)] == list(golden["rf_size"])
    assert [nets.multi_conv_receptive_field_center(f, K, S, Pd, D) for f in (0, 1, 588)] == list(golden["rf_center"])
    # tutorials/applying_a_model.ipynb:406: (1,1,160000) -> (1,60,589); frame step 270 samples, size 991
    assert nets.sincnet_num_frames(160000) == 589
    start, dur, step = nets.sincnet_receptive_field()
    assert (start, dur, step) == (0.0, 991 / 16000, 270 / 16000)


def test_vbx_matches_reference_module(golden):
    gamma, pi = P.cluster_vbx(golden["vbx_ahc"], golden["vbx_fea"], golden["vbx_phi"], Fa=0.07, Fb=0.8, maxIters=20)
    np.testing.assert_allclose(gamma, golden["vbx_gamma"], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(pi, golden["vbx_pi"], rtol=1e-12, atol=1e-14)


def test_plda_matches_reference_module(golden):
    from threadpoolctl import threadpool_limits

    # one BLAS thread, as the vectors were made (tests/golden/make_golden.py): the setup's inverses and generalised
    # eigh round differently with the number of threads
    with threadpool_limits(limits=1):
        plda = P.PLDA(**syn.make_plda(2))
        out = plda(golden["plda_in"])
    np.testing.assert_allclose(out, golden["plda_out"], rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(plda.phi, golden["plda_psi"][:128], rtol=1e-12)


def test_resnet_matches_reference_module(golden):
    net = nets.WeSpeakerResNet34()
    net.load_state_dict(syn.make_embedding_state_dict(1))
    net.eval()
    with torch.inference_mode():
        e = net.resnet(torch.from_numpy(golden["rn_fbank"]), weights=torch.from_numpy(golden["rn_weights"]))
        e0 = net.resnet(torch.from_numpy(golden["rn_fbank"]))
    np.testing.assert_allclose(e.numpy(), golden["rn_emb"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(e0.numpy(), golden["rn_emb_noweights"], rtol=0, atol=2e-5)


def test_agglomerative_known_answer():
    # /root/reference/tests/test_clustering.py:6-29 (issue 1525)
    emb = np.array([[1.0, 1.0, 1.0, 1.0], [1.0, 2.0, 1.0, 2.0]])
    clusters = P.ahc_cluster(emb, method="centroid", threshold=0.0, min_cluster_size=0, min_clusters=2,
                             max_clusters=2, num_clusters=2)
    assert np.array_equal(clusters, np.array([0, 1]))


def test_slide_plumbing_config0():
    """BASELINE.json configs[0]: Inference.slide on one 30 s waveform, CPU -> (21, 589, 3) in {0,1}."""
    seg = nets.PyanNet()
    seg.load_state_dict(syn.make_segmentation_state_dict(0))
    seg.eval()
    wav = syn.make_conversation(30.0, seed=3)
    out = P.slide(seg, wav)
    assert out.data.shape == (21, 589, 3)
    assert set(np.unique(out.data)) <= {0.0, 1.0}
    frames = P.SW(*nets.sincnet_receptive_field())
    count = P.speaker_count(out, frames)
    # 30 s -> closest_frame(10 + 20 + 0.5*dur) + 1 frames
    assert len(count.data) == frames.closest_frame(30.0 + 0.5 * frames.duration) + 1
    sf = P.chunk_start_frames(21, frames)
    assert sf[0] == 0 and sf[1] == 59 and sf[20] == 1185


def test_to_diarization_tie_rule_only_differs_from_numpy_default_on_ties():
    """np.argsort's default kind is not stable on every host (SURVEY.md Appendix A): the reference's top-`count`
    selection is ambiguous exactly where cluster activations tie at the selection boundary.  The oracle pins
    "descending activation, then ascending cluster index"; check that numpy's default order on THIS host agrees with
    it everywhere except at such ties (a reference ambiguity, not a parity failure)."""
    rng = np.random.default_rng(0)
    seg = (rng.uniform(size=(12, 589, 3)) < 0.4).astype(np.float64)
    hard = rng.integers(0, 4, size=(12, 3)).astype(np.int8)
    frames = P.SW(*nets.sincnet_receptive_field())
    swf = P.SWF(seg, P.SW(0.0, 10.0, 1.0))
    count = P.speaker_count(swf, frames)
    count.data = np.minimum(count.data, 3).astype(np.int8)
    a = P.reconstruct(swf, hard, count)
    clustered = np.nan * np.zeros((12, 589, 4))
    for c in range(12):
        for k in np.unique(hard[c]):
            clustered[c, :, k] = np.max(seg[c][:, hard[c] == k], axis=1)
    cl = P.SWF(clustered, swf.sw)
    b = P.to_diarization(cl, count, stable=False)
    act = P.aggregate(P.SWF(clustered.copy(), swf.sw), count.sw, hamming=False, missing=0.0, skip_average=True).data
    diff = np.nonzero((a.data != b.data).any(axis=1))[0]
    for t in diff:
        c = int(count.data[t, 0])
        srt = np.sort(act[t])[::-1]
        assert 0 < c < len(srt) and srt[c - 1] == srt[c], f"frame {t}: outputs differ without a boundary tie"
        assert a.data[t].sum() == b.data[t].sum() == c


def test_oracle_reports_assignment_scores():
    """OracleOutput.soft_clusters (used by the GPU parity tests to tell near-ties of the constrained assignment from
    real differences) is consistent with hard_clusters: every assigned (chunk, speaker) picks a valid cluster and the
    oracle's own choice is optimal under its scores."""
    import itertools

    from oracle import pipeline as P
    rng = np.random.default_rng(5)
    emb = rng.standard_normal((9, 3, 256)).astype(np.float32)
    emb[:, :2] += 4.0 * rng.standard_normal((1, 1, 256)).astype(np.float32)      # two similar speakers per chunk
    seg = (rng.random((9, 589, 3)) > 0.4).astype(np.float32)
    from pyannote_audio_b200 import synthetic as syn
    hard, soft, _ = P.vbx_clustering(emb, seg, P.PLDA(**syn.make_plda(2)), 0.6, 0.07, 0.8, num_clusters=None,
                                     min_clusters=1, max_clusters=np.inf)
    assert soft.shape[:2] == hard.shape and soft.shape[2] >= int(hard.max()) + 1
    K = soft.shape[2]
    for c in range(hard.shape[0]):
        got = sum(soft[c, s, k] for s, k in enumerate(hard[c]) if k >= 0)
        best = max(sum(soft[c, s, k] for s, k in zip(sp, ks))
                   for n in range(1, min(3, K) + 1)
                   for sp in itertools.permutations(range(3), n) for ks in itertools.combinations(range(K), n))
        assert got >= best - 1e-9

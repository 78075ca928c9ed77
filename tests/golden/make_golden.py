"""Generates tests/golden/reference_vectors.npz by EXECUTING the reference's own source files where they lie under
/root/reference (oracle/ref_loader.py) -- run once in the build container:

    PYTHONPATH=. python tests/golden/make_golden.py

Nothing here is needed at test time; the committed .npz is.  (The reference package as a whole cannot be imported
in this environment, see SURVEY.md section 8c; these five leaf modules can.)
"""
import numpy as np
import torch

from oracle import ref_loader
from pyannote_audio_b200 import synthetic as syn

ref = ref_loader.load_all()
out = {}
g = torch.Generator().manual_seed(123)

# ---- StatsPool (models/blocks/pooling.py) -------------------------------------------------------------------
sp = ref["pooling"].StatsPool()
x = torch.randn(3, 7, 11, generator=g)
w2 = torch.rand(3, 5, generator=g)
w3 = (torch.rand(3, 2, 5, generator=g) > 0.4).float()
out["sp_x"], out["sp_w2"], out["sp_w3"] = x.numpy(), w2.numpy(), w3.numpy()
out["sp_y_none"] = sp(x).numpy()
out["sp_y_w2"] = sp(x, weights=w2).numpy()
out["sp_y_w3"] = sp(x, weights=w3).numpy()

# ---- Powerset (utils/powerset.py) ---------------------------------------------------------------------------
ps = ref["powerset"].Powerset(3, 2)
out["ps_mapping"] = ps.mapping.numpy()
logits = torch.randn(4, 50, 7, generator=g)
out["ps_logits"] = logits.numpy()
out["ps_multilabel"] = ps.to_multilabel(logits).numpy()

# ---- receptive field arithmetic (utils/receptive_field.py) ----------------------------------------------------
rf = ref["receptive_field"]
K, S, P, D = [251, 3, 5, 3, 5, 3], [10, 3, 1, 3, 1, 3], [0] * 6, [1] * 6
out["rf_num_frames"] = np.array([rf.multi_conv_num_frames(n, K, S, P, D) for n in (160000, 32000, 80000, 991, 1261)])
out["rf_size"] = np.array([rf.multi_conv_receptive_field_size(n, K, S, P, D) for n in (1, 2, 589)])
out["rf_center"] = np.array([rf.multi_conv_receptive_field_center(f, K, S, P, D) for f in (0, 1, 588)])

# ---- VBx (utils/vbx.py) ----------------------------------------------------------------------------------------
rng = np.random.default_rng(5)
n, Dd, S0 = 60, 16, 5
fea = rng.standard_normal((n, Dd)) + 3.0 * rng.standard_normal((3, Dd))[rng.integers(0, 3, n)]
phi = np.sort(np.exp(rng.uniform(np.log(0.1), np.log(10.0), Dd)))[::-1].copy()
ahc = rng.integers(0, S0, n)
gamma, pi = ref["vbx"].cluster_vbx(ahc, fea, phi, Fa=0.07, Fb=0.8, maxIters=20)
out["vbx_fea"], out["vbx_phi"], out["vbx_ahc"], out["vbx_gamma"], out["vbx_pi"] = fea, phi, ahc, gamma, pi
plda = syn.make_plda(2)
import tempfile, os
from threadpoolctl import threadpool_limits

# the PLDA setup (inverses, generalised eigh) rounds differently with the number of BLAS threads: one thread here and
# in tests/test_oracle_golden.py, so that the comparison does not depend on the host's core count
with tempfile.TemporaryDirectory() as td, threadpool_limits(limits=1):
    np.savez(os.path.join(td, "xvec_transform.npz"), mean1=plda["mean1"], mean2=plda["mean2"], lda=plda["lda"])
    np.savez(os.path.join(td, "plda.npz"), mu=plda["mu"], tr=plda["tr"], psi=plda["psi"])
    xvec_tf, plda_tf, plda_psi = ref["vbx"].vbx_setup(os.path.join(td, "xvec_transform.npz"),
                                                      os.path.join(td, "plda.npz"))
    emb = rng.standard_normal((7, 256))
    out["plda_in"] = emb
    out["plda_out"] = plda_tf(xvec_tf(emb), lda_dim=128)
    out["plda_psi"] = plda_psi

# ---- ResNet34 trunk + TSTP + seg_1 (models/embedding/wespeaker/resnet.py) --------------------------------------
net = ref["resnet"].ResNet34(80, 256, pooling_func="TSTP", two_emb_layer=False)
sd = {k[len("resnet."):]: v for k, v in syn.make_embedding_state_dict(1).items()}
net.load_state_dict(sd, strict=True)
net.eval()
fb = torch.randn(2, 120, 80, generator=g)
wts = (torch.rand(2, 589, generator=g) > 0.5).float()
with torch.inference_mode():
    out["rn_fbank"], out["rn_weights"] = fb.numpy(), wts.numpy()
    out["rn_emb"] = net(fb.clone(), weights=wts)[1].numpy()
    out["rn_emb_noweights"] = net(fb.clone())[1].numpy()

np.savez_compressed("tests/golden/reference_vectors.npz", **out)
print({k: v.shape for k, v in out.items()})

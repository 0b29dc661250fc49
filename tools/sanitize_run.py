"""Small end-to-end run for compute-sanitizer: every kernel of the library on small inputs."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, pandas as pd, torch
import __graft_entry__ as g
g.build()
import muscle_synergies_b200 as ms
from muscle_synergies_b200.segment import Segmenter
from muscle_synergies_b200.pipeline import trial_synergies
from muscle_synergies_b200 import analysis, emg
from tools.synth_vicon import synth_layout

golden = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
data = ms.load_vicon_file(os.path.join(golden, "abridged_data.csv"))
print("abridged", data.emg.df.shape)
for name in sorted(os.listdir(os.path.join(golden, "variants")))[:40]:
    try:
        ms.load_vicon_file(os.path.join(golden, "variants", name))
    except Exception as exc:  # noqa: BLE001 - the variants include malformed files
        pass
blob = synth_layout("D", seed=0)
loader = ms.ViconLoader()
d = torch.empty(loader.padded_size(blob.nbytes), dtype=torch.uint8, device="cuda")
d[: blob.nbytes].copy_(torch.from_numpy(blob))
trial = loader.load_device(d, n=blob.nbytes, name="D", defer_check=True)
seg = Segmenter(trial, cut_phases_of=(trial.emg, trial.traj[0]))
print("transitions", len(seg.transitions), "cuts", len(seg.phase_cuts(trial.emg)))
res = trial_synergies(trial, 1, 5, n_restarts=2, max_iter=20, segmenter=seg)
print("pipeline", len(res.cycles))
x = np.abs(np.random.default_rng(0).normal(size=(3000, 6)))
analysis.nmf_mu_batched(x, [2, 3, 4], [0, 1, 2], max_iter=10, regime="stream")
analysis.nmf_cd_batched(x, [2, 3, 4], init="nndsvda", max_iter=10, regime="stream")
analysis.nmf_cd_batched(np.stack([x[:300], x[300:600]]), [1, 3, 6], init="nndsvd", x_index=[0, 1, 1], max_iter=10)
analysis.nmf_transform_batched(x, [np.ones((2, 6)), np.ones((4, 6))], solver="cd", max_iter=10, regime="stream")
analysis.nmf_transform_batched(x[:300], [np.ones((3, 6))], solver="mu", max_iter=30, regime="resident")
analysis.nmf_beta_batched(x, [2, 3, 4], "kullback-leibler", max_iter=25, tol=1e-4, regime="stream")
analysis.nmf_beta_batched(x[:300] + 0.01, [1, 3, 6], "itakura-saito", init="random", seeds=[0, 1, 2], max_iter=25)
analysis.nmf_beta_batched(x[:300], [2, 5], 1.5, max_iter=25, tol=1e-4, regime="resident")
analysis.nmf_transform_batched(x + 0.01, [np.ones((2, 6))], solver="mu", max_iter=25, regime="stream", beta_loss=0.5)
res = trial_synergies(trial, 1, 3, max_iter=20, segmenter=seg, solver="cd")
analysis.match_synergies_batched([np.ones((3, 6)), x[:3, :], x[3:5, :], x[5:7, :]], [[0, 1], [2, 3], [1, 1]], similarities=True, permutations=True)
df = pd.DataFrame(x, columns=list("abcdef"))
emg.linear_envelope(df, 6.0, 2000, 4); emg.rms(df, 100); emg.digital_filter(df, (20.0, 450.0), 2000, 2, band_type="bandpass", zero_lag=False)
torch.cuda.synchronize()
print("sanitize run done")

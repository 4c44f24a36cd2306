"""Generate tests/golden/a2h_*.npz from the UNMODIFIED reference (models/audio2headpose_model.py) - run in the container
that has /root/reference.  The fixture stores the reference loop's output and Sample_GMM's draws; weights and audio
features are regenerated from seeds (oracle/a2h_oracle.py), so the file stays small.

    PYTHONDONTWRITEBYTECODE=1 python oracle/make_golden_a2h.py
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from oracle import a2h_oracle as A  # noqa: E402


def main():
    torch.set_num_threads(8)          # tests/test_a2h_oracle.py GOLDEN_THREADS: the loop's last bits depend on it
    opt = A.default_opt()
    recipe, wseed, aseed, tseed, n_audio, sigma = "B", 0, 1, 5, 60, 0.3
    sd = A.make_state_dict(opt, recipe, wseed)
    m = A.reference_model(opt, sd)
    audio = A.make_audio_feats(n_audio, opt, aseed)
    pre = np.linspace(-0.25, 0.35, 12).astype(np.float32)
    noise = A.reference_noise(n_audio - opt.frame_future, opt.A2H_GMM_ndim, opt.A2H_GMM_ncenter, tseed)
    torch.manual_seed(tseed)
    with contextlib.redirect_stderr(io.StringIO()):
        pred = m.generate_sequences(audio.copy(), pre, fill_zero=True, sigma_scale=sigma, opt=opt)
    mine, params = A.generate_sequences(sd, audio, pre, noise, opt, sigma, return_params=True)
    assert np.abs(pred - mine).max() <= 1e-6, "restatement disagrees with the reference"
    out = os.path.join(ROOT, "tests", "golden", "a2h_B_60.npz")
    np.savez_compressed(out, recipe=recipe, weight_seed=wseed, audio_seed=aseed, torch_seed=tseed, n_audio=n_audio,
                        sigma_scale=sigma, pre_headpose=pre, noise=noise, pred=pred, params=params)
    print("wrote", out, "pred", pred.shape, "max|ref - restatement|", np.abs(pred - mine).max())


if __name__ == "__main__":
    main()

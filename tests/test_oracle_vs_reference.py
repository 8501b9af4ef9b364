"""CPU: the oracle against outputs of the unmodified reference (model.py, loss_function.py, stft.py) stored under
tests/golden by tools/make_golden.py refs."""
import numpy as np
import torch

from oracle import tacotron2_oracle as O
from tests.common import keep_mask, rand_text, rel_err, stft_inputs, synth_state_dict, weights_checksum
from tests.test_oracle_golden import check_grads_vs_fixture, grad_inputs, load, oracle_train_step

STFT_SETTINGS = ((1024, 256, 1024), (800, 200, 800), (512, 128, 400))     # (filter_length, hop_length, win_length)


def test_reference_inference_b1_live():
    """The reference's own Tacotron2.inference at B=1 (its stop loop, 12 steps, injected prenet masks)."""
    g = load("ref_inference_b1_t19")
    sd = synth_state_dict(5, gate_bias=-10.0, scale=2.0)
    assert abs(weights_checksum(sd) - float(g["wsum"])) < 1e-6 * float(g["wsum"]), "weight generator drifted"
    text = rand_text(1, 19, 3); keep = keep_mask((12, 2, 1, 256), 0.5, 4)
    with torch.no_grad():
        mel, post, gate, align, lengths = O.tacotron2_inference(sd, text, keep, 0.5, 12)
    assert int(lengths[0]) == g["mel"].shape[2] == 12
    for a, k in zip((mel, post, gate, align), ("mel", "mel_post", "gate", "align")):
        assert rel_err(a, torch.from_numpy(g[k])) < 2e-5, k


def test_reference_state_dict_layout():
    """The 84 keys / shapes the boundary must reproduce (SURVEY.md section 8(b1))."""
    from tests.common import state_dict_shapes
    g = load("ref_init_seed1234")
    want = state_dict_shapes()
    assert g["keys"].tolist() == list(want.keys())
    for k, s in zip(g["keys"].tolist(), g["shapes"].tolist()):
        assert tuple(int(n) for n in s.split(",") if n) == tuple(want[k]), k


def test_reference_training_step_gradients_live():
    """Full training step (forward + Tacotron2Loss + backward) of the unmodified reference vs torch autograd through
    the oracle: the loss, and per parameter the gradient's sum / abs-sum / max and 512 sampled entries."""
    g = load("grad_train_b3_t15_m8")
    sd, text, tl, ol, mels, gt, m = grad_inputs(g)
    o_loss, _, o_grads = oracle_train_step(sd, text, tl, ol, mels, gt, m, True)
    assert abs(float(g["loss"]) - float(o_loss)) < 1e-5 * abs(float(g["loss"]))
    assert set(o_grads) == {k[2:] for k in g if k.startswith("g/")}
    check_grads_vs_fixture(o_grads, g, 1e-4)


def test_stft_oracle_vs_reference_stft_live():
    """oracle/stft_oracle.py against the reference's own stft.STFT (functional stand-ins for the two librosa.util helpers
    stft.py imports): the windowed Fourier basis and the magnitudes for three filter / hop settings."""
    from oracle import stft_oracle as S
    g = load("stft_mag_settings")
    for fl, hop, win in STFT_SETTINGS:
        basis = torch.from_numpy(S.stft_forward_basis(fl, win)).reshape(-1)
        idx = torch.from_numpy(g["basis_index_%d" % fl]).long()
        assert float((basis[idx] - torch.from_numpy(g["basis_%d" % fl])).abs().max()) < 1e-6
        abs_sum = float(g["basis_abs_sum_%d" % fl])
        assert abs(float(np.abs(S.stft_forward_basis(fl, win)).sum(dtype=np.float64)) - abs_sum) < 1e-6 * abs_sum
        y = stft_inputs(seed=fl, n=5000)
        assert rel_err(S.stft_magnitude(y, fl, hop, win), torch.from_numpy(g["mag_%d" % fl])) < 1e-6

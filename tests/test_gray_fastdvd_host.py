"""CPU: the derived grayscale FastDVDnet loop ('fastdvd_gray') - its oracle's use of the global numpy RNG, the lr = 0
fine-tune, the write-back of the colour-shaped twin into the gray model, and the size check of the solver."""
import numpy as np
import pytest
import torch


def _oracle_model():
    from oracle import networks, synthetic
    m = networks.Wrapped(networks.FastDVDnet(5, 1))
    m.load_state_dict({"module." + k: v for k, v in synthetic.fastdvdnet_gray_synthetic_state_dict().items()}, strict=True)
    return m.eval()


@pytest.mark.parametrize("update_times", [-1, 1])
def test_oracle_draws_one_gray_noise_array_per_update(update_times):
    """Iterations k = 0..6, updates at k = 3 and 6 (k > 1, k % 3 == 0), the second one only with update_times = -1: the loop
    leaves the global RNG where that many (B,1,H,W) draws leave it."""
    from oracle import gray_fastdvd, synthetic
    H, W, B = 16, 16, 4
    meas, mask, orig = synthetic.make_case(H, W, B, 1001, bayer=False)
    np.random.seed(11)
    gray_fastdvd.twoStageAdmm_denoise_gray(meas, mask, 'fastdvd_gray', iter_max=[5, 2], sigma=[12 / 255, 6 / 255], X_orig=orig,
                                           model_denoise=_oracle_model(), lr_=2e-6, interval_iter=3, update_=True,
                                           update_per_iter=2, update_times=update_times)
    after = np.random.get_state()
    np.random.seed(11)
    for _ in range(2 if update_times < 0 else 1):
        np.random.normal(0, 5 / 255, (B, 1, H, W))
    want = np.random.get_state()
    assert after[0] == want[0] and np.array_equal(after[1], want[1]) and after[2:] == want[2:]


def test_oracle_update_with_zero_lr_is_inference():
    from oracle import gray_fastdvd, synthetic
    H, W, B = 16, 20, 5
    meas, mask, orig = synthetic.make_case(H, W, B, 1001, bayer=False)
    x = torch.from_numpy(np.ascontiguousarray(orig, dtype=np.float32))
    y, phi = torch.from_numpy(np.ascontiguousarray(meas)), torch.from_numpy(np.ascontiguousarray(mask))
    want = gray_fastdvd.fastdvdnet_gray_denoise_full_tensor(x, y, phi, 12 / 255, _oracle_model())
    np.random.seed(5)
    got, _ = gray_fastdvd.fastdvdnet_gray_denoise_full_tensor(x, y, phi, 12 / 255, _oracle_model(), lr_=0.0, updata_=True,
                                                              update_per_iter=2)
    assert got.shape == (H, W, B)
    assert np.array_equal(got.numpy().view(np.uint32), want.numpy().view(np.uint32))


def test_twin_restriction_inverts_the_embedding():
    """Embedding the gray weights into the colour-shaped twin and restricting them back is the identity, bit for bit; a
    change of the twin (what fine-tuning does) reaches the gray parameters, and the twin is then not re-copied over itself."""
    from adaptivepnp_sci_b200 import synthetic as syn
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    sd = syn.fastdvdnet_gray_synthetic_state_dict()
    m = FastDVDnet(num_input_frames=5, num_color_channels=1)
    m.load_state_dict(sd, strict=True)
    twin = m._colour_twin()
    m._restrict_twin()
    got = m.state_dict()
    assert list(got.keys()) == list(sd.keys())
    for k, v in sd.items():
        assert got[k].numpy().tobytes() == v.numpy().tobytes(), k
    with torch.no_grad():
        twin.temp2.inc.convblock[0].weight[:, 3].add_(0.25)          # the sigma column of every frame group
        twin.temp1.outc.convblock[3].weight[0].mul_(2.0)             # the one real output row
    m._restrict_twin()
    assert torch.equal(m.temp2.inc.convblock[0].weight[:, 1], sd["temp2.inc.convblock.0.weight"][:, 1] + 0.25)
    assert torch.equal(m.temp1.outc.convblock[3].weight[0], 2.0 * sd["temp1.outc.convblock.3.weight"][0])
    snapshot = {k: v.clone() for k, v in twin.state_dict().items()}
    assert m._colour_twin() is twin
    assert all(torch.equal(v, snapshot[k]) for k, v in twin.state_dict().items())
    assert float(twin.temp1.inc.convblock[0].weight.detach()[:, 1:3].abs().max()) == 0.0


def test_solver_refuses_sizes_that_are_not_multiples_of_4():
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_gray
    y = np.zeros((30, 32), np.float32)
    with pytest.raises(ValueError, match="multiples of 4"):
        twoStageAdmm_denoise_gray(y, np.zeros((30, 32, 4), np.float32), 'fastdvd_gray', iter_max=[1], sigma=[12 / 255])

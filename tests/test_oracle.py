"""The oracle against the golden vectors produced by the reference itself
(tests/golden/make_golden.py).  CPU only."""
import pytest
import torch

from conftest import load_golden, rel_l2
from oracle import unet3d_oracle as O

CASES = ["b2_f16_8x8", "b1_f3_16x24", "b2_f2_8x8_tvec"]


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_forward(name, synthetic_sd):
    g = load_golden(name)
    taps = {}
    out = O.unet_forward(synthetic_sd, g["sample"], g["timestep"], g["text"], taps=taps)
    assert out.shape == g["out"].shape
    assert rel_l2(out, g["out"]) < 2e-5
    assert (out - g["out"]).abs().max() < 2e-4
    for k, ref in g["taps"].items():
        got = taps[k][:, ::taps[k].shape[1] // ref.shape[1]]          # the golden keeps every 8th or 16th channel
        assert got.shape == ref.shape, k
        assert rel_l2(got, ref) < 2e-5, k


def test_synthetic_weights_are_reproducible(synthetic_sd):
    from lavie_b200.synthetic import synthetic_state_dict
    again = synthetic_state_dict(seed=0)
    for k in ("conv_in.weight", "mid_block.attentions.0.transformer_blocks.0.attn_temp.to_out.0.weight"):
        assert torch.equal(again[k], synthetic_sd[k])
    # the temporal-attention output projection must not be zero, or the path is invisible
    assert synthetic_sd["mid_block.attentions.0.transformer_blocks.0.attn_temp.to_out.0.weight"].abs().max() > 0


def test_temporal_attention_is_visible(synthetic_sd):
    """Zeroing attn_temp.to_out must move the output (SURVEY.md 8c trap (i))."""
    g = load_golden("b2_f2_8x8_tvec")
    sd = dict(synthetic_sd)
    for k in list(sd):
        if k.endswith("attn_temp.to_out.0.weight"):
            sd[k] = torch.zeros_like(sd[k])
    out = O.unet_forward(sd, g["sample"], g["timestep"], g["text"])
    assert rel_l2(out, g["out"]) > 1e-3


def test_rel_pos_bucket_known_values():
    # T5 bucketing with 32 buckets / max_distance 32 (attention.py:680-698): exact below 8, log above
    rel = torch.arange(-15, 16)
    b = O.rel_pos_bucket(rel, 32, 32)
    assert b[15] == 0                      # distance 0
    assert b[14] == 1 and b[16] == 17      # k one behind q -> n=+1 ; k one ahead -> 16 + 1
    assert int(b.max()) <= 31 and int(b.min()) >= 0
    assert b[0] == 8 + int(torch.log(torch.tensor(15.0 / 8)) / torch.log(torch.tensor(4.0)) * 8)


def test_rope_is_a_rotation():
    torch.manual_seed(0)
    x = torch.randn(3, 8, 16, 40)
    freqs = 1.0 / (10000.0 ** (torch.arange(0, 32, 2).float() / 32))
    y = O.rope(x, freqs)
    assert torch.allclose(y[..., 32:], x[..., 32:])
    assert torch.allclose(y[..., :32].pow(2).sum(-1), x[..., :32].pow(2).sum(-1), rtol=1e-5, atol=1e-5)
    assert torch.allclose(y[..., 0, :], x[..., 0, :])          # position 0 is unrotated


def test_ddim_schedule_and_step():
    acp, ts, ratio = O.ddim_schedule(50)
    assert ts[0] == 981 and ts[-1] == 1 and ratio == 20 and len(ts) == 50
    x = torch.randn(1, 4, 2, 4, 4)
    eps = torch.randn_like(x)
    # if eps is the true noise of x_t = sqrt(a) x0 + sqrt(1-a) eps, a DDIM step lands on the same x0/eps pair
    x0 = torch.randn_like(x)
    t = int(ts[3])
    xt = acp[t].sqrt() * x0 + (1 - acp[t]).sqrt() * eps
    prev = O.ddim_step(eps, t, xt, acp, ratio)
    want = acp[t - ratio].sqrt() * x0 + (1 - acp[t - ratio]).sqrt() * eps
    assert torch.allclose(prev, want, atol=1e-5)


def test_ddim_step_matches_reference_scheduler():
    """O.ddim_step / O.ddim_schedule against step() of the DDIMScheduler the reference vendors
    (vsr/diffusion/scheduling_ddim.py:292-414; fixture made by tests/golden/make_golden_ddim.py)."""
    g = load_golden("ddim_steps")
    acp, ts, ratio = O.ddim_schedule(g["num_inference_steps"])
    assert torch.equal(acp, g["alphas_cumprod"])
    for c in g["cases"]:
        got = O.ddim_step(c["model_output"], c["t"], c["sample"], acp, ratio)
        assert rel_l2(got, c["prev_sample"]) < 1e-6, c["t"]

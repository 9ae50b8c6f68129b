"""The VSR stage's caller: lavie_b200.pipeline.VSRSampler (v-prediction DDIM with scaled-linear betas, noise-augmented
low-resolution frames, 8-frame chunks, chunk parallelism over a process group) against oracle/vsr_sampler_oracle.py.

CPU: the schedule algebra, the noise augmentation, the chunk plan, the noise draw order and the argument checks; the
chunked loop itself with a stand-in denoiser (and the guidance + update kernel restated in PyTorch), also spread over
gloo ranks.  GPU: the loop through the VSR denoiser against the oracle loop, chunk independence, ``upscale`` through
the x4 VAE, and chunk-parallel ``upscale`` on two GPUs."""
import math
import os
import sys
from types import SimpleNamespace

import pytest
import torch

from conftest import ROOT, rel_l2

DEV = "cuda"


# ------------------------------------------------------------------------------------------------------------------ schedules
def test_scaled_linear_alphas_cumprod():
    from lavie_b200.pipeline import LOW_RES_ALPHAS_CUMPROD, DDIMSchedule, _alphas_cumprod
    from oracle import vsr_sampler_oracle as VS
    acp = _alphas_cumprod(1000, 1e-4, 2e-2, "scaled_linear")
    betas = torch.linspace(math.sqrt(1e-4), math.sqrt(2e-2), 1000, dtype=torch.float32) ** 2
    assert torch.equal(acp, torch.cumprod(1.0 - betas, dim=0))
    assert torch.equal(acp, VS.scaled_linear_alphas_cumprod()) and torch.equal(acp, LOW_RES_ALPHAS_CUMPROD)
    assert float(acp[0]) == pytest.approx(0.99990, abs=5e-6)
    assert float(acp[50]) == pytest.approx(0.990844, abs=5e-7)
    assert float(acp[999]) == pytest.approx(7.334e-4, rel=1e-4)
    s = DDIMSchedule(50, beta_schedule="scaled_linear", prediction_type="v_prediction")
    assert torch.equal(s.alphas_cumprod, acp)
    with pytest.raises(ValueError):
        _alphas_cumprod(1000, 1e-4, 2e-2, "cosine")
    with pytest.raises(ValueError):
        DDIMSchedule(50, prediction_type="sample")


def test_ddim_defaults_unchanged():
    """DDIMSchedule() is the base pipeline's schedule: linear betas, epsilon, stock 0.16 spacing."""
    from lavie_b200.pipeline import DDIMSchedule
    s = DDIMSchedule()
    assert s.prediction_type == "epsilon"
    assert s.timesteps == [981 - 20 * i for i in range(50)]
    acp = torch.cumprod(1.0 - torch.linspace(1e-4, 2e-2, 1000, dtype=torch.float32), dim=0)
    assert torch.equal(s.alphas_cumprod, acp)
    for i in (0, 1, 17, 48, 49):
        t = s.timesteps[i]
        a_t = float(acp[t])
        a_p = float(acp[t - 20]) if t >= 20 else float(acp[0])
        want = (math.sqrt(a_p / a_t), math.sqrt(1 - a_p) - math.sqrt(a_p) * math.sqrt(1 - a_t) / math.sqrt(a_t), 0.0)
        assert s.coefficients(i) == want


def test_v_prediction_fixed_point_and_coefficients():
    """v = sqrt(a_t) eps - sqrt(1-a_t) x0 is the true velocity of x_t: one step lands on sqrt(a_p) x0 + sqrt(1-a_p) eps;
    the product's (A, B) reproduce the oracle's explicit x0 / eps step."""
    from lavie_b200.pipeline import DDIMSchedule
    from oracle import vsr_sampler_oracle as VS
    ora = VS.DDIMV(50)
    prod = DDIMSchedule(50, beta_schedule="scaled_linear", prediction_type="v_prediction")
    assert prod.timesteps == ora.timesteps
    g = torch.Generator().manual_seed(3)
    for i in (0, 1, 17, 48, 49):
        x0 = torch.randn(1, 4, 2, 4, 4, generator=g, dtype=torch.float64)
        eps = torch.randn_like(x0)
        t = ora.timesteps[i]
        a_t = ora.acp[t]
        a_p = ora.acp[t - ora.ratio] if t >= ora.ratio else ora.acp[0]
        xt = a_t.sqrt() * x0 + (1 - a_t).sqrt() * eps
        v = a_t.sqrt() * eps - (1 - a_t).sqrt() * x0
        assert rel_l2(ora.step(v, i, xt), a_p.sqrt() * x0 + (1 - a_p).sqrt() * eps) < 1e-12
        a, b, c = prod.coefficients(i)
        assert c == 0.0 and isinstance(a, float) and isinstance(b, float)
        assert rel_l2(a * xt + b * v, ora.step(v, i, xt)) < 1e-12, i


def test_explicit_timesteps():
    from lavie_b200.pipeline import DDIMSchedule
    ts = [999, 800, 500, 200, 1]
    s = DDIMSchedule(beta_schedule="scaled_linear", prediction_type="v_prediction", timesteps=ts)
    assert s.timesteps == ts and s.ratio == 200
    assert s.alphas(500) == (float(s.alphas_cumprod[500]), float(s.alphas_cumprod[300]))
    assert s.alphas(1) == (float(s.alphas_cumprod[1]), float(s.alphas_cumprod[0]))
    with pytest.raises(ValueError):
        DDIMSchedule(timesteps=[1000])
    with pytest.raises(ValueError):
        DDIMSchedule(timesteps=[])


def test_add_low_res_noise():
    from lavie_b200.pipeline import add_low_res_noise
    from oracle import vsr_sampler_oracle as VS
    g = torch.Generator().manual_seed(1)
    x, n = torch.rand(1, 3, 2, 8, 8, generator=g) * 2 - 1, torch.randn(1, 3, 2, 8, 8, generator=g)
    ab = 0.9908438324928284
    got = add_low_res_noise(x, n, 50)
    assert rel_l2(got, math.sqrt(ab) * x.double() + math.sqrt(1 - ab) * n.double()) < 1e-6
    assert torch.equal(got, VS.add_noise(x, n, 50))
    assert torch.equal(add_low_res_noise(x, n, 350), VS.add_noise(x, n, 350))
    for bad in (351, -1):
        with pytest.raises(ValueError):
            add_low_res_noise(x, n, bad)


def test_chunk_plan_and_rank_assignment():
    from lavie_b200.pipeline import chunk_plan, rank_chunks
    assert chunk_plan(16, 8) == [(0, 8), (8, 8)]
    assert chunk_plan(61, 8) == [(8 * k, 8) for k in range(7)] + [(56, 5)]
    assert chunk_plan(5, 8) == [(0, 5)]
    for F in (5, 16, 61):
        plan = chunk_plan(F, 8)
        assert sum(n for _, n in plan) == F and all(s == i * 8 for i, (s, _) in enumerate(plan))
        for P in (1, 2, 3, 8):
            owned = sorted(k for r in range(P) for k in rank_chunks(len(plan), P, r))
            assert owned == list(range(len(plan))), (F, P)
    assert rank_chunks(8, 3, 1) == [1, 4, 7]


# -------------------------------------------------------------------------------- CPU: the loop with a stand-in denoiser
class _StandIn:
    """A deterministic stand-in for UNet3DVSRModel on the CPU: its output depends on every input, the CFG half, the
    timestep and the noise level, and mixes the chunk's frames (as the frame convolutions do)."""
    device = torch.device("cpu")

    def __init__(self):
        from lavie_b200.config import VSR_CONFIG
        self.cfg = VSR_CONFIG
        self.calls = []

    def __call__(self, sample, t, low_res, encoder_hidden_states=None, class_labels=None):
        self.calls.append(tuple(sample.shape))
        return SimpleNamespace(sample=_stand_in(sample, t, low_res, encoder_hidden_states, class_labels))


def _stand_in(x, t, lr, text, labels):
    half = text.float().mean(dim=(1, 2)).reshape(-1, 1, 1, 1, 1)
    lab = torch.as_tensor(labels).float().reshape(-1, 1, 1, 1, 1)
    return (0.5 * x + 0.2 * lr.mean(1, keepdim=True) + 0.1 * x.mean(2, keepdim=True) + half
            + 1e-4 * float(t) + 1e-3 * lab).float()


def _torch_cfg_linear_step(u, c, g, a, b, x, noise=None, c_noise=0.0, out=None):
    return a * x + b * (u + g * (c - u))


@pytest.fixture
def cpu_steps(monkeypatch):
    from lavie_b200 import ops
    monkeypatch.setattr(ops, "cfg_linear_step", _torch_cfg_linear_step)


def _cpu_inputs(F=7, h=16, w=16, seed=0):
    g = torch.Generator().manual_seed(seed)
    frames = torch.randint(0, 256, (1, F, h, w, 3), generator=g, dtype=torch.uint8)
    text = torch.randn(2, 8, 1024, generator=g)
    return frames, text


def _noises_in_order(plan, h, w, seed):
    """Per chunk, in chunk order: the low-resolution noise, then the initial latents (the documented draw order)."""
    g = torch.Generator().manual_seed(seed)
    lrn, lat = [], []
    for _, n in plan:
        lrn.append(torch.randn((1, 3, n, h, w), generator=g))
        lat.append(torch.randn((1, 4, n, h, w), generator=g))
    return torch.cat(lat, dim=2), torch.cat(lrn, dim=2)


def test_loop_matches_oracle_with_stand_in(cpu_steps):
    """Chunking (4 + 3 frames), uint8 normalisation, noise augmentation, guidance and the v-prediction update against
    the oracle loop driving the same stand-in denoiser."""
    from lavie_b200.pipeline import DDIMSchedule, VSRSampler, chunk_plan
    from oracle import vsr_sampler_oracle as VS
    frames, text = _cpu_inputs()
    lat, lrn = _noises_in_order(chunk_plan(7, 4), 16, 16, seed=9)
    unet = _StandIn()
    sched = DDIMSchedule(3, beta_schedule="scaled_linear", prediction_type="v_prediction")
    assert sched.timesteps == [667, 334, 1]
    got = VSRSampler(unet, 5.0, 50, chunk_frames=4, schedule=sched).loop(frames, text, latents=lat, low_res_noise=lrn)
    assert unet.calls == [(2, 4, 4, 16, 16)] * 3 + [(2, 4, 3, 16, 16)] * 3
    low = (frames.permute(0, 4, 1, 2, 3).float() / 255 - 0.5) / 0.5
    want = VS.vsr_loop(None, low, text, lat, lrn, VS.DDIMV(3), 5.0, 50, 4, forward=_stand_in)
    assert got.shape == (1, 4, 7, 16, 16) and got.dtype == torch.float32
    assert rel_l2(got, want) < 1e-5


def test_generator_path_equals_explicit_noise(cpu_steps):
    from lavie_b200.pipeline import VSRSampler, chunk_plan
    frames, text = _cpu_inputs()
    s = VSRSampler(_StandIn(), num_inference_steps=2, chunk_frames=4)
    a = s.loop(frames, text, generator=torch.Generator().manual_seed(9))
    lat, lrn = _noises_in_order(chunk_plan(7, 4), 16, 16, seed=9)
    assert torch.equal(a, s.loop(frames, text, latents=lat, low_res_noise=lrn))
    assert not torch.equal(a, s.loop(frames, text, generator=torch.Generator().manual_seed(10)))
    # float input in [-1, 1] == the uint8 frames it was normalised from
    low = (frames.permute(0, 4, 1, 2, 3).float() / 255 - 0.5) / 0.5
    assert torch.equal(a, s.loop(low, text, latents=lat, low_res_noise=lrn))


def test_argument_checks(cpu_steps):
    from lavie_b200.pipeline import DDPMSchedule, VSRSampler
    frames, text = _cpu_inputs(F=3)
    s = VSRSampler(_StandIn(), num_inference_steps=1)
    low = torch.zeros(1, 3, 3, 16, 16)
    bad = [
        lambda: s.loop(torch.zeros(2, 3, 3, 16, 16), torch.cat([text, text])[:2]),       # batch 2
        lambda: s.loop(torch.zeros(1, 4, 3, 16, 16), text),                              # channels
        lambda: s.loop(frames[..., :2], text),                                           # uint8 channels
        lambda: s.loop(frames.repeat(2, 1, 1, 1, 1), text),                              # uint8 batch 2
        lambda: s.loop(low, text[:1]),                                                   # text batch 1
        lambda: s.loop(low, torch.cat([text, text])),                                    # text batch 4
        lambda: s.loop(torch.zeros(1, 3, 3, 12, 16), text),                              # H % 8
        lambda: s.loop(torch.zeros(1, 3, 3, 16, 20), text),                              # W % 8
        lambda: s.loop(low, text, latents=torch.zeros(1, 4, 2, 16, 16)),                 # latents shape
        lambda: s.loop(low, text, low_res_noise=torch.zeros(1, 4, 3, 16, 16)),           # noise shape
        lambda: VSRSampler(_StandIn(), noise_level=351),
        lambda: VSRSampler(_StandIn(), chunk_frames=0),
        lambda: VSRSampler(_StandIn(), schedule=DDPMSchedule(10)),
    ]
    for f in bad:
        with pytest.raises(ValueError):
            f()


def _gloo_worker(rank, world, port, result):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from lavie_b200 import ops
    from lavie_b200.pipeline import VSRSampler
    ops.cfg_linear_step = _torch_cfg_linear_step
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        frames, text = _cpu_inputs(F=11, seed=3)
        s = VSRSampler(_StandIn(), num_inference_steps=2, chunk_frames=4)
        got = s.loop(frames, text, generator=torch.Generator().manual_seed(4), group=dist.group.WORLD)
        solo = s.loop(frames, text, generator=torch.Generator().manual_seed(4))
        result[rank] = (torch.equal(got, solo), tuple(got.shape))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_chunk_parallel_loop_over_gloo(world):
    """11 frames = 4 + 4 + 3 over 2, 3 and 4 ranks (the last one owning no chunk): every rank returns the single-process
    latents."""
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    result = mp.get_context("spawn").Manager().dict()
    mp.spawn(_gloo_worker, args=(world, port, result), nprocs=world, join=True)
    assert sorted(result.keys()) == list(range(world))
    assert all(v == (True, (1, 4, 11, 16, 16)) for v in result.values()), dict(result)


# ----------------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def vsr_sd():
    from lavie_b200.config import VSR_CONFIG
    from lavie_b200.synthetic import synthetic_state_dict
    return synthetic_state_dict(VSR_CONFIG, seed=0)


@pytest.fixture(scope="module")
def unet(vsr_sd):
    from lavie_b200.vsr import UNet3DVSRModel
    m = UNet3DVSRModel()
    m.load_state_dict(vsr_sd, strict=True)
    return m.to(DEV).eval()


def _gpu_case(seed=21):
    """F = 7 as a 4-frame chunk and a 3-frame tail, 16x16, text L = 8; noise for the whole video in the draw order."""
    from lavie_b200.pipeline import chunk_plan
    g = torch.Generator().manual_seed(seed)
    low = torch.rand(1, 3, 7, 16, 16, generator=g) * 2 - 1
    text = torch.randn(2, 8, 1024, generator=g)
    lat, lrn = _noises_in_order(chunk_plan(7, 4), 16, 16, seed=seed + 1)
    return low, text, lat, lrn


@pytest.mark.gpu
def test_loop_matches_oracle(unet, vsr_sd):
    """3 steps (t = 667, 334, 1: the last is the low-noise end, where errors of v reach the output), guidance 5, noise
    level 50.  Tolerance 5e-2, as for the interpolation loop: guidance amplifies the bf16 noise of both halves."""
    from lavie_b200.pipeline import VSRSampler
    from oracle import vsr_sampler_oracle as VS
    low, text, lat, lrn = _gpu_case()
    s = VSRSampler(unet, 5.0, 50, num_inference_steps=3, chunk_frames=4)
    assert s.schedule.timesteps == [667, 334, 1]
    out = s.loop(low.to(DEV), text.to(DEV), latents=lat, low_res_noise=lrn)
    assert out.shape == (1, 4, 7, 16, 16) and out.dtype == torch.float32 and out.device.type == "cuda"
    assert len([k for k in unet._graphs if k[0][2] in (3, 4)]) >= 2          # one step graph per chunk length
    want = VS.vsr_loop(vsr_sd, low, text, lat, lrn, VS.DDIMV(3), 5.0, 50, 4)
    err = rel_l2(out.cpu(), want)
    print(f"VSR loop 7 frames (4 + 3), 3 steps, guidance 5: rel-L2 vs oracle = {err:.3e}")
    assert torch.isfinite(out).all() and err <= 5e-2


@pytest.mark.gpu
def test_chunks_are_independent(unet):
    """Chunk k of a full run is bit-equal to a run on that chunk's frames alone with the same noise."""
    from lavie_b200.pipeline import VSRSampler
    low, text, lat, lrn = _gpu_case(seed=33)
    s = VSRSampler(unet, 5.0, 50, num_inference_steps=2, chunk_frames=4)
    full = s.loop(low.to(DEV), text.to(DEV), latents=lat, low_res_noise=lrn)
    for sl in (slice(0, 4), slice(4, 7)):
        alone = s.loop(low[:, :, sl].to(DEV), text.to(DEV), latents=lat[:, :, sl].contiguous(),
                       low_res_noise=lrn[:, :, sl].contiguous())
        assert torch.equal(alone, full[:, :, sl]), sl


@pytest.fixture(scope="module")
def vae_x4():
    from lavie_b200.vae import X4_BLOCK_OUT, VAEDecoder, vae_synthetic_state_dict
    m = VAEDecoder.x4_upscaler()
    m.load_state_dict(vae_synthetic_state_dict(seed=0, block_out_channels=X4_BLOCK_OUT), strict=True)
    return m.to(DEV).eval()


@pytest.mark.gpu
def test_upscale_is_decode_of_loop(unet, vae_x4):
    """uint8 frames in, uint8 [1, F, 4h, 4w, 3] out on the host: the x4 decode of every chunk's loop latents."""
    from lavie_b200.pipeline import VSRSampler
    g = torch.Generator().manual_seed(8)
    frames = torch.randint(0, 256, (1, 7, 16, 16, 3), generator=g, dtype=torch.uint8)
    text = torch.randn(2, 8, 1024, generator=g)
    s = VSRSampler(unet, 5.0, 50, num_inference_steps=2, chunk_frames=4)
    video = s.upscale(frames, text.to(DEV), vae_x4, generator=torch.Generator().manual_seed(3))
    assert video.shape == (1, 7, 64, 64, 3) and video.dtype == torch.uint8 and video.device.type == "cpu"
    lat = s.loop(frames, text.to(DEV), generator=torch.Generator().manual_seed(3))
    want = torch.cat([vae_x4.decode_latents(lat[:, :, sl]) for sl in (slice(0, 4), slice(4, 7))], dim=1)
    assert torch.equal(video, want)
    whole = vae_x4.decode_latents(lat)           # one decode of all 7 frames: the same per-frame work, regrouped
    print(f"upscale vs one decode of the whole video: bit-identical = {torch.equal(video, whole)}, "
          f"max |diff| = {int((video.int() - whole.int()).abs().max())}")


def _two_gpu_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from lavie_b200.config import VSR_CONFIG
    from lavie_b200.pipeline import VSRSampler
    from lavie_b200.synthetic import synthetic_state_dict
    from lavie_b200.vae import X4_BLOCK_OUT, VAEDecoder, vae_synthetic_state_dict
    from lavie_b200.vsr import UNet3DVSRModel
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    try:
        unet = UNet3DVSRModel()
        unet.load_state_dict(synthetic_state_dict(VSR_CONFIG, seed=0), strict=True)
        unet = unet.to(dev).eval()
        vae = VAEDecoder.x4_upscaler()
        vae.load_state_dict(vae_synthetic_state_dict(seed=0, block_out_channels=X4_BLOCK_OUT), strict=True)
        vae = vae.to(dev).eval()
        g = torch.Generator().manual_seed(8)
        frames = torch.randint(0, 256, (1, 7, 16, 16, 3), generator=g, dtype=torch.uint8)
        text = torch.randn(2, 8, 1024, generator=g).to(dev)
        s = VSRSampler(unet, 5.0, 50, num_inference_steps=2, chunk_frames=4)
        par = s.upscale(frames, text, vae, generator=torch.Generator().manual_seed(3), group=dist.group.WORLD)
        solo = s.upscale(frames, text, vae, generator=torch.Generator().manual_seed(3))
        q.put((rank, torch.equal(par, solo), tuple(par.shape), par.numpy().tobytes()))
        torch.cuda.synchronize()
        dist.barrier()
    finally:
        os._exit(0)        # captured NCCL graphs make process-group teardown hang (as in test_p2p_gpu.py)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_chunk_parallel_upscale():
    """7 frames = 4 + 3 over 2 ranks: each rank decodes its own chunk; both return the single-GPU bytes."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + os.getpid() % 90
    procs = [ctx.Process(target=_two_gpu_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=600) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
    for rank, same, shape, _ in got:
        print(f"rank {rank}: chunk-parallel upscale {shape} equals the single-GPU bytes: {same}")
        assert same and shape == (1, 7, 64, 64, 3)
    assert got[0][3] == got[1][3]

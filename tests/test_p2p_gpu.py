"""The peer-memory (p2p) frame-sharding back end: csrc/p2p.cu + lavie_b200/p2p.py.

* single GPU, P = 1: every p2p kernel (flag barrier, GroupNorm exchange, LayerNorm scatter, gather-add) with the rank
  as its own only peer -- epoch / parity-slot logic, layouts and arithmetic against the un-sharded kernels.  (Ranks that
  WAIT on each other must never share one GPU -- B200_PROFILING.md -- so P > 1 is not emulated on one device.)
* >= 2 GPUs (skipped otherwise): two processes, NCCL rendezvous, the frame-sharded forward of
  one CFG half (eager, then CUDA-graph replays over several consecutive steps) against the single-GPU forward.
"""
import os
import sys

import pytest
import torch

from conftest import ROOT, rel_l2

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def solo_ctx():
    """A PeerContext-like object for P = 1 built on plain device memory (no symmetric-memory rendezvous needed)."""
    import ctypes
    from lavie_b200 import p2p

    class Solo(p2p.PeerContext):
        def __init__(self, token_bytes, device):
            self.group, self.P, self.rank, self.device = None, 1, 0, device
            flags_b = 256
            slots_b = 2 * self.P * (2 * 64 * 2) * 8
            tok_b = (token_bytes + 255) // 256 * 256
            self.layout = {"flags": 0, "slots": flags_b, "recv": flags_b + slots_b, "y": flags_b + slots_b + tok_b,
                           "kvx": flags_b + slots_b + 2 * tok_b}
            self.frame_off, self.halo_bytes = -1, tok_b
            self.buf = torch.zeros(flags_b + slots_b + 3 * tok_b, dtype=torch.uint8, device=device)
            self.peer_base = [self.buf.data_ptr()]
            self.epoch = torch.zeros(1, dtype=torch.int32, device=device)
            self.ticket = torch.zeros(1, dtype=torch.int32, device=device)
            self.fault = torch.zeros(8, dtype=torch.int32).pin_memory()
            self.token_bytes = tok_b

    return Solo(64 * 160 * 640 * 2, torch.device("cuda", 0))


def test_p2p_kernels_with_a_single_peer(solo_ctx):
    from lavie_b200 import ops
    ctx = solo_ctx
    g = torch.Generator().manual_seed(0)
    f_loc, hw, C = 4, 160, 640
    x = torch.randn(f_loc * hw, C, generator=g).cuda().to(torch.bfloat16)
    gamma = (torch.randn(C, generator=g) * 0.1 + 1).cuda()
    beta = (torch.randn(C, generator=g) * 0.1).cuda()
    e0 = int(ctx.epoch)
    # LayerNorm whose store side is the all-to-all (here: into my own receive buffer) + flag barrier
    recv = ctx.layernorm_scatter(x, gamma, beta, hw)
    assert torch.equal(recv, ops.layernorm(x, gamma, beta))
    # gather-add: res + rows of the (only) peer's y buffer
    y = ctx.local("y", f_loc * hw, C)
    y.copy_(torch.randn(f_loc * hw, C, generator=g).cuda().to(torch.bfloat16))
    out = ctx.add_gathered(x, hw)
    assert torch.equal(out, (x.float() + y.float()).to(torch.bfloat16))
    # GroupNorm statistics exchange (both epoch parities) == the fused single-GPU statistics
    for _ in range(3):
        ss = ctx.gn_scale_shift(x, None, 1, f_loc * hw, gamma, beta, 1e-5)
        assert rel_l2(ss, ops.groupnorm_scale_shift(x, 1, f_loc * hw, gamma, beta, 1e-5)) < 1e-6
    # SparseCausal halo exchange with a single rank: frame 0 lands in halo block 0, block 1 stays untouched (no right
    # neighbour), and the attention over [halo | local] equals the un-sharded sparse-causal attention
    from lavie_b200.packing import head_pitch
    heads, d, frames, S = 8, 40, 3, 64
    hp = heads * head_pitch(d)
    ext = ctx.local("kvx", (2 + frames) * S, 3 * hp)
    ext.zero_()
    qkv = torch.zeros(frames * S, 3, heads, head_pitch(d))
    qkv[..., :d] = torch.randn(frames * S, 3, heads, d, generator=g)
    ext[2 * S:].copy_(qkv.reshape(frames * S, 3 * hp).to(torch.bfloat16))
    ctx.push_halo(ext, frames, S)
    assert torch.equal(ext[:S], ext[2 * S:3 * S]) and float(ext[S:2 * S].abs().max()) == 0.0
    loc = ext[2 * S:]
    got = ops.attention(loc[:, :hp], ext[:, hp:2 * hp], ext[:, 2 * hp:], frames, heads, S, S, d, head_pitch(d),
                        sparse_causal_frames=frames, sc_halo=2)
    want = ops.attention(loc[:, :hp], loc[:, hp:2 * hp], loc[:, 2 * hp:], frames, heads, S, S, d, head_pitch(d),
                         sparse_causal_frames=frames)
    assert torch.equal(got, want)
    torch.cuda.synchronize()
    assert int(ctx.epoch) == e0 + 2 + 3 + 1       # every exchange advanced the epoch exactly once
    assert ctx.describe_fault().startswith("no peer-wait timeout")


def _two_gpu_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from lavie_b200 import UNet3DConditionModel
    from lavie_b200.synthetic import synthetic_inputs, synthetic_state_dict
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    try:
        unet = UNet3DConditionModel()
        unet.load_state_dict(synthetic_state_dict(seed=0), strict=True)
        unet = unet.to(dev).eval()
        frames = 8
        sample, t, text = synthetic_inputs(1, frames, 16, 32, seed=5)
        sample, text = sample.to(dev), text.to(dev)
        ref = unet(sample, t, encoder_hidden_states=text).sample
        errs = {}
        for backend in ("p2p", "nccl"):
            unet.set_frame_sharding(dist.group.WORLD, backend=backend)
            fl = frames // world
            shard = sample[:, :, rank * fl:(rank + 1) * fl].contiguous()
            want = ref[:, :, rank * fl:(rank + 1) * fl]
            unet.use_cuda_graph = False
            errs[f"{backend}/eager"] = rel_l2(unet(shard, t, encoder_hidden_states=text).sample, want)
            unet.use_cuda_graph = True
            worst = 0.0
            for _ in range(4):                                       # capture + 3 replays: epochs keep advancing
                worst = max(worst, rel_l2(unet(shard, t, encoder_hidden_states=text).sample, want))
            errs[f"{backend}/graph"] = worst
            # a bigger geometry regrows the peer context: graphs of the old one must not be replayed (ADVICE r1)
            if backend == "p2p":
                s2, t2, e2 = synthetic_inputs(1, frames, 16, 64, seed=6)
                r2 = None
                unet.set_frame_sharding(None)
                r2 = unet(s2.to(dev), t2, encoder_hidden_states=e2.to(dev)).sample
                unet.set_frame_sharding(dist.group.WORLD, backend="p2p")
                unet(shard, t, encoder_hidden_states=text)            # small context + graph first
                big = unet(s2[:, :, rank * fl:(rank + 1) * fl].contiguous().to(dev), t2,
                           encoder_hidden_states=e2.to(dev)).sample  # regrow
                errs["p2p/regrow"] = rel_l2(big, r2[:, :, rank * fl:(rank + 1) * fl])
                errs["p2p/after-regrow"] = rel_l2(unet(shard, t, encoder_hidden_states=text).sample, want)
        # the interpolation model with UNEVEN shards (7 frames = 4 + 3), SparseCausal halo + plain temporal attention
        from lavie_b200.config import INTERP_CONFIG
        del unet
        torch.cuda.empty_cache()
        iu = UNet3DConditionModel(INTERP_CONFIG)
        iu.load_state_dict(synthetic_state_dict(INTERP_CONFIG, seed=0), strict=True)
        iu = iu.to(dev).eval()
        g = torch.Generator().manual_seed(17)
        xs = torch.randn(1, 8, 7, 16, 32, generator=g).to(dev)
        te = torch.randn(1, 77, 768, generator=g).to(dev)
        iref = iu(xs, 400, encoder_hidden_states=te).sample
        counts = [4, 3]
        off = sum(counts[:rank])
        iu.set_frame_sharding(dist.group.WORLD, backend="p2p", frame_counts=counts)
        ish = xs[:, :, off:off + counts[rank]].contiguous()
        iwant = iref[:, :, off:off + counts[rank]]
        iu.use_cuda_graph = False
        errs["interp/eager"] = rel_l2(iu(ish, 400, encoder_hidden_states=te).sample, iwant)
        iu.use_cuda_graph = True
        worst = 0.0
        for _ in range(3):
            worst = max(worst, rel_l2(iu(ish, 400, encoder_hidden_states=te).sample, iwant))
        errs["interp/graph"] = worst
        q.put((rank, errs))
        torch.cuda.synchronize()
        dist.barrier()
    finally:
        os._exit(0)        # captured NCCL graphs make process-group teardown hang


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_frame_sharding_matches_single_gpu():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 400
    procs = [ctx.Process(target=_two_gpu_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=600) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
    for rank, errs in sorted(got):
        print(f"rank {rank}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
        assert max(errs.values()) < 2e-2, errs


def _vsr_two_gpu_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from lavie_b200.config import VSR_CONFIG
    from lavie_b200.synthetic import synthetic_state_dict
    from lavie_b200.vsr import UNet3DVSRModel
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    try:
        unet = UNet3DVSRModel()
        unet.load_state_dict(synthetic_state_dict(VSR_CONFIG, seed=0), strict=True)
        unet = unet.to(dev).eval()
        frames = 8
        g = torch.Generator().manual_seed(21)
        sample, low = torch.randn(1, 4, frames, 16, 32, generator=g).to(dev), torch.randn(1, 3, frames, 16, 32, generator=g).to(dev)
        text = torch.randn(1, 77, 1024, generator=g).to(dev)
        labels = torch.tensor([40])
        ref = unet(sample, 300, low, encoder_hidden_states=text, class_labels=labels).sample
        unet.set_frame_sharding(dist.group.WORLD)
        fl = frames // world
        sl = slice(rank * fl, (rank + 1) * fl)
        errs = {}
        for i in range(2):
            out = unet(sample[:, :, sl].contiguous(), 300, low[:, :, sl].contiguous(), encoder_hidden_states=text,
                       class_labels=labels).sample
            errs[f"vsr/frames{world}/call{i}"] = rel_l2(out, ref[:, :, sl])
        q.put((rank, errs))
        torch.cuda.synchronize()
        dist.barrier()
    finally:
        os._exit(0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_vsr_frame_sharding_matches_single_gpu():
    """VSR denoiser, 8 frames over 2 ranks (4 each: enough for the 2-frame halo of the (5,1,1) convolutions): halo
    exchange of the frame convs, all-reduced GroupNorm sums, all-to-all around the temporal attention."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29900 + os.getpid() % 90
    procs = [ctx.Process(target=_vsr_two_gpu_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=600) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
    for rank, errs in sorted(got):
        print(f"rank {rank}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
        assert max(errs.values()) < 2e-2, errs

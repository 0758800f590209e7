"""Multi-GPU paths on real devices (need >= 2 GPUs; skipped otherwise).
* one process per GPU: rank 0 packs, one NCCL broadcast of the blob, every rank samples its contiguous shard of the batch, logits are
  gathered on rank 0 -- and must equal the single-GPU run of the whole batch bit for bit (samples are independent; the per-rank plans
  have the same per-GPU batch as the chunks of the single-GPU reference).
* one process, one engine per GPU: libmugd state is per handle and kernel attributes are per device, so the engine on the second GPU
  computes exactly what the first one does."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, L, B, S, out_path):
    import torch.distributed as dist
    from mug_diffusion_b200 import synth
    from mug_diffusion_b200.config import ModelConfig
    from mug_diffusion_b200.dist import broadcast_blob, sample_sharded
    from mug_diffusion_b200.sampler import DDIMSampler, MugDiffusionB200

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = torch.device(f"cuda:{rank}")
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    cfg = ModelConfig()
    sd = synth.synthetic_state_dict(L) if rank == 0 else None
    blob = broadcast_blob(sd, cfg, dev)
    m = MugDiffusionB200(None, cfg, z_length=L, device=dev, blob=blob)
    # the request lives on rank 0 only; the other ranks know its shapes
    shapes = dict(x_T=(B, 16, L), c=(B, 128, 21), uc=(B, 128, 21), w0=(B, 256, L), w1=(B, 512, L // 2), w2=(B, 512, L // 4), w3=(B, 512, L // 8))
    req = None
    if rank == 0:
        inp = synth.synthetic_inputs(B, L, seed=3)
        req = dict(x_T=inp["x_T"], c=inp["c"], uc=inp["uc"], w=list(inp["w"])[-4:])
    sampler = DDIMSampler(m)

    def run(xT, c, uc, w):
        z, _ = sampler.sample(S=S, c=c, w=w, batch_size=c.shape[0], verbose=False, x_T=xT, eta=0.0, shape=(16, L),
                              unconditional_guidance_scale=5.0, unconditional_conditioning=uc)
        return m.model.decode(z)

    full = sample_sharded(run, req, shapes, dev)
    if rank == 0:
        torch.save(full.cpu(), out_path)
    dist.destroy_process_group()


def test_two_rank_sharded_sampling_equals_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from mug_diffusion_b200 import synth
    from mug_diffusion_b200.sampler import DDIMSampler, MugDiffusionB200

    L, B, S, world = 96, 4, 4, 2
    out_path = str(tmp_path / "gathered.pt")
    mp.spawn(_worker, args=(world, _free_port(), L, B, S, out_path), nprocs=world, join=True)
    gathered = torch.load(out_path)
    # single-GPU reference: the same charts, sampled in the same per-GPU chunks (identical plans -> bit-identical results)
    m = MugDiffusionB200.from_state_dict(synth.synthetic_state_dict(L), z_length=L)
    inp = synth.synthetic_inputs(B, L, seed=3)
    sampler = DDIMSampler(m)
    chunks = []
    for lo in range(0, B, B // world):
        sl = slice(lo, lo + B // world)
        z, _ = sampler.sample(S=S, c=inp["c"][sl].cuda(), w=[t[sl].cuda() for t in inp["w"]], batch_size=B // world, verbose=False,
                              x_T=inp["x_T"][sl].cuda(), eta=0.0, shape=(16, L), unconditional_guidance_scale=5.0,
                              unconditional_conditioning=inp["uc"][sl].cuda())
        chunks.append(m.model.decode(z).cpu())
    single = torch.cat(chunks)
    assert gathered.shape == single.shape == (B, 16, 8 * L)
    assert torch.equal(gathered, single)


def test_engines_on_two_devices_of_one_process_agree(golden_dir):
    """The golden L=512 U-Net request four times over (Beff = 8) through session + eval on an engine on cuda:0 and one on cuda:1,
    built from the same blob: every kernel with more than 48 KB of shared memory (tensor-core GEMM and attention, S4 conv) must launch
    on the second device too, and both results must be bit-identical and match the reference's output."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import golden_cases as gc
    from gpu_util import rel_err
    from mug_diffusion_b200 import synth
    from mug_diffusion_b200.config import ModelConfig
    from mug_diffusion_b200.packer import pack_model
    from mug_diffusion_b200.runtime import MugEngine

    case, reps = gc.UNET_CASES["unet_L512_B2"], 4
    L, Beff = case["L"], reps * case["B"]
    cfg = ModelConfig()
    blob = pack_model(synth.synthetic_state_dict(L), cfg.unet, cfg.decoder)
    inp = synth.synthetic_inputs(case["B"], L)
    eps = []
    for d in (0, 1):
        dev = torch.device(f"cuda:{d}")
        with torch.cuda.device(dev):
            eng = MugEngine(None, cfg, device=dev, blob=blob)
            s = eng.session(Beff, L, per_sample_t=True)
            s.set_timestep_table(case["t"] * reps)
            s.set_context(torch.cat([inp["c"]] * reps).to(dev))
            s.set_audio([torch.cat([w] * reps).to(dev) for w in inp["w"]])
            s.load_x(torch.cat([inp["x_T"]] * reps).to(dev), dup=False)
            s.eval()
            eps.append(s.read_rows(s.eps, Beff, cfg.unet.out_channels, L).cpu())
    assert torch.equal(eps[0], eps[1])
    gold = gc.load_golden(os.path.join(golden_dir, "unet_L512_B2.npz"))["eps"]
    assert rel_err(eps[1], torch.cat([gold] * reps)) < 1e-4

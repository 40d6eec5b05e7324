"""GPU: the callers either side of the loop, on hardware (VERDICT r1 items 5 / 8 / 10):
  * CompMDMGeneratedDataset (evaluation-time generation, comp_v6_model_dataset.py:148-256) with a synthetic loader --
    variable lengths, multimodality repeats -- against the oracle run sequentially in the reference's call order;
  * parallel.sample_sharded over NCCL (2 ranks): bitwise equal to the 1-GPU run (skipped with < 2 GPUs)."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import b200mdm
from conftest import default_args, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-3
B, D, T, STEPS, L = 8, 263, 48, 6, 2


def _loader(n_batches):
    g = torch.Generator().manual_seed(1)
    batches = []
    for i in range(n_batches):
        lengths = torch.randint(4, T + 1, (B,), generator=g)
        lengths[0] = T
        y = dict(lengths=lengths, mask=(torch.arange(T)[None] < lengths[:, None]).view(B, 1, 1, T),
                 text=["caption %d %d" % (i, b) for b in range(B)], tokens=["sos/OTHER_walk/VERB_eos/OTHER_unk/OTHER"] * B,
                 text_embed=torch.randn(1, B, 512, generator=g))
        batches.append((torch.zeros(B, D, 1, T), {"y": y}))
    vec = {k: (np.zeros(3), np.zeros(2)) for k in ("sos/OTHER", "walk/VERB", "eos/OTHER", "unk/OTHER")}

    class DS(SimpleNamespace):
        def __len__(self):
            return n_batches * B

    class Ld(list):
        batch_size = B
        dataset = DS(mode="gt", w_vectorizer=vec)
    return Ld(batches)


@pytest.mark.parametrize("budget", [None, 1])
def test_eval_generation_caller_vs_sequential_oracle(monkeypatch, budget):
    from oracle import mdm_oracle as mo, schedule_oracle as so
    from b200mdm.data_loaders.humanml.motion_loaders import comp_v6_model_dataset as cv
    if budget is not None:          # force the long-loop path: per-repeat generator clones + chunked eps (1000-step evals)
        monkeypatch.setattr(cv, "TAPE_BUDGET_BYTES", budget)
    args = default_args(layers=L, diffusion_steps=STEPS)
    model, diffusion = b200mdm.create_model_and_diffusion(args, SimpleNamespace(dataset=SimpleNamespace()))
    sd = b200mdm.synthetic_state_dict(num_layers=L, seed=9)
    b200mdm.load_model_wo_clip(model, sd)
    cfg = b200mdm.ClassifierFreeSampleModel(model.to("cuda").eval())
    loader, repeats, scale = _loader(3), 3, 2.5
    np.random.seed(7)
    torch.manual_seed(123)
    ds = cv.CompMDMGeneratedDataset(args, cfg, diffusion, loader, mm_num_samples=B, mm_num_repeats=repeats,
                                    max_motion_length=T, num_samples_limit=None, scale=scale)
    assert len(ds) == 3 * B and len(ds.mm_generated_motion) >= B
    # the reference's order: per loader batch, `repeat_times` sequential p_sample_loop calls, each drawing x_T then one
    # eps per step from the default CUDA generator
    np.random.seed(7)
    mm_idxs = np.sort(np.random.choice(3, B // B + 1, replace=False))
    torch.manual_seed(123)
    W = mo.OracleWeights(sd, L)
    tabs = so.diffusion_tables(so.named_betas("cosine", STEPS))
    worst, mm_seen = 0.0, 0
    for i, (motion, kw) in enumerate(loader):
        y = kw["y"]
        reps = repeats if i in mm_idxs else 1
        outs = []
        for r in range(reps):
            xT = torch.randn(B, D, 1, T, device="cuda")
            tape = [xT.cpu()] + [torch.randn_like(xT).cpu() for _ in range(STEPS)]
            outs.append(mo.sample_loop(W, tabs, list(range(STEPS)), tape, y["text_embed"], torch.full((B,), scale), y["lengths"]))
        for b in range(B):
            got = torch.from_numpy(ds.generated_motion[i * B + b]["motion"])              # [T, D]
            worst = max(worst, rel_err(got, outs[0][b, :, 0].t()))
            assert ds.generated_motion[i * B + b]["length"] == int(y["lengths"][b])
        if reps > 1:
            for b in range(B):
                mm = ds.mm_generated_motion[mm_seen * B + b]["mm_motions"]
                assert len(mm) == reps
                for r in range(reps):
                    worst = max(worst, rel_err(torch.from_numpy(mm[r]["motion"]), outs[r][b, :, 0].t()))
            mm_seen += 1
    print("eval caller (budget=%r): worst relative error vs the sequential oracle %.3e" % (budget, worst))
    assert worst < RTOL
    # the default generator ends where the reference's sequential calls would leave it
    a = torch.randn(4, device="cuda")
    torch.manual_seed(123)
    for i in range(3):
        for r in range(repeats if i in mm_idxs else 1):
            torch.randn(B, D, 1, T, device="cuda")
            for _ in range(STEPS):
                torch.randn(B, D, 1, T, device="cuda")
    assert torch.equal(a, torch.randn(4, device="cuda"))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, path, seed):
    import torch.distributed as dist
    from b200mdm import parallel
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    cfg, diffusion, inp, shape = _sharded_setup(rank)
    y = dict(mask=inp["mask"].cuda(), lengths=inp["lengths"].cuda(), scale=inp["scale"].cuda(),
             text_embed=inp["text_embed"].cuda() if rank == 0 else torch.zeros_like(inp["text_embed"]).cuda())
    out = parallel.sample_sharded(diffusion.p_sample_loop, cfg, shape, {"y": y}, n_steps=diffusion.num_timesteps, seed=seed,
                                  clip_denoised=False)
    if rank == 0:
        torch.save(out.cpu(), path)
    dist.destroy_process_group()


def _sharded_setup(dev):
    args = default_args(layers=L, diffusion_steps=STEPS)
    model, diffusion = b200mdm.create_model_and_diffusion(args, SimpleNamespace(dataset=SimpleNamespace()))
    b200mdm.load_model_wo_clip(model, b200mdm.synthetic_state_dict(num_layers=L, seed=9))
    cfg = b200mdm.ClassifierFreeSampleModel(model.to("cuda:%d" % dev).eval())
    Bg = 7                                                       # odd: ranks get 4 + 3
    inp = b200mdm.synthetic_inputs(Bg, nframes=T, steps=1, seed=5, lengths=[T, 40, 30, 20, 10, 5, 1])
    return cfg, diffusion, inp, (Bg, D, 1, T)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sample_sharded_nccl_equals_single_gpu(tmp_path):
    import torch.multiprocessing as mp
    from b200mdm import parallel
    seed, path = 991, str(tmp_path / "sharded.pt")
    mp.spawn(_nccl_worker, args=(2, _free_port(), path, seed), nprocs=2, join=True)
    cfg, diffusion, inp, shape = _sharded_setup(0)
    y = dict(mask=inp["mask"].cuda(), lengths=inp["lengths"].cuda(), scale=inp["scale"].cuda(), text_embed=inp["text_embed"].cuda())
    single = parallel.sample_sharded(diffusion.p_sample_loop, cfg, shape, {"y": y}, n_steps=STEPS, seed=seed, clip_denoised=False)
    assert torch.equal(single.cpu(), torch.load(path))

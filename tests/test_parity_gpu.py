"""GPU: the CUDA path (through the C ABI / reference-shaped Python API) against
  (a) golden vectors produced by the unmodified reference (tests/golden, oracle/gen_golden.py),
  (b) the fp32 oracle (oracle/mdm_oracle.py) on the same seeded inputs,
  (c) size-independent properties at the benchmark size.
Tolerance (BASELINE.json north_star): 1e-3 relative, measured as ||out - ref||_F / ||ref||_F against the fp32
reference; the GEMM operands are fp16 with fp32 accumulation (in/out projections are hi/lo-split, ~fp32)."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import b200mdm
from conftest import default_args, inpaint_motion, rel_err

pytestmark = pytest.mark.gpu
RTOL = 1e-3


def _build(layers, steps, seed, guided=True, **over):
    args = default_args(layers=layers, diffusion_steps=steps, **over)
    model, diffusion = b200mdm.create_model_and_diffusion(args, SimpleNamespace(dataset=SimpleNamespace(**(
        {"num_actions": 12} if over.get("dataset") == "humanact12" else {}))))
    kw = {}
    if over.get("dataset") == "humanact12":
        kw = dict(input_feats=150, cond_mode="action", num_actions=12)
    b200mdm.load_model_wo_clip(model, b200mdm.synthetic_state_dict(num_layers=layers, seed=seed, **kw))
    model.to("cuda").eval()
    return (b200mdm.ClassifierFreeSampleModel(model) if guided else model), model, diffusion


def _small():
    cfg, model, diffusion = _build(2, 4, 1)
    inp = b200mdm.synthetic_inputs(3, nframes=24, steps=4, seed=11, lengths=[24, 17, 5], scale=torch.tensor([2.5, 1.0, 7.5]))
    return cfg, model, diffusion, inp


def _y(inp, scale=True, dev="cuda"):
    y = dict(mask=inp["mask"].to(dev), lengths=inp["lengths"].to(dev), text_embed=inp["text_embed"].to(dev))
    if scale:
        y["scale"] = inp["scale"].to(dev)
    return y


def _tape(inp):
    return torch.stack(inp["tape"][1:]).cuda(), inp["tape"][0].cuda()


def test_forward_vs_reference_golden(golden):
    g = golden("enc_small.npz")
    cfg, model, _, inp = _small()
    x = inp["tape"][0].cuda()
    t = torch.full((3,), 2, dtype=torch.long, device="cuda")
    assert rel_err(model(x, t, y=_y(inp, False)), g["fwd_cond"]) < RTOL
    yu = _y(inp, False)
    yu["uncond"] = True
    assert rel_err(model(x, t, y=yu), g["fwd_uncond"]) < RTOL
    assert rel_err(cfg(x, t, y=_y(inp)), g["fwd_cfg"]) < RTOL


def test_ddpm_loop_every_step_vs_reference_golden(golden):
    g = golden("enc_small.npz")
    cfg, _, diffusion, inp = _small()
    tape, xT = _tape(inp)
    outs = list(diffusion.p_sample_loop_progressive(cfg, (3, 263, 1, 24), noise=xT, clip_denoised=False,
                                                    model_kwargs={"y": _y(inp)}, noise_tape=tape))
    assert len(outs) == 4
    for k, o in enumerate(outs):
        assert rel_err(o["sample"], g["ddpm_steps"][k]) < RTOL, k
    for use_graph in (False, True):
        out = diffusion.p_sample_loop(cfg, (3, 263, 1, 24), noise=xT, clip_denoised=False, model_kwargs={"y": _y(inp)},
                                      noise_tape=tape, use_graph=use_graph)
        assert rel_err(out, g["ddpm_steps"][-1]) < RTOL
        assert torch.equal(out, outs[-1]["sample"])          # fused loop == step-by-step, bit for bit
    assert torch.equal(xT, inp["tape"][0].cuda())             # caller's noise is not clobbered by the in-place loop


def test_loop_variants_vs_reference_golden(golden):
    g = golden("enc_small.npz")
    cfg, model, diffusion, inp = _small()
    tape, xT = _tape(inp)
    shape = (3, 263, 1, 24)
    run = lambda **kw: diffusion.p_sample_loop(cfg, shape, noise=xT, model_kwargs={"y": _y(inp)}, noise_tape=tape, **kw)
    assert rel_err(run(clip_denoised=True), g["ddpm_clip"]) < RTOL
    assert rel_err(run(clip_denoised=False, const_noise=True), g["ddpm_const_noise"]) < RTOL
    for eta in (0.0, 0.5):
        o = diffusion.ddim_sample_loop(cfg, shape, noise=xT, clip_denoised=False, eta=eta, model_kwargs={"y": _y(inp)},
                                       noise_tape=tape)
        assert rel_err(o, g["ddim_eta%g" % eta]) < RTOL, eta
    motion = inpaint_motion().cuda()
    m = torch.zeros(shape, dtype=torch.bool, device="cuda")
    m[..., :8] = True
    yi = _y(inp)
    yi["inpainting_mask"], yi["inpainted_motion"] = m, motion
    o = diffusion.p_sample_loop(cfg, shape, noise=xT, clip_denoised=False, model_kwargs={"y": yi}, noise_tape=tape)
    assert rel_err(o, g["ddpm_inpaint"]) < RTOL
    o = diffusion.p_sample_loop(cfg, shape, noise=xT, clip_denoised=False, skip_timesteps=1, init_image=motion,
                                model_kwargs={"y": _y(inp)}, noise_tape=tape[:3])
    assert rel_err(o, g["ddpm_skip1_init"]) < RTOL
    o = diffusion.p_sample_loop(model, shape, noise=xT, clip_denoised=False, model_kwargs={"y": _y(inp, False)}, noise_tape=tape)
    assert rel_err(o, g["ddpm_noguide"]) < RTOL
    d = diffusion.p_sample_loop(cfg, shape, noise=xT, clip_denoised=False, model_kwargs={"y": _y(inp)}, noise_tape=tape,
                                dump_steps=[0, 3])
    assert len(d) == 2 and rel_err(d[0], g["ddpm_steps"][0]) < RTOL and rel_err(d[1], g["ddpm_steps"][3]) < RTOL
    with pytest.raises(NotImplementedError):
        diffusion.ddim_sample_loop(cfg, shape, dump_steps=[1], model_kwargs={"y": _y(inp)})


def test_a2m_vs_reference_golden(golden):
    g = golden("a2m_small.npz")
    model, _, diffusion = _build(2, 3, 2, guided=False, dataset="humanact12", cond_mask_prob=0.0)
    inp = b200mdm.synthetic_inputs(4, njoints=25, nfeats=6, nframes=60, steps=3, seed=12, lengths=[60, 60, 45, 30])
    tape, xT = _tape(inp)
    y = dict(mask=inp["mask"].cuda(), lengths=inp["lengths"].cuda(), action=torch.from_numpy(g["action"]).cuda())
    o = diffusion.p_sample_loop(model, (4, 25, 6, 60), noise=xT, clip_denoised=False, model_kwargs={"y": y}, noise_tape=tape)
    assert rel_err(o, g["sample"]) < RTOL


def test_c1_full_config_vs_reference_golden(golden):
    """BASELINE config 1: L=8, d=512, 196 frames, 50 steps, CFG 2.5 -- the reference's own CPU output."""
    g = golden("enc_c1.npz")
    cfg, _, diffusion = _build(8, 50, 0)
    inp = b200mdm.synthetic_inputs(1, nframes=196, steps=50, seed=10)
    tape, xT = _tape(inp)
    o = diffusion.p_sample_loop(cfg, (1, 263, 1, 196), noise=xT, clip_denoised=False, model_kwargs={"y": _y(inp)}, noise_tape=tape)
    e = rel_err(o, g["sample"])
    print("C1 relative error vs reference:", e)
    assert e < RTOL


def test_vs_oracle_fresh_seeds():
    """Same seeded inputs through the oracle (CPU fp32) and the CUDA path; ragged lengths, per-sample scales."""
    from oracle import mdm_oracle as mo, schedule_oracle as so
    L, steps, B, T = 3, 6, 5, 77
    cfg, model, diffusion = _build(L, steps, 5)
    inp = b200mdm.synthetic_inputs(B, nframes=T, steps=steps, seed=31, lengths=[77, 76, 40, 2, 1],
                                   scale=torch.tensor([2.5, 0.0, 1.0, 5.0, 2.5]))
    W = mo.OracleWeights(b200mdm.synthetic_state_dict(num_layers=L, seed=5), L)
    tabs = so.diffusion_tables(so.named_betas("cosine", steps))
    ref = mo.sample_loop(W, tabs, list(range(steps)), inp["tape"], inp["text_embed"], inp["scale"], inp["lengths"])
    tape, xT = _tape(inp)
    o = diffusion.p_sample_loop(cfg, (B, 263, 1, T), noise=xT, clip_denoised=False, model_kwargs={"y": _y(inp)}, noise_tape=tape)
    assert rel_err(o, ref) < RTOL


def test_benchmark_size_properties():
    """B=64, T=196 (BASELINE config 2 shape, fewer steps): properties that need no oracle run at this size --
    batch-slice invariance (what makes the multi-GPU shards bitwise equal to the 1-GPU run), determinism of
    graph replay, and the t == 0 identity x_0 = model output (coef1 = 1, coef2 = 0, no noise)."""
    steps, B, T = 3, 64, 196
    cfg, model, diffusion = _build(8, steps, 0)
    inp = b200mdm.synthetic_inputs(B, nframes=T, steps=steps, seed=10)
    tape, xT = _tape(inp)
    y = _y(inp)
    full = diffusion.p_sample_loop(cfg, (B, 263, 1, T), noise=xT, clip_denoised=False, model_kwargs={"y": y}, noise_tape=tape)
    again = diffusion.p_sample_loop(cfg, (B, 263, 1, T), noise=xT, clip_denoised=False, model_kwargs={"y": y}, noise_tape=tape)
    assert torch.equal(full, again)
    assert torch.isfinite(full).all()
    lo, hi = 16, 32
    ys = dict(mask=y["mask"][lo:hi], lengths=y["lengths"][lo:hi], text_embed=y["text_embed"][:, lo:hi].contiguous(),
              scale=y["scale"][lo:hi])
    part = diffusion.p_sample_loop(cfg, (hi - lo, 263, 1, T), noise=xT[lo:hi].contiguous(), clip_denoised=False,
                                   model_kwargs={"y": ys}, noise_tape=tape[:, lo:hi].contiguous())
    assert torch.equal(part, full[lo:hi])
    # last step: sample == pred_xstart exactly
    last = None
    for o in diffusion.p_sample_loop_progressive(cfg, (B, 263, 1, T), noise=xT, clip_denoised=False, model_kwargs={"y": y},
                                                 noise_tape=tape):
        last = o
    assert torch.equal(last["sample"], last["pred_xstart"])
    assert torch.equal(last["sample"], full)


def test_generator_stream_matches_reference_draw_order():
    """`noise=None`: x_T from th.randn(*shape) then one th.randn_like per step, including t == 0
    (gaussian_diffusion.py:691, :525) -- so a seeded run consumes the same CUDA generator stream as the reference."""
    cfg, _, diffusion, inp = _small()
    shape = (3, 263, 1, 24)
    torch.manual_seed(123)
    a = diffusion.p_sample_loop(cfg, shape, clip_denoised=False, model_kwargs={"y": _y(inp)})
    torch.manual_seed(123)
    xT = torch.randn(*shape, device="cuda")
    tape = torch.stack([torch.randn_like(xT) for _ in range(4)])
    b = diffusion.p_sample_loop(cfg, shape, noise=xT, clip_denoised=False, model_kwargs={"y": _y(inp)}, noise_tape=tape)
    assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# DiP: arch=trans_dec, BERT token memory, prefix completion (SURVEY.md section 8 rows a20/a22)
def _dip(layers, steps, seed, ctx=20, pred=40):
    args = default_args(layers=layers, diffusion_steps=steps, arch="trans_dec", text_encoder_type="bert", context_len=ctx,
                        pred_len=pred)
    model, diffusion = b200mdm.create_model_and_diffusion(args, SimpleNamespace(dataset=SimpleNamespace()))
    sd = b200mdm.synthetic_state_dict(arch="trans_dec", num_layers=layers, cond_dim=768, seed=seed)
    b200mdm.load_model_wo_clip(model, sd)
    model.to("cuda").eval()
    return b200mdm.ClassifierFreeSampleModel(model), model, diffusion, sd, args


def _dip_y(inp, enc, tmask, prefix, scale=True):
    y = dict(mask=inp["mask"].cuda(), lengths=inp["lengths"].cuda(), text_embed=(enc.cuda(), tmask.cuda()), prefix=prefix.cuda())
    if scale:
        y["scale"] = inp["scale"].cuda()
    return y


def test_dip_vs_reference_golden(golden):
    g = golden("dip_small.npz")
    cfg, model, diffusion, _, _ = _dip(2, 3, 4)
    enc, tmask, prefix = b200mdm.synthetic_dip_inputs(3, 7, 20)
    inp = b200mdm.synthetic_inputs(3, nframes=40, steps=3, seed=13, lengths=[40, 33, 12], scale=torch.tensor([7.5, 2.0, 1.0]))
    x = inp["tape"][0].cuda()
    t = torch.full((3,), 1, dtype=torch.long, device="cuda")
    y = _dip_y(inp, enc, tmask, prefix)
    assert rel_err(cfg(x, t, y=y), g["fwd_cfg"]) < RTOL
    assert y["mask"].shape[-1] == 40                      # y is not mutated
    tape, xT = _tape(inp)
    outs = []
    for use_graph in (False, True):
        out = diffusion.p_sample_loop(cfg, (3, 263, 1, 40), noise=xT, clip_denoised=False, model_kwargs={"y": y},
                                      noise_tape=tape, use_graph=use_graph)
        assert rel_err(out, g["ddpm"]) < RTOL
        outs.append(out)
    assert torch.equal(outs[0], outs[1])
    y.pop("prefix")
    with pytest.raises(KeyError):
        cfg(x, t, y=y)


def test_dip_full_depth_vs_oracle():
    """DiP at its released depth (8 layers, 20 + 40 frames), fresh seeds: single forwards (cond / uncond / CFG) and a
    5-step loop against the fp32 oracle."""
    from oracle import mdm_oracle as mo, schedule_oracle as so
    B, ctx, pred, Mt, steps = 5, 20, 40, 12, 5
    cfg, model, diffusion, sd, _ = _dip(8, steps, 21)
    W = mo.OracleWeights(sd, 8)
    enc, tmask, prefix = b200mdm.synthetic_dip_inputs(B, Mt, ctx, seed=31)
    inp = b200mdm.synthetic_inputs(B, nframes=pred, steps=steps, seed=32, lengths=[40, 40, 31, 7, 1],
                                   scale=torch.tensor([7.5, 7.5, 2.5, 1.0, 0.0]))
    x = inp["tape"][0]
    t = torch.tensor([0, 1, 2, 3, 4])
    for uncond in (False, True):
        y = _dip_y(inp, enc, tmask, prefix, scale=False)
        y["uncond"] = uncond
        want = torch.stack([mo.denoise_dec(W, x[b:b + 1], int(t[b]), enc[:, b:b + 1], tmask[b:b + 1], prefix[b:b + 1],
                                           inp["lengths"][b:b + 1], True, uncond)[0] for b in range(B)])
        assert rel_err(model(x.cuda(), t.cuda(), y=y), want) < RTOL, uncond
    tabs = so.diffusion_tables(so.named_betas("cosine", steps))
    want = mo.sample_loop_dec(W, tabs, list(range(steps)), inp["tape"], enc, tmask, prefix, inp["scale"], inp["lengths"])
    tape, xT = _tape(inp)
    out = diffusion.p_sample_loop(cfg, (B, 263, 1, pred), noise=xT, clip_denoised=False,
                                  model_kwargs={"y": _dip_y(inp, enc, tmask, prefix)}, noise_tape=tape)
    assert rel_err(out, want) < RTOL


def test_dip_autoregressive_vs_oracle():
    """AutoRegressiveSampler over the engine: 3 chunks of 40 frames cropped to 100, prefix handed from chunk to chunk."""
    from oracle import mdm_oracle as mo, schedule_oracle as so
    B, ctx, pred, Mt, steps, need = 2, 20, 40, 9, 3, 100
    cfg, model, diffusion, sd, args = _dip(2, steps, 22)
    W = mo.OracleWeights(sd, 2)
    enc, tmask, prefix = b200mdm.synthetic_dip_inputs(B, Mt, ctx, seed=33)
    scale = torch.tensor([7.5, 2.5])
    chunks = [b200mdm.synthetic_inputs(B, nframes=pred, steps=steps, seed=40 + i, scale=scale) for i in range(3)]
    tabs = so.diffusion_tables(so.named_betas("cosine", steps))
    cur, buf = prefix, []
    for c in chunks:
        s = mo.sample_loop_dec(W, tabs, list(range(steps)), c["tape"], enc, tmask, cur, scale, c["lengths"])
        buf.append(s)
        cur = s[..., -ctx:]
    want = torch.cat(buf, -1)[..., :need]
    y = dict(mask=chunks[0]["mask"].cuda(), lengths=chunks[0]["lengths"].cuda(), text_embed=(enc.cuda(), tmask.cuda()),
             prefix=prefix.cuda(), scale=scale.cuda(), text=["a", "b"])
    y.pop("text")                                           # cached embeddings only: no text tower on the box
    sampler = b200mdm.AutoRegressiveSampler(args, diffusion.p_sample_loop, required_frames=need)
    out = sampler.sample(cfg, (B, 263, 1, need), clip_denoised=False, model_kwargs={"y": y},
                         noise=torch.stack([c["tape"][0] for c in chunks]).cuda(),
                         noise_tape=torch.stack([torch.stack(c["tape"][1:]) for c in chunks]).cuda())
    assert out.shape == (B, 263, 1, need)
    assert rel_err(out, want) < RTOL
    assert torch.equal(y["prefix"], prefix.cuda())


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs 3 and 4 at their full sizes: the whole batch runs on the GPU, the fp32 oracle follows a few
# samples of it (every sample is independent of its batch neighbours, so a subset is a complete check of those rows).
def _gpu_tape(n_run, shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    xT = torch.randn(*shape, device="cuda", generator=g)
    tape = torch.randn(n_run, *shape, device="cuda", generator=g)
    return xT, tape


def test_dip_config_b128_autoregressive():
    """BASELINE config 3: DiP, B=128, 10 diffusion steps per 40-frame chunk, guidance 7.5 -- 3 chunks (120 -> 100 frames)."""
    from oracle import mdm_oracle as mo, schedule_oracle as so
    B, ctx, pred, Mt, steps, need, nchunk = 128, 20, 40, 16, 10, 100, 3
    cfg, model, diffusion, sd, args = _dip(8, steps, 23)
    enc, tmask, prefix = b200mdm.synthetic_dip_inputs(B, Mt, ctx, seed=35)
    scale = torch.full((B,), 7.5)
    lengths = torch.full((B,), pred, dtype=torch.long)
    shape = (B, 263, 1, pred)
    noise, tapes = zip(*[_gpu_tape(steps, shape, 50 + i) for i in range(nchunk)])
    y = dict(mask=torch.ones(B, 1, 1, pred, dtype=torch.bool, device="cuda"), lengths=lengths.cuda(),
             text_embed=(enc.cuda(), tmask.cuda()), prefix=prefix.cuda(), scale=scale.cuda())
    sampler = b200mdm.AutoRegressiveSampler(args, diffusion.p_sample_loop, required_frames=need)
    out = sampler.sample(cfg, (B, 263, 1, need), clip_denoised=False, model_kwargs={"y": y}, noise=torch.stack(noise),
                         noise_tape=torch.stack(tapes))
    again = sampler.sample(cfg, (B, 263, 1, need), clip_denoised=False, model_kwargs={"y": y}, noise=torch.stack(noise),
                           noise_tape=torch.stack(tapes))
    assert out.shape == (B, 263, 1, need) and torch.isfinite(out).all() and torch.equal(out, again)
    W = mo.OracleWeights(sd, 8)
    tabs = so.diffusion_tables(so.named_betas("cosine", steps))
    idx = [0, 77, 127]
    cur, buf = prefix[idx], []
    for c in range(nchunk):
        tape = [noise[c][idx].cpu()] + [tapes[c][k][idx].cpu() for k in range(steps)]
        s = mo.sample_loop_dec(W, tabs, list(range(steps)), tape, enc[:, idx], tmask[idx], cur, scale[idx], lengths[idx])
        buf.append(s)
        cur = s[..., -ctx:]
    want = torch.cat(buf, -1)[..., :need]
    e = rel_err(out[idx], want)
    print("DiP B=128, 3 chunks x 10 steps, guidance 7.5: relative error vs oracle", e)
    assert e < RTOL


def test_a2m_config_b256_1000_steps():
    """BASELINE config 4: HumanAct12 action2motion, B=256, 60 frames, 1000 steps, no guidance: 1000 recurrent steps of
    the fused loop (one graph replayed 1000 times) against the oracle on two samples."""
    from oracle import mdm_oracle as mo, schedule_oracle as so
    B, T, steps = 256, 60, 1000
    model, _, diffusion = _build(8, steps, 5, guided=False, dataset="humanact12", cond_mask_prob=0.0)
    sd = b200mdm.synthetic_state_dict(num_layers=8, seed=5, input_feats=150, cond_mode="action", num_actions=12)
    shape = (B, 25, 6, T)
    xT, tape = _gpu_tape(steps, shape, 60)
    lengths = torch.full((B,), T, dtype=torch.long)
    lengths[1] = 45
    action = (torch.arange(B) % 12).view(B, 1)
    y = dict(mask=(torch.arange(T)[None, :] < lengths[:, None]).view(B, 1, 1, T).cuda(), lengths=lengths.cuda(), action=action.cuda())
    out = diffusion.p_sample_loop(model, shape, noise=xT, clip_denoised=False, model_kwargs={"y": y}, noise_tape=tape)
    assert torch.isfinite(out).all()
    idx = [1, 200]
    W = mo.OracleWeights(sd, 8)
    tabs = so.diffusion_tables(so.named_betas("cosine", steps))
    tp = [xT[idx].cpu()] + [tape[k][idx].cpu() for k in range(steps)]
    want = mo.sample_loop(W, tabs, list(range(steps)), tp, None, None, lengths[idx], action=action[idx])
    e = rel_err(out[idx], want)
    print("a2m B=256, 1000 steps: relative error vs oracle", e)
    assert e < RTOL


# ---------------------------------------------------------------------------------------------------------------------
# Post-loop step (SURVEY.md 8f rank 2): inv_transform + recover_from_ric on the GPU (generate.py:161-166)
def _ric_close(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max())


def test_recover_from_ric_vs_reference_golden(golden):
    g = golden("ric.npz")
    for D, J in ((263, 22), (251, 21)):
        gen = torch.Generator().manual_seed(100 + D)
        sample = torch.randn(3, D, 1, 40, generator=gen) * 0.8
        mean, std = b200mdm.synthetic_norm_stats(D, seed=7)
        xyz = b200mdm.sample_to_xyz(sample.cuda(), mean.numpy(), std.numpy())
        assert xyz.shape == (3, J, 3, 40)
        assert _ric_close(xyz, g["xyz_%d" % D]) < 2e-6           # cosf / sinf are the only non-identical operations
        ric = b200mdm.recover_from_ric(sample.permute(0, 2, 3, 1).contiguous().cuda(), J)
        assert ric.shape == (3, 1, 40, J, 3)
        assert _ric_close(ric, g["ric_%d" % D]) < 2e-6
    with pytest.raises(RuntimeError):
        b200mdm.sample_to_xyz(sample, mean, std)                 # CPU tensor: no fallback


def test_recover_from_ric_benchmark_size_vs_oracle():
    """B=64, T=196 (what follows the BASELINE config 2 loop) against the CPU restatement; plus what the construction
    guarantees exactly: root height is the de-normalised feature 3, frame 0 sits at the origin."""
    from oracle import ric_oracle as ro
    gen = torch.Generator().manual_seed(5)
    sample = torch.randn(64, 263, 1, 196, generator=gen) * 0.5
    mean, std = b200mdm.synthetic_norm_stats(263, seed=8)
    xyz = b200mdm.sample_to_xyz(sample.cuda(), mean, std)
    want = ro.sample_to_xyz(sample, mean, std)
    assert _ric_close(xyz, want) < 1e-5                          # yaw accumulates over 196 frames
    h = (sample[:, 3, 0, :] * std[3] + mean[3])
    assert torch.equal(xyz[:, 0, 1, :].cpu(), h)
    assert torch.equal(xyz[:, 0, 0, 0].cpu(), torch.zeros(64)) and torch.equal(xyz[:, 0, 2, 0].cpu(), torch.zeros(64))

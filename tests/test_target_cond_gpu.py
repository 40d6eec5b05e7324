"""GPU: target-location conditioning through the engine (b200mdm_set_target + the conditioning-row fold) against
golden/target_small.npz (the unmodified reference) and the fp32 oracle; the no-target path stays bit for bit the path of
a plain model, and the step graph does not change."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import b200mdm
from conftest import default_args, rel_err
from oracle import mdm_oracle as mo
from oracle import schedule_oracle as so
from oracle import target_oracle as to
import target_cases as tc

pytestmark = pytest.mark.gpu
RTOL = 1e-3


def _cuda_case(name):
    model, diffusion, sd, inp, y, T = tc.build(name, device="cuda")
    model.to("cuda").eval()
    return b200mdm.ClassifierFreeSampleModel(model), model, diffusion, sd, inp, y, T


def _loop(cfg, diffusion, inp, y, B, T, use_graph=True):
    return diffusion.p_sample_loop(cfg, (B, 263, 1, T), noise=inp["tape"][0].cuda(), clip_denoised=False,
                                   model_kwargs={"y": y}, noise_tape=torch.stack(inp["tape"][1:]).cuda(), use_graph=use_graph)


@pytest.mark.parametrize("name", sorted(tc.CASES))
def test_target_cases_vs_reference_golden(golden, name):
    g = golden("target_small.npz")
    cfg, model, diffusion, sd, inp, y, T = _cuda_case(name)
    B = tc.CASES[name][4]
    x = inp["tape"][0].cuda()
    t = torch.full((B,), 1, dtype=torch.long, device="cuda")
    fwd = cfg(x, t, y=y())
    assert rel_err(fwd, g[name + "_fwd"]) < RTOL
    outs = [_loop(cfg, diffusion, inp, y(), B, T, use_graph=ug) for ug in (False, True)]
    assert rel_err(outs[1], g[name + "_ddpm"]) < RTOL
    assert torch.equal(outs[0], outs[1])
    # without targets the output is far from the reference's (the fold is not a no-op hiding in the tolerance)
    assert rel_err(cfg(x, t, y=tc.without_target(y())), g[name + "_fwd"]) > 20 * RTOL
    if name == "dip_multi":
        assert rel_err(cfg(x, t, y=y(target_uncond=True)), g[name + "_tuncond_fwd"]) < RTOL


@pytest.mark.parametrize("name", ["dip_multi", "enc_single"])
def test_no_target_is_the_plain_model_bit_for_bit(name):
    """target_uncond=True, a y without target_cond, and a plain model (no multi_target_cond) loaded with the same
    non-target weights: identical outputs, forward and loop."""
    cfg, model, diffusion, sd, inp, y, T = _cuda_case(name)
    arch, B = tc.CASES[name][0], tc.CASES[name][4]
    over = dict(arch="trans_dec", text_encoder_type="bert", context_len=tc.CTX, pred_len=tc.PRED) if arch == "trans_dec" else {}
    plain, _ = b200mdm.create_model_and_diffusion(default_args(layers=tc.L, diffusion_steps=tc.STEPS, **over),
                                                  SimpleNamespace(dataset=SimpleNamespace()))
    b200mdm.load_model_wo_clip(plain, {k: v for k, v in sd.items() if not k.startswith("embed_target_cond.")})
    plain_cfg = b200mdm.ClassifierFreeSampleModel(plain.to("cuda").eval())
    x = inp["tape"][0].cuda()
    t = torch.full((B,), 2, dtype=torch.long, device="cuda")
    want = plain_cfg(x, t, y=tc.without_target(y()))
    for yy in (y(target_uncond=True), tc.without_target(y())):
        assert torch.equal(cfg(x, t, y=yy), want)
    want = _loop(plain_cfg, diffusion, inp, tc.without_target(y()), B, T)
    assert torch.equal(_loop(cfg, diffusion, inp, y(target_uncond=True), B, T), want)
    assert torch.equal(_loop(cfg, diffusion, inp, tc.without_target(y()), B, T), want)


def test_launch_count_per_loop_and_alternation():
    """The step graph is the same with and without targets (same kernels per loop), and loops with and without targets
    alternate on one engine without a stale target."""
    cfg, model, diffusion, sd, inp, y, T = _cuda_case("dip_split")
    from b200mdm import _lib
    B = tc.CASES["dip_split"][4]
    eng = model.engine()
    counts = {}
    for with_t in (True, False):
        yy = y() if with_t else tc.without_target(y())
        eng.set_schedule(diffusion.schedule_rows(0.0), list(range(tc.STEPS)))
        eng.set_cond(B, T, yy, True, torch.device("cuda"))
        eng.set_inpaint(None, None)
        eng.launch_count(reset=True)
        eng.sample_loop(_lib.MODE_DDPM, inp["tape"][0].cuda(), torch.stack(inp["tape"][1:]).cuda())
        counts[with_t] = eng.launch_count()
    assert counts[True] == counts[False] > 0
    ref_t = _loop(cfg, diffusion, inp, y(), B, T)
    ref_n = _loop(cfg, diffusion, inp, tc.without_target(y()), B, T)
    assert rel_err(ref_t, ref_n) > 20 * RTOL
    for k in range(2):
        assert torch.equal(_loop(cfg, diffusion, inp, y(), B, T), ref_t), k
        assert torch.equal(_loop(cfg, diffusion, inp, tc.without_target(y()), B, T), ref_n), k


def _released_dip(encoder, seed):
    args = default_args(layers=8, diffusion_steps=10, arch="trans_dec", text_encoder_type="bert", context_len=20, pred_len=40,
                        multi_target_cond=True, multi_encoder_type=encoder, target_enc_layers=1)
    model, diffusion = b200mdm.create_model_and_diffusion(args, SimpleNamespace(dataset=SimpleNamespace()))
    sd = b200mdm.synthetic_state_dict(arch="trans_dec", num_layers=8, cond_dim=768, seed=seed, target_encoder=encoder)
    b200mdm.load_model_wo_clip(model, sd)
    return b200mdm.ClassifierFreeSampleModel(model.to("cuda").eval()), model, diffusion, sd, args


def _mixed_sets(B):
    pool = [[], ["traj"], ["left_wrist", "head"], ["pelvis"], ["right_foot", "left_foot", "traj"], ["right_wrist"]]
    return [pool[b % len(pool)] for b in range(B)], [b % 3 == 0 for b in range(B)]


def test_released_depth_dip_b128_autoregressive_with_targets():
    """DiP at its released depth, B=128, 10 steps per 40-frame chunk, guidance 7.5, 5 chunks (196 frames) through
    AutoRegressiveSampler with the same targets for every chunk (as the reference), mixed per-sample joint sets; the oracle
    follows four samples (samples are independent of their batch neighbours)."""
    B, ctx, pred, Mt, steps, need, nchunk = 128, 20, 40, 16, 10, 196, 5
    cfg, model, diffusion, sd, args = _released_dip("multi", 61)
    enc, tmask, prefix = b200mdm.synthetic_dip_inputs(B, Mt, ctx, seed=62)
    sets, heading = _mixed_sets(B)
    tgt = b200mdm.synthetic_targets(B, sets, heading, seed=63)
    scale = torch.full((B,), 7.5)
    shape = (B, 263, 1, pred)
    g = torch.Generator(device="cuda").manual_seed(64)
    noise = torch.randn(nchunk, *shape, device="cuda", generator=g)
    tapes = torch.randn(nchunk, steps, *shape, device="cuda", generator=g)
    y = dict(mask=torch.ones(B, 1, 1, pred, dtype=torch.bool, device="cuda"), lengths=torch.full((B,), pred, device="cuda"),
             text_embed=(enc.cuda(), tmask.cuda()), prefix=prefix.cuda(), scale=scale.cuda(),
             target_cond=tgt["target_cond"].cuda(), target_joint_names=tgt["target_joint_names"], is_heading=tgt["is_heading"].cuda())
    sampler = b200mdm.AutoRegressiveSampler(args, diffusion.p_sample_loop, required_frames=need)
    out = sampler.sample(cfg, (B, 263, 1, need), clip_denoised=False, model_kwargs={"y": y}, noise=noise, noise_tape=tapes)
    assert out.shape == (B, 263, 1, need) and torch.isfinite(out).all()
    W = mo.OracleWeights(sd, 8)
    tabs = so.diffusion_tables(so.named_betas("cosine", steps))
    idx = [0, 1, 2, 100]
    target = to.target_embedding(W, "multi", tc.ROWS, tgt["target_cond"][idx], [sets[i] for i in idx], tgt["is_heading"][idx])
    cur, buf = prefix[idx], []
    for c in range(nchunk):
        tape = [noise[c][idx].cpu()] + [tapes[c][k][idx].cpu() for k in range(steps)]
        s = to.sample_loop_dec(W, tabs, list(range(steps)), tape, enc[:, idx], tmask[idx], cur, scale[idx], target,
                               torch.full((len(idx),), pred))
        buf.append(s)
        cur = s[..., -ctx:]
    want = torch.cat(buf, -1)[..., :need]
    e = rel_err(out[idx], want)
    print("DiP + multi target encoder, B=128, 5 chunks x 10 steps, guidance 7.5: relative error vs oracle", e)
    assert e < RTOL


def test_philox_targets_match_two_sharded_halves():
    """Engine noise (Philox, keyed by global sample index): B=64 in one run equals the two halves run separately with
    their slices of the targets (parallel.shard_model_kwargs), bit for bit."""
    from b200mdm.parallel import shard_model_kwargs
    B, pred, Mt, steps = 64, 40, 12, 4
    cfg, model, diffusion, sd, args = _released_dip("single", 71)
    enc, tmask, prefix = b200mdm.synthetic_dip_inputs(B, Mt, 20, seed=72)
    sets, heading = _mixed_sets(B)
    tgt = b200mdm.synthetic_targets(B, sets, heading, seed=73)
    names = np.empty(B, dtype=object)
    names[:] = [np.array(s, dtype=str) for s in sets]
    y = dict(mask=torch.ones(B, 1, 1, pred, dtype=torch.bool, device="cuda"), lengths=torch.full((B,), pred, device="cuda"),
             text_embed=(enc.cuda(), tmask.cuda()), prefix=prefix.cuda(), scale=torch.full((B,), 7.5, device="cuda"),
             target_cond=tgt["target_cond"].cuda(), target_joint_names=names, is_heading=tgt["is_heading"].cuda())
    shape = (B, 263, 1, pred)
    full = diffusion.p_sample_loop(cfg, shape, clip_denoised=False, model_kwargs={"y": y}, noise_seed=99)
    parts = []
    for lo, hi in ((0, 32), (32, 64)):
        kw = shard_model_kwargs({"y": y}, lo, hi)
        parts.append(diffusion.p_sample_loop(cfg, (hi - lo,) + shape[1:], clip_denoised=False, model_kwargs=kw, noise_seed=99,
                                             sample_index_base=lo))
    assert torch.equal(torch.cat(parts), full)

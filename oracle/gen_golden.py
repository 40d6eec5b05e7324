"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, via oracle/ref_harness.py) on CPU in the build container:

    python -m oracle.gen_golden

The reference has no tests and no golden vectors of its own (SURVEY.md section 4), so these files are the pin:
every value below is an output of the reference's own code (fp32, torch CPU) for seeded inputs that can be
regenerated anywhere (numpy default_rng streams in motion-diffusion-model_b200/synthetic.py).

Files
  schedule.npz   fp64 tables + timestep maps of the reference for several (steps, respacing) settings, and
                 space_timesteps known answers (sorted lists) incl. the ValueError case
  enc_small.npz  trans_enc L=2, B=3, T=24, 4 steps, ragged lengths, per-sample scales: single forwards (cond,
                 uncond, CFG), every p_sample output of p_sample_loop, ddim (eta 0 and 0.5) loop outputs,
                 inpainting loop output, skip_timesteps/init_image output (the motion they start from is not stored:
                 tests/conftest.py inpaint_motion() draws it from the same seed, which keeps the file under 1 MB)
  enc_c1.npz     BASELINE config 1 shape: L=8, B=1, T=196, 50 steps, CFG 2.5 -> final sample
  enc_l3.npz     trans_enc L=3, B=2, T=31, 6 steps on seeds of its own: final sample, timestep map, diffusion tables
  a2m_small.npz  action-conditioned trans_enc (humanact12 shape 25x6, 12 classes), no CFG, 3 steps
  ric.npz        post-loop inv_transform + recover_from_ric (generate.py:161-166), 263- and 251-dim features
  dip_small.npz  trans_dec + BERT-token memory + prefix completion (DiP): L=2, ctx 20 + pred 40, 3 steps, ragged text
                 padding mask, per-sample scales: one CFG forward and the p_sample_loop output
"""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402

syn = importlib.import_module("motion-diffusion-model_b200.synthetic")
OUT = os.path.join(ROOT, "tests", "golden")
TABLE_NAMES = ["betas", "alphas_cumprod", "alphas_cumprod_prev", "alphas_cumprod_next", "sqrt_alphas_cumprod",
               "sqrt_one_minus_alphas_cumprod", "log_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod",
               "sqrt_recipm1_alphas_cumprod", "posterior_variance", "posterior_log_variance_clipped",
               "posterior_mean_coef1", "posterior_mean_coef2"]


def gen_schedule():
    ns = rh.load_reference()
    gd, rs = ns.gaussian_diffusion, ns.respace
    out = {}
    cases = [("cosine", 50, [50]), ("cosine", 1000, [1000]), ("cosine", 1000, "50"), ("cosine", 1000, "ddim50"),
             ("cosine", 10, [10]), ("linear", 1000, "10,15,20"), ("cosine", 300, [10, 15, 20])]
    for ci, (sched, steps, resp) in enumerate(cases):
        betas = gd.get_named_beta_schedule(sched, steps, 1.0)
        d = rs.SpacedDiffusion(use_timesteps=rs.space_timesteps(steps, resp), betas=betas,
                               model_mean_type=gd.ModelMeanType.START_X, model_var_type=gd.ModelVarType.FIXED_SMALL,
                               loss_type=gd.LossType.MSE, rescale_timesteps=False)
        out["case%d_meta" % ci] = np.array([sched, str(steps), repr(resp)])
        out["case%d_base_betas" % ci] = betas
        out["case%d_timestep_map" % ci] = np.array(d.timestep_map, dtype=np.int64)
        for n in TABLE_NAMES:
            out["case%d_%s" % (ci, n)] = getattr(d, n)
    kats = [(300, [10, 15, 20]), (1000, "ddim50"), (1000, "50"), (1000, "ddim25"), (50, [50]), (1000, "10,15,20"),
            (1000, [1]), (7, [3, 2]), (100, "ddim10"), (100, [100])]
    for ki, (n, sc) in enumerate(kats):
        out["space%d_args" % ki] = np.array([str(n), repr(sc)])
        out["space%d_steps" % ki] = np.array(sorted(rs.space_timesteps(n, sc)), dtype=np.int64)
    for n, sc in [(1000, "ddim333"), (10, [11])]:
        try:
            rs.space_timesteps(n, sc)
            raise AssertionError("expected ValueError")
        except ValueError:
            pass
    out["space_errors"] = np.array(["1000|'ddim333'", "10|[11]"])
    # _WrappedModel mapping (respace.py:125-127)
    tm = sorted(rs.space_timesteps(1000, "50"))
    wm = rs._WrappedModel(lambda x, ts, **kw: ts, tm, False, 1000)
    ts = torch.tensor([49, 0, 7, 25])
    out["wrapped_in"] = ts.numpy()
    out["wrapped_out"] = wm(None, ts).numpy()
    np.savez_compressed(os.path.join(OUT, "schedule.npz"), **out)
    print("schedule.npz:", len(out), "arrays")


def _y(inp, with_scale=True):
    y = dict(mask=inp["mask"], lengths=inp["lengths"], text_embed=inp["text_embed"])
    if with_scale:
        y["scale"] = inp["scale"]
    return y


def gen_enc_small():
    ns = rh.load_reference()
    L, steps, B, T = 2, 4, 3, 24
    args = rh.default_args(layers=L, diffusion_steps=steps)
    sd = syn.synthetic_state_dict(num_layers=L, seed=1)
    model, diff = rh.build(args, state_dict=sd)
    cfg = ns.sampler_util.ClassifierFreeSampleModel(model)
    inp = syn.synthetic_inputs(B, nframes=T, steps=steps, seed=11, lengths=[24, 17, 5],
                               scale=torch.tensor([2.5, 1.0, 7.5]))
    shape = (B, 263, 1, T)
    out = {"meta": np.array(["L=2 steps=4 B=3 T=24 weights_seed=1 inputs_seed=11 lengths=24,17,5 scales=2.5,1,7.5"])}
    x = inp["tape"][0]
    t = torch.full((B,), 2, dtype=torch.long)
    with torch.no_grad():
        out["fwd_cond"] = model(x, t, y=_y(inp, False)).numpy()
        yu = _y(inp, False)
        yu["uncond"] = True
        out["fwd_uncond"] = model(x, t, y=yu).numpy()
        out["fwd_cfg"] = cfg(x, t, y=_y(inp)).numpy()
        # full DDPM loop, every intermediate sample
        samples = []
        with rh.noise_tape(inp["tape"]):
            for o in diff.p_sample_loop_progressive(cfg, shape, clip_denoised=False, model_kwargs={"y": _y(inp)}):
                samples.append(o["sample"].numpy().copy())
        out["ddpm_steps"] = np.stack(samples)
        with rh.noise_tape(inp["tape"]):
            out["ddpm_clip"] = diff.p_sample_loop(cfg, shape, clip_denoised=True, model_kwargs={"y": _y(inp)}).numpy()
        with rh.noise_tape(inp["tape"]):
            out["ddpm_const_noise"] = diff.p_sample_loop(cfg, shape, clip_denoised=False, const_noise=True,
                                                         model_kwargs={"y": _y(inp)}).numpy()
        for eta in (0.0, 0.5):
            with rh.noise_tape(inp["tape"]):
                out["ddim_eta%g" % eta] = diff.ddim_sample_loop(cfg, shape, clip_denoised=False, eta=eta,
                                                                model_kwargs={"y": _y(inp)}).numpy()
        # inpainting (sample/edit.py style): keep the first 8 frames of a given motion
        rng = np.random.default_rng(5)
        motion = torch.from_numpy(rng.standard_normal(shape).astype(np.float32))
        imask = torch.zeros(shape, dtype=torch.bool)
        imask[..., :8] = True
        yi = _y(inp)
        yi["inpainting_mask"], yi["inpainted_motion"] = imask, motion
        with rh.noise_tape(inp["tape"]):
            out["ddpm_inpaint"] = diff.p_sample_loop(cfg, shape, clip_denoised=False, model_kwargs={"y": yi}).numpy()
        # skip_timesteps + init_image (q_sample at the first index)
        with rh.noise_tape(inp["tape"]):
            out["ddpm_skip1_init"] = diff.p_sample_loop(cfg, shape, clip_denoised=False, skip_timesteps=1,
                                                        init_image=motion, model_kwargs={"y": _y(inp)}).numpy()
        # no guidance wrapper (guidance_param == 1 path)
        with rh.noise_tape(inp["tape"]):
            out["ddpm_noguide"] = diff.p_sample_loop(model, shape, clip_denoised=False,
                                                     model_kwargs={"y": _y(inp, False)}).numpy()
    np.savez_compressed(os.path.join(OUT, "enc_small.npz"), **out)
    print("enc_small.npz:", {k: v.shape for k, v in out.items() if k != "meta"})


def gen_enc_c1():
    ns = rh.load_reference()
    L, steps, B, T = 8, 50, 1, 196
    args = rh.default_args(layers=L, diffusion_steps=steps)
    sd = syn.synthetic_state_dict(num_layers=L, seed=0)
    model, diff = rh.build(args, state_dict=sd)
    cfg = ns.sampler_util.ClassifierFreeSampleModel(model)
    inp = syn.synthetic_inputs(B, nframes=T, steps=steps, seed=10)
    with torch.no_grad(), rh.noise_tape(inp["tape"]):
        ref = diff.p_sample_loop(cfg, (B, 263, 1, T), clip_denoised=False, model_kwargs={"y": _y(inp)})
    np.savez_compressed(os.path.join(OUT, "enc_c1.npz"), sample=ref.numpy(),
                        meta=np.array(["L=8 steps=50 B=1 T=196 weights_seed=0 inputs_seed=10 scale=2.5"]))
    print("enc_c1.npz:", tuple(ref.shape), float(ref.abs().mean()))


def gen_enc_l3():
    """A third trans_enc setting on seeds no other fixture uses: L=3, 6 steps, B=2, T=31, ragged lengths, per-sample
    scales; the final sample, the timestep map and the diffusion tables of the reference."""
    ns = rh.load_reference()
    L, steps, B, T = 3, 6, 2, 31
    sd = syn.synthetic_state_dict(num_layers=L, seed=7)
    model, diff = rh.build(rh.default_args(layers=L, diffusion_steps=steps), state_dict=sd)
    cfg = ns.sampler_util.ClassifierFreeSampleModel(model)
    inp = syn.synthetic_inputs(B, nframes=T, steps=steps, seed=21, lengths=[31, 9], scale=torch.tensor([3.0, 0.5]))
    with torch.no_grad(), rh.noise_tape(inp["tape"]):
        ref = diff.p_sample_loop(cfg, (B, 263, 1, T), clip_denoised=False, model_kwargs={"y": _y(inp)})
    out = {"meta": np.array(["L=3 steps=6 B=2 T=31 weights_seed=7 inputs_seed=21 lengths=31,9 scales=3,0.5"]),
           "sample": ref.numpy(), "timestep_map": np.array(diff.timestep_map, dtype=np.int64)}
    for n in TABLE_NAMES:
        out["table_" + n] = getattr(diff, n)
    np.savez_compressed(os.path.join(OUT, "enc_l3.npz"), **out)
    print("enc_l3.npz:", tuple(ref.shape))


def gen_a2m_small():
    ns = rh.load_reference()
    L, steps, B, T = 2, 3, 4, 60
    args = rh.default_args(dataset="humanact12", layers=L, diffusion_steps=steps, cond_mask_prob=0.0)
    sd = syn.synthetic_state_dict(num_layers=L, input_feats=150, cond_mode="action", num_actions=12, seed=2)
    model, diff = rh.build(args, num_actions=12, state_dict=sd)
    inp = syn.synthetic_inputs(B, njoints=25, nfeats=6, nframes=T, steps=steps, seed=12, lengths=[60, 60, 45, 30])
    action = torch.tensor([[3], [0], [11], [7]])
    y = dict(mask=inp["mask"], lengths=inp["lengths"], action=action)
    with torch.no_grad(), rh.noise_tape(inp["tape"]):
        ref = diff.p_sample_loop(model, (B, 25, 6, T), clip_denoised=False, model_kwargs={"y": y})
    np.savez_compressed(os.path.join(OUT, "a2m_small.npz"), sample=ref.numpy(), action=action.numpy(),
                        meta=np.array(["humanact12 L=2 steps=3 B=4 T=60 weights_seed=2 inputs_seed=12 lengths=60,60,45,30"]))
    print("a2m_small.npz:", tuple(ref.shape))


def gen_dip_small():
    """trans_dec + bert dims (DiP): L=2, ctx 20 + pred 40, 3 steps, ragged text mask, per-sample scales."""
    ns = rh.load_reference()
    L, steps, B, ctx, pred, Mt = 2, 3, 3, 20, 40, 7
    args = rh.default_args(layers=L, diffusion_steps=steps, arch="trans_dec", text_encoder_type="bert", context_len=ctx, pred_len=pred)
    sd = syn.synthetic_state_dict(arch="trans_dec", num_layers=L, cond_dim=768, seed=4)
    model, diff = rh.build(args, state_dict=sd)
    cfg = ns.sampler_util.ClassifierFreeSampleModel(model)
    enc, tmask, prefix = syn.synthetic_dip_inputs(B, Mt, ctx)
    inp = syn.synthetic_inputs(B, nframes=pred, steps=steps, seed=13, lengths=[40, 33, 12], scale=torch.tensor([7.5, 2.0, 1.0]))

    def y():
        return dict(mask=inp["mask"].clone(), lengths=inp["lengths"], text_embed=(enc, tmask), scale=inp["scale"], prefix=prefix)
    out = {"meta": np.array(["DiP L=2 steps=3 B=3 ctx=20 pred=40 Mt=7 weights_seed=4 inputs_seed=13 dip_seed=3 lengths=40,33,12 scales=7.5,2,1"])}
    with torch.no_grad():
        t = torch.full((B,), 1, dtype=torch.long)
        out["fwd_cfg"] = cfg(inp["tape"][0], t, y=y()).numpy()
        with rh.noise_tape(inp["tape"]):
            out["ddpm"] = diff.p_sample_loop(cfg, (B, 263, 1, pred), clip_denoised=False, model_kwargs={"y": y()}).numpy()
    out["text_mask"] = tmask.numpy()
    np.savez_compressed(os.path.join(OUT, "dip_small.npz"), **out)
    print("dip_small.npz:", {k: v.shape for k, v in out.items() if k != "meta"})


def gen_ric():
    """Post-loop step of sample/generate.py:161-166 (inv_transform + recover_from_ric + permute) by the reference's own
    functions, HumanML3D (263 -> 22 joints) and KIT (251 -> 21 joints)."""
    rh.load_reference()
    mp = importlib.import_module("data_loaders.humanml.scripts.motion_process")
    out = {"meta": np.array(["sample = randn(torch seed 100+D) [3, D, 1, 40] * 0.8; mean/std = synthetic_norm_stats(D, seed 7)"])}
    for D, J in ((263, 22), (251, 21)):
        g = torch.Generator().manual_seed(100 + D)
        sample = torch.randn(3, D, 1, 40, generator=g) * 0.8
        mean, std = syn.synthetic_norm_stats(D, seed=7)
        data = (sample.cpu().permute(0, 2, 3, 1) * std.numpy() + mean.numpy()).float()      # dataset.py:309-310 on numpy stats
        xyz = mp.recover_from_ric(data, J)
        out["xyz_%d" % D] = xyz.view(-1, *xyz.shape[2:]).permute(0, 2, 3, 1).contiguous().numpy()
        out["ric_%d" % D] = mp.recover_from_ric(sample.permute(0, 2, 3, 1).contiguous(), J).numpy()   # no de-normalisation
    np.savez_compressed(os.path.join(OUT, "ric.npz"), **out)
    print("ric.npz:", {k: v.shape for k, v in out.items() if k != "meta"})


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    gen_schedule()
    gen_enc_small()
    gen_enc_c1()
    gen_enc_l3()
    gen_a2m_small()
    gen_dip_small()
    gen_ric()

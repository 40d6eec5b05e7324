"""Time target-location conditioning on the DiP configuration: trans_dec, 8 layers, B=128, 40-frame chunks with a
20-frame prefix, 10 diffusion steps per chunk, guidance 7.5, 5 chunks (196 frames) through AutoRegressiveSampler --
with and without targets (multi encoder, mixed per-sample joint sets), alternated, CUDA events around synchronised
batches; and b200mdm_set_target alone (each encoder type, B=128, many launches).  Prints the card and its power limit.

    python tools/time_target.py [--reps N]
"""
import ctypes
import os
import subprocess
import sys
from types import SimpleNamespace

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import b200mdm  # noqa: E402
from b200mdm import _lib  # noqa: E402

B, ctx, pred, Mt, steps, need = 128, 20, 40, 16, 10, 196
REPS = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 10


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name()


def dip(encoder, seed=23):
    args = SimpleNamespace(dataset="humanml", unconstrained=False, latent_dim=512, layers=8, cond_mask_prob=0.1,
                           arch="trans_dec", emb_trans_dec=False, text_encoder_type="bert", pos_embed_max_len=5000,
                           mask_frames=True, pred_len=pred, context_len=ctx, diffusion_steps=steps, noise_schedule="cosine",
                           sigma_small=True, lambda_vel=0.0, lambda_rcxyz=0.0, lambda_fc=0.0,
                           autoregressive_include_prefix=False, multi_target_cond=True, multi_encoder_type=encoder,
                           target_enc_layers=1)
    model, diffusion = b200mdm.create_model_and_diffusion(args, SimpleNamespace(dataset=SimpleNamespace()))
    b200mdm.load_model_wo_clip(model, b200mdm.synthetic_state_dict(arch="trans_dec", num_layers=8, cond_dim=768, seed=seed,
                                                                   target_encoder=encoder))
    model.to("cuda").eval()
    return b200mdm.ClassifierFreeSampleModel(model), model, diffusion, args


def main():
    torch.cuda.set_device(0)
    print("card:", card())
    pool = [[], ["traj"], ["left_wrist", "head"], ["pelvis"], ["right_foot", "left_foot", "traj"], ["right_wrist"]]
    sets, heading = [pool[b % len(pool)] for b in range(B)], [b % 3 == 0 for b in range(B)]
    tgt = b200mdm.synthetic_targets(B, sets, heading, seed=5)
    cfg, model, diffusion, args = dip("multi")
    enc, tmask, prefix = b200mdm.synthetic_dip_inputs(B, Mt, ctx, seed=35)
    y0 = dict(mask=torch.ones(B, 1, 1, pred, dtype=torch.bool, device="cuda"), lengths=torch.full((B,), pred, device="cuda"),
              text_embed=(enc.cuda(), tmask.cuda()), prefix=prefix.cuda(), scale=torch.full((B,), 7.5, device="cuda"))
    yt = dict(y0, target_cond=tgt["target_cond"].cuda(), target_joint_names=tgt["target_joint_names"],
              is_heading=tgt["is_heading"].cuda())
    g = torch.Generator(device="cuda").manual_seed(1)
    shape = (B, 263, 1, pred)
    n5 = torch.randn(5, *shape, device="cuda", generator=g)
    t5 = torch.randn(5, steps, *shape, device="cuda", generator=g)
    sampler = b200mdm.AutoRegressiveSampler(args, diffusion.p_sample_loop, required_frames=need)

    def run(y):
        return sampler.sample(cfg, (B, 263, 1, need), clip_denoised=False, model_kwargs={"y": y}, noise=n5, noise_tape=t5)

    for _ in range(3):
        run(y0), run(yt)
    torch.cuda.synchronize()
    times = {"without": [], "with": []}
    for _ in range(REPS):                          # alternate the two so that drift hits both alike
        for key, y in (("without", y0), ("with", yt)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            run(y)
            e1.record()
            torch.cuda.synchronize()
            times[key].append(e0.elapsed_time(e1))
    for key in ("without", "with"):
        ts = sorted(times[key])
        med = ts[len(ts) // 2]
        print("DiP B=%d, 5 chunks x %d steps, guidance 7.5, %s targets: median %.2f ms per 196-frame batch (min %.2f, max %.2f, "
              "%d reps) = %.3f ms per step incl. per-chunk set-up -> %.0f motions/s"
              % (B, steps, key, med, ts[0], ts[-1], len(ts), med / (5 * steps), B / med * 1e3))

    # the encoder alone: b200mdm_set_target over many launches, per encoder type
    lib = _lib.load()
    for encoder in ("single", "multi", "split"):
        _, m, _, _ = dip(encoder, seed=7)
        eng = m.engine()
        tc = tgt["target_cond"].cuda().contiguous()
        from b200mdm.engine import target_validity
        valid = target_validity(m.target_rows, sets, tgt["is_heading"])
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        call = lambda: _lib.check(lib.b200mdm_set_target(eng.h, B, ctypes.c_void_p(tc.data_ptr()),
                                                         valid.ctypes.data_as(ctypes.c_void_p), st))
        for _ in range(20):
            call()
        n = 500
        eng.launch_count(reset=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            call()
        e1.record()
        torch.cuda.synchronize()
        print("b200mdm_set_target %-6s B=%d: %.1f us per call (%d calls, %d kernels per call; includes the host-side "
              "validity staging and its host-to-device copy)" % (encoder, B, e0.elapsed_time(e1) * 1e3 / n, n,
                                                                       eng.launch_count() // n))
        lib.b200mdm_set_target(eng.h, B, None, None, st)


if __name__ == "__main__":
    main()

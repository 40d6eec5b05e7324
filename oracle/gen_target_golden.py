"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/target_small.npz by running the UNMODIFIED reference
(via oracle/ref_harness.py) on CPU in the build container:

    python -m oracle.gen_target_golden

target_small.npz: target-location conditioning (multi_target_cond, model/mdm.py:64-73,197-199,399-480): DiP L=2
(ctx 20 + pred 40) with the single encoder (target_enc_layers 1 and 2), multi and split, and trans_enc L=2 with single;
per case one CFG forward and a 3-step p_sample_loop; per-sample joint sets [], ['traj'], two joints, heading on and off;
one target_uncond=True forward (asserted here to equal the forward without target keys, bit for bit).  Weights and
inputs come from the seeded streams of motion-diffusion-model_b200/synthetic.py, so tests rebuild them
(tests/target_cases.py).  The other fixtures are written by oracle/gen_golden.py and are not touched here.
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

TARGET_SETS = [[], ["traj"], ["left_wrist", "head"]]
TARGET_HEADING = [True, False, True]


def gen_target_small():
    """multi_target_cond models of the reference (model/mdm.py:64-73,197-199) on the synthetic target weights."""
    ns = rh.load_reference()
    L, steps = 2, 3
    tgt3 = syn.synthetic_targets(3, TARGET_SETS, TARGET_HEADING, seed=19)
    out = {"meta": np.array(["L=2 steps=3; B=3 cases: samples 0-2 of the targets, B=2 cases: samples 1-2; target sets %r "
                             "heading %r target seed 19; DiP ctx=20 pred=40 Mt=7 dip_seed=3 inputs_seed=13 lengths=40,33,12 "
                             "scales=7.5,2,1 (B=2: the first two); trans_enc T=16 inputs_seed=11 lengths=16,11,5 scales=2.5,1,4"
                             % (TARGET_SETS, TARGET_HEADING)]),
           "target_cond": tgt3["target_cond"].numpy(), "is_heading": tgt3["is_heading"].numpy()}
    # (name, arch, encoder, target_enc_layers, weight seed, batch): B = 2 for three of the DiP cases keeps the file < 1 MB
    cases = [("dip_single1", "trans_dec", "single", 1, 41, 2), ("dip_single2", "trans_dec", "single", 2, 42, 2),
             ("dip_multi", "trans_dec", "multi", 1, 43, 3), ("dip_split", "trans_dec", "split", 1, 44, 2),
             ("enc_single", "trans_enc", "single", 1, 45, 3)]
    for name, arch, enc_type, layers, wseed, B in cases:
        tgt = {k: v[3 - B:] for k, v in tgt3.items()}
        tkw = dict(multi_target_cond=True, multi_encoder_type=enc_type, target_enc_layers=layers)
        if arch == "trans_dec":
            ctx, pred, Mt = 20, 40, 7
            args = rh.default_args(layers=L, diffusion_steps=steps, arch="trans_dec", text_encoder_type="bert",
                                   context_len=ctx, pred_len=pred, **tkw)
            sd = syn.synthetic_state_dict(arch="trans_dec", num_layers=L, cond_dim=768, seed=wseed, target_encoder=enc_type,
                                          target_enc_layers=layers)
            enc, tmask, prefix = syn.synthetic_dip_inputs(B, Mt, ctx)
            inp = syn.synthetic_inputs(B, nframes=pred, steps=steps, seed=13, lengths=[40, 33, 12][:B],
                                       scale=torch.tensor([7.5, 2.0, 1.0][:B]))

            def y(**extra):
                return dict(mask=inp["mask"].clone(), lengths=inp["lengths"], text_embed=(enc, tmask), scale=inp["scale"],
                            prefix=prefix, target_cond=tgt["target_cond"], target_joint_names=tgt["target_joint_names"],
                            is_heading=tgt["is_heading"], **extra)
            T = pred
        else:
            T = 16
            args = rh.default_args(layers=L, diffusion_steps=steps, **tkw)
            sd = syn.synthetic_state_dict(num_layers=L, seed=wseed, target_encoder=enc_type, target_enc_layers=layers)
            inp = syn.synthetic_inputs(B, nframes=T, steps=steps, seed=11, lengths=[16, 11, 5],
                                       scale=torch.tensor([2.5, 1.0, 4.0]))

            def y(**extra):
                return dict(mask=inp["mask"], lengths=inp["lengths"], text_embed=inp["text_embed"],
                            scale=inp["scale"], target_cond=tgt["target_cond"], target_joint_names=tgt["target_joint_names"],
                            is_heading=tgt["is_heading"], **extra)
        model, diff = rh.build(args, state_dict=sd)
        cfg = ns.sampler_util.ClassifierFreeSampleModel(model)
        with torch.no_grad():
            t = torch.full((B,), 1, dtype=torch.long)
            out[name + "_fwd"] = cfg(inp["tape"][0], t, y=y()).numpy()
            with rh.noise_tape(inp["tape"]):
                out[name + "_ddpm"] = diff.p_sample_loop(cfg, (B, 263, 1, T), clip_denoised=False, model_kwargs={"y": y()}).numpy()
            if name == "dip_multi":
                out[name + "_tuncond_fwd"] = cfg(inp["tape"][0], t, y=y(target_uncond=True)).numpy()
                yn = y()
                for k in ("target_cond", "target_joint_names", "is_heading"):
                    yn.pop(k)
                assert np.array_equal(out[name + "_tuncond_fwd"], cfg(inp["tape"][0], t, y=yn).numpy())
    np.savez_compressed(os.path.join(OUT, "target_small.npz"), **out)
    print("target_small.npz:", {k: v.shape for k, v in out.items() if k != "meta"})


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    gen_target_small()

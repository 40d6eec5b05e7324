"""The cases of golden/target_small.npz (oracle/gen_target_golden.py), rebuilt from their seeds: weights, inputs
and the reference-format `y` of each; shared by test_target_cond_cpu.py and test_target_cond_gpu.py."""
from types import SimpleNamespace

import torch

import b200mdm
from conftest import default_args

SETS = [[], ["traj"], ["left_wrist", "head"]]
HEADING = [True, False, True]
ROWS = ["pelvis", "left_foot", "right_foot", "left_wrist", "right_wrist", "head", "traj", "heading"]
# name -> (arch, encoder, target_enc_layers, weight seed, batch)
CASES = {"dip_single1": ("trans_dec", "single", 1, 41, 2), "dip_single2": ("trans_dec", "single", 2, 42, 2),
         "dip_multi": ("trans_dec", "multi", 1, 43, 3), "dip_split": ("trans_dec", "split", 1, 44, 2),
         "enc_single": ("trans_enc", "single", 1, 45, 3)}
L, STEPS, CTX, PRED, MT, T_ENC = 2, 3, 20, 40, 7, 16


def targets(B):
    t = b200mdm.synthetic_targets(3, SETS, HEADING, seed=19)
    return {k: v[3 - B:] for k, v in t.items()}


def args_of(name, layers=L, steps=STEPS):
    arch, enc, tl, _, _ = CASES[name]
    kw = dict(multi_target_cond=True, multi_encoder_type=enc, target_enc_layers=tl)
    if arch == "trans_dec":
        return default_args(layers=layers, diffusion_steps=steps, arch="trans_dec", text_encoder_type="bert",
                            context_len=CTX, pred_len=PRED, **kw)
    return default_args(layers=layers, diffusion_steps=steps, **kw)


def build(name, device=None):
    """(model, diffusion, state_dict, inputs dict, y(**extra) -> fresh y, T)."""
    arch, enc, tl, wseed, B = CASES[name]
    model, diffusion = b200mdm.create_model_and_diffusion(args_of(name), SimpleNamespace(dataset=SimpleNamespace()))
    dev = (lambda t: t.to(device)) if device else (lambda t: t)
    tgt = targets(B)
    if arch == "trans_dec":
        sd = b200mdm.synthetic_state_dict(arch="trans_dec", num_layers=L, cond_dim=768, seed=wseed, target_encoder=enc,
                                          target_enc_layers=tl)
        enc_t, tmask, prefix = b200mdm.synthetic_dip_inputs(B, MT, CTX)
        inp = b200mdm.synthetic_inputs(B, nframes=PRED, steps=STEPS, seed=13, lengths=[40, 33, 12][:B],
                                       scale=torch.tensor([7.5, 2.0, 1.0][:B]))
        inp.update(enc=enc_t, tmask=tmask, prefix=prefix)

        def y(**extra):
            d = dict(mask=dev(inp["mask"].clone()), lengths=dev(inp["lengths"]), text_embed=(dev(enc_t), dev(tmask)),
                     scale=dev(inp["scale"]), prefix=dev(prefix), target_cond=dev(tgt["target_cond"]),
                     target_joint_names=tgt["target_joint_names"], is_heading=dev(tgt["is_heading"]))
            d.update(extra)
            return d
        T = PRED
    else:
        sd = b200mdm.synthetic_state_dict(num_layers=L, seed=wseed, target_encoder=enc, target_enc_layers=tl)
        inp = b200mdm.synthetic_inputs(B, nframes=T_ENC, steps=STEPS, seed=11, lengths=[16, 11, 5],
                                       scale=torch.tensor([2.5, 1.0, 4.0]))

        def y(**extra):
            d = dict(mask=dev(inp["mask"]), lengths=dev(inp["lengths"]), text_embed=dev(inp["text_embed"]),
                     scale=dev(inp["scale"]), target_cond=dev(tgt["target_cond"]),
                     target_joint_names=tgt["target_joint_names"], is_heading=dev(tgt["is_heading"]))
            d.update(extra)
            return d
        T = T_ENC
    b200mdm.load_model_wo_clip(model, sd)
    return model, diffusion, sd, inp, y, T


def without_target(y):
    for k in ("target_cond", "target_joint_names", "is_heading", "target_uncond"):
        y.pop(k, None)
    return y

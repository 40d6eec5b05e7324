"""TEST INFRASTRUCTURE ONLY -- plain-torch fp32 restatement of the reference's target-location conditioning
(multi_target_cond), on top of oracle/mdm_oracle.py.  Only tests/ and tools may import this; the product path never does.

What is restated (paths relative to the reference repo):
  * EmbedTargetLoc{Single,Multi,Split} ... model/mdm.py:399-480, utils/misc.py:5-16 (target_embedding)
  * time_emb += embed_target_cond(...) ... model/mdm.py:197-199: the MDM.forward variants below take the embedding as
                                           `target` [B, d] and add it to the timestep embedding, which reaches the network
                                           only through emb = text_emb + time_emb (token 0 for trans_enc, every memory row
                                           for trans_dec)
Pinned by tests/golden/target_small.npz, produced by oracle/gen_target_golden.py from the reference itself.
"""
import torch
import torch.nn.functional as F

from . import mdm_oracle as mo


def target_validity(rows, target_joint_names, is_heading):
    """validity [B, n] of EmbedTarget*.forward (model/mdm.py:411-416); rows = all_goal_joint_names + ['traj', 'heading']."""
    v = torch.zeros(len(target_joint_names), len(rows))
    for b, names in enumerate(target_joint_names):
        for j in list(names) + (["heading"] if bool(is_heading[b]) else []):
            v[b, rows.index(j)] = 1.0
    return v


def target_embedding(W, encoder, rows, target_cond, target_joint_names, is_heading, layers=1):
    """embed_target_cond(y['target_cond'], y['target_joint_names'], y['is_heading']) -> [B, d] (model/mdm.py:399-480).
    encoder: 'single' | 'multi' | 'split' (args.multi_encoder_type); rows: all_goal_joint_names + ['traj', 'heading']."""
    p = "embed_target_cond."
    tc = target_cond.float()
    B, n = tc.shape[0], len(rows)
    valid = target_validity(rows, target_joint_names, is_heading)
    x = torch.cat([tc, valid[..., None]], dim=-1)                          # [B, n, 4]; invalid rows fed in as they are
    if encoder == "single":
        h = mo._lin(x.reshape(B, 4 * n), W[p + "mlp.0.weight"], W[p + "mlp.0.bias"])
        for l in range(1, layers + 1):
            h = mo._lin(F.silu(h), W[p + "mlp.%d.weight" % (2 * l)], W[p + "mlp.%d.bias" % (2 * l)])
        return h
    if encoder == "split":
        outs = []
        for j in range(n):
            q = p + "mini_mlps.%d." % j
            h = mo._lin(x[:, j], W[q + "0.weight"], W[q + "0.bias"])
            for l in range(1, layers + 1):
                h = mo._lin(F.silu(h), W[q + "%d.weight" % (2 * l)], W[q + "%d.bias" % (2 * l)])
            outs.append(h)
        return torch.cat(outs, dim=-1)
    w = W[p + "target_all_loc_emb.weights"]
    wn = w / w.sum()                                                        # utils/misc.py:12 (sum, not softmax)
    e = torch.zeros(B, n, W.d)
    for j, name in enumerate(rows):
        q = p + "target_loc_emb.%s." % name
        sel = valid[:, j] > 0
        if sel.any():
            h = F.silu(mo._lin(tc[sel, j], W[q + "0.weight"], W[q + "0.bias"]))
            e[sel, j] = mo._lin(h, W[q + "2.weight"], W[q + "2.bias"])
    return torch.einsum("j,bjd->bd", wn, e)


def _time_emb(W, t_model, target):
    """time_emb + target embedding, [B, d] (model/mdm.py:195-199)."""
    return mo.timestep_embedding(W, t_model)[None, :] + target


def denoise_enc(W, x, t_model, cond, target, lengths=None, mask_frames=True, uncond=False):
    """mdm_oracle.denoise_enc (text-conditioned trans_enc) with the target embedding [B, d] added to time_emb."""
    B, J, Fe, T = x.shape
    c = torch.zeros_like(cond[0]) if uncond else cond[0]                    # mask_cond force_mask
    tok0 = mo._lin(c, W["embed_text.weight"], W["embed_text.bias"]) + _time_emb(W, t_model, target)
    frames = x.permute(0, 3, 1, 2).reshape(B, T, J * Fe)
    hf = mo._lin(frames, W["input_process.poseEmbedding.weight"], W["input_process.poseEmbedding.bias"])
    h = torch.cat([tok0[:, None, :], hf], dim=1) + W.pe[: T + 1][None]
    keymask = None
    if mask_frames and lengths is not None and T > 1:
        keymask = torch.arange(T + 1)[None, :] >= (lengths[:, None] + 1)
    h = mo.encoder_stack(W, h, keymask)[:, 1:]
    out = mo._lin(h, W["output_process.poseFinal.weight"], W["output_process.poseFinal.bias"])
    return out.reshape(B, T, J, Fe).permute(0, 2, 3, 1).contiguous()


def denoise_dec(W, x, t_model, enc_text, text_mask, prefix, target, lengths=None, mask_frames=True, uncond=False):
    """mdm_oracle.denoise_dec (DiP) with the target embedding [B, d] added to time_emb, i.e. to every memory row."""
    B, J, Fe, Tp = x.shape
    ctx = prefix.shape[-1]
    enc = torch.zeros_like(enc_text) if uncond else enc_text
    mem = mo._lin(enc.permute(1, 0, 2), W["embed_text.weight"], W["embed_text.bias"]) + _time_emb(W, t_model, target)[:, None, :]
    xf = torch.cat([prefix, x], dim=-1)
    T = ctx + Tp
    frames = xf.permute(0, 3, 1, 2).reshape(B, T, J * Fe)
    h = mo._lin(frames, W["input_process.poseEmbedding.weight"], W["input_process.poseEmbedding.bias"]) + W.pe[:T][None]
    keymask = None
    if mask_frames and lengths is not None and T > 1:
        keymask = torch.arange(T)[None, :] >= (lengths[:, None] + ctx)
    h = mo.decoder_stack(W, h, mem, keymask, text_mask)[:, ctx:]
    out = mo._lin(h, W["output_process.poseFinal.weight"], W["output_process.poseFinal.bias"])
    return out.reshape(B, Tp, J, Fe).permute(0, 2, 3, 1).contiguous()


def cfg_denoise_enc(W, x, t_model, cond, scale, target, lengths=None, mask_frames=True):
    """ClassifierFreeSampleModel.forward: the guidance wrapper deep-copies y, so both halves carry the target."""
    oc = denoise_enc(W, x, t_model, cond, target, lengths, mask_frames, False)
    ou = denoise_enc(W, x, t_model, cond, target, lengths, mask_frames, True)
    return ou + scale.view(-1, 1, 1, 1) * (oc - ou)


def cfg_denoise_dec(W, x, t_model, enc_text, text_mask, prefix, scale, target, lengths=None, mask_frames=True):
    oc = denoise_dec(W, x, t_model, enc_text, text_mask, prefix, target, lengths, mask_frames, False)
    ou = denoise_dec(W, x, t_model, enc_text, text_mask, prefix, target, lengths, mask_frames, True)
    return ou + scale.view(-1, 1, 1, 1) * (oc - ou)


def sample_loop(W, tables, timestep_map, tape, cond, scale, target, lengths=None, mask_frames=True):
    """p_sample_loop with CFG (mdm_oracle.sample_loop's DDPM path) and a target."""
    n = len(tables["betas"])
    x = tape[0].clone()
    for k, i in enumerate(range(n - 1, -1, -1)):
        x0 = cfg_denoise_enc(W, x, int(timestep_map[i]), cond, scale, target, lengths, mask_frames)
        x, _ = mo.p_sample_step(tables, x0, x, i, tape[1 + k])
    return x


def sample_loop_dec(W, tables, timestep_map, tape, enc_text, text_mask, prefix, scale, target, lengths=None, mask_frames=True):
    n = len(tables["betas"])
    x = tape[0].clone()
    for k, i in enumerate(range(n - 1, -1, -1)):
        x0 = cfg_denoise_dec(W, x, int(timestep_map[i]), enc_text, text_mask, prefix, scale, target, lengths, mask_frames)
        x, _ = mo.p_sample_step(tables, x0, x, i, tape[1 + k])
    return x

"""TEST INFRASTRUCTURE ONLY -- plain-torch fp32 restatement of the reference's sampling hot path
(the floating-point oracle).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import this; the product path never does.

What is restated (paths relative to /root/reference):
  * MDM.forward, trans_enc branch .............. model/mdm.py:189-283  (+ :296-386 sub-modules)
  * nn.TransformerEncoderLayer (post-norm, gelu) . torch, built at model/mdm.py:77-84
  * ClassifierFreeSampleModel.forward ........... utils/sampler_util.py:27-34
  * p_mean_variance / q_posterior / p_sample .... diffusion/gaussian_diffusion.py:246-381, 489-541
  * ddim_sample ................................. diffusion/gaussian_diffusion.py:729-779
  * q_sample .................................... diffusion/gaussian_diffusion.py:226-244
  * p_sample_loop(_progressive) ................. diffusion/gaussian_diffusion.py:591-727

Layout: batch-major [B, S, d]; the cond/uncond CFG pair is evaluated as two halves of one batch.
Pinned by tests/golden/*.npz, produced by oracle/gen_golden.py from the reference itself
(tests/test_oracle_cpu.py).

`cast` (optional) rounds both GEMM operands through a narrower dtype and back; it exists only for
the precision studies behind DESIGN.md section 2 and is None for parity work.
"""
import math

import numpy as np
import torch
import torch.nn.functional as F

from . import schedule_oracle as so


class OracleWeights:
    """Reference state_dict -> tensors used by the restatement (names as in SURVEY.md A.4)."""

    def __init__(self, sd, num_layers, arch="trans_enc", num_heads=4, pos_embed_max_len=5000):
        self.sd = {k: v.detach().float() for k, v in sd.items() if torch.is_tensor(v)}
        self.L = num_layers
        self.H = num_heads
        self.arch = arch
        self.d = self.sd["input_process.poseEmbedding.weight"].shape[0]
        self.pe = so.positional_table(pos_embed_max_len, self.d)

    def __getitem__(self, k):
        return self.sd[k]


def _lin(x, w, b, cast=None):
    if cast is not None:
        x = x.to(cast).float()
        w = w.to(cast).float()
    y = x @ w.t()
    return y if b is None else y + b


def timestep_embedding(W, t_model, cast=None):
    """TimestepEmbedder.forward (model/mdm.py:329-330): MLP(pe[t]).  t_model: int (already mapped
    through timestep_map, respace.py:127)."""
    e = W.pe[int(t_model)]
    h = _lin(e, W["embed_timestep.time_embed.0.weight"], W["embed_timestep.time_embed.0.bias"])
    h = F.silu(h)
    return _lin(h, W["embed_timestep.time_embed.2.weight"], W["embed_timestep.time_embed.2.bias"])


def _mha_self(h, lw, keymask, H, cast=None):
    """nn.MultiheadAttention self-attention, eval mode.  h [B,S,d]; keymask [B,S] True = ignore."""
    B, S, d = h.shape
    dh = d // H
    qkv = _lin(h, lw["in_w"], lw["in_b"], cast)
    q, k, v = qkv.split(d, dim=-1)
    q = q.view(B, S, H, dh).transpose(1, 2)
    k = k.view(B, S, H, dh).transpose(1, 2)
    v = v.view(B, S, H, dh).transpose(1, 2)
    if cast is not None:
        q, k, v = (z.to(cast).float() for z in (q, k, v))
    s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
    if keymask is not None:
        s = s.masked_fill(keymask[:, None, None, :], float("-inf"))
    p = torch.softmax(s, dim=-1)
    if cast is not None:
        p = p.to(cast).float()
    a = (p @ v).transpose(1, 2).reshape(B, S, d)
    return _lin(a, lw["out_w"], lw["out_b"], cast)


def encoder_stack(W, h, keymask, cast=None):
    """8 x TransformerEncoderLayer, post-norm, exact-erf GELU, eps 1e-5, no final norm."""
    d = W.d
    for l in range(W.L):
        p = "seqTransEncoder.layers.%d." % l
        lw = dict(in_w=W[p + "self_attn.in_proj_weight"], in_b=W[p + "self_attn.in_proj_bias"],
                  out_w=W[p + "self_attn.out_proj.weight"], out_b=W[p + "self_attn.out_proj.bias"])
        a = _mha_self(h, lw, keymask, W.H, cast)
        h = F.layer_norm(h + a, (d,), W[p + "norm1.weight"], W[p + "norm1.bias"], 1e-5)
        f = F.gelu(_lin(h, W[p + "linear1.weight"], W[p + "linear1.bias"], cast))
        f = _lin(f, W[p + "linear2.weight"], W[p + "linear2.bias"], cast)
        h = F.layer_norm(h + f, (d,), W[p + "norm2.weight"], W[p + "norm2.bias"], 1e-5)
    return h


def denoise_enc(W, x, t_model, cond, lengths=None, mask_frames=True, uncond=False, action=None, cast=None):
    """MDM.forward for arch=trans_enc (model/mdm.py:189-283).

    x [B,J,F,T] fp32; t_model python int (same for the whole batch, gaussian_diffusion.py:709);
    cond: text_embed [1,B,C] (cond_mode text), or None (no_cond); action: [B,1] ints (cond_mode
    action); lengths [B] or None (=> no key mask, mdm.py:241-247)."""
    B, J, Fe, T = x.shape
    d = W.d
    temb = timestep_embedding(W, t_model)                                   # [d]
    if action is not None:                                                  # mdm.py:225-227
        aemb = W["embed_action.action_embedding"][action[:, 0].long()]
        tok0 = temb[None, :] + (torch.zeros_like(aemb) if uncond else aemb)
    elif cond is not None:                                                  # mdm.py:209-220
        c = cond[0]
        if uncond:                                                          # mask_cond force_mask
            c = torch.zeros_like(c)
        tok0 = _lin(c, W["embed_text.weight"], W["embed_text.bias"], None) + temb[None, :]
    else:
        tok0 = temb[None, :].expand(B, d)
    frames = x.permute(0, 3, 1, 2).reshape(B, T, J * Fe)                    # mdm.py:344-345
    hf = _lin(frames, W["input_process.poseEmbedding.weight"], W["input_process.poseEmbedding.bias"], cast)
    h = torch.cat([tok0[:, None, :], hf], dim=1) + W.pe[: T + 1][None]      # mdm.py:251-252
    keymask = None
    if mask_frames and lengths is not None and T > 1:                       # mdm.py:241-247
        keymask = torch.arange(T + 1)[None, :] >= (lengths[:, None] + 1)
    h = encoder_stack(W, h, keymask, cast)[:, 1:]                           # mdm.py:253
    out = _lin(h, W["output_process.poseFinal.weight"], W["output_process.poseFinal.bias"], cast)
    return out.reshape(B, T, J, Fe).permute(0, 2, 3, 1).contiguous()        # mdm.py:384-385


def cfg_denoise_enc(W, x, t_model, cond, scale, lengths=None, mask_frames=True, action=None, cast=None):
    """ClassifierFreeSampleModel.forward (utils/sampler_util.py:27-34)."""
    oc = denoise_enc(W, x, t_model, cond, lengths, mask_frames, False, action, cast)
    ou = denoise_enc(W, x, t_model, cond, lengths, mask_frames, True, action, cast)
    return ou + scale.view(-1, 1, 1, 1) * (oc - ou)


def f32(tab, i):
    """_extract_into_tensor (gaussian_diffusion.py:1602-1615): fp64 table value -> fp32 scalar."""
    return torch.tensor(np.float32(tab[i]))


def p_sample_step(tables, x0, x_t, i, eps, inpaint=None):
    """p_mean_variance START_X / FIXED_SMALL + p_sample (gaussian_diffusion.py:300-304, 325-369, 525-540).
    x0 = model output; i = index into the (respaced) schedule; eps = the randn_like draw."""
    if inpaint is not None:
        m, motion = inpaint
        x0 = (x0 * ~m) + (motion * m)
    mean = f32(tables["posterior_mean_coef1"], i) * x0 + f32(tables["posterior_mean_coef2"], i) * x_t
    nz = 0.0 if i == 0 else 1.0
    return mean + nz * torch.exp(0.5 * f32(tables["posterior_log_variance_clipped"], i)) * eps, x0


def ddim_step(tables, x0, x_t, i, eps, eta=0.0):
    """ddim_sample (gaussian_diffusion.py:729-779)."""
    e = (f32(tables["sqrt_recip_alphas_cumprod"], i) * x_t - x0) / f32(tables["sqrt_recipm1_alphas_cumprod"], i)
    ab = f32(tables["alphas_cumprod"], i)
    abp = f32(tables["alphas_cumprod_prev"], i)
    sigma = eta * torch.sqrt((1 - abp) / (1 - ab)) * torch.sqrt(1 - ab / abp)
    mean = x0 * torch.sqrt(abp) + torch.sqrt(1 - abp - sigma ** 2) * e
    nz = 0.0 if i == 0 else 1.0
    return mean + nz * sigma * eps


def q_sample(tables, x_start, i, noise):
    """q_sample (gaussian_diffusion.py:226-244)."""
    return f32(tables["sqrt_alphas_cumprod"], i) * x_start + f32(tables["sqrt_one_minus_alphas_cumprod"], i) * noise


def sample_loop(W, tables, timestep_map, tape, cond, scale, lengths=None, mask_frames=True, action=None,
                sampler="ddpm", eta=0.0, skip_timesteps=0, init_image=None, inpaint=None, cast=None,
                collect=None):
    """p_sample_loop / ddim_sample_loop with an explicit noise tape [x_T, eps_{T-1}, ..., eps_0].
    scale=None => no CFG wrapper (single conditional forward, guidance_param == 1)."""
    n = len(tables["betas"])
    x = tape[0].clone()
    idx = list(range(n - skip_timesteps))[::-1]
    if skip_timesteps and init_image is None:
        init_image = torch.zeros_like(x)
    if init_image is not None:                                              # gaussian_diffusion.py:698-700
        x = q_sample(tables, init_image, idx[0], x)
    for k, i in enumerate(idx):
        tm = int(timestep_map[i])
        if scale is None:
            x0 = denoise_enc(W, x, tm, cond, lengths, mask_frames, False, action, cast)
        else:
            x0 = cfg_denoise_enc(W, x, tm, cond, scale, lengths, mask_frames, action, cast)
        eps = tape[1 + k]
        if sampler == "ddpm":
            x, _ = p_sample_step(tables, x0, x, i, eps, inpaint)
        else:
            if inpaint is not None:
                m, motion = inpaint
                x0 = (x0 * ~m) + (motion * m)
            x = ddim_step(tables, x0, x, i, eps, eta)
        if collect is not None:
            collect.append(x.clone())
    return x


# ---------------------------------------------------------------------------------------------------------------
# trans_dec (DiP) -- model/mdm.py:203-206, 255-270, 278-280; torch nn.TransformerDecoderLayer (post-norm):
#   x = LN1(x + SelfAttn(x)); x = LN2(x + CrossAttn(x, memory)); x = LN3(x + FFN(x))
def _mha_cross(h, mem, lw, mem_mask, H, cast=None):
    """nn.MultiheadAttention with query = h [B,S,d], key = value = mem [B,Mt,d]; mem_mask [B,Mt] True = ignore."""
    B, S, d = h.shape
    Mt = mem.shape[1]
    dh = d // H
    wq, wk, wv = lw["in_w"].split(d, dim=0)
    bq, bk, bv = lw["in_b"].split(d, dim=0)
    q = _lin(h, wq, bq, cast).view(B, S, H, dh).transpose(1, 2)
    k = _lin(mem, wk, bk, cast).view(B, Mt, H, dh).transpose(1, 2)
    v = _lin(mem, wv, bv, cast).view(B, Mt, H, dh).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
    if mem_mask is not None:
        s = s.masked_fill(mem_mask[:, None, None, :], float("-inf"))
    a = (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(B, S, d)
    return _lin(a, lw["out_w"], lw["out_b"], cast)


def decoder_stack(W, h, mem, tgt_keymask, mem_keymask, cast=None):
    d = W.d
    for l in range(W.L):
        p = "seqTransDecoder.layers.%d." % l
        sa = dict(in_w=W[p + "self_attn.in_proj_weight"], in_b=W[p + "self_attn.in_proj_bias"],
                  out_w=W[p + "self_attn.out_proj.weight"], out_b=W[p + "self_attn.out_proj.bias"])
        ca = dict(in_w=W[p + "multihead_attn.in_proj_weight"], in_b=W[p + "multihead_attn.in_proj_bias"],
                  out_w=W[p + "multihead_attn.out_proj.weight"], out_b=W[p + "multihead_attn.out_proj.bias"])
        h = F.layer_norm(h + _mha_self(h, sa, tgt_keymask, W.H, cast), (d,), W[p + "norm1.weight"], W[p + "norm1.bias"], 1e-5)
        h = F.layer_norm(h + _mha_cross(h, mem, ca, mem_keymask, W.H, cast), (d,), W[p + "norm2.weight"], W[p + "norm2.bias"], 1e-5)
        f = _lin(F.gelu(_lin(h, W[p + "linear1.weight"], W[p + "linear1.bias"], cast)), W[p + "linear2.weight"], W[p + "linear2.bias"], cast)
        h = F.layer_norm(h + f, (d,), W[p + "norm3.weight"], W[p + "norm3.bias"], 1e-5)
    return h


def denoise_dec(W, x, t_model, enc_text, text_mask, prefix, lengths=None, mask_frames=True, uncond=False, cast=None):
    """MDM.forward for arch=trans_dec, text_encoder_type=bert, emb_trans_dec=False, prefix completion.

    x [B,J,F,pred]; prefix [B,J,F,ctx]; enc_text [Mt,B,768]; text_mask [B,Mt] True = padding;
    lengths [B] valid frames of x (the context frames are always valid, mdm.py:204-206)."""
    B, J, Fe, Tp = x.shape
    ctx = prefix.shape[-1]
    d = W.d
    temb = timestep_embedding(W, t_model)
    enc = torch.zeros_like(enc_text) if uncond else enc_text
    mem = _lin(enc.permute(1, 0, 2), W["embed_text.weight"], W["embed_text.bias"], None) + temb[None, None, :]   # [B,Mt,d]
    xf = torch.cat([prefix, x], dim=-1)
    T = ctx + Tp
    frames = xf.permute(0, 3, 1, 2).reshape(B, T, J * Fe)
    h = _lin(frames, W["input_process.poseEmbedding.weight"], W["input_process.poseEmbedding.bias"], cast) + W.pe[:T][None]
    keymask = None
    if mask_frames and lengths is not None and T > 1:
        keymask = torch.arange(T)[None, :] >= (lengths[:, None] + ctx)
    h = decoder_stack(W, h, mem, keymask, text_mask, cast)[:, ctx:]
    out = _lin(h, W["output_process.poseFinal.weight"], W["output_process.poseFinal.bias"], cast)
    return out.reshape(B, Tp, J, Fe).permute(0, 2, 3, 1).contiguous()


def cfg_denoise_dec(W, x, t_model, enc_text, text_mask, prefix, scale, lengths=None, mask_frames=True, cast=None):
    oc = denoise_dec(W, x, t_model, enc_text, text_mask, prefix, lengths, mask_frames, False, cast)
    ou = denoise_dec(W, x, t_model, enc_text, text_mask, prefix, lengths, mask_frames, True, cast)
    return ou + scale.view(-1, 1, 1, 1) * (oc - ou)


def sample_loop_dec(W, tables, timestep_map, tape, enc_text, text_mask, prefix, scale, lengths=None, mask_frames=True, cast=None):
    n = len(tables["betas"])
    x = tape[0].clone()
    for k, i in enumerate(range(n - 1, -1, -1)):
        x0 = cfg_denoise_dec(W, x, int(timestep_map[i]), enc_text, text_mask, prefix, scale, lengths, mask_frames, cast)
        x, _ = p_sample_step(tables, x0, x, i, tape[1 + k])
    return x

"""Deterministic synthetic checkpoints and inputs (no network => no released checkpoints).

`synthetic_state_dict` produces a reference-format ``state_dict`` (same key names and shapes as a
checkpoint written by the reference's train loop, SURVEY.md appendix A.4) from a numpy
``default_rng`` stream, so the very same weights can be regenerated in the build container, on the
GPU box and inside the reference oracle without shipping 70 MB files.  Scales follow the default
torch initialisers (Linear: U(+-1/sqrt(fan_in)); MHA in_proj: xavier-uniform) but biases and the
LayerNorm affine parameters are made non-trivial so that parity tests exercise them.
"""
import math

import numpy as np
import torch


def _uniform(rng, shape, bound):
    return torch.from_numpy(rng.uniform(-bound, bound, size=shape).astype(np.float32))


def _normal(rng, shape, std):
    return torch.from_numpy((rng.standard_normal(size=shape) * std).astype(np.float32))


HML_GOAL_ROWS = ["pelvis", "left_foot", "right_foot", "left_wrist", "right_wrist", "head", "traj", "heading"]


def synthetic_state_dict(arch="trans_enc", latent_dim=512, ff_size=1024, num_layers=8, input_feats=263,
                         cond_dim=512, cond_mode="text", num_actions=1, seed=0, target_encoder=None, target_enc_layers=1,
                         n_goal_rows=8):
    """target_encoder ('single' / 'multi' / 'split'): also the embed_target_cond.* keys of a multi_target_cond model
    (humanml rows: HML_GOAL_ROWS; n_goal_rows = 2 keeps 'traj' and 'heading' only).  They come from a stream of their
    own, so the other tensors are the same as without them."""
    sd = _base_state_dict(arch, latent_dim, ff_size, num_layers, input_feats, cond_dim, cond_mode, num_actions, seed)
    if target_encoder is not None:
        sd.update(_target_state_dict(target_encoder, latent_dim, target_enc_layers, n_goal_rows, seed))
    return sd


def _target_state_dict(encoder, d, layers, n, seed):
    """At the reference's default init the target moves a trans_enc output by only ~0.5 %; the last layer here is
    scaled up so that it moves it by several per cent (a missing target shows far outside the parity tolerance), and
    the multi encoder's row weights are positive so that their sum stays away from 0."""
    if n > len(HML_GOAL_ROWS) or n < 2:
        raise ValueError("n_goal_rows must be 2..%d" % len(HML_GOAL_ROWS))
    rows = HML_GOAL_ROWS[: n - 2] + ["traj", "heading"]
    rng = np.random.default_rng(seed + 7001)
    sd = {}
    gain = 6.0

    def linear(prefix, out_f, in_f, g=1.0):
        b = 1.0 / math.sqrt(in_f)
        sd[prefix + ".weight"] = _uniform(rng, (out_f, in_f), b * g)
        sd[prefix + ".bias"] = _uniform(rng, (out_f,), b * g)

    p = "embed_target_cond."
    if encoder == "single":
        linear(p + "mlp.0", d, 4 * n)
        for l in range(1, layers + 1):
            linear(p + "mlp.%d" % (2 * l), d, d, gain if l == layers else 1.0)
    elif encoder == "split":
        ds = d // n
        for j in range(n):
            linear(p + "mini_mlps.%d.0" % j, ds, 4)
            for l in range(1, layers + 1):
                linear(p + "mini_mlps.%d.%d" % (j, 2 * l), ds, ds, gain if l == layers else 1.0)
    elif encoder == "multi":
        for name in rows:
            linear(p + "target_loc_emb.%s.0" % name, d, 3)
            linear(p + "target_loc_emb.%s.2" % name, d, d, gain)
        sd[p + "target_all_loc_emb.weights"] = torch.from_numpy(rng.uniform(0.5, 1.5, size=n).astype(np.float32))
    else:
        raise ValueError("unsupported target encoder %r" % (encoder,))
    return sd


def synthetic_targets(batch, joint_sets, heading, n_goal_rows=8, seed=17):
    """y['target_cond'] [B, n, 3] (every row filled, valid or not -- the single and split encoders read them all),
    y['target_joint_names'] (the given per-sample name lists) and y['is_heading'] (bool [B])."""
    rng = np.random.default_rng(seed)
    tc = torch.from_numpy(rng.standard_normal((batch, n_goal_rows, 3)).astype(np.float32))
    assert len(joint_sets) == batch and len(heading) == batch
    return dict(target_cond=tc, target_joint_names=[list(s) for s in joint_sets],
                is_heading=torch.tensor([bool(h) for h in heading]))


def _base_state_dict(arch, latent_dim, ff_size, num_layers, input_feats, cond_dim, cond_mode, num_actions, seed):
    rng = np.random.default_rng(seed)
    d = latent_dim
    sd = {}

    def linear(prefix, out_f, in_f):
        b = 1.0 / math.sqrt(in_f)
        sd[prefix + ".weight"] = _uniform(rng, (out_f, in_f), b)
        sd[prefix + ".bias"] = _uniform(rng, (out_f,), b)

    def layer_norm(prefix):
        sd[prefix + ".weight"] = 1.0 + _normal(rng, (d,), 0.1)
        sd[prefix + ".bias"] = _normal(rng, (d,), 0.1)

    def mha(prefix):
        xb = math.sqrt(6.0 / (d + 3 * d))
        sd[prefix + ".in_proj_weight"] = _uniform(rng, (3 * d, d), xb)
        sd[prefix + ".in_proj_bias"] = _normal(rng, (3 * d,), 0.02)
        linear(prefix + ".out_proj", d, d)

    linear("input_process.poseEmbedding", d, input_feats)
    linear("embed_timestep.time_embed.0", d, d)
    linear("embed_timestep.time_embed.2", d, d)
    if "text" in cond_mode:
        linear("embed_text", d, cond_dim)
    if "action" in cond_mode:
        sd["embed_action.action_embedding"] = _normal(rng, (num_actions, d), 1.0)
    if arch == "trans_enc":
        for l in range(num_layers):
            p = "seqTransEncoder.layers.%d" % l
            mha(p + ".self_attn")
            linear(p + ".linear1", ff_size, d)
            linear(p + ".linear2", d, ff_size)
            layer_norm(p + ".norm1")
            layer_norm(p + ".norm2")
    elif arch == "trans_dec":
        for l in range(num_layers):
            p = "seqTransDecoder.layers.%d" % l
            mha(p + ".self_attn")
            mha(p + ".multihead_attn")
            linear(p + ".linear1", ff_size, d)
            linear(p + ".linear2", d, ff_size)
            layer_norm(p + ".norm1")
            layer_norm(p + ".norm2")
            layer_norm(p + ".norm3")
    else:
        raise ValueError("unsupported arch %r" % (arch,))
    linear("output_process.poseFinal", input_feats, d)
    return sd


def synthetic_inputs(batch, njoints=263, nfeats=1, nframes=196, steps=50, cond_dim=512, seed=10,
                     lengths=None, scale=2.5, dtype=torch.float32):
    """Noise tape [x_T, eps_{T-1} .. eps_0], text embedding [1,B,cond_dim], lengths, mask, scale."""
    rng = np.random.default_rng(seed)
    shape = (batch, njoints, nfeats, nframes)
    tape = [torch.from_numpy(rng.standard_normal(size=shape).astype(np.float32)) for _ in range(steps + 1)]
    text_embed = torch.from_numpy(rng.standard_normal(size=(1, batch, cond_dim)).astype(np.float32))
    if lengths is None:
        lengths = [nframes] * batch
    lengths = torch.tensor(lengths, dtype=torch.int64)
    mask = (torch.arange(nframes)[None, :] < lengths[:, None]).view(batch, 1, 1, nframes)
    if not torch.is_tensor(scale):
        scale = torch.full((batch,), float(scale), dtype=torch.float32)
    return dict(tape=tape, text_embed=text_embed, lengths=lengths, mask=mask, scale=scale)


def synthetic_dip_inputs(batch, n_tokens, context_len, njoints=263, nfeats=1, cond_dim=768, seed=3):
    """Deterministic DiP conditioning in the reference's layouts (model/mdm.py:180-187,204): BERT token features
    [n_tokens, B, 768], ragged padding mask [B, n_tokens] (True = padding; sample 0 has none), prefix [B, J, F, ctx]."""
    g = torch.Generator().manual_seed(seed)
    enc = torch.randn(n_tokens, batch, cond_dim, generator=g)
    tmask = torch.zeros(batch, n_tokens, dtype=torch.bool)
    for b in range(1, batch):
        tmask[b, n_tokens - (b * 2) % n_tokens:] = True
    prefix = torch.randn(batch, njoints, nfeats, context_len, generator=g)
    return enc, tmask, prefix


def synthetic_norm_stats(dim=263, seed=7):
    """Stand-in for the dataset's Mean.npy / Std.npy (data_loaders/humanml/data/dataset.py:248-249): fp32 [dim]."""
    rng = np.random.default_rng(seed)
    mean = rng.standard_normal(dim).astype(np.float32)
    std = rng.uniform(0.2, 2.0, size=dim).astype(np.float32)
    return torch.from_numpy(mean), torch.from_numpy(std)

"""Host mirror of the reference denoiser class (model/mdm.py in the reference tree).

`MDM` keeps the reference's constructor keywords, attribute surface and -- crucially -- parameter names and
shapes, so reference checkpoints load with the reference's own `load_state_dict(strict=False)` call
(utils/model_util.py:8-15).  The parameters are plain storage: `forward` never multiplies by them in PyTorch.
It uploads them once into the B200 engine (fp16 repack) and calls `b200mdm_denoise`.

Implemented: arch='trans_enc' with cond_mode in {no_cond, text (CLIP features), action}; arch='trans_dec' with
text_encoder_type='bert' (DiP: BERT token memory, prefix completion, model/mdm.py:203-206,255-270); hml_vec / rot6d /
xyz data_rep; target-location conditioning (multi_target_cond, the CLoSD "DiP with target conditioning" checkpoint:
y['target_cond'] / y['target_joint_names'] / y['is_heading'], model/mdm.py:197-199) with the single, multi and split
target encoders.
Not implemented (raise): arch 'gru', data_rep 'rot_vel', emb_trans_dec, emb_policy != 'add', trans_dec with CLIP
features.
"""
import numpy as np
import torch
import torch.nn as nn

from ..engine import Engine


def positional_table(max_len, d_model):
    """The `pe` buffer of the reference's PositionalEncoding (model/mdm.py:301-308), built with the same fp32 op
    sequence so the table is bit-identical; shape [max_len, d_model]."""
    pe = torch.zeros(max_len, d_model)
    position = torch.arange(0, max_len, dtype=torch.float).unsqueeze(1)
    div_term = torch.exp(torch.arange(0, d_model, 2).float() * (-np.log(10000.0) / d_model))
    pe[:, 0::2] = torch.sin(position * div_term)
    pe[:, 1::2] = torch.cos(position * div_term)
    return pe


class _Bag(nn.Module):
    """Parameter container: gives nested, reference-compatible state_dict keys without any compute."""

    def add(self, dotted, tensor, buffer=False):
        head, _, rest = dotted.partition(".")
        if not rest:
            if buffer:
                self.register_buffer(head, tensor, persistent=False)
            else:
                self.register_parameter(head, nn.Parameter(tensor, requires_grad=False))
            return
        if head not in self._modules:
            self.add_module(head, _Bag())
        self._modules[head].add(rest, tensor, buffer)


def target_row_names(all_goal_joint_names):
    """The rows of y['target_cond']: EmbedTarget*.extended_goal_joint_names (model/mdm.py:402,425,453)."""
    return list(all_goal_joint_names) + ["traj", "heading"]


def _target_spec(encoder, d, layers, rows):
    """embed_target_cond.* keys of EmbedTargetLocSingle / Multi / Split (model/mdm.py:399-480, utils/misc.py:5-9)."""
    n = len(rows)
    p = "embed_target_cond."
    if encoder == "single":
        s = [(p + "mlp.0.weight", (d, 4 * n), "lin"), (p + "mlp.0.bias", (d,), "lin")]
        for l in range(1, layers + 1):
            s += [(p + "mlp.%d.weight" % (2 * l), (d, d), "lin"), (p + "mlp.%d.bias" % (2 * l), (d,), "lin")]
        return s
    if encoder == "split":
        ds = d // n
        s = []
        for j in range(n):
            s += [(p + "mini_mlps.%d.0.weight" % j, (ds, 4), "lin"), (p + "mini_mlps.%d.0.bias" % j, (ds,), "lin")]
            for l in range(1, layers + 1):
                s += [(p + "mini_mlps.%d.%d.weight" % (j, 2 * l), (ds, ds), "lin"), (p + "mini_mlps.%d.%d.bias" % (j, 2 * l), (ds,), "lin")]
        return s
    s = []
    for name in rows:
        q = p + "target_loc_emb.%s." % name
        s += [(q + "0.weight", (d, 3), "lin"), (q + "0.bias", (d,), "lin"), (q + "2.weight", (d, d), "lin"), (q + "2.bias", (d,), "lin")]
    return s + [(p + "target_all_loc_emb.weights", (n,), "normal")]


def _spec(arch, d, ff, layers, input_feats, cond_mode, cond_dim, num_actions):
    """(key, shape, init) for every learned tensor -- SURVEY.md appendix A.4."""
    s = [("input_process.poseEmbedding.weight", (d, input_feats), "lin"), ("input_process.poseEmbedding.bias", (d,), "lin"),
         ("embed_timestep.time_embed.0.weight", (d, d), "lin"), ("embed_timestep.time_embed.0.bias", (d,), "lin"),
         ("embed_timestep.time_embed.2.weight", (d, d), "lin"), ("embed_timestep.time_embed.2.bias", (d,), "lin")]
    if "text" in cond_mode:
        s += [("embed_text.weight", (d, cond_dim), "lin"), ("embed_text.bias", (d,), "lin")]
    if "action" in cond_mode:
        s += [("embed_action.action_embedding", (num_actions, d), "normal")]
    dec = arch == "trans_dec"
    for l in range(layers):
        p = ("seqTransDecoder.layers.%d." if dec else "seqTransEncoder.layers.%d.") % l
        if dec:   # nn.TransformerDecoderLayer: cross-attention block + third norm
            s += [(p + "multihead_attn.in_proj_weight", (3 * d, d), "xavier"), (p + "multihead_attn.in_proj_bias", (3 * d,), "zero"),
                  (p + "multihead_attn.out_proj.weight", (d, d), "lin"), (p + "multihead_attn.out_proj.bias", (d,), "zero"),
                  (p + "norm3.weight", (d,), "one"), (p + "norm3.bias", (d,), "zero")]
        s += [(p + "self_attn.in_proj_weight", (3 * d, d), "xavier"), (p + "self_attn.in_proj_bias", (3 * d,), "zero"),
              (p + "self_attn.out_proj.weight", (d, d), "lin"), (p + "self_attn.out_proj.bias", (d,), "zero"),
              (p + "linear1.weight", (ff, d), "lin"), (p + "linear1.bias", (ff,), "lin"),
              (p + "linear2.weight", (d, ff), "lin"), (p + "linear2.bias", (d,), "lin"),
              (p + "norm1.weight", (d,), "one"), (p + "norm1.bias", (d,), "zero"),
              (p + "norm2.weight", (d,), "one"), (p + "norm2.bias", (d,), "zero")]
    s += [("output_process.poseFinal.weight", (input_feats, d), "lin"), ("output_process.poseFinal.bias", (input_feats,), "lin")]
    return s


def _init(shape, kind):
    if kind == "zero":
        return torch.zeros(shape)
    if kind == "one":
        return torch.ones(shape)
    if kind == "normal":
        return torch.randn(shape)
    fan_in = shape[-1] if len(shape) > 1 else shape[0]
    bound = (6.0 / (shape[0] + shape[1])) ** 0.5 if kind == "xavier" else 1.0 / fan_in ** 0.5
    return torch.empty(shape).uniform_(-bound, bound)


class MDM(_Bag):
    def __init__(self, modeltype, njoints, nfeats, num_actions, translation, pose_rep, glob, glob_rot,
                 latent_dim=256, ff_size=1024, num_layers=8, num_heads=4, dropout=0.1, ablation=None, activation="gelu",
                 legacy=False, data_rep="rot6d", dataset="amass", clip_dim=512, arch="trans_enc", emb_trans_dec=False,
                 clip_version=None, **kargs):
        super().__init__()
        # attribute surface read by the reference's callers (SURVEY.md section 8b)
        self.legacy, self.modeltype, self.njoints, self.nfeats, self.num_actions = legacy, modeltype, njoints, nfeats, num_actions
        self.data_rep, self.dataset, self.pose_rep, self.glob, self.glob_rot = data_rep, dataset, pose_rep, glob, glob_rot
        self.translation, self.latent_dim, self.ff_size, self.num_layers = translation, latent_dim, ff_size, num_layers
        self.num_heads, self.dropout, self.ablation, self.activation = num_heads, dropout, ablation, activation
        self.clip_dim, self.clip_version = clip_dim, clip_version
        self.action_emb = kargs.get("action_emb", None)
        self.input_feats = njoints * nfeats
        self.cond_mode = kargs.get("cond_mode", "no_cond")
        self.cond_mask_prob = kargs.get("cond_mask_prob", 0.0)
        self.mask_frames = kargs.get("mask_frames", False)
        self.arch, self.emb_trans_dec = arch, emb_trans_dec
        self.emb_policy = kargs.get("emb_policy", "add")
        self.pred_len, self.context_len = kargs.get("pred_len", 0), kargs.get("context_len", 0)
        self.total_len = self.pred_len + self.context_len
        self.is_prefix_comp = self.total_len > 0
        self.all_goal_joint_names = kargs.get("all_goal_joint_names", [])
        self.multi_target_cond = kargs.get("multi_target_cond", False)
        self.multi_encoder_type = kargs.get("multi_encoder_type", "multi")
        self.target_enc_layers = kargs.get("target_enc_layers", 1)
        self.text_encoder_type = kargs.get("text_encoder_type", "clip")
        self.pos_embed_max_len = kargs.get("pos_embed_max_len", 5000)
        self.temb_rows = min(self.pos_embed_max_len, kargs.get("num_model_timesteps", 1000))
        self.rot2xyz = _identity_rot2xyz            # hml_vec: Rotation2xyz is an identity (rotation2xyz.py:20-21)
        self.clip_model = None                      # the frozen text tower stays outside the engine

        if arch not in ("trans_enc", "trans_dec"):
            raise NotImplementedError("arch=%r: the engine implements the trans_enc and trans_dec (DiP) denoisers; gru is "
                                      "an ablation and out of scope" % (arch,))
        if activation != "gelu":
            raise NotImplementedError("the fused FFN epilogue implements exact GELU only (model_util.py:63)")
        if data_rep == "rot_vel" or self.emb_policy != "add":
            raise NotImplementedError("rot_vel / emb_policy='cat' variants are outside the hot path")
        self.target_rows = target_row_names(self.all_goal_joint_names) if self.multi_target_cond else None
        if self.multi_target_cond:
            if self.multi_encoder_type not in ("single", "multi", "split"):
                raise NotImplementedError("multi_encoder_type=%r: the single, multi and split target encoders are "
                                          "implemented (model/mdm.py:67-73)" % (self.multi_encoder_type,))
            if self.multi_encoder_type == "split" and latent_dim % len(self.target_rows):
                raise AssertionError("split target encoder needs latent_dim %% %d == 0 (model/mdm.py:430)" % len(self.target_rows))
        if arch == "trans_enc":
            if self.is_prefix_comp:
                raise NotImplementedError("prefix completion is implemented for arch='trans_dec' (DiP) only")
            if "text" in self.cond_mode and self.text_encoder_type != "clip":
                raise AssertionError("BERT text conditioning requires arch='trans_dec' (model/mdm.py:114)")
        else:
            if "text" not in self.cond_mode or self.text_encoder_type != "bert" or emb_trans_dec:
                raise NotImplementedError("arch='trans_dec' is implemented for the DiP configuration: cond_mode='text', "
                                          "text_encoder_type='bert', emb_trans_dec=False")
            self.clip_dim = 768                     # model/mdm.py:117

        for key, shape, kind in _spec(arch, latent_dim, ff_size, num_layers, self.input_feats, self.cond_mode,
                                      self.clip_dim, num_actions):
            self.add(key, _init(shape, kind))
        if self.multi_target_cond:
            for key, shape, kind in _target_spec(self.multi_encoder_type, latent_dim, self.target_enc_layers, self.target_rows):
                self.add(key, _init(shape, kind))
        self.add("sequence_pos_encoder.pe", positional_table(self.pos_embed_max_len, latent_dim).unsqueeze(1), buffer=True)
        self._engine = None
        self._engine_dirty = True
        self._engine_device = None

    # ------------------------------------------------------------------ torch.nn.Module plumbing
    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._engine_dirty = True
        return out

    def load_state_dict(self, state_dict, strict=True, **k):
        out = super().load_state_dict(state_dict, strict=strict, **k)
        self._engine_dirty = True
        return out

    def parameters_wo_clip(self):
        return [p for n, p in self.named_parameters() if not n.startswith("clip_model.")]

    # ------------------------------------------------------------------ text
    def encode_text(self, raw_text):
        """clip_encode_text / bert_encode_text (reference model/mdm.py:163-187).  The text tower is third-party, frozen,
        and runs once per loop outside the replaced path; plug it in with `model.clip_model = clip.load(...)[0]`
        (or the DistilBERT wrapper for DiP)."""
        if self.clip_model is None:
            raise RuntimeError("no text encoder attached: pass y['text_embed'] (cached CLIP features [1,B,512], or the "
                               "(tokens [Mt,B,768], padding mask [B,Mt]) pair for DiP) or set model.clip_model")
        if self.text_encoder_type == "bert":
            enc_text, mask = self.clip_model(raw_text)          # mask: True = token present
            return enc_text.permute(1, 0, 2), ~mask
        import clip  # noqa -- only when a real encoder was attached
        device = next(self.parameters()).device
        if self.dataset in ("humanml", "kit"):
            texts = clip.tokenize(raw_text, context_length=22, truncate=True).to(device)
            texts = torch.cat([texts, torch.zeros([texts.shape[0], 77 - 22], dtype=texts.dtype, device=device)], dim=1)
        else:
            texts = clip.tokenize(raw_text, truncate=True).to(device)
        return self.clip_model.encode_text(texts).float().unsqueeze(0)

    # ------------------------------------------------------------------ engine
    def engine(self):
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("b200mdm runs on a B200 only (model is on %s); move it with model.to('cuda'). "
                               "There is no CPU / eager fallback." % dev)
        if self._engine is None or self._engine_device != dev:
            with torch.cuda.device(dev):
                self._engine = Engine(arch=self.arch, latent_dim=self.latent_dim, ff_size=self.ff_size,
                                      num_layers=self.num_layers, num_heads=self.num_heads, njoints=self.njoints,
                                      nfeats=self.nfeats, cond_mode=self.cond_mode, cond_dim=self.clip_dim,
                                      num_actions=max(1, self.num_actions), mask_frames=self.mask_frames,
                                      pos_embed_max_len=self.pos_embed_max_len, temb_rows=self.temb_rows,
                                      context_len=self.context_len if self.arch == "trans_dec" else 0,
                                      target_encoder=self.multi_encoder_type if self.multi_target_cond else None,
                                      target_rows=self.target_rows, target_enc_layers=self.target_enc_layers)
            self._engine_device = dev
            self._engine_dirty = True
        if self._engine_dirty:
            sd = self.engine_state_dict()
            with torch.cuda.device(dev):
                self._engine.load_state_dict(sd)
            self._engine_dirty = False
        return self._engine

    def engine_state_dict(self):
        """The tensors b200mdm_load_weight receives: the state_dict plus the positional table, with the multi target
        encoder's per-joint MLPs renamed from joint name to row index (the C side addresses rows; only the host knows
        all_goal_joint_names)."""
        sd = {k: v for k, v in self.state_dict().items()}
        if self.multi_target_cond and self.multi_encoder_type == "multi":
            pre = "embed_target_cond.target_loc_emb."
            for j, name in enumerate(self.target_rows):
                for suffix in ("0.weight", "0.bias", "2.weight", "2.bias"):
                    sd["%s%d.%s" % (pre, j, suffix)] = sd.pop("%s%s.%s" % (pre, name, suffix))
        sd["sequence_pos_encoder.pe"] = self.sequence_pos_encoder.pe.squeeze(1)
        return sd

    def forward(self, x, timesteps, y=None):
        """x [B, njoints, nfeats, T] fp32, timesteps [B] (model timesteps), y dict -> [B, njoints, nfeats, T]
        (reference model/mdm.py:189-283)."""
        return _run_model(self, x, timesteps, y, guided=False)


def _identity_rot2xyz(x, mask=None, pose_rep="xyz", **kw):
    if pose_rep != "xyz":
        raise NotImplementedError("SMPL forward kinematics is post-processing, outside the engine")
    return x


def _run_model(model, x, timesteps, y, guided):
    eng = model.engine()
    B, T = x.shape[0], x.shape[-1]
    with torch.cuda.device(x.device):
        eng.set_cond(B, T, y if y is not None else {}, guided, x.device)
        eng.set_inpaint(None, None)
        return eng.denoise(x, timesteps)


def engine_for(model):
    """(engine, guided) for a bare MDM or a ClassifierFreeSampleModel wrapper (possibly behind respace._WrappedModel).

    Only wrappers this package knows are looked through: an unknown object that merely has a `.model` attribute (for
    instance a guidance wrapper class from another import of this package, or the reference's own
    ClassifierFreeSampleModel) would otherwise be unwrapped down to the bare denoiser and sampled WITHOUT guidance,
    silently."""
    from ..utils.sampler_util import ClassifierFreeSampleModel
    from ..diffusion.respace import _WrappedModel
    inner = model
    while isinstance(inner, _WrappedModel):
        inner = inner.model
    if isinstance(inner, ClassifierFreeSampleModel):
        if not isinstance(inner.model, MDM):
            raise TypeError("ClassifierFreeSampleModel must wrap a b200mdm MDM (got %r)" % type(inner.model))
        return inner.model.engine(), True
    if isinstance(inner, MDM):
        return inner.engine(), False
    raise TypeError("b200mdm diffusion objects drive b200mdm.MDM or b200mdm.ClassifierFreeSampleModel only (got %r); "
                    "wrap the model with the classes of this package" % type(model))

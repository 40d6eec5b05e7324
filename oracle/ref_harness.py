"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

Loads the UNMODIFIED reference (GuyTevet/motion-diffusion-model) on CPU: oracle/gen_golden.py runs
it to write the golden vectors under tests/golden/, oracle/build_ref.py to list its hot-path files,
and bench.py's CPU reference arm to time it.  No test imports this module; the tests compare
against the stored vectors.

Two third-party imports of the reference are absent here and are stubbed *before* import
(SURVEY.md section 8c): `clip` (model/mdm.py:5) and `model.rotation2xyz` -> smplx
(model/rotation2xyz.py:6).  Neither is on the per-step path.  `model.BERT.BERT_encoder.load_bert`
is stubbed for the DiP (trans_dec + bert) configuration.

Noise injection: `diffusion.gaussian_diffusion` draws with the module alias `th`
(gaussian_diffusion.py:14, used at :525, :691, :770).  We swap that alias for a proxy whose
randn / randn_like pop from a caller-provided tape; every other attribute delegates to torch.
Tape order = [x_T, eps_{T-1}, ..., eps_0].
"""
import os
import sys
import types
from types import SimpleNamespace

import torch
import torch.nn as nn

_HERE = os.path.dirname(os.path.abspath(__file__))


def _reference_root():
    """MDM_REFERENCE_ROOT if set; else the read-only reference tree of the build container; else `oracle/_ref/`, the
    byte-for-byte copy of the 15 hot-path files made by oracle/build_ref.py (what travels to the GPU box)."""
    env = os.environ.get("MDM_REFERENCE_ROOT")
    if env:
        return env
    if os.path.isdir("/root/reference/diffusion"):
        return "/root/reference"
    return os.path.join(_HERE, "_ref")


REFERENCE_ROOT = _reference_root()


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "diffusion"))


_loaded = {}


def load_reference():
    """Import the reference modules with the stubs in place; returns a namespace of modules."""
    if _loaded:
        return _loaded["ns"]
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    # The reference uses top-level package names (utils, model, diffusion, data_loaders).
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    clip = types.ModuleType("clip")
    clip.model = types.ModuleType("clip.model")
    clip.load = lambda v, device="cpu", jit=False: (nn.Identity(), None)
    clip.model.convert_weights = lambda m: None
    sys.modules["clip"] = clip
    sys.modules["clip.model"] = clip.model

    r2x = types.ModuleType("model.rotation2xyz")

    class Rotation2xyz:  # MDM only touches .smpl_model._apply / .train (mdm.py:286-293)
        def __init__(self, device, dataset="amass"):
            self.smpl_model = nn.Identity()

        def __call__(self, x, **kw):
            return x

    r2x.Rotation2xyz = Rotation2xyz
    sys.modules["model.rotation2xyz"] = r2x

    bert = types.ModuleType("model.BERT.BERT_encoder")
    bert.load_bert = lambda p: nn.Identity()
    sys.modules["model.BERT.BERT_encoder"] = bert

    import io
    import contextlib

    with contextlib.redirect_stdout(io.StringIO()):
        from utils import model_util, sampler_util  # noqa
        from diffusion import gaussian_diffusion, respace  # noqa
        from model import mdm  # noqa
    ns = SimpleNamespace(model_util=model_util, sampler_util=sampler_util,
                         gaussian_diffusion=gaussian_diffusion, respace=respace, mdm=mdm)
    _loaded["ns"] = ns
    return ns


def default_args(**over):
    """The Namespace the reference's parser would produce for the released humanml models
    (utils/parser_util.py:74-131 defaults; see SURVEY.md section 8c)."""
    a = dict(dataset="humanml", unconstrained=False, latent_dim=512, layers=8, cond_mask_prob=0.1,
             arch="trans_enc", emb_trans_dec=False, text_encoder_type="clip", pos_embed_max_len=5000,
             mask_frames=True, pred_len=0, context_len=0, diffusion_steps=50,
             noise_schedule="cosine", sigma_small=True, lambda_vel=0.0, lambda_rcxyz=0.0, lambda_fc=0.0)
    a.update(over)
    return SimpleNamespace(**a)


def build(args=None, num_actions=None, state_dict=None):
    """create_model_and_diffusion of the reference (utils/model_util.py:18-21), eval mode."""
    import io
    import contextlib
    ns = load_reference()
    args = args or default_args()
    ds = SimpleNamespace()
    if num_actions is not None:
        ds.num_actions = num_actions
    with contextlib.redirect_stdout(io.StringIO()):
        model, diffusion = ns.model_util.create_model_and_diffusion(args, SimpleNamespace(dataset=ds))
    if state_dict is not None:
        missing, unexpected = model.load_state_dict(state_dict, strict=False)
        assert not unexpected, unexpected
        assert all(k.startswith("clip_model.") or "sequence_pos_encoder" in k for k in missing), missing
    model.eval()
    return model, diffusion


class _TapeTorch:
    """Stand-in for the `th` alias inside gaussian_diffusion: randn / randn_like pop the tape."""

    def __init__(self, tape):
        self._tape = list(tape)
        self._pos = 0

    def _pop(self, shape):
        t = self._tape[self._pos]
        self._pos += 1
        assert tuple(t.shape) == tuple(shape), (t.shape, shape)
        return t.clone()

    def randn(self, *shape, **kw):
        if len(shape) == 1 and isinstance(shape[0], (tuple, list)):
            shape = tuple(shape[0])
        return self._pop(shape)

    def randn_like(self, x, **kw):
        return self._pop(x.shape)

    def __getattr__(self, name):
        return getattr(torch, name)


class noise_tape:
    """Context manager: `with noise_tape([x_T, eps, ...]): diffusion.p_sample_loop(...)`."""

    def __init__(self, tape):
        self.tape = tape

    def __enter__(self):
        gd = load_reference().gaussian_diffusion
        self._saved = gd.th
        self.proxy = _TapeTorch(self.tape)
        gd.th = self.proxy
        return self.proxy

    def __exit__(self, *exc):
        load_reference().gaussian_diffusion.th = self._saved
        return False

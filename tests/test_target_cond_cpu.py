"""CPU: target-location conditioning (multi_target_cond; reference model/mdm.py:64-73,197-199,399-480) -- parameter layout,
validity construction and input errors of the host mirror, the fp32 oracle against golden/target_small.npz (written by
the unmodified reference), batch sharding of the target keys, and the C-ABI checks that run without a GPU."""
import ctypes
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

TOL = 2e-5


def _model(**over):
    model, _ = b200mdm.create_model_and_diffusion(default_args(layers=1, **over), SimpleNamespace(dataset=SimpleNamespace()))
    return model


@pytest.mark.parametrize("encoder,layers", [("single", 1), ("single", 3), ("multi", 1), ("split", 1), ("split", 2)])
def test_target_keys_match_reference_layout(encoder, layers):
    model = _model(multi_target_cond=True, multi_encoder_type=encoder, target_enc_layers=layers)
    assert model.target_rows == tc.ROWS
    got = {k: tuple(v.shape) for k, v in model.state_dict().items() if k.startswith("embed_target_cond.")}
    if encoder == "single":
        want = {"embed_target_cond.mlp.0.weight": (512, 32), "embed_target_cond.mlp.0.bias": (512,)}
        for l in range(1, layers + 1):
            want.update({"embed_target_cond.mlp.%d.weight" % (2 * l): (512, 512), "embed_target_cond.mlp.%d.bias" % (2 * l): (512,)})
    elif encoder == "split":
        want = {}
        for j in range(8):
            want.update({"embed_target_cond.mini_mlps.%d.0.weight" % j: (64, 4), "embed_target_cond.mini_mlps.%d.0.bias" % j: (64,)})
            for l in range(1, layers + 1):
                want.update({"embed_target_cond.mini_mlps.%d.%d.weight" % (j, 2 * l): (64, 64),
                             "embed_target_cond.mini_mlps.%d.%d.bias" % (j, 2 * l): (64,)})
    else:
        want = {"embed_target_cond.target_all_loc_emb.weights": (8,)}
        for name in tc.ROWS:
            p = "embed_target_cond.target_loc_emb.%s." % name
            want.update({p + "0.weight": (512, 3), p + "0.bias": (512,), p + "2.weight": (512, 512), p + "2.bias": (512,)})
    assert got == want
    sd = b200mdm.synthetic_state_dict(num_layers=1, target_encoder=encoder, target_enc_layers=layers)
    assert set(sd) == set(model.state_dict())
    b200mdm.load_model_wo_clip(model, sd)          # the reference's loader: no unexpected, no missing keys
    assert torch.equal(model.state_dict()[sorted(want)[0]], sd[sorted(want)[0]])
    # plain models have no target keys, and a target state_dict does not load into them
    plain = _model()
    assert not any(k.startswith("embed_target_cond.") for k in plain.state_dict())
    with pytest.raises(AssertionError):
        b200mdm.load_model_wo_clip(plain, sd)


def test_multi_keys_map_to_row_indices_by_name():
    """The reference's ParameterDict lists the joints alphabetically (head, heading, left_foot, ...); the engine gets
    them by row index of all_goal_joint_names + ['traj', 'heading'], matched by name."""
    model = _model(multi_target_cond=True, multi_encoder_type="multi")
    sd = b200mdm.synthetic_state_dict(num_layers=1, target_encoder="multi")
    b200mdm.load_model_wo_clip(model, sd)
    names = sorted({k.split(".")[2] for k in sd if k.startswith("embed_target_cond.target_loc_emb.")})
    assert names == sorted(tc.ROWS) and names[:2] == ["head", "heading"]
    seen = model.engine_state_dict()
    for j, name in enumerate(tc.ROWS):
        assert torch.equal(seen["embed_target_cond.target_loc_emb.%d.2.weight" % j],
                           sd["embed_target_cond.target_loc_emb.%s.2.weight" % name])
    assert not any(k.startswith("embed_target_cond.target_loc_emb.%s." % n) for k in seen for n in tc.ROWS)


def test_validity_from_name_sets_and_heading():
    from b200mdm.engine import target_validity
    names = np.empty(4, dtype=object)                       # what sample_goal returns
    names[:] = [np.array([], dtype="<U5"), np.array(["traj"]), np.array(["left_wrist", "head"]), ["pelvis"]]
    heading = torch.tensor([True, False, True, False])
    v = target_validity(tc.ROWS, names, heading)
    want = np.zeros((4, 8), np.uint8)
    want[0, 7] = 1
    want[1, 6] = 1
    want[2, [3, 5, 7]] = 1
    want[3, 0] = 1
    assert v.dtype == np.uint8 and np.array_equal(v, want)
    assert np.array_equal(target_validity(tc.ROWS, [list(s) for s in names], heading.numpy()), want)
    assert np.array_equal(to.target_validity(tc.ROWS, [list(s) for s in names], heading).numpy(), want)
    with pytest.raises(ValueError):
        target_validity(tc.ROWS, [["left_hand"]], torch.tensor([False]))


def test_target_input_errors():
    """Unknown joint name -> ValueError, a missing target_joint_names / is_heading -> KeyError, target_cond on a model
    without a target encoder -> AttributeError (as in the reference); checked before any CUDA call."""
    from b200mdm.engine import Engine
    calls = []
    lib = SimpleNamespace(b200mdm_set_target=lambda *a: calls.append(a) or 0)
    eng = Engine.__new__(Engine)
    eng.lib, eng.h, eng._keep, eng.target_rows = lib, None, {}, list(tc.ROWS)
    y = dict(target_cond=torch.zeros(2, 8, 3), target_joint_names=[["traj"], ["nose"]], is_heading=torch.tensor([False, True]))
    with pytest.raises(ValueError):
        eng.set_target(2, y, "cpu")
    for k in ("target_joint_names", "is_heading"):
        with pytest.raises(KeyError):
            eng.set_target(2, {kk: v for kk, v in y.items() if kk != k}, "cpu")
    with pytest.raises(ValueError):
        eng.set_target(2, dict(y, target_cond=torch.zeros(2, 6, 3)), "cpu")
    assert not calls
    plain = Engine.__new__(Engine)
    plain.target_rows = None
    with pytest.raises(AttributeError):
        plain.set_target(2, y, "cpu")
    plain.set_target(2, {"text_embed": None}, "cpu")        # no target key: nothing to do
    with pytest.raises(NotImplementedError):
        _model(multi_target_cond=True, multi_encoder_type="transformer")


def _oracle_case(name):
    model, diffusion, sd, inp, y, T = tc.build(name)
    arch, enc, tl, _, B = tc.CASES[name]
    W = mo.OracleWeights(sd, tc.L)
    yy = y()
    target = to.target_embedding(W, enc, tc.ROWS, yy["target_cond"], yy["target_joint_names"], yy["is_heading"], tl)
    return W, inp, yy, target, arch, B, T


@pytest.mark.parametrize("name", sorted(tc.CASES))
def test_oracle_vs_reference_golden(golden, name):
    g = golden("target_small.npz")
    W, inp, y, target, arch, B, T = _oracle_case(name)
    assert np.array_equal(g["target_cond"][3 - B:], y["target_cond"].numpy())
    tabs = so.diffusion_tables(so.named_betas("cosine", tc.STEPS))
    x = inp["tape"][0]
    if arch == "trans_dec":
        fwd = to.cfg_denoise_dec(W, x, 1, inp["enc"], inp["tmask"], inp["prefix"], inp["scale"], target, inp["lengths"])
        loop = to.sample_loop_dec(W, tabs, list(range(tc.STEPS)), inp["tape"], inp["enc"], inp["tmask"], inp["prefix"],
                                  inp["scale"], target, inp["lengths"])
        plain = mo.cfg_denoise_dec(W, x, 1, inp["enc"], inp["tmask"], inp["prefix"], inp["scale"], inp["lengths"])
    else:
        fwd = to.cfg_denoise_enc(W, x, 1, inp["text_embed"], inp["scale"], target, inp["lengths"])
        loop = to.sample_loop(W, tabs, list(range(tc.STEPS)), inp["tape"], inp["text_embed"], inp["scale"], target, inp["lengths"])
        plain = mo.cfg_denoise_enc(W, x, 1, inp["text_embed"], inp["scale"], inp["lengths"])
    assert rel_err(fwd, g[name + "_fwd"]) < TOL
    assert rel_err(loop, g[name + "_ddpm"]) < TOL
    # the synthetic target weights move the output far outside the 1e-3 parity tolerance
    assert rel_err(plain, g[name + "_fwd"]) > 0.05
    if name == "dip_multi":                                  # target_uncond: exactly the forward without targets
        assert rel_err(plain, g[name + "_tuncond_fwd"]) < TOL


def test_shard_model_kwargs_slices_targets():
    from b200mdm.parallel import shard_model_kwargs
    names = np.empty(4, dtype=object)
    names[:] = [[], ["traj"], ["head", "pelvis"], ["left_foot"]]
    y = dict(target_cond=torch.arange(96.).view(4, 8, 3), is_heading=torch.tensor([True, False, True, False]),
             target_joint_names=names, target_uncond=False)
    out = shard_model_kwargs({"y": y}, 1, 3)["y"]
    assert torch.equal(out["target_cond"], y["target_cond"][1:3]) and torch.equal(out["is_heading"], y["is_heading"][1:3])
    assert list(out["target_joint_names"]) == [["traj"], ["head", "pelvis"]] and out["target_uncond"] is False
    out = shard_model_kwargs({"y": dict(y, target_joint_names=list(names))}, 2, 4)["y"]
    assert out["target_joint_names"] == [["head", "pelvis"], ["left_foot"]]


def test_c_abi_target_contract_without_gpu():
    """b200mdm_create validates the target fields before touching CUDA; b200mdm_set_target refuses a null engine."""
    from b200mdm import _lib
    lib = _lib.load()
    h = ctypes.c_void_p()
    base = dict(arch=_lib.ARCH["trans_dec"], latent_dim=512, ff_size=1024, num_layers=8, num_heads=4, njoints=263, nfeats=1,
                cond_mode=_lib.COND_TEXT, cond_dim=768, num_actions=1, mask_frames=1, pos_embed_max_len=5000,
                temb_rows=1000, context_len=20)
    for bad, msg in ((dict(target_encoder=4, n_goal_rows=8, target_enc_layers=1), b"target_encoder 4"),
                     (dict(target_encoder=1, n_goal_rows=0, target_enc_layers=1), b"n_goal_rows"),
                     (dict(target_encoder=1, n_goal_rows=8, target_enc_layers=0), b"target_enc_layers"),
                     (dict(target_encoder=3, n_goal_rows=7, target_enc_layers=1), b"latent_dim % n_goal_rows")):
        cfg = _lib.Config(**base, **bad)
        assert lib.b200mdm_create(ctypes.byref(cfg), ctypes.byref(h)) == _lib.ENOTIMPL, bad
        assert msg in lib.b200mdm_last_error(), (bad, lib.b200mdm_last_error())
    assert not h.value
    assert ctypes.sizeof(_lib.Config) == 80
    buf = (ctypes.c_float * 24)()
    mask = (ctypes.c_uint8 * 8)()
    assert lib.b200mdm_set_target(None, 1, buf, mask, None) == _lib.EINVAL and b"null engine" in lib.b200mdm_last_error()
    assert lib.b200mdm_set_target(None, 1, None, None, None) == _lib.EINVAL

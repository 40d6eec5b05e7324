"""CPU: the floating-point oracle (oracle/mdm_oracle.py, plain torch fp32) against the golden vectors produced by the
unmodified reference (tests/golden/, generator oracle/gen_golden.py).  Tolerance: fp32 round-off (different summation
order only)."""
import numpy as np
import torch

import b200mdm
from conftest import inpaint_motion, rel_err
from oracle import mdm_oracle as mo
from oracle import schedule_oracle as so

TOL = 2e-5


def _setup_small():
    sd = b200mdm.synthetic_state_dict(num_layers=2, seed=1)
    W = mo.OracleWeights(sd, 2)
    inp = b200mdm.synthetic_inputs(3, nframes=24, steps=4, seed=11, lengths=[24, 17, 5], scale=torch.tensor([2.5, 1.0, 7.5]))
    tabs = so.diffusion_tables(so.named_betas("cosine", 4))
    return W, inp, tabs


def test_forward_vs_golden(golden):
    g = golden("enc_small.npz")
    W, inp, _ = _setup_small()
    x = inp["tape"][0]
    oc = mo.denoise_enc(W, x, 2, inp["text_embed"], inp["lengths"], True, False)
    ou = mo.denoise_enc(W, x, 2, inp["text_embed"], inp["lengths"], True, True)
    cf = mo.cfg_denoise_enc(W, x, 2, inp["text_embed"], inp["scale"], inp["lengths"])
    assert rel_err(oc, g["fwd_cond"]) < TOL
    assert rel_err(ou, g["fwd_uncond"]) < TOL
    assert rel_err(cf, g["fwd_cfg"]) < TOL


def test_loops_vs_golden(golden):
    g = golden("enc_small.npz")
    W, inp, tabs = _setup_small()
    tmap = list(range(4))
    col = []
    out = mo.sample_loop(W, tabs, tmap, inp["tape"], inp["text_embed"], inp["scale"], inp["lengths"], collect=col)
    for k in range(4):
        assert rel_err(col[k], g["ddpm_steps"][k]) < TOL, k
    assert rel_err(out, g["ddpm_steps"][-1]) < TOL
    for eta in (0.0, 0.5):
        o = mo.sample_loop(W, tabs, tmap, inp["tape"], inp["text_embed"], inp["scale"], inp["lengths"], sampler="ddim", eta=eta)
        assert rel_err(o, g["ddim_eta%g" % eta]) < TOL
    motion = inpaint_motion()
    m = torch.zeros(motion.shape, dtype=torch.bool)
    m[..., :8] = True
    o = mo.sample_loop(W, tabs, tmap, inp["tape"], inp["text_embed"], inp["scale"], inp["lengths"], inpaint=(m, motion))
    assert rel_err(o, g["ddpm_inpaint"]) < TOL
    o = mo.sample_loop(W, tabs, tmap, inp["tape"], inp["text_embed"], inp["scale"], inp["lengths"], skip_timesteps=1,
                       init_image=motion)
    assert rel_err(o, g["ddpm_skip1_init"]) < TOL
    o = mo.sample_loop(W, tabs, tmap, inp["tape"], inp["text_embed"], None, inp["lengths"])
    assert rel_err(o, g["ddpm_noguide"]) < TOL


def test_c1_vs_golden(golden):
    g = golden("enc_c1.npz")
    W = mo.OracleWeights(b200mdm.synthetic_state_dict(num_layers=8, seed=0), 8)
    inp = b200mdm.synthetic_inputs(1, nframes=196, steps=50, seed=10)
    tabs = so.diffusion_tables(so.named_betas("cosine", 50))
    o = mo.sample_loop(W, tabs, list(range(50)), inp["tape"], inp["text_embed"], inp["scale"], inp["lengths"])
    assert rel_err(o, g["sample"]) < 1e-4   # 50 recurrent steps of fp32 round-off


def test_a2m_vs_golden(golden):
    g = golden("a2m_small.npz")
    sd = b200mdm.synthetic_state_dict(num_layers=2, input_feats=150, cond_mode="action", num_actions=12, seed=2)
    W = mo.OracleWeights(sd, 2)
    inp = b200mdm.synthetic_inputs(4, njoints=25, nfeats=6, nframes=60, steps=3, seed=12, lengths=[60, 60, 45, 30])
    tabs = so.diffusion_tables(so.named_betas("cosine", 3))
    o = mo.sample_loop(W, tabs, [0, 1, 2], inp["tape"], None, None, inp["lengths"], action=torch.from_numpy(g["action"]))
    assert rel_err(o, g["sample"]) < TOL


def _setup_dip():
    L, steps, B, ctx, pred, Mt = 2, 3, 3, 20, 40, 7
    W = mo.OracleWeights(b200mdm.synthetic_state_dict(arch="trans_dec", num_layers=L, cond_dim=768, seed=4), L)
    enc, tmask, prefix = b200mdm.synthetic_dip_inputs(B, Mt, ctx)
    inp = b200mdm.synthetic_inputs(B, nframes=pred, steps=steps, seed=13, lengths=[40, 33, 12], scale=torch.tensor([7.5, 2.0, 1.0]))
    return W, enc, tmask, prefix, inp


def test_dip_vs_golden(golden):
    """trans_dec + BERT memory + prefix completion (DiP): decoder restatement against the unmodified reference."""
    g = golden("dip_small.npz")
    W, enc, tmask, prefix, inp = _setup_dip()
    assert np.array_equal(tmask.numpy(), g["text_mask"])
    out = mo.cfg_denoise_dec(W, inp["tape"][0], 1, enc, tmask, prefix, inp["scale"], inp["lengths"])
    assert rel_err(out, g["fwd_cfg"]) < TOL
    tabs = so.diffusion_tables(so.named_betas("cosine", 3))
    o = mo.sample_loop_dec(W, tabs, [0, 1, 2], inp["tape"], enc, tmask, prefix, inp["scale"], inp["lengths"])
    assert rel_err(o, g["ddpm"]) < TOL


def test_oracle_vs_live_reference(golden):
    """The unmodified reference's p_sample_loop on seeds no other fixture uses (L=3, 6 steps, T=31), with its diffusion
    tables and timestep map, as run by oracle/gen_golden.py into golden/enc_l3.npz."""
    g = golden("enc_l3.npz")
    L, steps, B, T = 3, 6, 2, 31
    sd = b200mdm.synthetic_state_dict(num_layers=L, seed=7)
    inp = b200mdm.synthetic_inputs(B, nframes=T, steps=steps, seed=21, lengths=[31, 9], scale=torch.tensor([3.0, 0.5]))
    W = mo.OracleWeights(sd, L)
    tabs = so.diffusion_tables(so.named_betas("cosine", steps))
    for k in tabs:
        assert np.array_equal(tabs[k], g["table_" + k]), k
    tmap = [int(t) for t in g["timestep_map"]]
    o = mo.sample_loop(W, tabs, tmap, inp["tape"], inp["text_embed"], inp["scale"], inp["lengths"])
    assert tuple(o.shape) == (B, 263, 1, T)
    assert rel_err(o, g["sample"]) < TOL


def test_recover_from_ric_vs_golden(golden):
    """Post-loop step (generate.py:161-166): the restatement in oracle/ric_oracle.py against the reference's own
    inv_transform + recover_from_ric outputs, bit for bit (same torch CPU ops in the same order)."""
    from oracle import ric_oracle as ro
    g = golden("ric.npz")
    for D, J in ((263, 22), (251, 21)):
        gen = torch.Generator().manual_seed(100 + D)
        sample = torch.randn(3, D, 1, 40, generator=gen) * 0.8
        mean, std = b200mdm.synthetic_norm_stats(D, seed=7)
        assert torch.equal(ro.sample_to_xyz(sample, mean, std), torch.from_numpy(g["xyz_%d" % D]))
        assert torch.equal(ro.recover_from_ric(sample.permute(0, 2, 3, 1).contiguous(), J), torch.from_numpy(g["ric_%d" % D]))

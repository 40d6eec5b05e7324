import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        return np.load(os.path.join(GOLDEN, name), allow_pickle=False)
    return load


def default_args(**over):
    """The Namespace utils/parser_util.py of the reference produces for the released humanml models."""
    from types import SimpleNamespace
    a = dict(dataset="humanml", unconstrained=False, latent_dim=512, layers=8, cond_mask_prob=0.1, arch="trans_enc",
             emb_trans_dec=False, text_encoder_type="clip", pos_embed_max_len=5000, mask_frames=True, pred_len=0,
             context_len=0, diffusion_steps=50, noise_schedule="cosine", sigma_small=True, lambda_vel=0.0,
             lambda_rcxyz=0.0, lambda_fc=0.0)
    a.update(over)
    return SimpleNamespace(**a)


def inpaint_motion():
    """The motion [3, 263, 1, 24] the inpainting and init_image outputs of golden/enc_small.npz start from, drawn from the
    same seeded stream as in oracle/gen_golden.py (an input, so it is regenerated instead of stored)."""
    import numpy as np
    import torch
    return torch.from_numpy(np.random.default_rng(5).standard_normal((3, 263, 1, 24)).astype(np.float32))


def rel_err(a, b):
    import torch
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm())

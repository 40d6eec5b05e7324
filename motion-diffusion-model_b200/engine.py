"""Thin Python wrapper over the C ABI (include/b200mdm.h): torch tensors in, torch tensors out.

Everything numeric happens inside libb200mdm.so; this module only marshals pointers, keeps the tensors that
the engine references alive, and canonicalises the reference's untyped ``y`` dict into the POD arguments of
``b200mdm_set_cond``.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import check


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def target_validity(rows, target_joint_names, is_heading):
    """The validity mask EmbedTarget*.forward builds (model/mdm.py:411-416): uint8 [B, n], 1 at row(name) for every name
    in target_joint_names[b] and at row('heading') when is_heading[b].  target_joint_names: a list of name lists or the
    object ndarray sample_goal returns (empty sets allowed); an unknown name raises ValueError like the reference's
    list.index."""
    heading = np.asarray(torch.as_tensor(is_heading).detach().cpu()).reshape(-1).astype(bool)
    if len(target_joint_names) != heading.shape[0]:
        raise ValueError("target_joint_names has %d entries, is_heading %d" % (len(target_joint_names), heading.shape[0]))
    valid = np.zeros((heading.shape[0], len(rows)), dtype=np.uint8)
    for b, names in enumerate(target_joint_names):
        names = [str(j) for j in np.asarray(names, dtype=object).reshape(-1)] + (["heading"] if heading[b] else [])
        for j in names:
            valid[b, rows.index(j)] = 1
    return valid


class Engine:
    """One engine per model instance (weights + workspace live on the current CUDA device)."""

    def __init__(self, *, arch, latent_dim, ff_size, num_layers, num_heads, njoints, nfeats, cond_mode, cond_dim,
                 num_actions, mask_frames, pos_embed_max_len, temb_rows, context_len=0, target_encoder=None,
                 target_rows=None, target_enc_layers=1):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("b200mdm needs a CUDA device (sm_100a); there is no CPU fallback")
        cm = _lib.COND_TEXT if "text" in cond_mode else _lib.COND_ACTION if "action" in cond_mode else _lib.COND_NONE
        self.cfg = _lib.Config(arch=_lib.ARCH[arch], latent_dim=latent_dim, ff_size=ff_size, num_layers=num_layers,
                               num_heads=num_heads, njoints=njoints, nfeats=nfeats, cond_mode=cm, cond_dim=cond_dim,
                               num_actions=num_actions, mask_frames=int(bool(mask_frames)),
                               pos_embed_max_len=pos_embed_max_len, temb_rows=temb_rows, context_len=context_len,
                               target_encoder=_lib.TARGET[target_encoder], n_goal_rows=len(target_rows or ()),
                               target_enc_layers=target_enc_layers)
        self.target_rows = list(target_rows) if target_encoder is not None else None
        self.dec = arch == "trans_dec"
        self.context_len = context_len
        h = ctypes.c_void_p()
        check(self.lib.b200mdm_create(ctypes.byref(self.cfg), ctypes.byref(h)))
        self.h = h
        self.cond_mode = cm
        self._keep = {}
        self._cond_key = None
        self._sched_key = None
        self.batch = self.nframes = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.b200mdm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ weights
    def load_state_dict(self, sd):
        for name, t in sd.items():
            if not torch.is_tensor(t):
                continue
            t = t.detach().to(torch.float32).contiguous()
            shape = (ctypes.c_int64 * t.dim())(*t.shape)
            check(self.lib.b200mdm_load_weight(self.h, name.encode(), _ptr(t), shape, t.dim()))
        check(self.lib.b200mdm_finalize_weights(self.h, _stream()))
        self._cond_key = None

    # ------------------------------------------------------------------ schedule
    def set_schedule(self, rows, timestep_map, key=None):
        if key is not None and key == self._sched_key:
            return
        rows = np.ascontiguousarray(rows, dtype=np.float32)
        tmap = np.ascontiguousarray(timestep_map, dtype=np.int32)
        assert rows.shape == (len(tmap), _lib.SCHED_STRIDE)
        check(self.lib.b200mdm_set_schedule(self.h, len(tmap), rows.ctypes.data_as(ctypes.c_void_p),
                                            tmap.ctypes.data_as(ctypes.c_void_p)))
        self._sched_key = key

    # ------------------------------------------------------------------ conditioning
    def set_target(self, batch, y, device):
        """y['target_cond'] [B, n, 3] (+ y['target_joint_names'], y['is_heading']) -> b200mdm_set_target, for the next
        set_cond*.  No 'target_cond' key, or y['target_uncond'] (mask_cond zeros the embedding, model/mdm.py:199): the
        target is cleared, and the loop is exactly the one without targets.  The target is the same for both halves of a
        CFG pair (the reference's guidance wrapper deep-copies y, targets included)."""
        if self.target_rows is None:
            if y is not None and "target_cond" in y:
                raise AttributeError("y['target_cond'] given to a model without target conditioning: 'MDM' object has "
                                     "no attribute 'embed_target_cond' (create it with multi_target_cond=True)")
            return
        tc = y.get("target_cond") if y is not None else None
        if tc is None or bool(y.get("target_uncond", False)):
            check(self.lib.b200mdm_set_target(self.h, batch, None, None, _stream()))
            self._keep.pop("target", None)
            return
        names, heading = y["target_joint_names"], y["is_heading"]      # KeyError, as the reference's y[...]
        n = len(self.target_rows)
        tc = torch.as_tensor(tc).detach().to(device=device, dtype=torch.float32).contiguous()
        if tuple(tc.shape) != (batch, n, 3):
            raise ValueError("y['target_cond'] must be [batch, %d, 3] (rows %s), got %s" % (n, self.target_rows, tuple(tc.shape)))
        valid = target_validity(self.target_rows, names, heading)
        if valid.shape[0] != batch:
            raise ValueError("target_joint_names / is_heading describe %d samples, the batch has %d" % (valid.shape[0], batch))
        check(self.lib.b200mdm_set_target(self.h, batch, _ptr(tc), valid.ctypes.data_as(ctypes.c_void_p), _stream()))
        self._keep["target"] = (tc, valid)

    def set_cond(self, batch, nframes, y, guided, device):
        """Canonicalise model_kwargs['y'] (data_loaders/tensors.py:22-64 schema).  `guided` => CFG pair."""
        self.set_target(batch, y, device)
        text_embed = y.get("text_embed") if y is not None else None
        if self.dec:
            return self._set_cond_dec(batch, nframes, y, guided, device)
        if isinstance(text_embed, tuple):
            raise NotImplementedError("BERT (tokens, mask) conditioning belongs to the trans_dec path")
        lengths = y.get("lengths") if y is not None else None
        mask = y.get("mask") if y is not None else None
        if mask is not None and mask.shape[-1] <= 1:      # model/mdm.py:242 "is_valid_mask"
            lengths = None
        elif lengths is None and mask is not None:        # prefix mask -> lengths (tensors.py:3-6)
            lengths = mask.reshape(mask.shape[0], -1).sum(-1)
        scale = y.get("scale") if (guided and y is not None) else None
        if guided and scale is None:
            raise AssertionError("ClassifierFreeSampleModel needs y['scale'] (sampler_util.py:34)")
        uncond = bool(y.get("uncond", False)) if y is not None else False
        action = y.get("action") if y is not None else None
        te = None
        if text_embed is not None and self.cond_mode == _lib.COND_TEXT:
            te = text_embed.detach().to(device=device, dtype=torch.float32)
            te = te.reshape(-1, te.shape[-1])
            if te.shape[0] == 1 and batch > 1:             # single prompt for the whole batch (sample/predict.py)
                te = te.expand(batch, -1)
            te = te.contiguous()
            assert te.shape == (batch, self.cfg.cond_dim), (te.shape, batch, self.cfg.cond_dim)
        ln = None
        if lengths is not None:
            ln = np.ascontiguousarray(lengths.detach().reshape(-1).cpu().numpy().astype(np.int64))
            assert ln.shape[0] == batch
        sc = None
        if scale is not None:
            sc = scale.detach().to(device=device, dtype=torch.float32).reshape(-1).contiguous()
            assert sc.shape[0] == batch
        ac = None
        if action is not None and self.cond_mode == _lib.COND_ACTION:
            ac = np.ascontiguousarray(action.detach().reshape(batch, -1)[:, 0].cpu().numpy().astype(np.int64))
        check(self.lib.b200mdm_set_cond(self.h, batch, nframes, _ptr(te),
                                        None if ln is None else ln.ctypes.data_as(ctypes.c_void_p), _ptr(sc),
                                        int(uncond), None if ac is None else ac.ctypes.data_as(ctypes.c_void_p),
                                        _stream()))
        self._keep["cond"] = (te, sc)
        self.batch, self.nframes = batch, nframes

    def _set_cond_dec(self, batch, nframes, y, guided, device):
        """DiP: y['text_embed'] = (BERT tokens [Mt,B,768], padding mask [B,Mt] True = pad), y['prefix'] [B,J,F,ctx]
        (reference model/mdm.py:203-206,210-217,264)."""
        te = y.get("text_embed")
        if not isinstance(te, tuple):
            raise RuntimeError("trans_dec (DiP) needs y['text_embed'] = (tokens, mask) from bert_encode_text "
                               "(model/mdm.py:180-187)")
        enc, tmask = te
        enc = enc.detach().to(device=device, dtype=torch.float32)
        if enc.shape[1] == 1 and batch > 1:
            enc = enc.expand(-1, batch, -1)
        enc = enc.contiguous()
        if tmask.shape[0] == 1 and batch > 1:                  # model/mdm.py:215-216
            tmask = torch.repeat_interleave(tmask, batch, dim=0)
        Mt = enc.shape[0]
        assert enc.shape == (Mt, batch, self.cfg.cond_dim) and tuple(tmask.shape) == (batch, Mt), (enc.shape, tmask.shape)
        tm = np.ascontiguousarray(tmask.detach().cpu().numpy().astype(np.uint8))
        lengths, mask = y.get("lengths"), y.get("mask")
        if mask is not None and mask.shape[-1] <= 1:
            lengths = None
        elif lengths is None and mask is not None:
            lengths = mask.reshape(mask.shape[0], -1).sum(-1)
        ln = None
        if lengths is not None:
            ln = np.ascontiguousarray(lengths.detach().reshape(-1).cpu().numpy().astype(np.int64))
            assert ln.shape[0] == batch
        scale = y.get("scale") if guided else None
        if guided and scale is None:
            raise AssertionError("ClassifierFreeSampleModel needs y['scale'] (sampler_util.py:34)")
        sc = None
        if scale is not None:
            sc = scale.detach().to(device=device, dtype=torch.float32).reshape(-1).contiguous()
            assert sc.shape[0] == batch
        check(self.lib.b200mdm_set_cond_dec(self.h, batch, nframes, _ptr(enc), tm.ctypes.data_as(ctypes.c_void_p), Mt,
                                            None if ln is None else ln.ctypes.data_as(ctypes.c_void_p), _ptr(sc),
                                            int(bool(y.get("uncond", False))), _stream()))
        pf = None
        if self.context_len > 0:
            if "prefix" not in y:
                raise KeyError("prefix completion needs y['prefix'] [B, njoints, nfeats, context_len] (model/mdm.py:204)")
            pf = y["prefix"].detach().to(device=device, dtype=torch.float32).contiguous()
            assert tuple(pf.shape) == (batch, self.cfg.njoints, self.cfg.nfeats, self.context_len), pf.shape
            check(self.lib.b200mdm_set_prefix(self.h, _ptr(pf), _stream()))
        self._keep["cond"] = (enc, sc, pf)
        self.batch, self.nframes = batch, nframes

    def set_inpaint(self, mask, motion):
        if mask is None:
            check(self.lib.b200mdm_set_inpaint(self.h, None, None))
            self._keep.pop("inpaint", None)
            return
        m8 = mask.to(torch.uint8).contiguous()
        mo = motion.to(torch.float32).contiguous()
        check(self.lib.b200mdm_set_inpaint(self.h, _ptr(m8), _ptr(mo)))
        self._keep["inpaint"] = (m8, mo)

    # ------------------------------------------------------------------ compute
    def denoise(self, x, timesteps):
        x = x.to(torch.float32).contiguous()
        ts = np.ascontiguousarray(timesteps.detach().reshape(-1).cpu().numpy().astype(np.int32))
        assert ts.shape[0] == x.shape[0]
        out = torch.empty_like(x)
        check(self.lib.b200mdm_denoise(self.h, _ptr(x), ts.ctypes.data_as(ctypes.c_void_p), _ptr(out), _stream()))
        return out

    def sample_step(self, mode, index, x_t, noise, flags=0, want_pred=True):
        x_t = x_t.to(torch.float32).contiguous()
        noise = noise.to(torch.float32).contiguous()
        out = torch.empty_like(x_t)
        pred = torch.empty_like(x_t) if want_pred else None
        check(self.lib.b200mdm_sample_step(self.h, mode, index, _ptr(x_t), _ptr(noise), flags, _ptr(out), _ptr(pred),
                                           _stream()))
        return out, pred

    def sample_loop(self, mode, x, tape, skip_timesteps=0, flags=0, use_graph=True):
        """x: [B,J,F,T] fp32 (x_T, left untouched); tape: [n_run, B,J,F,T] fp32.  Returns x_0 (new tensor)."""
        x = x.to(torch.float32).contiguous()
        assert tape.is_contiguous() and tape.dtype == torch.float32
        out = torch.empty_like(x)
        check(self.lib.b200mdm_sample_loop(self.h, mode, skip_timesteps, _ptr(x), _ptr(out), _ptr(tape), tape.stride(0),
                                           flags, int(use_graph), _stream()))
        # the loop is asynchronous and runs on the engine's own stream, which torch's caching allocator knows nothing
        # about: the inputs are kept referenced here until the next loop replaces them
        self._keep["loop"] = (x, tape)
        return out

    def sample_loop_range(self, mode, first_index, n_run, x_in, x_out, tape, flags=0, use_graph=True):
        """Steps first_index .. first_index-n_run+1 on the engine's working buffer (b200mdm_sample_loop_range).
        x_in None: continue; x_out None: leave the state in the engine; tape None: B200MDM_FLAG_PHILOX_NOISE."""
        if tape is not None:
            assert tape.is_contiguous() and tape.dtype == torch.float32 and tape.shape[0] >= n_run
        else:
            flags |= _lib.FLAG_PHILOX_NOISE
        check(self.lib.b200mdm_sample_loop_range(self.h, mode, first_index, n_run, _ptr(x_in), _ptr(x_out), _ptr(tape),
                                                 tape.stride(0) if tape is not None else 0, flags, int(use_graph), _stream()))

    def set_noise_stream(self, seed, sample_index_base=0):
        check(self.lib.b200mdm_set_noise_stream(self.h, ctypes.c_uint64(int(seed) & (2 ** 64 - 1)), int(sample_index_base)))

    def philox_normal(self, shape, seed, sample_index_base, step_id, device):
        """[B, ...] fp32 from the engine's counter-based stream (x_T: step_id = -1)."""
        out = torch.empty(tuple(shape), device=device, dtype=torch.float32)
        n = out[0].numel()
        check(self.lib.b200mdm_philox_normal(_ptr(out), int(shape[0]), n, ctypes.c_uint64(int(seed) & (2 ** 64 - 1)),
                                             int(sample_index_base), int(step_id), _stream()))
        return out

    def q_sample(self, sqrt_ac, sqrt_1mac, x_start, noise):
        out = torch.empty_like(noise)
        check(self.lib.b200mdm_q_sample(self.h, float(sqrt_ac), float(sqrt_1mac), _ptr(x_start), _ptr(noise), _ptr(out),
                                        noise.numel(), _stream()))
        return out

    def launch_count(self, reset=False):
        return int(self.lib.b200mdm_launch_count(self.h, int(reset)))

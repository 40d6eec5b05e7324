"""Batch-of-prompts data parallelism over the GPUs of one box (SURVEY.md section 8e).

Samples never interact inside the sampling loop (attention is per sample, LayerNorm per token), so the batch is cut
into contiguous per-rank slices; the ONLY collective of the path is one broadcast of the cached text embedding
(the reference encodes the prompts once per loop, diffusion/gaussian_diffusion.py:633-635), plus an optional gather
of the finished motions.  Nothing crosses GPUs inside the loop.

Determinism: ``noise_mode="philox"`` (default) uses the engine's counter-based noise stream keyed by (seed, step,
GLOBAL sample index) -- each rank generates exactly its own samples' noise inside the step graph (no tape, no redundant
draws) and the G-GPU result is bitwise identical to the 1-GPU result for that seed.  ``noise_mode="global"`` gets the same
property from torch's generator by drawing the global batch on every rank and keeping a slice (G-fold redundant RNG, done
step by step so that only one step of global noise is alive at a time); ``noise_mode="per_rank"`` lets each rank draw
its slice from its own torch stream (rank-dependent results).

One process per GPU, ``torch.distributed`` (backend nccl on GPUs; the same code runs on gloo/CPU in the tests).
"""
import numpy as np
import torch
import torch.distributed as dist


def shard_range(global_batch, rank, world):
    """Contiguous slice [lo, hi) of rank `rank`; the first (global_batch % world) ranks get one extra sample."""
    base, extra = divmod(global_batch, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def broadcast_text_embed(text_embed, src=0, group=None):
    """The one collective of the path: rank `src` owns the encoded prompts -- CLIP features [1, B, C], or for DiP the
    (BERT tokens [Mt, B, 768], padding mask [B, Mt]) pair; everybody receives them."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        for t in (text_embed if isinstance(text_embed, tuple) else (text_embed,)):
            if t.dtype == torch.bool:                 # gloo / nccl broadcast byte tensors, not bool
                b = t.to(torch.uint8)
                dist.broadcast(b, src=src, group=group)
                t.copy_(b.to(torch.bool))
            else:
                dist.broadcast(t, src=src, group=group)
    return text_embed


def shard_replications(replication_times, rank=None, world=None):
    """Evaluation (eval/eval_humanml.py:262-329 runs the whole generate-and-score pass `replication_times` times, each
    with its own `CompMDMGeneratedDataset`): replications are independent, so rank r takes replications
    r, r + world, ... and the per-replication metrics are gathered afterwards (`gather_objects`).  No traffic between the
    ranks while a replication runs."""
    if rank is None:
        rank = dist.get_rank() if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size() if dist.is_initialized() else 1
    return list(range(rank, replication_times, world))


def gather_objects(obj, group=None):
    """All ranks' python objects (e.g. {replication index: metrics dict}) on every rank, in rank order."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return [obj]
    out = [None] * dist.get_world_size(group)
    dist.all_gather_object(out, obj, group=group)
    return out


_BATCH_KEYS = ("mask", "lengths", "scale", "action", "inpainting_mask", "inpainted_motion", "prefix", "target_cond",
               "is_heading")


def shard_model_kwargs(model_kwargs, lo, hi):
    """Slice the reference's `y` dict (data_loaders/tensors.py:22-64 schema) along the batch dimension."""
    y = model_kwargs["y"]
    out = {}
    for k, v in y.items():
        if k == "text_embed" and torch.is_tensor(v):
            out[k] = v[:, lo:hi].contiguous() if v.shape[1] > 1 else v      # [1, B, C]; a single prompt is shared
        elif k == "text_embed" and isinstance(v, tuple):                     # DiP: (tokens [Mt, B, C], mask [B, Mt])
            tok, msk = v
            out[k] = (tok[:, lo:hi].contiguous() if tok.shape[1] > 1 else tok, msk[lo:hi].contiguous() if msk.shape[0] > 1 else msk)
        elif k in _BATCH_KEYS and torch.is_tensor(v):
            out[k] = v[lo:hi].contiguous()
        elif k in ("text", "tokens") and isinstance(v, (list, tuple)):
            out[k] = list(v[lo:hi])
        elif k == "target_joint_names" and isinstance(v, (list, tuple, np.ndarray)):   # a name set per sample
            out[k] = v[lo:hi] if isinstance(v, np.ndarray) else list(v[lo:hi])
        else:
            out[k] = v
    return {**model_kwargs, "y": out}


def sample_sharded(sample_fn, model, shape, model_kwargs, *, n_steps, noise_mode="philox", seed=None, device=None,
                   gather=True, group=None, **kwargs):
    """Run `sample_fn` (e.g. ``diffusion.p_sample_loop``) on this rank's slice of the batch.

    shape: GLOBAL shape (B, J, F, T).  `model_kwargs['y']['text_embed']` needs to be valid on rank 0 only (it is
    broadcast); the other entries must be present on every rank.  Returns the gathered [B, J, F, T] tensor on every
    rank when `gather` (all_gather), else the local slice.
    """
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    B = int(shape[0])
    if B < world:
        # a rank with an empty shard would skip the loop but still has to meet the others in the collectives; the
        # reference never samples fewer motions than it has GPUs -- refuse up front instead of hanging in all_gather
        raise ValueError("global batch %d is smaller than the number of ranks %d" % (B, world))
    lo, hi = shard_range(B, rank, world)
    y = model_kwargs["y"]
    if torch.is_tensor(y.get("text_embed")) or isinstance(y.get("text_embed"), tuple):
        broadcast_text_embed(y["text_embed"], 0, group)
    local_kwargs = shard_model_kwargs(model_kwargs, lo, hi)
    local_shape = (hi - lo,) + tuple(shape[1:])
    if device is None:
        te = y.get("text_embed")
        te = te[0] if isinstance(te, tuple) else te
        device = te.device if torch.is_tensor(te) else torch.device("cpu")
    if noise_mode == "philox":
        # engine stream: x_T and every eps are functions of (seed, step, global sample index) -- nothing is drawn here
        local = sample_fn(model, local_shape, model_kwargs=local_kwargs, noise_seed=0 if seed is None else seed,
                          sample_index_base=lo, **kwargs)
    else:
        gen = None
        if seed is not None:
            gen = torch.Generator(device=device)
            gen.manual_seed(seed if noise_mode == "global" else seed + 7919 * rank)
        if noise_mode == "global":
            # identical stream on every rank, in the reference's draw order: x_T, then one eps per step; one global
            # step is alive at a time (the local tape is still O(n_steps): use "philox" for 1000-step loops)
            x_T = torch.randn(tuple(shape), device=device, generator=gen)[lo:hi].contiguous()
            tape = torch.empty((n_steps,) + local_shape, device=device)
            for k in range(n_steps):
                tape[k] = torch.randn(tuple(shape), device=device, generator=gen)[lo:hi]
        elif noise_mode == "per_rank":
            x_T = torch.randn(local_shape, device=device, generator=gen)
            tape = torch.randn((n_steps,) + local_shape, device=device, generator=gen)
        else:
            raise ValueError("noise_mode must be 'philox', 'global' or 'per_rank'")
        local = sample_fn(model, local_shape, noise=x_T, model_kwargs=local_kwargs, noise_tape=tape, **kwargs)
    if not gather or world == 1:
        return local
    # all_gather wants equal shapes: pad every shard to the largest one, trim after the exchange
    sizes = [h - l for l, h in (shard_range(B, r, world) for r in range(world))]
    top = max(sizes)
    padded = torch.zeros((top,) + tuple(shape[1:]), device=local.device, dtype=local.dtype)
    padded[: hi - lo] = local
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    return torch.cat([p[:n] for p, n in zip(parts, sizes)], dim=0)

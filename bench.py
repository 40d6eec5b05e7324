#!/usr/bin/env python
"""bench.py -- motions/sec of the MDM sampling hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config c2|c3|dip|a2m] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one complete sampling loop over one batch.  Default (--config c2) = BASELINE config 2 -- HumanML3D shapes,
B=64 motions per GPU, 196 frames x 263 features, 50 DDPM steps, classifier-free guidance 2.5 (cond/uncond packed to 128
sequences), trans_enc L=8 d=512 -- synthetic weights / text embeddings / noise (no network for checkpoints).
Other BASELINE configs (same JSON line, their own FLOP count from SURVEY.md section 8d):
  c3  : HumanML3D, 1000 steps, 64 motions per GPU, through parallel.sample_sharded (NCCL broadcast of the text embedding,
        engine-side Philox noise: no 13 GB tape)          dip : DiP trans_dec, B=128, 5 chunks x 10 steps, guidance 7.5
  a2m : HumanAct12 action2motion, 64 motions per GPU (B=256 on 4 GPUs), 60 frames, 1000 steps, no guidance
  value : whole-job motions/s, inputs (x_T, 660 MB noise tape, text embedding) resident in HBM, CUDA events, max over ranks
  e2e   : the same metric through the public API call a user makes (diffusion.p_sample_loop(model, shape, model_kwargs)),
          conditioning copied from pinned host memory and the sample read back to the host inside the timed region;
          noise is drawn on the device by the API exactly as the reference does on a GPU
  roofline     : the dominant kernel of the step (see DESIGN.md section 4) timed alone with CUDA events, L2 flushed
  cpu_baseline : the reference's own CPU p_sample_loop (unmodified files in oracle/_ref, kind "reference") on a bounded
                 sample: full 50 steps, as many of the 64 motions as the time box allows; the oracle port if _ref is absent
--dump-outputs DIR writes DIR/sample.npy (float32): the motions the last timed resident loop returned to its caller (rank
0's shard with several GPUs).  Weights, conditioning and noise come from fixed seeds (torch's default generators, which
DiP draws its noise from, are seeded per rank at start-up), so two builds run with the same arguments can be compared
output for output.
Multi-GPU: batch sharded, one NCCL broadcast of the text embedding per loop, nothing inside the loop ("weak" scaling:
64 motions per GPU).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, T, J, STEPS, L, D, FF, SCALE = 64, 196, 263, 50, 8, 512, 1024, 2.5


WORKLOAD = "HumanML3D text2motion B=64/GPU T=196 J=263 50 DDPM steps CFG 2.5 trans_enc L8 d512 ff1024 h4"


def flops_per_forward_sample(S=T + 1, d=D, ff=FF, layers=L, jf=J, t=T):
    """SURVEY.md section 8d: F_fwd = L*2S*(3d^2 + d^2 + 2*d*ff + 2*S*d) + 2*(2*T*JF*d)."""
    return layers * 2 * S * (3 * d * d + d * d + 2 * d * ff + 2 * S * d) + 2 * (2 * t * jf * d)


FLOP_PER_MOTION = flops_per_forward_sample() * 2 * STEPS   # two CFG forwards per step


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d["bf16_tflops"], sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), hbm=d["hbm_gbs"],
                    source="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback")


class ClockSampler:
    """SM clock + throttle reasons DURING the timed region (B200_PROFILING.md clocks line).

    Two independent sources, both opened BEFORE the warm-up so that their start-up cost (nvmlInit, the first nvidia-smi
    line) is not paid inside the region: an in-process NVML poll every 20 ms (a 0.4 s region still gets ~20 samples) and
    an `nvidia-smi -lms 100` child whose lines are time-stamped on arrival.  stop() reports the NVML samples taken between
    start() and stop(); if there are none (r02_p: one run in five came back empty, every poll raising), the nvidia-smi
    lines of the same window; if there are none either, one synchronous sample taken at stop() -- the GPU has just
    finished the last step -- and says so in `source`."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = (0x8, 0x40, 0x20, 0x4)   # hw_slowdown, hw_thermal_slowdown, sw_thermal_slowdown, sw_power_cap
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index, enabled=True):
        self.idx, self.proc, self.nvml, self.handle = gpu_index, None, None, None
        self.nvml_rows, self.smi_rows, self.errors = [], [], []
        self.t0, self.t1, self.stop_flag, self.thread = None, None, False, None
        if not enabled:
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                import torch
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(gpu_index).uuid)).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nvml, self.handle = pynvml, h
            self._nvml_sample()           # pays the first-call cost outside the region; raises if NVML is unusable
        except Exception as e:            # noqa: BLE001
            self.errors.append("nvml open: %r" % (e,))
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            import atexit
            atexit.register(lambda p=self.proc: p.poll() is None and p.terminate())   # never leave the child behind
        except Exception as e:            # noqa: BLE001
            self.errors.append("nvidia-smi: %r" % (e,))
            self.proc = None

    def _nvml_sample(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = int(get(self.handle))
        return (time.perf_counter(), int(sm), int(mx), [nm for b, nm in zip(self.BITS, self.NAMES) if bits & b])

    def _nvml_poll(self):
        while not self.stop_flag:
            try:
                self.nvml_rows.append(self._nvml_sample())
            except Exception as e:        # noqa: BLE001
                if len(self.errors) < 4:
                    self.errors.append("nvml poll: %r" % (e,))
            time.sleep(0.02)

    def _pump(self):
        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(",")]
            if len(c) >= 9 and c[1].isdigit() and c[2].isdigit():
                self.smi_rows.append((time.perf_counter(), int(c[1]), int(c[2]),
                                      [nm for nm, v in zip(self.NAMES, c[5:9]) if v.lower().startswith("active")]))

    def start(self):
        self.t0 = time.perf_counter()
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._nvml_poll, daemon=True)
            self.thread.start()

    def stop(self):
        self.t1 = time.perf_counter()
        if self.t0 is None:
            self.t0 = self.t1
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=1.0)
        if self.proc is not None:
            time.sleep(0.12)              # the line that covers the end of the region
            self.proc.terminate()
        window = lambda rows: [r for r in rows if self.t0 <= r[0] <= self.t1 + 0.12]
        rows, source = window(self.nvml_rows), "nvml 20 ms"
        if not rows:
            rows, source = window(self.smi_rows), "nvidia-smi -lms 100"
        if not rows and self.nvml is not None:
            try:
                rows, source = [self._nvml_sample()], "nvml, ONE sample at the end of the timed region (no in-region sample)"
            except Exception as e:        # noqa: BLE001
                self.errors.append("nvml final: %r" % (e,))
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0,
                    "source": "none", "errors": self.errors}
        sm = sorted(r[1] for r in rows)
        out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[2] for r in rows),
               "reasons": sorted({nm for r in rows for nm in r[3]}), "samples": len(rows), "source": source}
        if self.errors:
            out["errors"] = self.errors
        return out


def make_args(**over):
    from types import SimpleNamespace
    a = dict(dataset="humanml", unconstrained=False, latent_dim=D, layers=L, cond_mask_prob=0.1,
             arch="trans_enc", emb_trans_dec=False, text_encoder_type="clip", pos_embed_max_len=5000,
             mask_frames=True, pred_len=0, context_len=0, diffusion_steps=STEPS, noise_schedule="cosine",
             sigma_small=True, lambda_vel=0.0, lambda_rcxyz=0.0, lambda_fc=0.0)
    a.update(over)
    return SimpleNamespace(**a)


# FLOPs per denoiser forward per sample, SURVEY.md section 8d
def flops_dec_forward(S=60, Mt=16, d=D, ff=FF, layers=L, jf=J, pred=40):
    """trans_dec (DiP): self-attention + cross-attention (K/V projection of the Mt memory tokens) + FFN + in/out proj."""
    per_layer = 2 * S * (3 * d * d + d * d) + 4 * S * S * d            # self-attn projections + core
    per_layer += 2 * S * d * d + 2 * Mt * 2 * d * d + 4 * S * Mt * d + 2 * S * d * d   # cross-attn: q, kv(memory), core, out
    per_layer += 4 * S * d * ff
    return layers * per_layer + 2 * S * jf * d + 2 * pred * jf * d      # input projection on ctx+pred frames, output on pred


CONFIGS = {
    "c2": dict(workload=WORKLOAD, steps=STEPS, per_gpu=64, flop_per_motion=FLOP_PER_MOTION),
    "c3": dict(workload="HumanML3D text2motion B=64/GPU T=196 J=263 1000 DDPM steps CFG 2.5 trans_enc L8 d512 (BASELINE config 3 "
                        "shard; parallel.sample_sharded, engine Philox noise)", steps=1000, per_gpu=64,
               flop_per_motion=flops_per_forward_sample() * 2 * 1000),
    "a2m": dict(workload="HumanAct12 action2motion B=64/GPU (256 on 4 GPUs) T=60 25x6 feats 1000 DDPM steps no guidance trans_enc L8 d512",
                steps=1000, per_gpu=64, flop_per_motion=flops_per_forward_sample(S=61, jf=150, t=60) * 1000),
    "dip": dict(workload="DiP trans_dec L8 d512 B=128/GPU, 5 autoregressive chunks of 40 frames (context 20), 10 steps per chunk, "
                         "guidance 7.5, 16 BERT tokens", steps=10, per_gpu=128, flop_per_motion=flops_dec_forward() * 2 * 10 * 5),
}


# ----------------------------------------------------------------------------------------------------- CPU arms
def host_threads():
    """Threads the CPU arm may use: the cgroup quota if there is one, else the affinity mask (capped at 64)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, min(n, 64))


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ReferenceCpu:
    """The reference's own CPU sampling loop, UNMODIFIED: `diffusion.p_sample_loop(ClassifierFreeSampleModel(MDM), ...)` of
    GuyTevet/motion-diffusion-model imported from oracle/_ref (the byte-for-byte copy of its 15 hot-path files made by
    oracle/build_ref.py), random-init weights of the released architecture, torch fp32 on all host threads."""

    def __init__(self, threads, steps=STEPS):
        import torch
        from oracle import ref_harness as rh
        if not rh.available():
            raise RuntimeError("oracle/_ref is absent (run __graft_entry__.build() in the build container)")
        torch.set_num_threads(threads)
        self.torch, self.rh, self.steps = torch, rh, steps
        import b200mdm
        self.model, self.diffusion = rh.build(rh.default_args(diffusion_steps=steps),
                                              state_dict=b200mdm.synthetic_state_dict(num_layers=L, seed=0))
        ns = rh.load_reference()
        self.cfg = ns.sampler_util.ClassifierFreeSampleModel(self.model)

    def loop(self, batch):
        """One full p_sample_loop (all `steps` steps, CFG 2.5) over `batch` motions; returns seconds."""
        torch = self.torch
        g = torch.Generator().manual_seed(10)
        y = {"mask": torch.ones(batch, 1, 1, T, dtype=torch.bool), "lengths": torch.full((batch,), T),
             "text_embed": torch.randn(1, batch, 512, generator=g), "scale": torch.full((batch,), SCALE)}
        t0 = time.perf_counter()
        with torch.no_grad():
            out = self.diffusion.p_sample_loop(self.cfg, (batch, J, 1, T), clip_denoised=False, model_kwargs={"y": y},
                                               skip_timesteps=0, init_image=None, progress=False, dump_steps=None,
                                               noise=None, const_noise=False)
        assert tuple(out.shape) == (batch, J, 1, T)
        return time.perf_counter() - t0


def reference_cpu_measure(n_loops, warm, budget_s):
    """Times the unmodified reference on the host cores.  The batch is the largest of 4, 8, 16, 32, 64 for which
    (n_loops + warm) full loops fit the time budget (measured with one warm loop of 4).  Returns a dict."""
    threads = host_threads()
    ref = ReferenceCpu(threads)
    t4 = ref.loop(4)                                     # warm-up (thread pools, allocator) + the sizing probe
    per_motion = t4 / 4
    batch = 4
    for b in (64, 32, 16, 8):
        if per_motion * b * (n_loops + warm) <= budget_s:
            batch = b
            break
    for _ in range(warm):
        ref.loop(batch)
    secs = [ref.loop(batch) for _ in range(n_loops)]
    sec = sum(secs) / len(secs)
    return dict(value=batch / sec, sec_per_loop=sec, batch=batch, threads=threads, kind="reference",
                sample="UNMODIFIED reference p_sample_loop (oracle/_ref: gaussian_diffusion.py + ClassifierFreeSampleModel + MDM), "
                       "%d of 64 motions per loop, all %d steps timed (x2 CFG forwards each), no extrapolation, %d loops of %.1f s; "
                       "torch fp32, %d threads; %s" % (batch, STEPS, n_loops, sec, threads, cpu_model_name()))


def port_cpu_measure(budget_s):
    """Fallback when oracle/_ref is absent: the oracle PORT of the reference loop (oracle/mdm_oracle.py), 4 motions, as many
    of the 50 steps as fit the budget, extrapolated."""
    import torch
    import b200mdm
    from oracle import mdm_oracle as mo, schedule_oracle as so
    threads = host_threads()
    torch.set_num_threads(threads)
    W = mo.OracleWeights(b200mdm.synthetic_state_dict(num_layers=L, seed=0), L)
    inp = b200mdm.synthetic_inputs(4, nframes=T, steps=STEPS, seed=10)
    tabs = so.diffusion_tables(so.named_betas("cosine", STEPS))
    x = inp["tape"][0].clone()
    times = []
    with torch.no_grad():
        for k, i in enumerate(range(STEPS - 1, -1, -1)):
            t0 = time.perf_counter()
            x0 = mo.cfg_denoise_enc(W, x, i, inp["text_embed"], inp["scale"], inp["lengths"])
            x, _ = mo.p_sample_step(tabs, x0, x, i, inp["tape"][1 + k])
            times.append(time.perf_counter() - t0)
            if sum(times) > budget_s and len(times) >= 2:
                break
    steady = times[1:] if len(times) > 1 else times
    per_step = sum(steady) / len(steady)
    sec = per_step * STEPS
    return dict(value=4 / sec, sec_per_loop=sec, batch=4, threads=threads, kind="port",
                sample="oracle PORT of the reference loop (oracle/_ref absent): 4 of 64 motions, %d of 50 steps timed, extrapolated; "
                       "torch fp32, %d threads; %s" % (len(times), threads, cpu_model_name()))


def cpu_arm(n_loops, warm, budget_s):
    try:
        return reference_cpu_measure(n_loops, warm, budget_s)
    except Exception as e:                                 # noqa: BLE001 -- any import problem => the port, and say so
        sys.stderr.write("[bench] reference arm unavailable (%s); timing the oracle port instead\n" % (e,))
        return port_cpu_measure(min(budget_s, 20.0))


def run_reference_arm(a, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, rank 0 only."""
    if rank != 0:
        return
    if a.config != "c2":
        print(json.dumps({"impl": "reference", "unavailable": "the CPU reference arm is defined for --config c2 (BASELINE config 1/2)"}), flush=True)
        return
    m = cpu_arm(max(1, a.steps), min(a.warmup, 1), 200.0)
    line = {"impl": "reference", "metric": "motions/sec", "value": round(m["value"], 4), "unit": "motions/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(m["sec_per_loop"] * 1e3, 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": 64 * max(1, a.gpus),
                       "sample": "%d of 64 motions per loop (one step = one full 50-step loop over that sample)" % m["batch"]},
            "cpu_baseline": {"value": round(m["value"], 4), "unit": "motions/s", "cores": m["threads"], "kind": m["kind"],
                             "sample": m["sample"]},
            "e2e": {"value": round(m["value"], 4), "unit": "motions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------- GPU arm
def build_workload(cfg_name, B, rank, world, dev):
    """Returns (engine, one_loop_resident, one_loop_e2e, h2d_bytes, d2h_bytes, l2_note)."""
    import torch
    import torch.distributed as dist
    from types import SimpleNamespace
    import b200mdm
    from b200mdm import parallel
    if cfg_name in ("c2", "c3"):
        steps = CONFIGS[cfg_name]["steps"]
        model, diffusion = b200mdm.create_model_and_diffusion(make_args(diffusion_steps=steps), SimpleNamespace(dataset=SimpleNamespace()))
        b200mdm.load_model_wo_clip(model, b200mdm.synthetic_state_dict(num_layers=L, seed=0))
        model = b200mdm.ClassifierFreeSampleModel(model.to(dev).eval())
        eng = model.model.engine()
        shape = (B, J, 1, T)
        inp = b200mdm.synthetic_inputs(B, nframes=T, steps=1, seed=10 + rank)
        text = torch.zeros(1, B * world, 512, device=dev)
        if rank == 0:
            text.copy_(torch.randn(1, B * world, 512, generator=torch.Generator().manual_seed(1234)))
        lengths, mask, scale = inp["lengths"].to(dev), inp["mask"].to(dev), inp["scale"].to(dev)
        text_h = torch.randn(1, B, 512).pin_memory()
        scale_h = torch.full((B,), SCALE).pin_memory()
        lengths_h = torch.full((B,), T, dtype=torch.int64).pin_memory()
        out_h = torch.empty(shape, dtype=torch.float32).pin_memory()
        h2d = int(text_h.numel() * 4 + scale_h.numel() * 4 + lengths_h.numel() * 8)
        if cfg_name == "c2":
            g = torch.Generator(device=dev).manual_seed(77 + rank)
            xT = torch.randn(*shape, device=dev, generator=g)
            tape = torch.randn(steps, *shape, device=dev, generator=g)          # 50 x 13.2 MB = 660 MB  (> 126 MB L2)

            def resident():
                if world > 1:
                    dist.broadcast(text, src=0)                                  # the one collective of the path
                y = dict(mask=mask, lengths=lengths, text_embed=text[:, rank * B:(rank + 1) * B], scale=scale)
                return diffusion.p_sample_loop(model, shape, noise=xT, clip_denoised=False, model_kwargs={"y": y}, noise_tape=tape)

            def e2e():
                te, sc, ln = (t.to(dev, non_blocking=True) for t in (text_h, scale_h, lengths_h))
                if world > 1:
                    dist.broadcast(te, src=0)
                y = dict(mask=mask, lengths=ln, text_embed=te, scale=sc)
                s = diffusion.p_sample_loop(model, shape, clip_denoised=False, model_kwargs={"y": y})
                out_h.copy_(s, non_blocking=True)
                return s
            note = "inputs larger than L2 (660 MB noise tape streamed per loop)"
        else:
            gmask = torch.ones(B * world, 1, 1, T, dtype=torch.bool, device=dev)
            glen = torch.full((B * world,), T, dtype=torch.int64, device=dev)
            gscale = torch.full((B * world,), SCALE, device=dev)
            gshape = (B * world, J, 1, T)

            def resident():
                y = dict(mask=gmask, lengths=glen, text_embed=text, scale=gscale)
                return parallel.sample_sharded(diffusion.p_sample_loop, model, gshape, {"y": y}, n_steps=steps, seed=5, device=dev,
                                               gather=False, clip_denoised=False)

            def e2e():
                te = text_h.to(dev, non_blocking=True)
                tg = te if world == 1 else te.repeat(1, world, 1)
                y = dict(mask=gmask, lengths=glen, text_embed=tg, scale=gscale)
                s = parallel.sample_sharded(diffusion.p_sample_loop, model, gshape, {"y": y}, n_steps=steps, seed=5, device=dev,
                                            gather=False, clip_denoised=False)
                out_h.copy_(s, non_blocking=True)
                return s
            note = "activations of one step (~0.5 GB) exceed L2; 1000 recurrent steps per loop; noise generated in-engine"
        return eng, resident, e2e, h2d, int(out_h.numel() * 4), note
    if cfg_name == "a2m":
        steps, Ta = 1000, 60
        args = make_args(dataset="humanact12", cond_mask_prob=0.0, diffusion_steps=steps)
        model, diffusion = b200mdm.create_model_and_diffusion(args, SimpleNamespace(dataset=SimpleNamespace(num_actions=12)))
        b200mdm.load_model_wo_clip(model, b200mdm.synthetic_state_dict(num_layers=L, seed=5, input_feats=150, cond_mode="action", num_actions=12))
        model = model.to(dev).eval()
        eng = model.engine()
        shape = (B, 25, 6, Ta)
        mask = torch.ones(B, 1, 1, Ta, dtype=torch.bool, device=dev)
        lengths = torch.full((B,), Ta, dtype=torch.int64, device=dev)
        action = (torch.arange(B) % 12).view(B, 1).to(dev)
        action_h = (torch.arange(B) % 12).view(B, 1).pin_memory()
        out_h = torch.empty(shape, dtype=torch.float32).pin_memory()

        def resident():
            y = dict(mask=mask, lengths=lengths, action=action)
            return diffusion.p_sample_loop(model, shape, clip_denoised=False, model_kwargs={"y": y}, noise_seed=5, sample_index_base=rank * B)

        def e2e():
            y = dict(mask=mask, lengths=lengths, action=action_h.to(dev, non_blocking=True))
            s = diffusion.p_sample_loop(model, shape, clip_denoised=False, model_kwargs={"y": y})      # torch generator, chunked draws
            out_h.copy_(s, non_blocking=True)
            return s
        return eng, resident, e2e, int(action_h.numel() * 8), int(out_h.numel() * 4), "1000 recurrent steps per loop; workspace ~150 MB"
    if cfg_name == "dip":
        steps, ctx, pred, Mt, need = 10, 20, 40, 16, 196
        args = make_args(arch="trans_dec", text_encoder_type="bert", context_len=ctx, pred_len=pred, diffusion_steps=steps)
        model, diffusion = b200mdm.create_model_and_diffusion(args, SimpleNamespace(dataset=SimpleNamespace()))
        b200mdm.load_model_wo_clip(model, b200mdm.synthetic_state_dict(arch="trans_dec", num_layers=L, cond_dim=768, seed=23))
        model = b200mdm.ClassifierFreeSampleModel(model.to(dev).eval())
        eng = model.model.engine()
        enc, tmask, prefix = b200mdm.synthetic_dip_inputs(B, Mt, ctx, seed=35)
        tmask[:] = False
        enc_d, tmask_d, prefix_d = enc.to(dev), tmask.to(dev), prefix.to(dev)
        enc_h, prefix_h = enc.pin_memory(), prefix.pin_memory()
        scale = torch.full((B,), 7.5, device=dev)
        mask = torch.ones(B, 1, 1, pred, dtype=torch.bool, device=dev)
        lengths = torch.full((B,), pred, dtype=torch.int64, device=dev)
        sampler = b200mdm.AutoRegressiveSampler(args, diffusion.p_sample_loop, required_frames=need)
        out_h = torch.empty((B, J, 1, need), dtype=torch.float32).pin_memory()

        def resident():
            y = dict(mask=mask, lengths=lengths, text_embed=(enc_d, tmask_d), prefix=prefix_d, scale=scale)
            return sampler.sample(model, (B, J, 1, need), clip_denoised=False, model_kwargs={"y": y})

        def e2e():
            y = dict(mask=mask, lengths=lengths, text_embed=(enc_h.to(dev, non_blocking=True), tmask_d),
                     prefix=prefix_h.to(dev, non_blocking=True), scale=scale)
            s = sampler.sample(model, (B, J, 1, need), clip_denoised=False, model_kwargs={"y": y})
            out_h.copy_(s, non_blocking=True)
            return s
        return eng, resident, e2e, int(enc_h.numel() * 4 + prefix_h.numel() * 4), int(out_h.numel() * 4), "5 chunks x 10 steps per loop; activations of one step ~0.3 GB"
    raise ValueError(cfg_name)


def kernel_roofline(dev, peaks, B):
    """The step's kernels timed alone at the c2 shapes (M = 128 sequences x 197 tokens) through the kernel-level C-ABI hooks:
    CUDA events on the launching stream, L2 flushed (256 MB memset) between timed launches."""
    import ctypes
    import torch
    from b200mdm import _lib
    lib = _lib.load()
    n_seq, S = 2 * B, T + 1
    M = n_seq * S
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def time_kernel(call):
        for _ in range(3):
            call()
        ts = []
        for _ in range(10):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); call(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sum(ts) / len(ts)

    def gemm_case(N, K, act):
        A = torch.randn(M, K, device=dev).half()
        Wt = (torch.randn(N, K, device=dev) / K ** 0.5).half()
        bias = torch.zeros(N, device=dev)
        O = torch.empty(M, N, device=dev, dtype=torch.float16)
        ms = time_kernel(lambda: _lib.check(lib.b200mdm_test_gemm_f16(A.data_ptr(), Wt.data_ptr(), bias.data_ptr(), O.data_ptr(), M, N, K, act, 513 if K <= 512 else 512, st)))   # 513: the W-resident pair GEMM the step dispatches at K <= 512
        return 2.0 * M * N * K, ms

    def ln_case(K):
        A = torch.randn(M, K, device=dev).half()
        Wt = (torch.randn(512, K, device=dev) / K ** 0.5).half()
        vec = [torch.zeros(512, device=dev), torch.ones(512, device=dev), torch.zeros(512, device=dev)]
        hres = torch.randn(M, 1024, device=dev).half()
        hres[:, 512:] *= 1e-3
        ms = time_kernel(lambda: _lib.check(lib.b200mdm_test_gemm_resid_ln(A.data_ptr(), Wt.data_ptr(), vec[0].data_ptr(), vec[1].data_ptr(), vec[2].data_ptr(), hres.data_ptr(), M, K, st)))
        return 2.0 * M * 512 * K, ms

    def qkv_attn_case():
        h = torch.randn(M, 1024, device=dev).half()
        Wt = (torch.randn(1536, 512, device=dev) / 512 ** 0.5).half()
        bias = torch.zeros(1536, device=dev)
        kv = torch.full((n_seq,), S, dtype=torch.int32, device=dev)
        O = torch.empty(M, 512, device=dev, dtype=torch.float16)
        ms = time_kernel(lambda: _lib.check(lib.b200mdm_test_qkv_attention(h.data_ptr(), 1024, Wt.data_ptr(), bias.data_ptr(), O.data_ptr(), kv.data_ptr(), n_seq, S, st)))
        # SURVEY section 8d accounting for the fused kernel: QKV projection 2*S*d*3d + attention core 4*S^2*d per sequence,
        # padding FLOPs (197 -> 256) NOT counted
        return n_seq * (2.0 * S * 512 * 1536 + 4.0 * S * S * 512), ms

    cases = [("qkv_attention_kernel (fused QKV projection + softmax attention, 128 sequences x 4 heads, S=197)", qkv_attn_case),
             ("gemm_resid_ln_cluster FFN-down + residual + LayerNorm M=%d N=512 K=1024" % M, lambda: ln_case(FF)),
             ("gemm_resid_ln_cluster out-proj + residual + LayerNorm K=512", lambda: ln_case(D)),
             ("gemm2w_f16_tcgen05<gelu> (W-resident pair GEMM) FFN-up N=1024 K=512", lambda: gemm_case(FF, D, 1))]
    rows = []
    for name, fn in cases:
        fl, ms = fn()
        tf = fl / (ms * 1e-3) / 1e12
        rows.append({"kernel": name, "achieved": round(tf, 1), "frac": round(tf / peaks["burst"], 4), "us": round(ms * 1e3, 1),
                     "flop": fl})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the sample the last timed step returned as DIR/sample.npy (float32)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs the GPU path (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        return run_reference_arm(a, rank, world)

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a B200"
    torch.cuda.set_device(local)
    torch.manual_seed(7 + rank)   # the paths that draw from torch's default generators (DiP, e2e) start from a fixed state
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    cfg = CONFIGS[a.config]
    B = cfg["per_gpu"]
    eng, one_loop_resident, one_loop_e2e, h2d, d2h, l2_note = build_workload(a.config, B, rank, world, dev)

    def timed(fn, iters):
        """Milliseconds of `iters` calls of fn between two CUDA events, and what the last call returned."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters - 1):
            fn()                  # results dropped at once, as in the warm-up: the allocator reuses one output block
        last = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), last

    def log(msg):
        if rank == 0:
            print("[bench %.1fs] %s" % (time.perf_counter() - t_start, msg), file=sys.stderr, flush=True)

    t_start = time.perf_counter()
    try:
        sampler = ClockSampler(local, enabled=(rank == 0))   # NVML / nvidia-smi opened before the warm-up, sampled in the region
    except Exception as e:   # noqa: BLE001  (a broken sampler must not take the measurement down with it)
        sampler = ClockSampler(local, enabled=False)
        sampler.errors.append("sampler: %r" % (e,))
    for _ in range(max(a.warmup, 3)):
        one_loop_resident()
    torch.cuda.synchronize()
    log("warm-up done")
    eng.launch_count(reset=True)
    if rank == 0:
        try:
            sampler.start()
        except Exception as e:   # noqa: BLE001
            sampler.errors.append("start: %r" % (e,))
    ms_total, last_sample = timed(one_loop_resident, a.steps)
    try:
        clocks = sampler.stop() if rank == 0 else None
    except Exception as e:   # noqa: BLE001
        clocks = {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling failed"], "samples": 0, "source": "none",
                  "errors": ["stop: %r" % (e,)]}
    launches = eng.launch_count(reset=True)
    log("resident loops timed: %.2f ms per loop" % (ms_total / a.steps))
    for _ in range(2):
        one_loop_e2e()
    ms_e2e, _ = timed(one_loop_e2e, a.steps)
    log("e2e loops timed: %.2f ms per loop" % (ms_e2e / a.steps))

    ms_step = ms_total / a.steps
    value = B * world / (ms_step * 1e-3)
    e2e_value = B * world / (ms_e2e / a.steps * 1e-3)
    peaks = measured_peaks()

    if rank == 0:
        path_tflops = value / world * cfg["flop_per_motion"] / 1e12            # per GPU
        if a.config == "c2":
            rows = kernel_roofline(dev, peaks, B)
            top = rows[0]
            roof = {"bound": "tensor", "kernel": top["kernel"], "achieved": top["achieved"], "peak": peaks["burst"], "unit": "TFLOP/s",
                    "frac": top["frac"], "us": top["us"], "flop_per_launch": top["flop"],
                    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel per launch: taken from the committed ncu
                    # capture, not re-measured per run (a profiler cannot run inside a timed bench)
                    "traffic": 17.5e6, "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full, "
                                                        "profiles/r02_f_ncu_qkv_attention_kernel.txt (14.5 MB + 3.0 MB: the operands are "
                                                        "L2-resident; algorithmic operand bytes 164 MB per launch come from the L2)",
                    "peak_source": peaks["source"] + " bf16 burst (cuBLAS 8192^3)",
                    "other_kernels": [{k: r[k] for k in ("kernel", "achieved", "frac", "us")} for r in rows[1:]]}
            log("kernel roofline timed: %s" % ", ".join("%.0f us" % r["us"] for r in rows))
        else:
            roof = {"bound": "tensor", "kernel": "whole sampling path of this config (per-kernel figures: --config c2)",
                    "achieved": round(path_tflops, 1), "peak": peaks["sustained"], "unit": "TFLOP/s",
                    "frac": round(path_tflops / peaks["sustained"], 4), "traffic": None,
                    "peak_source": peaks["source"] + " bf16 sustained (cuBLAS 8192^3 back to back)"}
        roof["path_achieved_tflops_per_gpu"] = round(path_tflops, 1)
        roof["path_frac_of_sustained"] = round(path_tflops / peaks["sustained"], 4)
        cpu = None
        if world == 1 and not a.no_cpu_baseline and a.config == "c2":
            m = cpu_arm(1, 0, 25.0)
            cpu = {"value": round(m["value"], 4), "unit": "motions/s", "cores": m["threads"], "kind": m["kind"], "sample": m["sample"]}
        line = {"metric": "motions/sec", "value": round(value, 2), "unit": "motions/s", "n_gpus": world, "steps": a.steps,
                "warmup": max(a.warmup, 3), "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "fp16 operands / fp32 accumulate (in/out projections hi-lo split)",
                "data": "synthetic",
                "config": {"workload": cfg["workload"], "name": a.config,
                           "global_batch": B * world, "parallelism": "batch-sharded x%d, 1 NCCL broadcast of text_embed per loop" % world,
                           "l2": l2_note, "cuda_graph": True},
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": round(e2e_value, 2), "unit": "motions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "roofline": roof, "cpu_baseline": cpu,
                "flop_per_motion": cfg["flop_per_motion"]}
        print(json.dumps(line), flush=True)
        if a.dump_outputs:
            import numpy as np
            os.makedirs(a.dump_outputs, exist_ok=True)
            path = os.path.join(a.dump_outputs, "sample.npy")
            np.save(path, last_sample.float().cpu().numpy())
            log("last timed sample %s -> %s" % (tuple(last_sample.shape), path))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

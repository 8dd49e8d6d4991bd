#!/usr/bin/env python
"""bench.py -- headline benchmark of the CMGAN hot path on B200 (contract in the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--workload train_gd|gen_only] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[2], metric: utterances/sec, 2 s @ 16 kHz): per rank, one step = the reference's whole
``train_step`` (train.py:176-205) on a batch of B = 16 synthetic 2 s clips:
  generator: RMS normalise -> STFT -> power compression -> TSCNet forward (train mode: dropout, BatchNorm batch statistics) ->
  un-compression -> iSTFT -> loss (RI + magnitude + time + metric-GAN term through the discriminator) -> backward through all of it ->
  (one NCCL all-reduce of the flat gradient buffer when N > 1) -> AdamW;
  discriminator: D(clean, est) and D(clean, clean) forward (train mode: spectral-norm power iterations, dropout), loss against a
  fixed synthetic PESQ target (the ``pesq`` package is host code and absent), backward, (all-reduce), AdamW.
All of it is one CUDA graph per step.  Prints ONE JSON line on rank 0.
"""
import argparse
import io
import json
import os
import subprocess
import sys
import threading
import time

# the benchmark leaves the tree it runs from untouched (it may be read-only): no __pycache__ for the modules it imports
sys.dont_write_bytecode = True

# stdout carries exactly one JSON line.  Libraries print there too (NCCL's version banner), so file descriptor 1 is pointed at
# stderr for the whole run and the JSON line is written to the saved original descriptor by emit().
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
sys.stdout.flush()
_STDOUT_FD = os.dup(1)
os.dup2(2, 1)


def emit(obj) -> None:
    os.write(_STDOUT_FD, (json.dumps(obj) + "\n").encode())


ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "utterances/sec (2 s @16 kHz) generator fwd+bwd"
UNIT = "utt/s"
CLIP = 32000
FWD_GFLOP_PER_UTT = 145.96            # SURVEY.md section 8(d): mm + bmm + conv, 2*MAC, 2 s clip
STEP_GFLOP_PER_UTT = 3 * FWD_GFLOP_PER_UTT
TSCB_FWD_GFLOP_PER_UTT = 4 * 19.58    # SURVEY.md section 8(d): four two-stage conformer blocks
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def synth_batch(B, seed, device=None, pin=False):
    import torch
    g = torch.Generator().manual_seed(seed)
    clean = 0.05 * torch.randn(B, CLIP, generator=g)
    noisy = clean + 0.05 * torch.randn(B, CLIP, generator=g)
    if pin:
        return clean.pin_memory(), noisy.pin_memory()
    if device is not None:
        return clean.to(device), noisy.to(device)
    return clean, noisy


def workload_name(B, kind):
    if kind == "gen_only":
        return (f"generator training step fwd+bwd+AdamW (train mode: dropout + BatchNorm batch stats), "
                f"stft->compress->TSCNet->uncompress->istft->loss->backward->update, batch {B} x 2 s @16 kHz per GPU, fp32 storage")
    return (f"configs[2]: train.py train_step = generator fwd+bwd+AdamW (train mode, loss incl. the metric-GAN term through D) + discriminator step "
            f"(2 more D forwards, 2 D backwards, AdamW; fixed synthetic PESQ target 0.5), batch {B} x 2 s @16 kHz per GPU, "
            f"tf32 tensor-core operands / fp32 storage + accumulation")


# ------------------------------------------------------------------------------------------------ reference arms
class RefModules:
    """The reference's own generator / discriminator (unmodified files staged under baseline/_ref by tools/stage_reference.py) driven
    by the train.py:72-151 glue restated with the torch >= 2 complex STFT API (SURVEY.md section 8c); when the staged files are
    absent, the oracle port (oracle/cmgan_oracle.py) stands in.  Used by ``--impl reference`` (CPU) and ``gpu_eager_reference``."""

    def __init__(self, device, with_disc=True):
        import torch
        from oracle import cmgan_oracle as O
        self.torch, self.O, self.dev = torch, O, device
        w = O.load_weights_npz(os.path.join(ROOT, "tests", "golden", "weights_g.npz"))
        self.kind = "port"
        self.model = self.disc = None
        if os.path.isdir(os.path.join(REF_DIR, "models")):
            try:
                import types
                if "pesq" not in sys.modules:           # discriminator.py imports pesq at module level; the bench never calls it
                    stub = types.ModuleType("pesq")
                    stub.pesq = lambda *a, **k: 0.0
                    sys.modules["pesq"] = stub
                sys.path.insert(0, REF_DIR)
                from models.generator import TSCNet
                import utils as ref_utils
                self.ref_utils = ref_utils
                self.model = TSCNet(num_channel=64, num_features=201)
                self.model.load_state_dict(w, strict=True)
                self.model = self.model.to(device).train()
                if with_disc:
                    from models.discriminator import Discriminator
                    torch.manual_seed(7)
                    self.disc = Discriminator(ndf=16).to(device).train()
                self.kind = "reference"
            except Exception as e:       # noqa: BLE001 -- report and fall back to the port
                print(f"[bench] staged reference modules unusable ({type(e).__name__}: {e}); using the oracle port", file=sys.stderr)
                self.model = self.disc = None
                self.kind = "port"
        if self.model is None:
            self.sd = {k: (v.clone().to(device).requires_grad_(True) if v.is_floating_point() and "running_" not in k else v.to(device)) for k, v in w.items()}
            self.params = [v for v in self.sd.values() if v.is_floating_point() and v.requires_grad]
        else:
            self.params = list(self.model.parameters())

    def _stft(self, x):
        t = self.torch
        return t.view_as_real(t.stft(x, 400, 100, window=t.hamming_window(400, device=x.device), onesided=True, return_complex=True))

    def _istft(self, spec):
        t = self.torch
        return t.istft(t.view_as_complex(spec.contiguous()), 400, 100, window=t.hamming_window(400, device=spec.device), onesided=True)

    def gen_fwd(self, clean, noisy):
        t, F = self.torch, self.torch.nn.functional
        if self.model is None:
            go = self.O.forward_generator_step(clean, noisy, self.sd, training=True)
        else:
            c = t.sqrt(noisy.size(-1) / t.sum(noisy ** 2.0, dim=-1))
            n2, c2 = (noisy.t() * c).t(), (clean.t() * c).t()
            nspec = self.ref_utils.power_compress(self._stft(n2)).permute(0, 1, 3, 2)
            cspec = self.ref_utils.power_compress(self._stft(c2))
            er, ei = self.model(nspec)
            er, ei = er.permute(0, 1, 3, 2), ei.permute(0, 1, 3, 2)
            go = dict(est_real=er, est_imag=ei, est_mag=t.sqrt(er ** 2 + ei ** 2), clean_real=cspec[:, 0:1], clean_imag=cspec[:, 1:2],
                      clean_mag=t.sqrt(cspec[:, 0:1] ** 2 + cspec[:, 1:2] ** 2),
                      est_audio=self._istft(self.ref_utils.power_uncompress(er, ei).squeeze(1)))
        loss = 0.1 * (F.mse_loss(go["est_real"], go["clean_real"]) + F.mse_loss(go["est_imag"], go["clean_imag"])) \
            + 0.9 * F.mse_loss(go["est_mag"], go["clean_mag"]) + 0.2 * t.mean(t.abs(go["est_audio"] - clean))
        return go, loss

    def step(self, clean, noisy, with_disc):
        """generator forward + backward (+ the GAN term and the discriminator's loss/backward when the reference D is available)"""
        t, F = self.torch, self.torch.nn.functional
        for p in self.params:
            p.grad = None
        go, loss = self.gen_fwd(clean, noisy)
        B = clean.shape[0]
        if with_disc and self.disc is not None:
            fake = self.disc(go["clean_mag"], go["est_mag"])
            loss = loss + 0.05 * F.mse_loss(fake.flatten(), t.ones(B, device=clean.device))
        loss.backward()
        if with_disc and self.disc is not None:
            for p in self.disc.parameters():
                p.grad = None
            d_enh = self.disc(go["clean_mag"], go["est_mag"].detach())
            d_max = self.disc(go["clean_mag"], go["clean_mag"])
            dl = F.mse_loss(d_max.flatten(), t.ones(B, device=clean.device)) + F.mse_loss(d_enh.flatten(), t.full((B,), 0.5, device=clean.device))
            dl.backward()
        return loss


def host_threads():
    """threads for the CPU arm: the cores this process may run on, capped at 32 (the reference's ~700 small ATen ops per
    forward stop scaling well before that; 128 threads measured 17x slower than 8 on the GPU box's host)"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, 32))


def time_cpu(n_steps, warm, with_disc=True):
    import torch
    torch.set_num_threads(host_threads())
    ref = RefModules(torch.device("cpu"), with_disc)
    clean, noisy = synth_batch(1, 123)
    for _ in range(warm):
        ref.step(clean, noisy, with_disc)
    t0 = time.perf_counter()
    for _ in range(n_steps):
        ref.step(clean, noisy, with_disc)
    return (time.perf_counter() - t0) / n_steps, ref.kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_threads()
    with_disc = args.workload == "train_gd"
    dt, kind = time_cpu(args.steps, args.warmup, with_disc)
    v = 1.0 / dt
    sample = ("1 utterance (B=1 x 2 s) per step of the workload: " + ("the reference's own TSCNet / Discriminator modules (baseline/_ref)" if kind == "reference"
              else "oracle CPU port of the reference") + ", generator forward+backward" + (" + discriminator step" if with_disc and kind == "reference" else "")
              + ", fp32, torch CPU threads = cores")
    emit(({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.batch, args.workload), "reference_sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ our arm (GPU)
def run_ours(args):
    import torch
    import torch.distributed as dist
    import cmgan_b200
    from cmgan_b200 import ops as _ops
    _ops.set_precision(args.precision)
    from cmgan_b200 import ops, training
    from cmgan_b200.trainer import FusedTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    if args.global_batch:
        assert args.global_batch % world == 0, "--global-batch must divide by the number of ranks"
        args.batch = args.global_batch // world
    B = args.batch
    gd = args.workload == "train_gd"
    torch.manual_seed(0)
    model = cmgan_b200.TSCNet(64, 201).to(dev).train()
    disc = cmgan_b200.Discriminator(16).to(dev).train() if gd else None
    trainer = FusedTrainer(model, disc)          # flat parameter/gradient buffers; rank-0 parameters win (train.py:68)
    start_state = None
    if args.dump_outputs:                        # the seeded state before any step: the dumped step starts from it
        start_state = io.BytesIO()
        trainer.save_checkpoint(start_state, full=True)
    clean, noisy = synth_batch(B, 1000 + rank, device=dev)
    hclean, hnoisy = synth_batch(B, 1000 + rank, pin=True)
    pesq_t = torch.full((B,), 0.5, device=dev)
    hpesq = torch.full((B,), 0.5).pin_memory()

    def eager_step(c, n):          # every kernel launched from Python (gradient all-reduce when N > 1, AdamW updates)
        lg = trainer.generator_step(c, n)
        return (lg, trainer.discriminator_step(pesq_t)) if gd else (lg, None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = [0.0]

    def timed(fn, K):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        for _ in range(K):
            fn()
        host_ms[0] = (time.perf_counter() - t0) * 1e3 / K       # host time to enqueue one step
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    for _ in range(2):
        eager_step(clean, noisy)
    K_eager = min(args.steps, 3)
    ms_eager = timed(lambda: eager_step(clean, noisy), K_eager) / K_eager
    eager_host_ms = host_ms[0]

    # ---- the whole step as one CUDA graph.  N > 1: the NCCL all-reduces (generator: two segments, the first overlapped with the encoder's
    # backward; discriminator: one) and both AdamW updates are captured too; CMGAN_GRAPH_NCCL=0 keeps them eager after a backward-only graph.
    graph_nccl = world == 1 or os.environ.get("CMGAN_GRAPH_NCCL", "1") != "0"
    l0 = ops.LAUNCHES
    if gd:
        if graph_nccl:
            trainer.capture_train_step(clean, noisy)
        else:
            raise SystemExit("the G+D workload needs the collectives inside the graph (CMGAN_GRAPH_NCCL=1)")
    else:
        trainer.capture_generator_step(clean, noisy, update=graph_nccl, allreduce=graph_nccl)
    launches_per_step = trainer.graph_launches

    def gstep(c, n, p=None):
        if gd:
            return trainer.replay_train_step(c, n, p)
        loss = trainer.replay_generator_step(c, n)
        if not graph_nccl:
            from cmgan_b200 import parallel
            parallel.allreduce_mean_(trainer.gg)
            trainer.opt_g.step()
            if trainer.pack is not None:
                trainer.pack.refresh()
        return loss, None

    for _ in range(max(args.warmup, 3)):
        gstep(clean, noisy, pesq_t)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(lambda: gstep(clean, noisy, pesq_t), args.steps)
    if args.dump_outputs:
        trained_state = io.BytesIO()
        trainer.save_checkpoint(trained_state, full=True)
        start_state.seek(0)
        trainer.load_checkpoint(start_state)
        gstep(clean, noisy, pesq_t)
        barrier()
        if rank == 0:
            dump_outputs(args.dump_outputs, trainer, gd)
        trained_state.seek(0)
        trainer.load_checkpoint(trained_state)
    losses = gstep(clean, noisy, pesq_t)
    loss_after = float(losses[0].item())
    dloss_after = float(losses[1].item()) if gd else None
    assert loss_after == loss_after and abs(loss_after) < 1e30, f"training step diverged: loss {loss_after}"
    launches = launches_per_step * args.steps
    host_enqueue_ms = host_ms[0]
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms * 1e-3)

    # ---- end to end: pinned host buffers in (waveforms + PESQ targets), loss scalars out, every step
    host_loss = torch.empty(2).pin_memory()

    def e2e_step():
        lg, ld = gstep(hclean, hnoisy, hpesq)             # H2D copies of the pinned batch into the graph's input buffers
        host_loss[0:1].copy_(lg.detach().reshape(1), non_blocking=True)
        if ld is not None:
            host_loss[1:2].copy_(ld.detach().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()       # the caller reads the losses every step (train.py:205)
    e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    e2e_value = world * B * args.steps / (ms_e2e * 1e-3)
    h2d = 2 * B * CLIP * 4 + (B * 4 if gd else 0)
    d2h = 8 if gd else 4

    out = None
    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": workload_name(B, args.workload), "global_batch": B * world, "clip_samples": CLIP, "parallelism": f"dp{world}",
                       "l2": "per-step working set (activations saved for backward, several GB) >> 126 MB L2; no explicit flush",
                       "weights": "torch.manual_seed(0) default init, updated by AdamW every step (lr 5e-4 / 1e-3)", "loss_after": loss_after,
                       "disc_loss_after": dloss_after,
                       "launch": "one CUDA graph per step (cmgan_b200.trainer.FusedTrainer): forward, losses, backward, "
                                 + ("NCCL gradient all-reduces, " if world > 1 and graph_nccl else "") + "AdamW"
                                 + ("" if graph_nccl else " -- all-reduce + AdamW eager after the graph")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "gpu_launches_per_step": launches_per_step, "host_enqueue_ms_per_step": host_enqueue_ms,
            "eager": {"value": world * B / (ms_eager * 1e-3), "unit": UNIT, "ms_per_step": ms_eager,
                      "host_enqueue_ms_per_step": eager_host_ms, "note": "same step launched kernel by kernel from Python (no CUDA graph)"},
            "clocks": clocks,
            "model_tflops": value * STEP_GFLOP_PER_UTT / 1e3,
        }
    if world == 1 and not args.no_extras:
        extras(args, out, trainer, model, dev, ms / args.steps)
    if rank == 0:
        emit(out)
    if world > 1:
        # the captured graphs hold NCCL kernels: tearing the process group down underneath them can block, so leave together and at once
        dist.barrier()
        torch.cuda.synchronize()
        sys.stderr.flush()
        os._exit(0)


DUMP_AUDIO_BYTES = 32 << 20


def dump_outputs(path, trainer, gd):
    """write what one replay of the timed step computed from the seeded batch and the seeded start state, as float32 .npy files:
    the losses, the enhanced waveforms (the first rows only, when the batch's exceed 32 MB) and the gradients.

    The step starts from the state before any training step because the timed steps' weights carry every earlier step's rounding:
    the gradient, statistics and loss reductions accumulate with float atomics in whatever order they land, and AdamW turns a
    rounding-level gradient (conv biases in front of an InstanceNorm, mathematically zero) into a +-lr move.  For the same reason
    the updated parameters are not written: the gradients are what the step computed from them."""
    import numpy as np
    audio = trainer.last["est_audio"]
    arrays = {"generator_loss": trainer.static_losses[0] if gd else trainer.static_loss,
              "est_audio": audio[:max(1, DUMP_AUDIO_BYTES // (audio.shape[1] * audio.element_size()))],
              "generator_grads": trainer.gg}
    if gd:
        arrays.update(discriminator_loss=trainer.static_losses[1], discriminator_grads=trainer.gd)
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def extras(args, out, trainer, model, dev, step_ms):
    """single-GPU explanatory numbers: forward-only (configs[1]), the TSCB stack's roofline, the GEMM family's roofline, the same-box
    GPU-eager reference, the CPU baseline"""
    import torch
    from cmgan_b200 import conformer_block as G, ops, training
    peaks, psrc = _peaks()
    hbm_peak = peaks.get("hbm_gbs", 6500.0)
    tf32_peak = peaks.get("bf16_tflops_sustained", 1400.0) / 2.0      # dense tf32 = half the bf16 rate on the same tensor pipe

    def time_graph(fn, reps):
        """capture ``fn`` (after two warm-up passes) and time ``reps`` replays with CUDA events"""
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        for _ in range(2):
            g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    # ---- forward only (configs[1]: eval forward, batch 4)
    Bf = 4
    clean4, noisy4 = synth_batch(Bf, 77, device=dev)
    model.eval()
    with torch.no_grad():
        ms_f = time_graph(lambda: training.forward_generator_step(model, clean4, noisy4)["est_audio"], args.steps)
    model.train()
    out["forward_only"] = {"value": Bf / (ms_f * 1e-3), "unit": UNIT, "ms_per_step": ms_f, "workload": f"configs[1]: eval forward, batch {Bf} x 2 s"}

    # ---- the TSCB stack alone (the kernel group the north-star puts a number on): 8 conformer blocks forward + backward, train mode,
    # on the bench batch's (B, 321, 101, 64) activation, as one graph; algorithmic flops = SURVEY 8(d) 4 x 19.58 GFLOP forward per utterance, x3
    B = args.batch
    T, F2 = CLIP // 100 + 1, 101
    M = B * T * F2
    P = model._tensor_dict()
    h0 = torch.randn(M, 64, device=dev)
    dy0 = torch.randn(M, 64, device=dev)
    grads = trainer.model._flat_views
    cache = trainer.pack

    def tscb_stack():
        ops.PACK_CACHE = cache
        try:
            sums = G._Sums(8 * 2 * 128 * 2 * 2 + 64, dev)
            saves, h = [], h0
            for i in range(1, 5):
                for axis, name in ((0, "time_conformer"), (1, "freq_conformer")):
                    sv = {}
                    h = G.conformer_fwd(h, P, f"TSCB_{i}.{name}", B, T, F2, axis, True, 1, (i - 1) * 2 + axis, sums, sv)
                    saves.append(sv)
            d = dy0
            sums2 = G._Sums(8 * 2 * 128 * 2 * 2 + 64, dev)
            for sv in reversed(saves):
                d = G.conformer_bwd(d, sv, P, grads, B, T, F2, sums2)
            ops.join_wgrad()
            return d
        finally:
            ops.PACK_CACHE = None
    bufs = [b.clone() for b in model.buffers()]
    ms_tscb = time_graph(tscb_stack, max(3, args.steps // 2))
    for b, v in zip(model.buffers(), bufs):
        b.copy_(v)
    tscb_flop = 3 * TSCB_FWD_GFLOP_PER_UTT * B * 1e9
    out["tscb"] = {"what": "4 x TSCB (8 conformer blocks) forward + backward, train mode, one CUDA graph, CUDA events", "batch": B, "ms": ms_tscb,
                   "share_of_step": ms_tscb / step_ms, "algorithmic_gflop": tscb_flop / 1e9, "achieved_tflops": tscb_flop / (ms_tscb * 1e-3) / 1e12,
                   "peak_tflops": tf32_peak, "frac_of_tensor_roofline": tscb_flop / (ms_tscb * 1e-3) / 1e12 / tf32_peak,
                   "peak_source": f"{psrc}: bf16_tflops_sustained / 2 (tf32 runs at half the bf16 rate)", "target": 0.70}

    # ---- dominant kernel family: every GEMM launch of one generator step is recorded (arguments + operands kept alive) and the whole list is
    # replayed back to back between two CUDA events, so the durations carry no host gaps (an eager step is host-bound)
    import ctypes as _ct
    from cmgan_b200._lib import lib as _lib
    clean, noisy = synth_batch(B, 1000, device=dev)
    ops.PROBE = []
    trainer.generator_step(clean, noisy, update=False)
    torch.cuda.synchronize()
    probe, ops.PROBE = ops.PROBE, None

    def replay(entries, reps=3):
        L, st = _lib(), ops.stream()

        def once():
            for p in entries:
                L.call(p[0], _ct.byref(p[5]), st)
        once()
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(reps):
            once()
        r1.record()
        torch.cuda.synchronize()
        return r0.elapsed_time(r1) / reps * 1e-3

    rows = [p for p in probe if p[0] == "cmgan_gemm_rows_f32"]
    wgs = [p for p in probe if p[0] == "cmgan_gemm_wgrad_f32"]
    t_rows, t_wg = replay(rows), replay(wgs)
    if os.environ.get("CMGAN_PROBE_DUMP"):      # per-shape replay timings for analysis (not part of the JSON line)
        shapes = {}
        for p in probe:
            shapes.setdefault((p[0], p[1], p[2], p[3], p[4]), []).append(p)
        dump = [[k[0], k[1], k[2], k[3], replay(v, 2) / len(v) * 1e6, k[4], len(v)] for k, v in shapes.items()]
        with open(os.environ["CMGAN_PROBE_DUMP"], "w") as fh:
            json.dump(dump, fh)
    f_rows = sum(2.0 * p[1] * p[2] * p[3] for p in rows)
    f_wg = sum(2.0 * p[1] * p[2] * p[3] for p in wgs)
    b_rows = float(sum(p[4] for p in rows))
    b_wg = float(sum(p[4] for p in wgs))
    del probe
    step_s = step_ms * 1e-3
    achieved = b_rows / t_rows / 1e9 if t_rows > 0 else 0.0
    # The row-parallel GEMM family (tcgen05 tf32): K = 64 .. 256 against N = 64 .. 256 is 13 - 64 flop/byte, far below the ~110 flop/byte
    # balance point of tf32 tensor cores vs HBM, so the family is HBM-bound and is reported as such (algorithmic bytes of each launch).
    out["gemm_family"] = {"bound": "hbm", "kernel": "gemm_rows_tc_kernel (every dense contraction of the generator step outside the fused FFN: linear, "
                                                    "pointwise, dilated/strided conv)",
                          "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                          "how": "sum of algorithmic bytes (A once, C, epilogue operands, weights) over every launch of one generator step / CUDA-event time "
                                 "of those launches replayed back to back",
                          "launches_per_step": len(rows), "share_of_step": t_rows / step_s, "algorithmic_gb_per_step": b_rows / 1e9,
                          "tensor": {"achieved_tflops": f_rows / t_rows / 1e12 if t_rows > 0 else 0.0, "peak_tflops": tf32_peak,
                                     "algorithmic_gflop_per_step": f_rows / 1e9},
                          "wgrad": {"achieved": (b_wg / t_wg / 1e9) if t_wg > 0 else 0.0, "unit": "GB/s",
                                    "frac": (b_wg / t_wg / 1e9 / hbm_peak) if t_wg > 0 else 0.0, "share_of_step": t_wg / step_s,
                                    "achieved_tflops": (f_wg / t_wg / 1e12) if t_wg > 0 else 0.0}}

    # ---- the dominant single kernel of the step (profiles/r2_launch_summary.md: 17.6 % of the kernel time, 8 launches): attention backward
    # dq / dE (attn_bwd_dq_mma_kernel).  Timed alone here, on the bench batch's shapes, both sequence axes (4 launches each per step).
    # Algorithmic flops (SURVEY 8d counts attention as L^2 d MACs per contraction, rel-pos term included): this kernel owns three of the six
    # backward contractions -- dQ = dS K, dQ += dR E, dE = dR^T Q -- = 3 x 2 x 16 = 96 flop per (query, key) pair and head.  It also recomputes
    # S, R and dP (not counted).  Bound: tensor pipe (compulsory traffic ~0.9 GB per launch = 0.14 ms at HBM speed vs 0.09 ms of tf32 math).
    H_, D_ = 4, 16
    Ew = torch.randn(1025, D_, device=dev) * 0.1
    dq_us, dq_flop = [], []
    for axis, L, nseq in ((0, T, B * F2), (1, F2, B * T)):
        qkv = torch.randn(M, 3 * 64, device=dev) * 0.5
        dctx = torch.randn(M, 64, device=dev) * 0.1
        ctx, lse = torch.empty(M, 64, device=dev), torch.empty(M, H_, device=dev)
        delta, dqkv, dE = torch.empty(M, H_, device=dev), torch.empty(M, 3 * 64, device=dev), torch.zeros(1025, D_, device=dev)
        ops.call("cmgan_attention_fwd_tf32", qkv, Ew, B, T, F2, axis, ctx, lse)
        ops.call("cmgan_attention_bwd_tf32_parts", qkv, Ew, ctx, dctx, lse, B, T, F2, axis, delta, dqkv, dE, 1)       # delta only
        nws = _lib().cdll.cmgan_attention_bwd_ws_floats(B, T, F2, axis) if ops.ATTN_BWD_WS else 0
        wsb = torch.empty(max(nws, 1), device=dev) if nws else None
        for _ in range(2):
            ops.call("cmgan_attention_bwd_tf32_ws", qkv, Ew, ctx, dctx, lse, B, T, F2, axis, delta, dqkv, dE, 2, wsb, nws)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(4):
            ops.call("cmgan_attention_bwd_tf32_ws", qkv, Ew, ctx, dctx, lse, B, T, F2, axis, delta, dqkv, dE, 2, wsb, nws)   # dq + dE kernel only, as the step runs it
        a1.record()
        torch.cuda.synchronize()
        dq_us.append(a0.elapsed_time(a1) / 4 * 1e3)
        dq_flop.append(96.0 * nseq * H_ * L * L)
        del qkv, dctx, ctx, lse, delta, dqkv, dE
    dq_t = sum(dq_us) / len(dq_us) * 1e-6                    # average launch duration over the step's 4 + 4 launches
    dq_f = sum(dq_flop) / len(dq_flop)
    traffic, traffic_note = None, "no ncu capture committed for this batch size"
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tp):           # dram read + write per launch of the same kernel at the same batch, from the committed ncu launch list
        tj = json.load(open(tp))
        if tj.get("batch") == B:
            traffic, traffic_note = tj.get("traffic_bytes_per_launch"), tj.get("note", "")
    tf32_burst = peaks.get("bf16_tflops", 1590.0) / 2.0        # kernel timed alone: the burst figure
    out["roofline"] = {"bound": "tensor", "kernel": "attn_bwd_dq_mma_kernel (attention backward: dQ, dE; mma.sync tf32)", "achieved": dq_f / dq_t / 1e12,
                       "peak": tf32_burst, "unit": "TFLOP/s", "frac": dq_f / dq_t / 1e12 / tf32_burst,
                       "peak_source": f"{psrc}: bf16_tflops (burst, kernel timed alone) / 2 (tf32 runs at half the bf16 rate)",
                       "how": "96 algorithmic flop per (query, key) pair and head x pairs of one launch / CUDA-event duration of that launch, averaged over "
                              "the time-axis and frequency-axis shapes of the bench batch (4 launches each per step); the kernel timed alone, 4 repeats",
                       "launch_us": {"time_axis": dq_us[0], "freq_axis": dq_us[1]}, "launches_per_step": 8,
                       "share_of_step": 4 * (dq_us[0] + dq_us[1]) * 1e-6 / step_s, "algorithmic_gflop_per_launch": dq_f / 1e9,
                       "traffic": traffic, "traffic_note": traffic_note}

    # ---- the same-box competitor (SURVEY 8d / BASELINE.md 4.5): the reference's modules in PyTorch eager on this B200, generator forward +
    # backward, B = 4, fp32 and with TF32 allowed
    if not args.no_gpu_eager:
        try:
            ref = RefModules(dev, with_disc=False)
            cl, nz = synth_batch(4, 55, device=dev)
            res = {}
            for name, flag in (("fp32", False), ("tf32", True)):
                torch.backends.cuda.matmul.allow_tf32 = flag
                torch.backends.cudnn.allow_tf32 = flag
                for _ in range(2):
                    ref.step(cl, nz, False)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(3):
                    ref.step(cl, nz, False)
                e1.record()
                torch.cuda.synchronize()
                res[name] = {"value": 4 * 3 / (e0.elapsed_time(e1) * 1e-3), "unit": UNIT, "ms_per_step": e0.elapsed_time(e1) / 3}
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = True
            out["gpu_eager_reference"] = {"kind": ref.kind, "workload": "generator forward + backward (train mode), batch 4 x 2 s, PyTorch eager on this GPU",
                                          **res}
            del ref
            torch.cuda.empty_cache()
        except Exception as e:      # noqa: BLE001
            out["gpu_eager_reference"] = {"unavailable": f"{type(e).__name__}: {e}"}

    if not args.no_cpu:
        cores = host_threads()
        dt, kind = time_cpu(2, 1, with_disc=args.workload == "train_gd")
        out["cpu_baseline"] = {"value": 1.0 / dt, "unit": UNIT, "cores": cores, "kind": kind,
                               "sample": "2 timed steps (after 1 warm-up) of B=1 x 2 s of the same workload through "
                                         + ("the reference's own modules (baseline/_ref)" if kind == "reference" else "the oracle CPU port") + ", fp32, all host threads"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="utterances per GPU (configs[2]: 16; configs[3] = 8 per GPU on 8 GPUs)")
    ap.add_argument("--global-batch", type=int, default=0, help="strong scaling: total utterances split over the ranks (overrides --batch)")
    ap.add_argument("--workload", default="train_gd", choices=["train_gd", "gen_only"],
                    help="train_gd: generator + discriminator train step (configs[2], default); gen_only: generator step without the GAN term")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the GPU-eager reference leg")
    ap.add_argument("--no-extras", action="store_true", help="headline only (no forward-only / roofline / baseline legs)")
    ap.add_argument("--precision", default="tf32", choices=["tf32", "fp32"], help="dense contractions: tcgen05 tf32 (default) or exact fp32 FFMA")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, replay the timed step once from the seeded start state and write what it computed to "
                         "DIR/<name>.npy (float32; the same inputs every run, so two builds compare output for output)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

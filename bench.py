#!/usr/bin/env python
"""bench.py — headline benchmarks of the B200 Tacotron-2 hot paths (BASELINE.json metric:
"WaveNet train audio-samples/sec/GPU; Tacotron mel-frames/sec; 1/2/4/8 B200").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME]      # our arm (CUDA, one process per GPU)
  python bench.py [...] --dump-outputs DIR                                   # + one timed step from the seeded state, as DIR/*.npy
  python bench.py --impl reference [...]                                     # CPU arm: the oracle restatement of the reference
                                                                             # graph on the host cores (TF1 cannot be installed
                                                                             # here; DESIGN.md §2)
Workloads (SURVEY.md §8d):
  wavenet_ce       (default; BASELINE.json configs[1], "Cfg-2") 24 layers / 4 stacks, R256/G512/S256, mu-law-256 one-hot input and
                   softmax-CE, local conditioning through the learnable upsampling net, dropout 0.05, 2 x 7680 samples per GPU
  wavenet_mol      (configs[3], "Cfg-4") same stack, raw input + MoL-10 NLL, 8 x 16128 samples per GPU
  wavenet_default  the reference's DEFAULT widths (hparams.py:203-207: R128/G256/S128, 20 layers / 2 stacks) with mu-law-256 CE,
                   8 x 16128 samples per GPU — the HBM-bound shape of SURVEY §8d (north-star ">= 70 % HBM roofline" line)
  tacotron         (configs[2], "Cfg-3") encoder + decoder + postnet training step, r = 1, B = 32 per GPU, T_in 160, T_out 800
One step = forward + loss + backward + gradient all-reduce (N > 1) + clip + Adam (+ EMA) + re-pack of the bf16 operand copies.
Prints ONE JSON line (rank 0)."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


# ---------------------------------------------------------------------------------------------------------------------
# workload definitions
# ---------------------------------------------------------------------------------------------------------------------
def workload_hparams(name="wavenet_ce"):
    from hparams import hparams
    hp = hparams.copy()
    if name == "wavenet_ce":
        hp.parse("input_type=mulaw-quantize,quantize_channels=256,out_channels=256,layers=24,stacks=4,"
                 "residual_channels=256,gate_channels=512,skip_out_channels=256,upsample_scales=[16,16],hop_size=256,"
                 "wavenet_dropout=0.05")
    elif name == "wavenet_mol":
        hp.parse("input_type=raw,quantize_channels=65536,out_channels=30,layers=24,stacks=4,residual_channels=256,"
                 "gate_channels=512,skip_out_channels=256,upsample_scales=[16,16],hop_size=256,wavenet_dropout=0.05")
    elif name == "wavenet_default":
        hp.parse("input_type=mulaw-quantize,quantize_channels=256,out_channels=256,layers=20,stacks=2,"
                 "residual_channels=128,gate_channels=256,skip_out_channels=128,upsample_scales=[16,16],hop_size=256,"
                 "wavenet_dropout=0.05")
    elif name == "tacotron":
        hp.parse("predict_linear=False")
    else:
        raise ValueError(name)
    return hp


B_PER_GPU, T_STEP = 2, 7680           # Cfg-2 (kept as module constants: tools/ import them)
WN_SHAPES = {"wavenet_ce": (2, 7680), "wavenet_mol": (8, 16128), "wavenet_default": (8, 16128)}
TACO_SHAPE = (32, 160, 800)


def synth_batch(hp, B, T, seed, quantize):
    """Synthetic LJSpeech-shaped batch: AR(2) 'speech-like' noise -> mu-law indices (or raw floats); mels ~ U[0,1].
    quantize: float32 [B,T] -> int indices (the CUDA mu-law kernel on the GPU arm, the oracle on the CPU arm); None = raw input."""
    import numpy as np
    from scipy.signal import lfilter
    rng = np.random.default_rng(seed)
    e = rng.standard_normal((B, T + 64))
    w = lfilter([1.0], [1.0, -1.6, 0.8], e, axis=1)[:, 64:]
    w = (w / np.abs(w).max() * 0.6).astype(np.float32)
    x = w if quantize is None else quantize(w).astype(np.int32)
    c = rng.random((B, hp.cin_channels, T // 256), dtype=np.float32)
    lengths = np.full((B,), T, dtype=np.int32)
    return x, c, lengths


def taco_batch(hp, B, T_in, T_out, seed):
    """SURVEY §8d Cfg-3: ids U{2..65} ending in EOS, sorted input lengths U{60..160}, targets clip(N(-1,1.5),-4,4) padded with -4
    (tacotron/feeder.py:64-65), stop targets 0 then 1-padding (:69,240-252)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    inputs = rng.integers(2, 66, (B, T_in)).astype(np.int32)
    lens = np.sort(rng.integers(60, T_in + 1, (B,)))[::-1].astype(np.int32).copy()
    lens[0] = T_in
    tl = rng.integers(T_out // 2, T_out + 1, (B,))
    mel = np.clip(rng.normal(-1.0, 1.5, (B, T_out, hp.num_mels)), -4, 4).astype(np.float32)
    stop = np.zeros((B, T_out), dtype=np.float32)
    for b in range(B):
        inputs[b, lens[b] - 1] = 1
        inputs[b, lens[b]:] = 0
        mel[b, tl[b]:] = -4.0
        stop[b, tl[b] - 1:] = 1.0
    return inputs, lens, mel, stop


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm, reasons, mx = [], set(), 0
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _traffic(key):
    """measured DRAM bytes (read + write) from the committed ncu pass (profiles/r02_dram_traffic.json), or None"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_dram_traffic.json"))).get(key)
    except Exception:
        return None


def _pick_threads(fn):
    """fastest torch intra-op thread count for this graph on this host (oversubscribing a 128-core box is ~5x slower)"""
    import torch
    ncores = os.cpu_count() or 1
    best = (1, 1e30)
    for nt in sorted({ncores, min(ncores, 64), min(ncores, 32), min(ncores, 16)}):
        torch.set_num_threads(nt)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (nt, dt)
    torch.set_num_threads(best[0])
    return best[0], ncores


# ---------------------------------------------------------------------------------------------------------------------
class WaveNetWorkload(object):
    metric, unit = "wavenet_train_audio_samples_per_sec", "samples/s"

    def __init__(self, name):
        self.name = name
        self.hp = workload_hparams(name)
        self.B, self.T = WN_SHAPES[name]
        self.scalar = self.hp.input_type != "mulaw-quantize"
        self.units_per_gpu_step = self.B * self.T

    def config(self, world):
        hp = self.hp
        return {"workload": "%s: WaveNet %d layers / %d stacks, R%d/G%d/S%d, %s, fwd+bwd+clip+Adam+EMA, batch %d x %d samples per GPU, "
                            "dropout %.2f, dp%d" % (self.name, hp.layers, hp.stacks, hp.residual_channels, hp.gate_channels, hp.skip_out_channels,
                                                    "raw input + MoL-%d NLL" % (hp.out_channels // 3) if self.scalar else "mu-law-256 one-hot + softmax-CE",
                                                    self.B, self.T, hp.wavenet_dropout, world),
                "per_gpu_batch": self.B, "samples_per_item": self.T, "parallelism": "dp%d" % world,
                "l2": "per-step working set (activations stashed for backward, GBs) >> 126 MB L2: no explicit flush"}

    def setup(self, dev, rank, use_graph):
        import torch
        from t2_import import t2
        self.model = t2.wavenet.WaveNet(self.hp, self.B, self.T, device=dev)
        self.model.init_variables(seed=5339)
        q = None if self.scalar else (lambda w: t2.audio.mulaw_quantize(torch.from_numpy(w).to(dev)).cpu().numpy())
        x, c, lengths = synth_batch(self.hp, self.B, self.T, 2 + rank, q)
        self.pin = [torch.from_numpy(a).pin_memory() for a in (x, c, x, lengths)]
        self.static = [p.to(dev) for p in self.pin]
        self.loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
        self.use_graph = use_graph
        if use_graph:
            # data parallel: the step is cut into 3 graphs after each third of the stack's weight gradients so that the NCCL
            # all-reduce of a third overlaps the next third's GEMM (3 x 8 layers = 3 x 144 tiles = 3 full waves of 148 SMs)
            world = int(os.environ.get("WORLD_SIZE", "1"))
            self.model.capture(*self.static, overlap_groups=3 if (world >= 4 and self.hp.layers % 3 == 0 and os.environ.get("T2_AR_OVERLAP", "1") != "0") else 1)

    def step(self, e2e, world):
        import torch
        if e2e:
            self.model.train_step(*self.pin, world_size=world)
            self.loss_host.copy_(self.model.loss_buf, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        else:
            self.model.train_step(*((None, None, None, None) if self.use_graph else self.static), world_size=world)

    def h2d_bytes(self):
        return int(sum(p.numel() * p.element_size() for p in self.pin))

    d2h_bytes = 8

    def loss(self):
        return self.model.loss_value()

    def launches_per_step(self):
        return int(self.model.launches_per_step)

    def roofline(self, ms_per_step):
        hp, m = self.hp, self.model
        L = hp.layers
        probe = sorted({L // 8, (3 * L) // 8, (5 * L) // 8, (7 * L) // 8})
        gate_ms = sum(m.time_kernel(0, l, reps=20) for l in probe) / len(probe)
        R, G, S, C = hp.residual_channels, hp.gate_channels, hp.skip_out_channels, hp.cin_channels
        BT = self.B * self.T
        flops_gate = 2.0 * BT * G * (3 * R + C)
        pk = _peaks()
        burst, sustained, hbm = float(pk.get("bf16_tflops", 1590.0)), float(pk.get("bf16_tflops_sustained", 1400.0)), float(pk.get("hbm_gbs", 6650.0))
        src = "MEASURED_PEAKS.json" if pk else "fallback (B200_PROFILING.md)"
        # whole residual stack, SURVEY §8d accounting: FLOPs fwd = 2(3RG + CG + (G/2)S + (G/2)R) per (b,t,layer), x3 for fwd+bwd;
        # algorithmic bytes fwd+bwd = (5R + 2C + 3S) * sizeof(activation); activations are stored as bf16 here
        flops_step = 3.0 * 2.0 * (3 * R * G + C * G + (G // 2) * S + (G // 2) * R) * BT * L
        bytes_step = (5 * R + 2 * C + 3 * S) * 2.0 * BT * L
        sec = ms_per_step * 1e-3
        step = {"algorithmic_tflop": flops_step / 1e12, "tflops": flops_step / sec / 1e12, "frac_of_sustained_bf16": flops_step / sec / 1e12 / sustained,
                "algorithmic_gb_bf16_act": bytes_step / 1e9, "gbs": bytes_step / sec / 1e9, "frac_of_hbm": bytes_step / sec / 1e9 / hbm,
                "t_min_ms": 1e3 * max(flops_step / (sustained * 1e12), bytes_step / (hbm * 1e9)),
                "dram_bytes_measured": _traffic(self.name + "_step_dram_bytes"),
                "note": "residual stack only (head, upsampling net and optimizer excluded from the algorithmic figures, included in the time)"}
        gate = {"kernel": "act_gemm_kernel<EPI_GATE,256,NT=2> (per-layer dilated-conv + conditioning gate GEMM, %d launches / step)" % L,
                "timing": "CUDA events around 20 back-to-back launches replayed from one CUDA graph on a private stream (kernel timed ALONE), "
                          "averaged over layers %s" % probe,
                "flops_per_launch": flops_gate, "ms_per_launch": gate_ms, "tflops": flops_gate / (gate_ms * 1e-3) / 1e12,
                "frac_of_burst_bf16": flops_gate / (gate_ms * 1e-3) / 1e12 / burst,
                "dram_bytes_measured": _traffic(self.name + "_gate_dram_bytes_per_launch")}
        if self.name == "wavenet_default":
            # the HBM-bound shape: the roofline object is the whole dilated stack against the measured copy bandwidth
            return {"bound": "hbm", "kernel": "residual stack (gate / out / dz / dx / wgrad GEMM chain), whole training step",
                    "achieved": step["gbs"], "peak": hbm, "unit": "GB/s", "frac": step["frac_of_hbm"], "traffic": step["dram_bytes_measured"],
                    "peak_source": src + " hbm_gbs (kernel chain timed inside the long step)", "step": step, "gate_gemm": gate}
        return {"bound": "tensor", "kernel": gate["kernel"], "timing": gate["timing"], "achieved": gate["tflops"], "peak": burst,
                "unit": "TFLOP/s", "frac": gate["frac_of_burst_bf16"], "traffic": gate["dram_bytes_measured"],
                "flops_per_launch": flops_gate, "ms_per_launch": gate_ms,
                "peak_source": src + " bf16_tflops (burst: the kernel is timed in isolation)", "step": step}

    def cpu_reference(self, steps, warmup):
        """oracle (fp32 PyTorch-CPU restatement of the reference graph): forward + loss + autograd backward + clip + Adam + EMA on a
        bounded sample of the same workload (at most 2 x 7680 samples per step)."""
        import torch
        from oracle import audio as oa
        from oracle import wavenet as ow
        hp = self.hp
        B, T = min(self.B, 2), min(self.T, 7680)
        params = ow.init_params(hp, seed=5339)
        x, c, lengths = synth_batch(hp, B, T, 2, None if self.scalar else oa.mulaw_quantize)
        if self.scalar:
            xt = torch.from_numpy(x).unsqueeze(1)
            y = torch.from_numpy(x)
        else:
            y = torch.from_numpy(x).long()
            xt = torch.nn.functional.one_hot(y, hp.quantize_channels).float().transpose(1, 2).contiguous()
        c_t, len_t = torch.from_numpy(c), torch.from_numpy(lengths).long()
        px, pc = xt[:1, :, :2048].contiguous(), c_t[:1, :, :8].contiguous()

        def probe():
            with torch.no_grad():
                ow.step(px, pc, params, hp)
        nthreads, ncores = _pick_threads(probe)
        state, times = {}, []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            loss, grads, _ = ow.train_step(params, xt, c_t, y, len_t, hp)
            ow.adam_step(params, grads, state, hp, i)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        total = sum(times)
        return {"value": B * T * len(times) / total, "ms_per_step": 1e3 * total / len(times), "cores": nthreads,
                "sample": "B=%d x T=%d samples per step, %d timed steps, fp32, torch.set_num_threads(%d) of %d host cores (fastest probed)" % (
                    B, T, len(times), nthreads, ncores)}


class TacotronWorkload(object):
    metric, unit = "tacotron_train_mel_frames_per_sec", "frames/s"
    name = "tacotron"

    def __init__(self):
        self.hp = workload_hparams("tacotron")
        self.B, self.Ti, self.To = TACO_SHAPE
        self.units_per_gpu_step = self.B * self.To

    def config(self, world):
        return {"workload": "tacotron: encoder (3 conv + BiLSTM) + 2-layer zoneout-LSTM decoder with location-sensitive attention + postnet, "
                            "r=1, predict_linear=False, conv dropout 0.5 / prenet dropout 0.5 / zoneout 0.1 ON, fwd+bwd+global-norm clip+Adam, "
                            "batch %d per GPU, T_in %d, T_out %d, bf16 GEMM operands / fp32 state, dp%d" % (self.B, self.Ti, self.To, world),
                "per_gpu_batch": self.B, "frames_per_item": self.To, "parallelism": "dp%d" % world,
                "l2": "per-step working set (state histories for BPTT, GBs) >> 126 MB L2: no explicit flush"}

    def setup(self, dev, rank, use_graph):
        import torch
        from t2_import import t2
        self.model = t2.tacotron.Tacotron(self.hp, self.B, self.Ti, self.To, device=dev)
        self.model.init_variables(seed=5339)
        arrs = taco_batch(self.hp, self.B, self.Ti, self.To, 3 + rank)
        self.pin = [torch.from_numpy(a).pin_memory() for a in arrs]
        self.static = [p.to(dev) for p in self.pin]
        self.loss_host = torch.zeros(4, dtype=torch.float32).pin_memory()
        self.use_graph = use_graph
        if use_graph:
            self.model.capture(*self.static)

    def step(self, e2e, world):
        import torch
        if e2e:
            if self.use_graph:
                self.model.train_step(*self.pin, world_size=world)
            else:
                self.model.train_step(*[p.to(self.static[0].device, non_blocking=True) for p in self.pin], world_size=world)
            self.loss_host.copy_(self.model.loss_buf, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        else:
            self.model.train_step(*((None, None, None, None) if self.use_graph else self.static), world_size=world)

    def h2d_bytes(self):
        return int(sum(p.numel() * p.element_size() for p in self.pin))

    d2h_bytes = 16

    def loss(self):
        return self.model.losses()["total"]

    def launches_per_step(self):
        return int(self.model.launches_per_step)

    def roofline(self, ms_per_step):
        # SURVEY §8d: the decoder recurrence is weight-streaming / latency bound (M = 32 rows): every decoder step must read the LSTM-1/2,
        # attention-query and projection weights once forward and (transposed) once in BPTT, plus once for the weight gradients
        hp = self.hp
        D, H, A, P2, M = hp.decoder_lstm_units, hp.encoder_lstm_units, hp.attention_dim, hp.prenet_layers[-1], hp.num_mels
        w_params = (2 * H + D) * 4 * D + 2 * D * 4 * D + D * A + (D + 2 * H) * (M + 1)       # per-step recurrent operand set (prenet part batched)
        bytes_step = 2.0 * w_params * 2 * self.To                                           # bf16, forward + BPTT sweeps
        pk = _peaks()
        hbm = float(pk.get("hbm_gbs", 6650.0))
        sec = ms_per_step * 1e-3
        flops = 3.0 * 34.0e6 * self.B * self.To + 3.0 * (11.0e6 * self.B * self.Ti + 10.98e6 * self.B * self.To)
        return {"bound": "hbm", "kernel": "decoder recurrence (EPI_LSTM swapped GEMMs + attention, %d dependent steps fwd and bwd)" % self.To,
                "achieved": bytes_step / sec / 1e9, "peak": hbm, "unit": "GB/s", "frac": bytes_step / sec / 1e9 / hbm,
                "traffic": _traffic("tacotron_step_dram_bytes"),
                "algorithmic_bytes_per_step": bytes_step,
                "peak_source": ("MEASURED_PEAKS.json" if pk else "fallback") + " hbm_gbs; weights are L2-resident in practice, so this is the floor "
                               "set by re-streaming them once per decoder step (SURVEY §8d), not a DRAM-traffic claim",
                "step": {"algorithmic_tflop": flops / 1e12, "tflops": flops / sec / 1e12,
                         "frac_of_sustained_bf16": flops / sec / 1e12 / float(pk.get("bf16_tflops_sustained", 1400.0))}}

    def cpu_reference(self, steps, warmup):
        import torch
        from oracle import tacotron as ot
        hp = self.hp
        B = 4
        arrs = taco_batch(hp, B, self.Ti, self.To, 3)
        inputs, lens, mel, stop = (torch.from_numpy(a) for a in arrs)
        inputs, lens = inputs.long(), lens.long()
        params = ot.init_params(hp, seed=5339)

        def probe():
            with torch.no_grad():
                ot.forward(params, inputs[:, :40], torch.clamp(lens, max=40), mel[:, :16], hp, training=True)
        nthreads, ncores = _pick_threads(probe)
        state, times = {}, []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            _, grads, _, _ = ot.train_step(params, inputs, lens, mel, stop, hp)
            ot.adam_step(params, grads, state, hp, i)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        total = sum(times)
        return {"value": B * self.To * len(times) / total, "ms_per_step": 1e3 * total / len(times), "cores": nthreads,
                "sample": "B=%d x T_out=%d frames per step (T_in %d), %d timed steps, fp32 autograd, torch.set_num_threads(%d) of %d host cores" % (
                    B, self.To, self.Ti, len(times), nthreads, ncores)}


def make_workload(name):
    return TacotronWorkload() if name == "tacotron" else WaveNetWorkload(name)


DUMP_SAMPLE = 1 << 22          # elements kept of a larger flat buffer: 3 buffers x 16 MB + the loss stay under 64 MB


def restore_initial_state(model, params0):
    """Puts a model back where setup() left it: the seeded variables, no Adam moments or EMA shadows yet, step counters at zero
    (the dropout seed of the next step is then the first step's)."""
    model.params.copy_(params0)
    model.m = model.v = None
    if hasattr(model, "ema"):
        model.ema = None
    model.global_step = 0
    model.step_dev.zero_()
    for flag in ("_packed_dirty", "_dirty"):        # the eager path re-packs the bf16 operand copies before its next forward
        if hasattr(model, flag):
            setattr(model, flag, True)


def dump_outputs(model, out_dir):
    """Writes what a training step hands its caller as float32 .npy files: the loss buffer, the gradients, the updated parameters
    and (WaveNet) their EMA shadows. A flat buffer longer than DUMP_SAMPLE is written as a fixed, seeded sample of its elements in
    index order, the same indices for every buffer of that length."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name in ("loss_buf", "grads", "params", "ema"):
        t = getattr(model, name, None)
        if t is None:
            continue
        a = t.detach().float().cpu().numpy()
        if a.size > DUMP_SAMPLE:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="wavenet_ce", choices=["wavenet_ce", "wavenet_mol", "wavenet_default", "tacotron"])
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the bounded oracle timing on rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, run the timed step once more from the seeded initial "
                                                         "variables and write what it computed to DIR/<name>.npy (rank 0), so that "
                                                         "runs with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    heavy = args.workload != "wavenet_ce"
    steps = args.steps if args.steps is not None else (20 if heavy else 200)
    warmup = args.warmup if args.warmup is not None else (3 if heavy else 10)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = make_workload(args.workload)
    config = wl.config(max(world, 1))

    if args.impl == "reference":
        if rank != 0:
            return
        k, w = min(steps, 2), min(warmup, 1)
        r = wl.cpu_reference(k, w)
        line = {"impl": "reference", "metric": wl.metric, "value": r["value"], "unit": wl.unit, "n_gpus": args.gpus, "steps": k, "warmup": w,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": wl.unit, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "oracle/ (fp32 PyTorch-CPU restatement of the reference TF1 graph; TF1 is not installable here)"}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl.setup(dev, rank, not args.no_graph)
    params0 = wl.model.params.clone() if args.dump_outputs else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    results, clocks, sampler = {}, None, None
    for mode in ("resident", "e2e"):
        for _ in range(max(warmup, 3)):
            wl.step(mode == "e2e", world)
        barrier()
        if mode == "resident":
            sampler = ClockSampler(local_rank)
            if rank == 0:
                sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            wl.step(mode == "e2e", world)
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if mode == "resident" and rank == 0:
            clocks = sampler.stop()
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        results[mode] = t.item()
    loss = wl.loss()
    ms_per_step = results["resident"] / steps
    roof = wl.roofline(ms_per_step)
    if args.dump_outputs:
        # The state after the timed steps is not reproducible: the kernels reduce with float atomics, and over many steps the bf16
        # re-rounding of the weights and Adam on gradients that are zero up to rounding amplify that order noise far beyond
        # rounding. One step of the timed call from the seeded variables and batch carries only that one step's order noise.
        restore_initial_state(wl.model, params0)
        wl.step(False, world)
        barrier()
        if rank == 0:
            dump_outputs(wl.model, args.dump_outputs)

    if rank == 0:
        total_units = world * wl.units_per_gpu_step * steps
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            r = wl.cpu_reference(1, 1)
            cpu = {"value": r["value"], "unit": wl.unit, "cores": r["cores"], "kind": "port", "sample": r["sample"]}
        line = {"metric": wl.metric, "value": total_units / (results["resident"] * 1e-3), "unit": wl.unit, "n_gpus": world,
                "steps": steps, "warmup": max(warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config, "loss": loss, "clocks": clocks,
                "e2e": {"value": total_units / (results["e2e"] * 1e-3), "unit": wl.unit, "h2d_bytes_per_step": wl.h2d_bytes(),
                        "d2h_bytes_per_step": wl.d2h_bytes, "ms_per_step": results["e2e"] / steps},
                "gpu_launches": wl.launches_per_step() * steps,
                "parity": _parity_record(wl.name),
                "roofline": roof, "cpu_baseline": cpu}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _parity_record(name):
    """bf16-mode deviation from the fp32 oracle at this workload's shape, from the committed measurement of the GPU parity tests
    (profiles/r02_measured_parity.jsonl; tests/test_parity_full_gpu.py)"""
    key = {"wavenet_ce": "wavenet_cfg2_24L_2x7680_ce_dropout", "wavenet_mol": "wavenet_cfg4_24L_2x4096_mol",
           "wavenet_default": "wavenet_small_mulaw-quantize_L4_R128_B2xT512", "tacotron": "tacotron_cfg3_fullwidth_B32_Tin160_Tout200_stochastic"}[name]
    try:
        for ln in open(os.path.join(ROOT, "profiles", "r02_measured_parity.jsonl")):
            d = json.loads(ln)
            if d.get("test") == key:
                keep = ("loss_abs_err", "logits_max_err", "logits_mean_err", "mel_l1", "dec_l1", "align_max_err", "loss_before_err", "loss_after_err")
                out = {"mode": "bf16 operands + bf16-stored activations, fp32 accumulate; oracle fp32", "measured_at": key}
                out.update({k: d[k] for k in keep if k in d})
                return out
    except Exception:
        pass
    return None


if __name__ == "__main__":
    main()

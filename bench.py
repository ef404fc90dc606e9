#!/usr/bin/env python
"""Benchmark of the speech-encoder hot path: one train step (zero_grad + forward + backward + gradient all-reduce + Adam)
of a BASELINE.json configuration on synthetic 16 kHz utterances.

    python bench.py --gpus 1 --steps 20 --warmup 5             # config 3 (the headline), this repo's sm_100a path
    python bench.py --config {2,3,3s,4,5}                       # the other BASELINE configs (3s = config 3, strong scaling)
    torchrun --nproc-per-node N bench.py --gpus N ...           # one process per GPU, NCCL
    python bench.py --impl reference ...                        # the reference's CPU execution (oracle port)

Prints ONE JSON line (rank 0).  `e2e` (the headline) = utterances/s through the public API (models.Model.forward /
PretrainedModel.forward) from pinned HOST buffers with the H2D copy and the D2H loss read inside the timed region;
`value` = the same step with inputs already resident in HBM (device-timed, max over ranks).  `roofline` describes the
dominant kernel, `cpu_baseline` the reference-style CPU execution on this box's host cores, `reference_gpu` (N=1) the
reference-structured port on this GPU (cuDNN RNN / cuDNN conv / cuBLAS, its 80x conv loop included) timed with CUDA events.
"""
import argparse
import importlib
import json
import os
import statistics
import string
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs 2-5 (config 1 is the CPU decode_intents plumbing case: tests/test_models_cpu.py).
#   batch: per GPU (weak scaling) | global_batch: split over the ranks (strong scaling)
CONFIGS = {
    "2": dict(cfg="no_unfreezing", kind="frozen", T=64000, batch=64, scaling="weak",
              workload="experiments/no_unfreezing.cfg SLU train step, encoder frozen (freeze_all_layers): full forward, backward through the "
                       "intent GRU + head only, dropout 0.5, Adam; 4 s @16 kHz synthetic utterances"),
    "3": dict(cfg="unfreeze_all_layers", kind="slu", T=64000, batch=256, scaling="weak",
              workload="experiments/unfreeze_all_layers.cfg SLU train step (all layers unfrozen, dropout 0.5, Adam), "
                       "4 s @16 kHz synthetic utterances"),
    "3s": dict(cfg="unfreeze_all_layers", kind="slu", T=64000, global_batch=256, scaling="strong",
               workload="experiments/unfreeze_all_layers.cfg SLU train step (all layers unfrozen, dropout 0.5, Adam), "
                        "4 s @16 kHz synthetic utterances, GLOBAL batch 256 split over the ranks"),
    "4": dict(cfg="no_unfreezing", kind="asr", T=240000, global_batch=128, scaling="strong",
              workload="--pretrain ASR path: PretrainedModel.forward (pretraining_type 2: frame-wise CE phoneme + word heads, "
                       "not CTC), dropout 0.5, Adam; 15 s @16 kHz synthetic utterances, GLOBAL batch 128 split over the ranks"),
    "5": dict(cfg="seq2seq", kind="seq2seq", T=64000, batch=64, scaling="weak",
              workload="repaired all_real_seq2seq cfg: SLU train step with the seq2seq attention decoder (teacher forced, 40 symbols, "
                       "alphabet 102) on top of the encoder kernels, nothing frozen, Adam; 4 s @16 kHz synthetic utterances"),
}
U_SEQ, N_LABELS = 40, 102


def gru_lengths(T, kind):
    L0 = (T - 1) // 80 + 1
    t = (L0 + 1) // 2
    out = []
    for _ in range(4):
        out.append(t)
        t = (t + 1) // 2
    if kind != "asr":
        out.append(t)               # intent GRU / seq2seq encoder GRU on the word-module output (no downsample before it)
    return out


def host_threads():
    """Threads for the CPU reference legs: torch's intra-op pool gets SLOWER beyond ~16-32 threads on this op mix
    (measured: 128 threads = 0.18 utt/s vs 8 threads = 12 utt/s), so use the cores it can actually exploit."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("SLU_REF_THREADS", "16"))))


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["hbm_gbs"], p["bf16_tflops"], p.get("bf16_tflops_sustained", p["bf16_tflops"]), "measured"
    except Exception:
        return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, interval_ms=25, query=None):
        self.rows, self.proc, self.index, self.lo, self.hi = [], None, index, 0, None
        self.interval_ms, self.query = interval_ms, query or self.Q

    def __enter__(self):
        self.lo = len(self.rows)             # rows from here on were sampled inside the timed region
        return self

    def __exit__(self, *a):
        time.sleep(0.12)                     # at least one 100 ms sample lands inside short regions
        self.hi = len(self.rows)

    def start(self):
        """Launch nvidia-smi ahead of the timed region (its start-up takes longer than a short run)."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.query,
                                          "--format=csv,noheader,nounits", "-lms", str(self.interval_ms)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=lambda: [self.rows.append(l) for l in self.proc.stdout], daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)    # gone before anything else is timed
            except Exception:
                self.proc.kill()
            self.thread.join(timeout=2)
            self.proc = None

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.rows[self.lo:self.hi]:
            f = [v.strip() for v in l.split(",")]
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
                reasons |= {n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")}
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


_JSON_FD = None


def _claim_stdout():
    """Everything libraries print to fd 1 (NCCL's version banner, warnings) goes to stderr; the one JSON line is written to the
    real stdout by _emit()."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, (json.dumps(line) + "\n").encode())


def ref_sample_batch(spec, args):
    """Utterances per step of the bounded CPU sample (about 0.07 s of CPU work per utterance-4-s)."""
    if args.ref_batch:
        return args.ref_batch
    return 8 if spec["T"] <= 64000 else 4


def cpu_port_seconds(spec, B, steps, warmup):
    import torch
    from oracle import ref_port, torch_ref as R
    torch.set_num_threads(host_threads())
    return ref_port.train_steps(R.synthetic_params(seed=0, asr=spec["kind"] == "asr"), B, spec["T"], steps, warmup, device="cpu",
                                loop80=True, kind=spec["kind"])


def run_reference(args, spec, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle port with the
    reference's execution structure incl. its 80x conv loop), all host threads it can use, bounded sample."""
    if rank != 0:
        return
    cores = host_threads()
    B = ref_sample_batch(spec, args)
    steps, warmup = max(1, args.steps), max(0, args.warmup)      # a step = one train step on a bounded sample (B utterances)
    sec = cpu_port_seconds(spec, B, steps, warmup)
    val = B / sec
    line = {"impl": "reference", "metric": "utterances_per_sec_train_step", "value": val, "unit": "utt/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": spec["scaling"],
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": spec["workload"], "baseline_config": args.config, "samples_per_utt": spec["T"], "batch_per_step": B,
                       "note": "bounded sample of the workload: the same train step on batch_per_step utterances per step"},
            "cpu_baseline": {"value": val, "unit": "utt/s", "cores": cores, "kind": "port",
                             "sample": "%d train steps of batch %d x %g s (reference execution structure incl. 80x conv loop), "
                                       "torch CPU %d threads" % (steps, B, spec["T"] / 16000, cores)},
            "e2e": {"value": val, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


def build_workload(spec, B, rank, pkg):
    """-> (model, labels(generator) -> tuple of host tensors, loss_of(outputs))."""
    import torch
    import models
    cfgmod = importlib.import_module("end-to-end-slu_b200.config")
    cfg = cfgmod.read_config(os.path.join(ROOT, "configs", spec["cfg"] + ".cfg"))
    kind = spec["kind"]
    cfg.num_phonemes = 42
    cfg.Sy_intent, cfg.values_per_slot = cfgmod.fsc_intent_table()
    if kind == "seq2seq":
        cfg.Sy_intent = ["<sos>"] + list(string.printable) + ["<eos>"]          # alphabet of 102 (data.py:202-207)
        assert len(cfg.Sy_intent) == N_LABELS
    if kind == "asr":
        cfg.pretraining_type = 2
        torch.manual_seed(cfg.seed)
        model = models.PretrainedModel(cfg)
    else:
        cfg.pretraining_type = 0                             # random init, nothing frozen == fully unfrozen (SURVEY 5.6)
        torch.manual_seed(cfg.seed)
        model = models.Model(cfg)
        if kind == "frozen":
            model.freeze_all_layers()                        # what Model.__init__ does after loading a pretrained checkpoint

    def labels(gen):
        if kind in ("slu", "frozen"):
            return (torch.stack([torch.randint(0, v, (B,), generator=gen) for v in (6, 14, 4)], 1),)
        if kind == "asr":
            T = spec["T"]
            return (torch.randint(-1, 42, (B, -(-T // 640)), generator=gen), torch.randint(-1, 10000, (B, -(-T // 2560)), generator=gen))
        idx = torch.randint(1, N_LABELS - 1, (B, U_SEQ), generator=gen)
        idx[:, 0] = 0
        idx[:, -1] = N_LABELS - 1
        return (torch.nn.functional.one_hot(idx, N_LABELS).float(),)

    def loss_of(out):
        if kind == "asr":
            return out[0] + out[1]                           # pretraining_type 2: phoneme + word loss (training.py:61-63)
        return out[0]
    return model, labels, loss_of


OUTPUT_NAMES = {"asr": ("phoneme_loss", "word_loss", "phoneme_acc", "word_acc")}     # PretrainedModel.forward; Model.forward: loss, acc
DUMP_LIMIT = 64 * 10 ** 6


def dump_outputs(out_dir, kind, out, model, opt):
    """What the last train step computed: the model's outputs, the gradients of the loss and Adam's first and second moments
    after its update, each as out_dir/<out|grad|adam_m|adam_v>.<name>.npy in float32 or float64.  When dumping, every step
    starts from the same weights (see `step` in main), so with the same arguments these agree from run to run up to the
    rounding of the kernels' atomic gradient sums (<= 2e-6 of each tensor's largest element, measured on a B200 at 1000 W,
    configs 3 and 4).  A gradient that is exactly zero in exact arithmetic holds only that rounding (config 5: the attention
    key bias, to which the softmax is invariant), so compare it with an absolute tolerance.  The updated weights are not written: Adam divides each moment by its own magnitude + 1e-8, which turns
    that rounding of near-zero gradients into weight differences of up to lr."""
    import numpy as np
    arrays = {"out." + n: t for n, t in zip(OUTPUT_NAMES.get(kind, ("loss", "acc")), out)}
    for n, p in model.named_parameters():
        if p.grad is not None:
            arrays["grad." + n] = p.grad
        st = opt.state.get(p, {})
        if "exp_avg" in st:
            arrays["adam_m." + n], arrays["adam_v." + n] = st["exp_avg"], st["exp_avg_sq"]
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes, more than the %d allowed" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="3", choices=sorted(CONFIGS), help="BASELINE.json config (3s = config 3 at global batch 256)")
    ap.add_argument("--batch", type=int, default=0, help="utterances per GPU per step (default: the config's)")
    ap.add_argument("--ref-batch", type=int, default=0, help="utterances per step of the bounded CPU sample")
    ap.add_argument("--background-prefetch", action="store_true", help="stage batch i+1 in a helper thread instead of the consumer's")
    ap.add_argument("--launch-detail", action="store_true", help="print every launch of one step with its sizes and device time")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference-structured port on this GPU (cuDNN), N=1 only")
    ap.add_argument("--sampler-probe", action="store_true", help="developer: time the step under several clock-sampler settings (stderr)")
    ap.add_argument("--eval-dropout", action="store_true", help="disable dropout (debug)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed (model "
                    "outputs, gradients, Adam moments) to DIR/<name>.npy, for comparing two builds output for output; every step "
                    "then starts from the initial weights, which makes the results reproducible and the steps slower")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    spec = CONFIGS[args.config]
    if args.impl == "reference":
        return run_reference(args, spec, rank, world)

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = importlib.import_module("end-to-end-slu_b200")
    pkg._lib.load()                                          # fail loudly if the CUDA library is missing
    pkg.dp.install()
    kind, T_SAMPLES = spec["kind"], spec["T"]
    if args.batch:
        B = args.batch
    elif "global_batch" in spec:
        assert spec["global_batch"] % world == 0
        B = spec["global_batch"] // world
    else:
        B = spec["batch"]
    model, labels, loss_of = build_workload(spec, B, rank, pkg)
    model.train()
    if args.eval_dropout:
        model.eval()
    params = [p for p in model.parameters()]
    lr = 1e-3
    opt = torch.optim.Adam(params, lr=lr)                    # what training.py:19 constructs
    NB = 4 if T_SAMPLES * B * 4 * 4 > 130e6 else 8           # rotating input sets, together larger than the 126 MB L2
    gen = torch.Generator().manual_seed(1234 + rank)
    xs_host = [(0.1 * torch.randn(B, T_SAMPLES, generator=gen)).pin_memory() for _ in range(NB)]
    ys_host = [tuple(y.pin_memory() for y in labels(gen)) for _ in range(NB)]
    xs_dev = [x.cuda(non_blocking=True) for x in xs_host]
    ys_dev = [tuple(y.cuda(non_blocking=True) for y in ys) for ys in ys_host]
    h2d_bytes = xs_host[0].numel() * 4 + sum(y.numel() * y.element_size() for y in ys_host[0])

    last = {}                                                # outputs of the most recent step, for --dump-outputs
    # With --dump-outputs every step trains from the initial weights.  The kernels sum gradients with atomics (last-bit order
    # effects) and Adam amplifies those across steps into a different trajectory on every run; from fixed weights, batch and
    # dropout seeds a step computes the same result each run.  The restore adds ~0.17 ms to a config-3 step (B200, 1000 W), so
    # the times of a dumping run are not comparable with those of a plain one.
    init_weights = [p.detach().clone() for p in params] if args.dump_outputs else None

    def step(x, ys):
        if init_weights is not None:
            with torch.no_grad():
                torch._foreach_copy_(params, init_weights)
        out = model(x, *ys)
        loss = loss_of(out)
        opt.zero_grad()
        loss.backward()
        opt.step()                                           # pre-step hook = the single gradient all-reduce
        last["out"] = out
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(k, host):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        if host == "prefetch":                                        # the Trainer loop over a DevicePrefetcher-wrapped loader
            batches = ((xs_host[i % NB],) + ys_host[i % NB] for i in range(k))
            for batch in pkg.loader.DevicePrefetcher(batches, background=args.background_prefetch):   # H2D of batch i+1 under step i
                loss = step(batch[0], batch[1:])
                loss.item()                                           # D2H read of the step's result, every step
        for i in range(k if host != "prefetch" else 0):
            if host == "serial":
                loss = step(xs_host[i % NB], ys_host[i % NB])         # H2D inside forward (models.py: x.cuda())
                loss.item()
            else:
                step(xs_dev[i % NB], ys_dev[i % NB])
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    clk = ClockSampler(local).start()
    for i in range(max(args.warmup, 3)):
        step(xs_dev[i % NB], ys_dev[i % NB])
    timed(3, host="prefetch")                                # untimed warm-up of the host-fed paths too (copy stream, its
    timed(3, host="serial")                                  # allocator pool, pinned staging)
    for _ in range(30):                                      # nvidia-smi is up and sampling before the timed region starts
        if clk.rows or clk.proc is None:
            break
        time.sleep(0.1)
    for i in range(max(args.warmup, 3)):                     # the GPU idled while nvidia-smi started: warm it again (untimed)
        step(xs_dev[i % NB], ys_dev[i % NB])
    torch.cuda.synchronize()
    calls0 = pkg._lib.stats["calls"]
    with clk:
        ms_dev = timed(args.steps, host=None)
    launches = pkg._lib.stats["calls"] - calls0
    clk.stop()
    if args.dump_outputs and rank == 0:                      # before any later step overwrites what the timed run left
        dump_outputs(args.dump_outputs, kind, last["out"], model, opt)
    if args.sampler_probe and rank == 0:                     # developer: how much does the clock sampler perturb the timed region?
        for name, kw in [("none", None), ("25 ms full query", {}), ("25 ms, clocks + reasons only", {"query": ClockSampler.Q.replace("power.draw,", "")}),
                         ("100 ms full query", {"interval_ms": 100}), ("200 ms full query", {"interval_ms": 200}), ("none", None)]:
            c = ClockSampler(local, **kw).start() if kw is not None else None
            time.sleep(1.0)
            runs = [timed(args.steps, host=None) / args.steps for _ in range(5)]
            if c is not None:
                c.stop()
            print("sampler %-30s ms/step: %s" % (name, " ".join("%.3f" % r for r in runs)), file=sys.stderr)
    ms_e2e = timed(args.steps, host="prefetch")
    ms_e2e_serial = timed(args.steps, host="serial")
    per_step = ms_dev / args.steps
    value = world * B / (per_step * 1e-3)
    e2e_value = world * B / (ms_e2e / args.steps * 1e-3)

    # ---- per-kernel device time (CUDA events around every C-ABI launch, separate untimed pass) -----
    pkg.ops.OVERLAP = False                                  # serialise the side-stream launches: clean per-kernel durations
    pkg._lib.profile_begin(detail=args.launch_detail)
    for i in range(3):
        step(xs_dev[i % NB], ys_dev[i % NB])
    if args.launch_detail and rank == 0:                     # per-launch table (sizes, ms) of the last profiled step -> stderr
        det = pkg._lib.profile_detail()
        for n, a, ms in det[2 * len(det) // 3:]:
            print("launch %-22s %-60s %8.1f us" % (n, a, ms * 1e3), file=sys.stderr)
    prof = pkg._lib.profile_end()                            # {name: [ms, ...]}
    pkg.ops.OVERLAP = True
    hbm_peak, tf_burst, tf_sust, how = peaks()
    kern = {k: {"launches_per_step": len(v) / 3, "ms_per_step": sum(v) / 3} for k, v in prof.items()}
    GRU_T = gru_lengths(T_SAMPLES, kind)
    L1 = GRU_T[0]
    gru_names = [k for k in prof if k.startswith("slu_gru_fwd")]
    roofline, extra = None, {}

    def traffic_of(name):
        # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture (config 3, B=256)
        if args.config != "3" or B != 256:
            return None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                return json.load(f).get(name, {}).get("bytes_per_launch")
        except Exception:
            return None
    if gru_names:
        name = gru_names[0]
        # algorithmic flops of the recurrent contraction h.W_hh^T per launch, summed over the layers / step
        flops = sum(2 * 2 * t * 384 * 128 * B for t in GRU_T)
        sec = kern[name]["ms_per_step"] * 1e-3
        ach = flops / sec / 1e12
        nr_rows = pkg.ops.gru_rows_per_cta(B)
        ex = pkg.ops.gru_executed_flop_factor(B)
        roofline = {"kernel": name, "bound": "tensor", "achieved": ach, "peak": tf_sust, "unit": "TFLOP/s",
                    "frac": ach / tf_sust, "traffic": traffic_of(name), "peak_source": how + " bf16 sustained (kernel timed inside a step)",
                    "traffic_note": "bytes of the layer-0 launch (the longest of the %d); null outside the profiled config" % len(GRU_T),
                    "executed_tflops": ex * ach if pkg.ops.GRU_IMPL == "tc" else ach,
                    "note": "persistent-GRU forward, %d launches/step summed; algorithmic flops = 2 dirs * T_l * 2*384*128 * B over the "
                            "layers (h.W_hh only).  The N=16 MMA tile carries %d batch rows, hi and lo stacked along N, times the W_hi / "
                            "W_lo passes: the tensor core executes %dx the algorithmic flops.  The recurrence is a dependency chain "
                            "(%d CTAs of %d batch rows): see DESIGN.md section 4" % (len(GRU_T), nr_rows, ex,
                                                                                    2 * ((B + nr_rows - 1) // nr_rows), nr_rows)}
    sinc_names = [k for k in prof if k.startswith("slu_sincconv_fwd")]
    if sinc_names:
        name = sinc_names[0]
        bytes_ = B * (4 * T_SAMPLES + 4 * 80 * L1)
        sec = kern[name]["ms_per_step"] * 1e-3
        extra["roofline_sincconv"] = {"kernel": name, "bound": "hbm", "achieved": bytes_ / sec / 1e9, "peak": hbm_peak,
                                      "unit": "GB/s", "frac": bytes_ / sec / 1e9 / hbm_peak, "traffic": traffic_of(name),
                                      "note": "algorithmic bytes = B*(4*T + 4*80*L1) = read the waveform once, write the pooled frames once"}

    line = None
    if rank == 0:
        cpu_base = None
        if not args.no_cpu_baseline and world == 1:
            cores = host_threads()
            Bc = ref_sample_batch(spec, args)
            sec = cpu_port_seconds(spec, Bc, 2, 1)
            cpu_base = {"value": Bc / sec, "unit": "utt/s", "cores": cores, "kind": "port",
                        "sample": "2 train steps of batch %d x %g s, reference execution structure (80x conv loop, nn.GRU), "
                                  "torch CPU %d threads" % (Bc, T_SAMPLES / 16000, cores)}
        if not args.no_ref_gpu and world == 1:
            # the north-star comparison: the reference's cuDNN build on THIS GPU, same config and batch, CUDA-event timed
            from oracle import ref_port, torch_ref as R
            xs_dev.clear(); ys_dev.clear()
            torch.cuda.empty_cache()
            rsteps, rwarm = 8, 5
            sec_g = ref_port.train_steps(R.synthetic_params(seed=0, asr=kind == "asr"), B, T_SAMPLES, rsteps, rwarm, device="cuda",
                                         loop80=True, kind=kind)
            ref_v = B / sec_g
            extra["reference_gpu"] = {
                "value": ref_v, "unit": "utt/s", "ms_per_step": sec_g * 1e3, "batch": B, "steps": rsteps, "warmup": rwarm,
                "kind": "port", "timing": "CUDA events around the timed steps (device resident inputs, loss.item() per step)",
                "what": "oracle/ref_port.py: the reference's execution structure on this GPU -- nn.GRU (cuDNN RNN), F.conv1d (cuDNN) "
                        "inside the reference's 80-iteration filter loop with its per-filter host->device copies (models.py:12-13,21,"
                        "98-108), nn.Linear (cuBLAS), torch.optim.Adam; cuDNN TF32 allowed as in the reference's defaults",
                "omits": "nothing on the timed path for configs 2/3/4; config 5's decoder is this repo's seq2seq.py (same per-step "
                         "library calls as models.py:413-556).  It is a port, not the unmodified reference: /root/reference does "
                         "not exist on the GPU box and has no installable package",
                "speedup_device_timed": value / ref_v, "speedup_e2e": e2e_value / ref_v}
        line = {"metric": "utterances_per_sec_train_step", "value": value, "unit": "utt/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": per_step, "higher_is_better": True,
                "scaling": spec["scaling"], "vs_baseline": None,
                "dtype": "f32 (tensor-core contractions as bf16 hi/lo 3-pass split, fp32 accumulate)",
                "data": "synthetic", "impl": "ours",
                "config": {"workload": spec["workload"], "baseline_config": args.config, "batch_per_gpu": B, "global_batch": B * world,
                           "samples_per_utt": T_SAMPLES, "parallelism": "dp%d" % world,
                           "l2": "inputs rotate over %d batches (%d MB) > 126 MB L2; activations ~1 GB/step" % (NB, NB * B * T_SAMPLES * 4 // 1000000)},
                "e2e": {"value": e2e_value, "unit": "utt/s", "h2d_bytes_per_step": h2d_bytes,
                        "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps,
                        "h2d": "pinned host batches, copy of batch i+1 on a copy stream under step i (loader.DevicePrefetcher)",
                        "ms_per_step_serial_copy": ms_e2e_serial / args.steps},
                "gpu_launches": launches, "kernels": kern, "roofline": roofline, "cpu_baseline": cpu_base,
                "clocks": clk.summary(), "allreduce": dict(pkg.dp.stats)}
        line.update(extra)
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

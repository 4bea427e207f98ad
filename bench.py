#!/usr/bin/env python
"""bench.py — MotifNet-SGCls training throughput (images/sec), BASELINE.json's headline metric.

    python bench.py --gpus N --steps K --warmup W            # this framework, one rank per GPU
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU reference arm (oracle port)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also write the last timed step's outputs

With --dump-outputs the inputs, the seeds and the number of steps before the dumped one are fixed by the arguments,
so two builds of the project can be compared output for output (dump_outputs lists what is written).

Workload (BASELINE.json configs[1]): models/train_rels.py step of MotifNet SGCls — VGG16 backbone
(frozen), batch 6 x 3 x 592 x 592 synthetic images per GPU, 20 GT boxes and 15 GT relations per image
(-> 1536 sampled relation triples), forward + backward + grad-clip + SGD(momentum) step, fp32 semantics.
A "step" is one such training step on one batch per GPU (weak scaling: 6 images per GPU).

Timing: W >= 3 untimed warm-up steps, then exactly K steps bracketed by barrier + cuda synchronize
on both sides, CUDA events on the launching stream, max over ranks. The per-step working set
(1.7 GB of parameters + 25 MB fresh images + activations) is far larger than the 126 MB L2, so no
explicit L2 flush is needed (stated in `config`).

One JSON line on rank 0 with `value` (inputs already resident in HBM), `e2e` (through the public
`detector[blob]` API from pinned host buffers, H2D of the batch and D2H of the loss inside the timed
region), `roofline` (dominant kernel = the tcgen05 bf16x3 GEMM/conv, algorithmic fp32 FLOPs per
launch / CUDA-event duration vs the measured bf16 peak), `cpu_baseline` (oracle port on host cores,
bounded sample) and `clocks`.
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
sys.path.insert(0, os.path.join(ROOT, "neural-motifs_b200"))

BATCH_PER_GPU = 6
BOXES, RELS = 20, 15
METRIC = "MotifNet-SGCls train images/sec"
UNIT = "img/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0; see dump_outputs)")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc, self.lines, self.gpu = None, [], gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------ model setup
def build_model(device, seed=0):
    import numpy as np
    import torch
    from lib.rel_model import RelModel
    from dataloaders.synthetic import synthetic_model_state
    classes = ['__background__'] + ['obj%d' % i for i in range(150)]
    rels = ['__background__'] + ['rel%d' % i for i in range(50)]
    torch.manual_seed(seed)
    np.random.seed(seed)        # the relation / RoI sampling draws from numpy's global RNG
    # scripts/train_models_sgcls.sh:19-21
    m = RelModel(classes, rels, mode='sgcls', num_gpus=1, require_overlap_det=True, use_resnet=False, order='leftright',
                 nl_edge=4, nl_obj=2, hidden_dim=512, use_proposals=False, pass_in_obj_feats_to_decoder=False,
                 pass_in_obj_feats_to_edge=False, pooling_dim=4096, rec_dropout=0.1, use_bias=True, use_tanh=False,
                 limit_vision=False)
    synthetic_model_state(m, seed)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.Conv2d):
                torch.nn.init.kaiming_normal_(mod.weight, nonlinearity='relu')
    for p in m.detector.parameters():       # models/train_rels.py:51-52
        p.requires_grad = False
    return m.to(device).train()


def get_optim(model, lr):
    """models/train_rels.py:57-70 (SGD branch: fc layers of roi_fmap* at lr/10, momentum 0.9, l2 1e-4) and
    :145-150 (clip 5) as the fused flat-buffer optimizer (lib/fused_optim.py, csrc/optim.cu)."""
    from lib.fused_optim import FlatSGD
    fc = [p for n, p in model.named_parameters() if n.startswith('roi_fmap') and p.requires_grad]
    non_fc = [p for n, p in model.named_parameters() if not n.startswith('roi_fmap') and p.requires_grad]
    # defer_step: the gradient all-reduce + the fused clip/SGD kernel run on a side stream underneath the NEXT step's
    # frozen backbone; RelModel.forward joins the streams before it reads the first trainable parameter.
    return FlatSGD([(fc, lr / 10.0), (non_fc, lr)], momentum=0.9, weight_decay=1e-4, max_norm=5.0, defer_step=True)


def train_step(model, optimizer, reducer=None, fwd_tuple=None, blob=None, keep=None):
    """models/train_rels.py:118-152 (train_batch): forward, two cross-entropies, backward, clip 5, step.
    The data-parallel gradient average is one all-reduce per flat gradient buffer.
    `keep` (a dict), when given, receives the step's Result and loss tensor."""
    from torch.nn import functional as F
    import torch.distributed as dist
    result = model[blob] if blob is not None else model(*fwd_tuple)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        # the reference averages over the objects / relations of ALL GPUs (gather_res, then one mean): count-weighted
        from lib.data_parallel import count_weighted_loss
        loss = count_weighted_loss([
            (F.cross_entropy(result.rm_obj_dists, result.rm_obj_labels, reduction='sum'), result.rm_obj_labels.size(0)),
            (F.cross_entropy(result.rel_dists, result.rel_labels[:, -1], reduction='sum'), result.rel_labels.size(0))])
    else:
        loss = F.cross_entropy(result.rm_obj_dists, result.rm_obj_labels) + \
            F.cross_entropy(result.rel_dists, result.rel_labels[:, -1])
    optimizer.zero_grad()
    loss.backward()
    optimizer.all_reduce_grads()
    optimizer.step()
    if keep is not None:
        keep["result"], keep["loss"] = result, loss.detach()
    return float(loss.detach())  # the reference's train_batch reads the losses back every step (train_rels.py:151)


DUMP_MAX_ELEMS = 1 << 18        # per array: 1 MB as float32, 2 MB as float64 (< 64 MB over all Result fields)
PARAM_SAMPLE = 1 << 14


def dump_outputs(out_dir, model, last):
    """--dump-outputs: what a caller of the timed step receives from its last step, one DIR/<name>.npy each:
    `loss`, every tensor field of the training Result (`rm_obj_dists`, `rel_dists`, `rel_labels`, ...) and
    `trainable_params` (the parameters the step's update left, PARAM_SAMPLE seeded elements of each trainable
    parameter in named_parameters() order, all of a smaller one). An array larger than DUMP_MAX_ELEMS elements is
    written as `<name>_sample`, a seeded sample of its flattened elements. Floating arrays are float32, integer ones
    float64 (exact)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)

    def sample(flat, k, seed):
        idx = np.random.RandomState(seed).randint(0, flat.numel(), k)
        return flat[torch.from_numpy(idx).to(flat.device)]

    arrays = {"loss": last["loss"].reshape(1)}
    for name, v in vars(last["result"]).items():
        if not torch.is_tensor(v):
            continue
        v = v.detach()
        if v.numel() > DUMP_MAX_ELEMS:
            name, v = name + "_sample", sample(v.reshape(-1), DUMP_MAX_ELEMS, 0)
        arrays[name] = v
    params = [p.detach().reshape(-1) for _, p in model.named_parameters() if p.requires_grad]
    arrays["trainable_params"] = torch.cat([p if p.numel() <= PARAM_SAMPLE else sample(p, PARAM_SAMPLE, i)
                                            for i, p in enumerate(params)])
    for name, v in arrays.items():
        v = v.cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (v.float() if v.is_floating_point() else v.double()).numpy())


def settle_warmup(step, sync, world, dev, min_steps=12, max_steps=60, tol=1.03):
    """Untimed warm-up steps until the step time has settled: at least `min_steps`, then the last five within
    `tol` of each other and of the best, or `max_steps`. `step(i)` may hold collectives (the gradient all-reduce),
    so with world > 1 the decision to stop is itself collective: every rank leaves in the same iteration.
    Returns the number of steps run."""
    import torch
    import torch.distributed as dist
    recent, n = [], 0
    while n < max_steps:
        sync(); t0 = time.perf_counter()
        step(n)
        sync(); recent.append(time.perf_counter() - t0); n += 1
        settled = len(recent) >= min_steps and max(recent[-5:]) <= tol * min(recent[-5:]) and \
            min(recent[-5:]) <= tol * min(recent)
        if world > 1:
            flag = torch.tensor([1 if settled else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            settled = bool(flag.item())
        if settled:
            break
    return n


# ------------------------------------------------------------------------------------------ b200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    import motifs_cabi
    from lib import fused_optim, tc_ops
    from lib.data_parallel import init_from_env
    from dataloaders.synthetic import make_numpy_batch, SyntheticBlob

    # NCCL prints its INFO lines (version banner, "comm ... rank r nranks N ... Init COMPLETE") on STDOUT; the contract
    # wants exactly one JSON line there. Keep the lines (they are the evidence of the communicator's size) but move
    # everything that is not the JSON line to stderr: fd 1 is pointed at fd 2 for the run, the JSON line is written to
    # the saved original stdout at the end.
    if "MOTIFS_KEEP_NCCL_DEBUG" not in os.environ:       # (the image presets NCCL_DEBUG=VERSION: only the banner would appear)
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ["NCCL_DEBUG_SUBSYS"] = "INIT"
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = init_from_env("nccl")
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl b200) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    motifs_cabi.load()
    model = build_model(dev, seed=0)
    opt = get_optim(model, lr=1e-3 * BATCH_PER_GPU)      # train_rels.py:193: lr * num_gpus * batch_size
    reducer = None
    pool = [make_numpy_batch(BATCH_PER_GPU, seed=100 * rank + i, boxes_per_img=BOXES, rels_per_img=RELS,
                             image_offset=0) for i in range(4)]
    blobs = [SyntheticBlob(nb, dev) for nb in pool]
    for b in blobs:
        b.scatter()
    resident = [b[0] for b in blobs]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        marks = []
        e0.record()
        for i in range(steps):
            fn(i)
            ev = torch.cuda.Event(enable_timing=True); ev.record(); marks.append(ev)
        fused_optim.wait_pending_updates()      # the last step's deferred update belongs to the timed region
        e1.record()
        barrier()
        per_step = [a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks)]
        timed.last_per_step = per_step
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    W = max(args.warmup, 5)      # >= 3 required; 5 so that allocator, cuDNN autotuning and clocks are all settled
    sampler = ClockSampler(local)
    sampler.start()
    # nvidia-smi needs ~1 s to initialise NVML (and pokes the driver while doing so): wait for its first
    # sample BEFORE the warm-up, so that the warm-up steps also bring the clocks back up from idle and
    # only the steady 10 Hz polling overlaps the timed region.
    t_wait = time.time()
    while sampler.proc is not None and len(sampler.lines) == 0 and time.time() - t_wait < 8.0:
        time.sleep(0.05)
    for i in range(W):
        train_step(model, opt, reducer, fwd_tuple=resident[i % len(resident)])
    # A fresh box keeps paging libraries in and autotuning for a while: keep warming up (untimed) until
    # the step time has settled — at least 12 extra steps and the last five within 3 % of each other and of the best — or 60 extra steps.
    # With --dump-outputs every run takes the longest warm-up, so that the dumped step starts from the same parameters,
    # optimizer state and RNG state whatever the timings were.
    extra = settle_warmup(lambda i: train_step(model, opt, reducer, fwd_tuple=resident[i % len(resident)]),
                          torch.cuda.synchronize, world, dev, min_steps=60 if args.dump_outputs else 12)
    W += extra
    # Python's cyclic GC pauses the host for tens of ms when a generation-2 pass lands in a step (seen as one
    # 90 ms step among 21.7 ms ones): collect now, freeze what survived, and keep the collector off inside the
    # timed regions (collected again between them) — the usual arrangement of a training loop.
    import gc
    gc_log = []
    gc_t0 = [0.0]

    def gc_cb(phase, info):
        if phase == "start":
            gc_t0[0] = time.perf_counter()
        else:
            gc_log.append((info.get("generation"), round((time.perf_counter() - gc_t0[0]) * 1e3, 2)))
    gc.callbacks.append(gc_cb)
    gc.collect(); gc.freeze(); gc.disable()
    # the collection just released cyclic garbage that held device buffers: two more untimed steps let the caching
    # allocator settle again (round 2: one 700 MB cudaMalloc — 58 ms — landed in the first timed step otherwise)
    for i in range(2):
        train_step(model, opt, reducer, fwd_tuple=resident[i % len(resident)])
    W += 2
    mem0 = torch.cuda.memory_stats(dev)
    calls0 = motifs_cabi.LAUNCHER_CALLS
    last = {} if args.dump_outputs and rank == 0 else None
    ms_res = timed(lambda i: train_step(model, opt, reducer, fwd_tuple=resident[i % len(resident)],
                                        keep=last if i == args.steps - 1 else None), args.steps)
    calls = motifs_cabi.LAUNCHER_CALLS - calls0
    steps_res = list(timed.last_per_step)
    if last is not None:
        dump_outputs(args.dump_outputs, model, last)
        last.clear()
    # e2e: public API with host buffers; H2D of the batch and D2H of the loss every step
    losses = []

    def e2e_step(i):
        losses.append(train_step(model, opt, reducer, blob=blobs[i % len(blobs)]))

    gc.collect()
    for i in range(6):          # the e2e leg allocates the device batch every step: let the allocator settle on that too
        e2e_step(i)
    ms_e2e = timed(e2e_step, args.steps)
    clocks = sampler.stop()
    gc.enable(); gc.callbacks.remove(gc_cb)
    mem1 = torch.cuda.memory_stats(dev)
    host_notes = {"gc": "collector disabled inside the timed regions, gc.collect() between them",
                  "gc_passes_ms": gc_log[-6:],
                  "cuda_mallocs_in_timed_legs": int(mem1.get("num_device_alloc", 0) - mem0.get("num_device_alloc", 0)),
                  "alloc_retries_in_timed_legs": int(mem1.get("num_alloc_retries", 0) - mem0.get("num_alloc_retries", 0))}

    # roofline leg: one extra profiled step, CUDA events around every tensor-core launch
    tc_ops.PROFILE = []
    train_step(model, opt, reducer, fwd_tuple=resident[0])
    torch.cuda.synchronize()
    prof, tc_ops.PROFILE = tc_ops.PROFILE, None
    flops = sum(f for _, f, _, _ in prof)
    tc_ms = sum(a.elapsed_time(b) for _, _, a, b in prof)
    conv = [(f, a.elapsed_time(b)) for k, f, a, b in prof if k == "conv3x3"]
    pk, kind = peaks()
    peak_tf = float(pk.get("bf16_tflops_sustained", pk["bf16_tflops"]))
    achieved = flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    lstm_mb = lstm_microbench(dev) if world == 1 else None
    imgs = BATCH_PER_GPU * world * args.steps
    value = imgs / (ms_res * 1e-3)
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "MotifNet SGCls train_rels.py step, VGG16 backbone, batch 6x592x592 per GPU, "
                               "20 GT boxes + 15 GT rels per image (1536 rel triples), fwd+bwd+clip+SGD",
                   "global_batch": BATCH_PER_GPU * world, "parallelism": "dp%d" % world,
                   "dp_comm": {"nvls": "sharded update over NVSwitch multicast (own kernels: multimem.ld_reduce / multimem.st)",
                               "nccl": "NCCL all-reduce of the flat gradient", "ce": "sharded update, gradient shards and updated parameters moved by copy engines over NVLink (peer-mapped symmetric memory)", "none": "single GPU"}[opt.comm],
                   "warmup_steps_run": W,
                   "arithmetic": "fp32 semantics: tcgen05 bf16x3 split-operand GEMM/conv, fp32 accumulate",
                   "l2": "per-step working set (1.7 GB params + activations) >> 126 MB L2; 4 rotating batches"},
        "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": blobs[0].h2d_bytes(), "d2h_bytes_per_step": 4,
                "api": "RelModel.__getitem__(blob) (models/train_rels.py:137) from pinned host tensors"},
        "gpu_launches": calls,
        "gpu_launches_note": "C-ABI launcher calls of libmotifs_b200.so in the timed region (each >= 1 kernel)",
        "roofline": {"kernel": "gemm_bf16x3_kernel (tcgen05 GEMM + implicit-GEMM 3x3 conv)", "bound": "tensor",
                     "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                     "peak_kind": "%s bf16 sustained" % kind, "launches_per_step": len(prof),
                     "algorithmic_gflop_per_step": flops / 1e9, "kernel_ms_per_step": tc_ms,
                     "share_of_step": tc_ms / (ms_res / args.steps),
                     "backbone_conv_tflops": (sum(f for f, _ in conv) / (sum(t for _, t in conv) * 1e-3) / 1e12) if conv else None,
                     "note": "algorithmic fp32-equivalent FLOPs; the bf16x3 scheme issues 3 tensor-core MACs per "
                             "algorithmic MAC, so tensor-pipe busy fraction is ~3x frac",
                     "traffic": None,
                     "traffic_note": "not measured inside this run (needs ncu); per-launch dram__bytes of one step vs the "
                                     "algorithmic bytes: profiles/r02_gemm_traffic.json"},
        "clocks": clocks,
        "host": host_notes,
        "step_ms": {"value_leg": [round(t, 2) for t in steps_res], "e2e_leg": [round(t, 2) for t in timed.last_per_step]},
        "final_loss": losses[-1] if losses else None,
    }
    if world == 1:
        out["roi_align"] = roi_align_microbench(dev, pk, kind)
        out["lstm"] = lstm_mb
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(sample_images=2)
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(out) + "\n").encode())


def lstm_microbench(dev):
    """BASELINE.json metric (iv) / configs[4]: AlternatingHighwayLSTM, H=512, 2 layers (forward, backward), B=256,
    T in {32, 64, 128, 256}, inputs 712 (edge context) and 4424 (object context), all lengths = T. Forward in eval mode
    and forward+backward in training mode, median of 5 after 2 warm-ups, CUDA events. FLOPs (SURVEY.md section 8d):
    sum_l T * (2*B*In_l*6H + 2*B*H*5H). The reference kernels' times beside these: profiles/ (tools/microbench_ops.py)."""
    import numpy as np
    import torch
    from torch.nn.utils.rnn import pack_padded_sequence
    from lib.lstm.highway_lstm_cuda.alternating_highway_lstm import AlternatingHighwayLSTM
    H, L, B = 512, 2, 256
    rows = []
    for In in (712, 4424):
        torch.manual_seed(0)
        m = AlternatingHighwayLSTM(In, H, L, recurrent_dropout_probability=0.1).to(dev)
        for T in (32, 64, 128, 256):
            x = torch.randn(T, B, In, device=dev)
            packed = pack_padded_sequence(x, [T] * B)
            flops = sum(T * (2.0 * B * (In if l == 0 else H) * 6 * H + 2.0 * B * H * 5 * H) for l in range(L))

            def fwd():
                with torch.no_grad():
                    m.eval()
                    m(packed)

            def fwd_bwd():
                m.train()
                xr = x.detach().requires_grad_(True)
                out, _ = m(pack_padded_sequence(xr, [T] * B))
                out.data.sum().backward()
                m.weight.grad = None; m.bias.grad = None

            def t(fn):
                ts = []
                for i in range(7):
                    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
                    a.record(); fn(); b.record(); torch.cuda.synchronize()
                    if i >= 2:
                        ts.append(a.elapsed_time(b))
                return float(np.median(ts))
            f_ms, fb_ms = t(fwd), t(fwd_bwd)
            rows.append({"In": In, "T": T, "fwd_ms": f_ms, "fwd_tflops": flops / f_ms / 1e9,
                         "fwd_bwd_ms": fb_ms, "gflop_fwd": flops / 1e9})
        del m
    return {"config": "AlternatingHighwayLSTM H=512, L=2, B=256, all lengths = T (BASELINE configs[4])", "rows": rows}


def roi_align_microbench(dev, pk, kind):
    """BASELINE.json metric (ii): RoIAlign achieved GB/s vs the measured HBM peak, config 4
    (1024 boxes x 7x7 x 512 ch on a 37x37 map). Algorithmic bytes (SURVEY.md section 8d): output write +
    each feature element once + rois = 105.6 MB. L2 flushed between iterations (256 MB memset)."""
    import numpy as np
    import torch
    import motifs_cabi as C
    from lib.fpn.roi_align.functions.roi_align import normalize_rois
    rng = np.random.RandomState(0)
    N, Cn, B = 1024, 512, 1
    x1 = rng.uniform(0, 400, N); y1 = rng.uniform(0, 400, N)
    w = rng.uniform(32, 190, N); h = rng.uniform(32, 190, N)
    rois = np.concatenate([np.zeros((N, 1)), np.stack([x1, y1, np.minimum(x1 + w, 591), np.minimum(y1 + h, 591)], 1)], 1)
    rn = normalize_rois(torch.from_numpy(rois.astype(np.float32)).to(dev), 37, 37, 1 / 16)
    feat = torch.randn(B, Cn, 37, 37, device=dev)
    feat_nhwc = feat.permute(0, 2, 3, 1).contiguous()
    out = torch.empty(N, Cn, 7, 7, device=dev)
    flush = torch.empty(64 * 1024 * 1024, device=dev)
    lib = C.load()
    alg = N * Cn * 49 * 4 + B * Cn * 37 * 37 * 4 + N * 20

    def run(fn):
        ts = []
        for i in range(13):
            flush.zero_()
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            if i >= 3:
                ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts))
    st = C.cur_stream()
    t_nchw = run(lambda: lib.ROIAlignForwardLaucher(C.ptr(feat), C.ptr(rn), N, B, 37, 37, 7, 7, Cn, 0.0, C.ptr(out), st))
    t_nhwc = run(lambda: lib.mb200_roi_align_forward_nhwc(C.ptr(feat_nhwc), C.ptr(rn), N, B, 37, 37, 7, 7, Cn, 0.0, C.ptr(out), st))
    peak = float(pk["hbm_gbs"])
    return {"config": "N=1024 boxes, 7x7, C=512, B=1 (BASELINE configs[3])", "algorithmic_bytes": alg, "bound": "hbm",
            "peak": peak, "peak_kind": "%s copy bandwidth" % kind, "unit": "GB/s",
            "drop_in_nchw": {"us": t_nchw, "achieved": alg / t_nchw / 1e3, "frac": alg / t_nchw / 1e3 / peak},
            "pipeline_nhwc": {"us": t_nhwc, "achieved": alg / t_nhwc / 1e3, "frac": alg / t_nhwc / 1e3 / peak}}


# ------------------------------------------------------------------------------------------ CPU arm (oracle port)
def oracle_step_time(B, reps=1, threads=None, warm=1):
    """Seconds for one oracle (CPU, torch fp32) SGCls training step on a B-image batch of the same
    per-image shape; returns (seconds_per_step, cores_used)."""
    import numpy as np
    import torch
    from tests.model_utils import make_masks, CLASSES, RELS as RELCLS, KW
    from oracle import model as OM
    from dataloaders.synthetic import make_numpy_batch
    cores = threads or min(len(os.sched_getaffinity(0)), 32)   # >32 torch threads only oversubscribe here
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    orc = OM.RelModel(CLASSES, RELCLS, mode='sgcls', **KW)
    with torch.no_grad():
        for mod in orc.modules():
            if isinstance(mod, torch.nn.Conv2d):
                torch.nn.init.kaiming_normal_(mod.weight, nonlinearity='relu')
        orc.freq_bias.obj_baseline.weight.normal_(0, 1)
    for p in orc.detector.parameters():
        p.requires_grad = False
    orc.train()
    opt = torch.optim.SGD([p for p in orc.parameters() if p.requires_grad], lr=1e-3, momentum=0.9, weight_decay=1e-4)
    F = torch.nn.functional
    times = []
    for r in range(reps + warm):
        nb = make_numpy_batch(B, seed=r, boxes_per_img=BOXES, rels_per_img=RELS)
        n_obj, n_rel = B * BOXES, min(B * BOXES * (BOXES - 1), 256 * B)
        det, top, ctx = make_masks(n_obj, n_rel, B, seed=r)
        orc.detector.masks, orc.masks, orc.context.masks = det, top, ctx
        orc.detector.rng = np.random.RandomState(r)
        t0 = time.perf_counter()
        res = orc(torch.from_numpy(nb["imgs"]), nb["im_sizes"], 0, torch.from_numpy(nb["gt_boxes"]),
                  torch.from_numpy(nb["gt_classes"]), torch.from_numpy(nb["gt_rels"]))
        loss = F.cross_entropy(res.rm_obj_dists, res.rm_obj_labels) + F.cross_entropy(res.rel_dists, res.rel_labels[:, -1])
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_([p for p in orc.parameters() if p.requires_grad], 5.0)
        opt.step()
        if r >= warm:                   # first pass(es) warm the allocator / oneDNN primitives
            times.append(time.perf_counter() - t0)
    return sum(times) / len(times), cores


def cpu_baseline(sample_images=2):
    sec, cores = oracle_step_time(sample_images, reps=3)
    return {"value": sample_images / sec, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "mean of 3 timed SGCls train steps (after 1 untimed) of the oracle port on a %d-image batch of the same "
                      "per-image shape (20 boxes, 256 rel triples / image); the reference has no CPU path and "
                      "PyTorch 0.3 is not installable here (SURVEY.md section 8c)" % sample_images,
            "seconds_per_step": sec}


def run_reference(args):
    """CPU arm: the oracle port (the reference has no CPU path and PyTorch 0.3 is not installable, SURVEY.md section 8c)
    stepping the SAME workload as the b200 arm — one SGCls train step on a 6-image batch per step, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = BATCH_PER_GPU
    W = max(args.warmup, 1)
    sec, cores = oracle_step_time(B, reps=args.steps, warm=W)
    value = B / sec
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": W, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": "MotifNet SGCls train_rels.py step, VGG16 backbone, batch 6x592x592 per GPU, "
                                  "20 GT boxes + 15 GT rels per image (1536 rel triples), fwd+bwd+clip+SGD",
                      "global_batch": B, "parallelism": "cpu"},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": "oracle port (oracle/model.py, torch fp32 CPU, all host threads), the full 6-image batch "
                                      "per step; mean over %d steps after %d warm-up" % (args.steps, W)},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    import faulthandler
    wd = int(os.environ.get("MOTIFS_WATCHDOG_S", "0"))
    if wd > 0:      # dump every thread's Python stack and exit if the run wedges (debugging aid)
        faulthandler.dump_traceback_later(wd, exit=True)
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)

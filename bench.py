"""bench.py - learner frames/sec of the B200-native IMPALA learner hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one full learn() step (AtariNet forward, fused V-trace + losses + their gradients,
network backward, [NCCL all-reduce of the flat gradient], global-norm clip + RMSprop, actor-weight
publication) on one synthetic [T+1, B, 4, 84, 84] uint8 rollout batch per GPU (BASELINE.json
configs[1]: T=80, B=32 per GPU; weak scaling: the global batch is 32*N columns).

Printed JSON (one line, rank 0):
  value   frames/s with the rollout batches already resident in HBM (T*B*N / step time, the
          reference's own accounting, polybeast_learner.py:372), CUDA events, max over ranks.
  e2e     same metric through the public API (torchbeast_b200.monobeast.learn) with HOST pinned
          buffers: every step's inputs are copied host->device and the step's stats are read back
          inside the timed region.
  roofline / roofline_ops / vtrace / cpu_baseline / clocks / gpu_launches: see DESIGN.md section 5.
`--impl reference` times the CPU restatement of the reference's learner step (oracle/, kind
"port") on the host cores: the reference itself is PyTorch-on-CPU code that cannot travel to the box.
`--dump-outputs DIR` saves what the last timed device-resident step returned, plus the updated parameters, as
DIR/<name>.npy; the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--T", type=int, default=80)
    ap.add_argument("--B", type=int, default=32, help="batch columns per GPU")
    ap.add_argument("--use_lstm", type=int, default=1)
    ap.add_argument("--net", default="atari", choices=["atari", "resnet"],
                    help="atari: monobeast AtariNet (BASELINE configs[1]); resnet: polybeast IMPALA ResNet (configs[3])")
    ap.add_argument("--precision", default=None, choices=["fp32", "bf16", "bf16x3"],
                    help="GEMM backend (default: the package default, bf16x3 = split-bf16 tensor-core products, parity-green)")
    ap.add_argument("--num_actions", type=int, default=6)
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_profile", action="store_true")
    ap.add_argument("--graph", type=int, default=1, help="replay the step as one CUDA graph (falls back to eager)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --B columns per GPU (default, the driver's scaling run); strong: --B columns in total, B/N per GPU")
    ap.add_argument("--no_dp_check", action="store_true", help="skip the multi-GPU gradient / replica check before the timed runs")
    ap.add_argument("--actors", type=int, default=0,
                    help="BASELINE configs[2]: N synthetic host actor threads -> pinned slots -> learner queue -> "
                         "polybeast_learner.learn on --learner_threads threads; prints the end-to-end SPS line")
    ap.add_argument("--learner_threads", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, save what the last device-resident step computed as DIR/<name>.npy "
                         "(float32, at most 64 MB in all); the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.actors > 0 or args.impl == "reference"):
        ap.error("--dump-outputs saves the device-resident learn step; it does not apply to --actors or --impl reference")
    return args


# what the arithmetic is, per backend (the line's `dtype`)
DTYPE_NAMES = {
    "bf16x3": "bf16x3 (split-bf16 hi+lo operands, 3 tcgen05 MMAs per product, fp32 accumulate; fp32 state/loss/optimizer)",
    "bf16": "bf16 (single-plane bf16 operands, fp32 accumulate)",
    "fp32": "f32",
}


def flags_ns(T, B):
    return types.SimpleNamespace(
        reward_clipping="abs_one", discounting=0.99, baseline_cost=0.5, entropy_cost=0.0006,
        grad_norm_clipping=40.0, unroll_length=T, batch_size=B)


def synthetic_host_batch(T, B, A, seed, pin):
    """SURVEY.md 8(d) M2 synthetic rollout (numpy RandomState), host tensors (pinned if asked)."""
    rs = np.random.RandomState(seed)
    b = dict(
        frame=torch.from_numpy(rs.randint(0, 256, size=(T + 1, B, 4, 84, 84), dtype=np.uint8)),
        reward=torch.from_numpy(rs.randn(T + 1, B).astype(np.float32)),
        done=torch.from_numpy(rs.rand(T + 1, B) < 0.01),
        episode_return=torch.from_numpy(rs.randn(T + 1, B).astype(np.float32)),
        policy_logits=torch.from_numpy(rs.randn(T + 1, B, A).astype(np.float32)),
        action=torch.from_numpy(rs.randint(0, A, size=(T + 1, B)).astype(np.int64)),
        last_action=torch.from_numpy(rs.randint(0, A, size=(T + 1, B)).astype(np.int64)),
    )
    if pin:
        b = {k: v.pin_memory() for k, v in b.items()}
    return b


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 50 ms.  Started before the warm-up (nvidia-smi needs ~0.2 s to
    produce its first line and a step is ~2 ms) and filtered to the timed region by nvidia-smi's own timestamps; if
    that filter leaves nothing (clock skew, parse trouble) every collected sample is used."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        try:
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    @staticmethod
    def _stamp(text):
        import datetime
        try:
            return datetime.datetime.strptime(text, "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except Exception:
            return None

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return None
        try:
            time.sleep(0.12)
            self.proc.terminate()
            self.thread.join(timeout=2)
            rows = [r for r in list(self.rows) if len(r) >= 2 and r[1].replace(".", "").isdigit()]
            if not rows:
                return None
            window = []
            if t0 is not None and t1 is not None:
                for r in rows:
                    ts = self._stamp(r[0])
                    if ts is not None and t0 - 0.06 <= ts <= t1 + 0.06:
                        window.append(r)
            used = window if window else rows
            sm = [float(r[1]) for r in used]
            reasons = []
            for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                if any(len(r) > 4 + i and r[4 + i].lower().startswith("active") for r in used):
                    reasons.append(name)
            mx = [float(r[2]) for r in used if len(r) > 2 and r[2].replace(".", "").isdigit()]
            return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(sm),
                        in_timed_region=bool(window))
        except Exception:
            return None


def host_cpu_info():
    """os.cpu_count() and the CPU model string, reported next to every CPU number (SURVEY 8(d) M5)."""
    info = {"host_cpu_count": os.cpu_count()}
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    info["host_cpu_model"] = ln.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    return info


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, so the pinned rollout
    staging buffers are allocated next to the GPU's PCIe root (first touch) - H2D bandwidth on a
    2-socket host depends on it.  Returns the node id or None."""
    try:
        bus = torch.cuda.get_device_properties(index).pci_bus_id
        dom = torch.cuda.get_device_properties(index).pci_domain_id
        dev = torch.cuda.get_device_properties(index).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0" % (dom, bus, dev)
        node = int(open(path + "/numa_node").read())
        cpus = open(path + "/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            if "-" in part:
                a, b = part.split("-")
                ids.update(range(int(a), int(b) + 1))
            elif part:
                ids.add(int(part))
        if ids:
            os.sched_setaffinity(0, ids)
        return node
    except Exception:
        return None


def measure_h2d_gbs(dev):
    """Pinned-host -> device copy bandwidth of this process (256 MB, best of 3)."""
    src = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    dst = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    best = 0.0
    for _ in range(3):
        a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); dst.copy_(src, non_blocking=True); z.record(); torch.cuda.synchronize()
        best = max(best, src.numel() / (a.elapsed_time(z) * 1e-3) / 1e9)
    return best


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return dict(hbm=p["hbm_gbs"], tensor=p["bf16_tflops_sustained"], tensor_burst=p["bf16_tflops"], source="measured")
    except Exception:
        return dict(hbm=6650.0, tensor=1400.0, tensor_burst=1590.0, source="fallback")


def gemm_flops_table(N, A, use_lstm):
    """2*M*N*K of every tagged GEMM op per step (N = (T+1)*B frames) - DESIGN.md section 4."""
    M1, M2, M3 = N * 400, N * 81, N * 49
    core = 512 + 1 + A
    t = {
        "conv1_fwd": 2 * M1 * 32 * 256, "conv2_fwd": 2 * M2 * 64 * 512, "conv3_fwd": 2 * M3 * 64 * 576,
        "fc_fwd": 2 * N * 512 * 3136, "heads_fwd": 2 * N * (A + 1) * core,
        "conv1_wgrad": 2 * M1 * 32 * 256, "conv2_wgrad": 2 * M2 * 64 * 512, "conv3_wgrad": 2 * M3 * 64 * 576,
        "fc_wgrad": 2 * N * 512 * 3136, "heads_wgrad": 2 * N * (A + 1) * core,
        "conv2_dgrad": 2 * M2 * 64 * 512, "conv3_dgrad": 2 * M3 * 64 * 576, "fc_dgrad": 2 * N * 512 * 3136,
        "heads_dgrad": 2 * N * (A + 1) * core,
    }
    if use_lstm == "resnet":
        return resnet_flops_table(N, A)
    if use_lstm:
        H = core
        t.update({
            "lstm_xproj_fwd": 2 * 2 * N * 4 * H * H, "lstm_recurrence_fwd": 2 * 2 * N * 4 * H * H,
            "lstm_recurrence_bwd": 2 * 2 * N * 4 * H * H, "lstm_wgrad": 2 * 2 * 2 * N * 4 * H * H,
            "lstm_xproj_dgrad": 2 * 2 * N * 4 * H * H,
        })
    return t


def gemm_bytes_table(N, A, use_lstm, precision):
    """ALGORITHMIC operand + result bytes of the tagged AtariNet GEMM ops - with K of 64..576 most of these products
    are HBM streams, not tensor-pipe work.  Activations count 2 B (bf16), 4 B (bf16x3: hi + lo plane, or fp32); conv1's
    input counts as the 1-byte uint8 frames (the bf16 image the kernels stage is an implementation cost, not algorithmic)."""
    bf16 = precision != "fp32"
    e = {"bf16": 2, "bf16x3": 4}.get(precision, 4)
    M1, M2, M3 = N * 400, N * 81, N * 49
    e1 = 2 if bf16 else 1  # conv1 patch matrix: bf16 (tensor-core backend) or uint8 (fp32 backend)
    t = {
        "conv1_fwd": M1 * 256 * e1 + M1 * 32 * e, "conv2_fwd": M2 * 512 * e + M2 * 64 * e, "conv3_fwd": M3 * 576 * e + M3 * 64 * e,
        "fc_fwd": N * 3136 * e + 512 * 3136 * e + N * 512 * 4,
        "conv1_wgrad": M1 * 256 * e1 + M1 * 32 * e, "conv2_wgrad": M2 * 512 * e + M2 * 64 * e, "conv3_wgrad": M3 * 576 * e + M3 * 64 * e,
        "fc_wgrad": N * 3136 * e + N * 512 * e + 512 * 3136 * 4,
        "conv2_dgrad": M2 * 64 * e + M2 * 512 * e, "conv3_dgrad": M3 * 64 * e + M3 * 576 * e,
        "fc_dgrad": N * 512 * e + 512 * 3136 * e + 2 * N * 3136 * e,
    }
    if bf16:  # implicit-GEMM convolutions: the activation (or the frames) is the operand - read once, no patch matrix
        img = N * 28224  # uint8 frames
        t.update({"conv1_fwd": img + M1 * 32 * e, "conv1_wgrad": img + M1 * 32 * e,
                  "conv2_fwd": M1 * 32 * e + M2 * 64 * e, "conv2_wgrad": M1 * 32 * e + M2 * 64 * e,
                  "conv3_fwd": M2 * 64 * e + M3 * 64 * e, "conv3_wgrad": M2 * 64 * e + M3 * 64 * e,
                  "conv2_dgrad": M2 * 64 * e + M1 * 32 * 2 + M1 * 32 * e, "conv3_dgrad": M3 * 64 * e + M2 * 64 * 2 + M2 * 64 * e})  # dY + mask + dX
    if use_lstm:
        H = 512 + 1 + A
        t.update({"lstm_xproj_fwd": 2 * (N * H * e + 4 * H * H * e + N * 4 * H * 4),
                  "lstm_wgrad": 4 * (N * 4 * H * e + N * H * e + 4 * H * H * 4),
                  "lstm_xproj_dgrad": 2 * (N * 4 * H * e + 4 * H * H * e + N * H * 4)})
    return t


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(out, model):
    """Host copies of what one learn step hands its caller: the fused loss kernel's outputs (losses, V-trace targets,
    policy-gradient advantages, log-rhos, action log-probs, loss gradients) and the updated flat parameters (the actor's
    copy is identical)."""
    arrays = dict(out["vtrace"]._asdict(), params=model.flat_params)
    return {k: v.detach().cpu().numpy() for k, v in arrays.items() if v is not None}


def write_outputs(arrays, out_dir, limit=DUMP_LIMIT_BYTES):
    """Save each array as out_dir/<name>.npy in float32 (float64 stays float64).  When together they exceed `limit`
    bytes, each array above an even share of it is stored as a sample of its flattened elements at sorted positions
    drawn from RandomState(0): the same arguments give the same positions, so two builds can be compared."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: a if a.dtype == np.float64 else a.astype(np.float32) for k, a in arrays.items()}
    share = limit // max(len(arrays), 1) - 4096  # room for each file's .npy header
    sample = sum(a.nbytes + 4096 for a in arrays.values()) > limit
    for name, a in arrays.items():
        if sample and a.nbytes > share:
            a = a.reshape(-1)[np.sort(np.random.RandomState(0).choice(a.size, share // a.itemsize, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def resnet_flops_table(N, A):
    """2*M*N*K per tagged op of the IMPALA ResNet trunk (aggregated over the 15 convs)."""
    secs = [(84, 42, 4, 16), (42, 21, 16, 32), (21, 11, 32, 32)]
    feat = sum(2 * N * S * S * ch * cin * 9 for S, So, cin, ch in secs)
    feat_d = sum(2 * N * S * S * ch * cin * 9 for S, So, cin, ch in secs[1:])
    res = sum(4 * 2 * N * So * So * ch * ch * 9 for S, So, cin, ch in secs)
    fc = 2 * N * 256 * 3872
    return {"feat_conv_fwd": feat, "feat_conv_wgrad": 2 * N * 84 * 84 * 16 * 36, "res_conv_fwd": res,
            "res_conv_wgrad": res + feat_d, "res_conv_dgrad": res + feat_d, "fc_fwd": fc, "fc_wgrad": fc, "fc_dgrad": fc}


def resnet_bytes_table(N):
    """ALGORITHMIC bytes of the tagged ResNet trunk ops on the bf16x3 backend (aggregated over the convs): every tensor moves
    once - conv inputs as zero-padded split-bf16 images (4 B per element, (S+2)^2 pixels; written by the previous conv's
    epilogue where there is one), outputs / gradients / ReLU masks / residuals in fp32.  With 16..32 channels these products
    are HBM streams, not tensor-pipe work."""
    secs = [(84, 42, 4, 16), (42, 21, 16, 32), (21, 11, 32, 32)]
    t = dict(feat_conv_fwd=0, feat_conv_wgrad=0, res_conv_fwd=0, res_conv_wgrad=0, res_conv_dgrad=0, pad_split=0,
             bias_grad_colsum=0, frames_to_image=0, maxpool_fwd=0, maxpool_bwd=0)
    for i, (S, So, cin, ch) in enumerate(secs):
        cin16 = max(cin, 16)
        M, Mp, Mo, Mop = N * S * S, N * (S + 2) ** 2, N * So * So, N * (So + 2) ** 2
        t["feat_conv_fwd"] += Mp * cin16 * 4 + M * ch * 4
        wg = Mp * ch * 4 + Mp * cin16 * 4                       # dY image + input image
        t["feat_conv_wgrad" if i == 0 else "res_conv_wgrad"] += wg
        if i > 0:
            t["res_conv_dgrad"] += Mp * ch * 4 + M * cin * 4 + Mp * cin * 4   # dY image -> dX fp32 + the previous section's dY image
        else:
            t["frames_to_image"] += N * 4 * S * S + Mp * 16 * 4
        t["maxpool_fwd"] += M * ch * 4 + Mo * ch * 5            # + argmax byte
        t["maxpool_bwd"] += Mo * ch * 5 + Mp * ch * 4           # pooled gradient + argmax -> the feat conv's dY image
        t["pad_split"] += Mo * ch * 4 + Mop * ch * 4            # relu(X0) of the first block conv
        # four block convs: image + output (+ residual on two of them) + the next conv's image from the epilogue;
        # backward: dY image + dX + ReLU mask (+ skip on two) + the next dY image on three
        t["res_conv_fwd"] += 4 * (Mop * ch * 4 + Mo * ch * 4) + 2 * Mo * ch * 4 + (4 if i < 2 else 3) * Mop * ch * 4
        t["res_conv_wgrad"] += 4 * (2 * Mop * ch * 4)
        t["res_conv_dgrad"] += 4 * (Mop * ch * 4 + 2 * Mo * ch * 4) + 2 * Mo * ch * 4 + 3 * Mop * ch * 4
    del t["bias_grad_colsum"]   # now the column-sum reduces of the epilogue partials + one small image pass: no meaningful byte count
    return t


def hbm_bytes_table(N, T, B, A, use_lstm, nparams):
    """Algorithmic bytes of the bandwidth-bound ops per step."""
    M1, M2, M3 = N * 400, N * 81, N * 49
    return {
        "im2col_u8": N * 28224 + M1 * 256,                       # read frames once, write the patch matrix
        "im2col_f32": 4 * (M1 * 32 + M2 * 512) + 4 * (M2 * 64 + M3 * 576),
        "col2im": 4 * (M3 * 576 + 2 * M2 * 64) + 4 * (M2 * 512 + 2 * M1 * 32),
        "impala_loss_fwd_bwd": (12 * A + 32 + 12 - 3) * T * B + 4 * B + 16,
        "clip_rmsprop": 4 * nparams * 5, "grad_sumsq": 4 * nparams,
    }


def run_reference(args, world=1):
    """CPU arm: the oracle port of the reference's learn step on the host cores (the reference itself is PyTorch-on-CPU
    code that cannot travel to the box; the port is pinned to the reference's outputs by tests/test_oracle_golden.py).
    Honours --steps / --warmup.  Each step trains on the job's GLOBAL batch (B per GPU x N columns) unless that would
    exceed the time budget (TB_CPU_BASELINE_BUDGET_S, default 240 s for the whole run): then every step is a bounded
    sample of `cols` batch columns of the same rollout shape - frames/s is per column, so the sample does not bias it."""
    from oracle import learner_torch as LT
    T, B, A = args.T, args.B, args.num_actions
    Bg = B * world if args.scaling == "weak" else B
    budget_s = float(os.environ.get("TB_CPU_BASELINE_BUDGET_S", "240"))
    net = getattr(args, "net", "atari")
    shapes = (LT.resnet_param_shapes if net == "resnet" else LT.atarinet_param_shapes)(A, bool(args.use_lstm))
    p = LT.random_params(shapes, seed=0)
    # Thread count: the op-by-op CPU path is dispatch-bound and gets SLOWER with many threads
    # (measured on the 128-thread B200 host: 250 s/step at 128 threads; SURVEY.md section 6), so pick
    # the fastest of a few counts on a small calibration rollout and report it as `cores`.
    ncpu = os.cpu_count() or 1
    cal = synthetic_host_batch(8, 8, A, seed=2, pin=False)
    st_shape = (lambda b: (1, b, 256)) if net == "resnet" else (lambda b: (2, b, 512 + A + 1))
    cal_state = tuple(torch.zeros(*st_shape(8)) for _ in range(2)) if args.use_lstm else ()
    best = None
    for nt in sorted({min(ncpu, n) for n in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(nt)
        LT.learner_step(p, cal, cal_state, net=net, num_actions=A)
        t0 = time.perf_counter()
        LT.learner_step(p, cal, cal_state, net=net, num_actions=A)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
        if dt > 4 * best[0]:
            break
    torch.set_num_threads(best[1])
    steps, warm = max(1, args.steps), max(0, args.warmup)
    # size the per-step sample: time one step on min(Bg, 8) columns, extrapolate linearly in columns
    probe_cols = min(Bg, 8)
    pb = synthetic_host_batch(T, probe_cols, A, seed=1, pin=False)
    ps = tuple(torch.zeros(*st_shape(probe_cols)) for _ in range(2)) if args.use_lstm else ()
    t0 = time.perf_counter()
    LT.learner_step(p, pb, ps, net=net, num_actions=A)
    per_col = (time.perf_counter() - t0) / probe_cols
    cols = int(max(1, min(Bg, budget_s / max(per_col * (steps + warm), 1e-9))))
    batch = synthetic_host_batch(T, cols, A, seed=1, pin=False)
    state = tuple(torch.zeros(*st_shape(cols)) for _ in range(2)) if args.use_lstm else ()
    sq = None
    for _ in range(warm):
        o = LT.learner_step(p, batch, state, net=net, square_avg=sq, num_actions=A)
        p, sq = o["params"], o["square_avg"]
    t0 = time.perf_counter()
    for _ in range(steps):
        o = LT.learner_step(p, batch, state, net=net, square_avg=sq, num_actions=A)
        p, sq = o["params"], o["square_avg"]
    dt = (time.perf_counter() - t0) / steps
    return dict(value=T * cols / dt, ms_per_step=dt * 1e3 * (Bg / cols), steps=steps, warmup=warm, cores=torch.get_num_threads(),
                cols=cols, global_cols=Bg,
                sample="%d timed + %d warm-up learn steps of oracle/learner_torch.py (port of monobeast.learn) on %d of the %d "
                       "batch columns of the global T=%d rollout per step" % (steps, warm, cols, Bg, T))


def make_config(args, world):
    T, B, A = args.T, args.B, args.num_actions
    per_gpu = B if args.scaling == "weak" else B // max(world, 1)
    if args.net == "resnet":
        workload = "IMPALA ResNet(84x84x4 u8)%s + V-trace learner step, T=%d B=%d per GPU, synthetic frames" % (
            "+LSTM(257->256)" if args.use_lstm else "", T, per_gpu)
    else:
        workload = "AtariNet(84x84x4 u8)%s + V-trace learner step, T=%d B=%d per GPU, synthetic frames" % (
            "+LSTM(2x519)" if args.use_lstm else "", T, per_gpu)
    return dict(workload=workload, T=T, B_per_gpu=per_gpu, global_batch=per_gpu * max(world, 1), num_actions=A,
                use_lstm=bool(args.use_lstm), scaling=args.scaling,
                parallelism="dp%d over batch columns, one SUM all-reduce of the flat gradient (two buckets, the LSTM + heads "
                            "bucket overlapped with the trunk backward)" % world)


def dp_check(args, world, rank, dev, A):
    """Multi-GPU correctness on the hardware (VERDICT r1 item 2): one step on a full global batch by rank 0 alone vs the
    same batch column-sharded over all ranks + the SUM all-reduce -> flat gradient difference; then every rank steps and
    the replicas' parameters must be BIT-identical."""
    import torch.distributed as dist
    from torchbeast_b200 import learner, monobeast, optim
    T = args.T
    Bg = max(world, (args.B // world) * world)
    flags = flags_ns(T, Bg)
    full = {k: v.to(dev) for k, v in synthetic_host_batch(T, Bg, A, seed=4242, pin=False).items()}

    def fresh():
        m = monobeast.AtariNet((4, 84, 84), A, bool(args.use_lstm), precision=args.precision)
        m.reset_parameters_like_torch(seed=7)
        return m

    def grads(m, batch, state, reduce):
        out = m.learner_forward(batch, state)
        loss = learner.impala_loss_fwd_bwd(batch["policy_logits"][1:], out.policy_logits[:-1], batch["action"][1:], batch["reward"][1:],
                                           batch["done"][1:], out.baseline[:-1], out.baseline[-1])
        if reduce:
            fg = learner._backward_with_overlapped_all_reduce(m, loss.grad_logits, loss.grad_values)
        else:
            fg = m.learner_backward(loss.grad_logits, loss.grad_values)
        return fg, loss.losses

    m = fresh()
    st_full = m.initial_state(Bg)
    shard, st = learner.shard_rollout(full, st_full, rank, world)
    g_dp, l_dp = grads(m, shard, st, True)
    g_dp = g_dp.clone()
    l_sum = l_dp.clone()
    dist.all_reduce(l_sum)
    res = {}
    if rank == 0:
        m1 = fresh()
        g_full, l_full = grads(m1, full, m1.initial_state(Bg), False)
        d = (g_dp.double() - g_full.double())
        res["grad_rel_l2"] = float(d.norm() / g_full.double().norm())
        res["grad_max_over_max"] = float(d.abs().max() / g_full.abs().max())
        res["loss_rel"] = float((l_sum[3] - l_full[3]).abs() / l_full[3].abs())
    opt = optim.RMSprop(m, lr=0.00048, momentum=0, eps=0.01, alpha=0.99)
    opt.step(max_grad_norm=flags.grad_norm_clipping)
    torch.cuda.synchronize()
    bits = m.flat_params.view(torch.int32).to(torch.int64)
    sig = torch.stack([bits.sum(), (bits * torch.arange(1, bits.numel() + 1, device=dev) % 1000003).sum()])
    sigs = [torch.zeros_like(sig) for _ in range(world)]
    dist.all_gather(sigs, sig)
    res["replicas_bit_identical"] = bool(all(torch.equal(sigs[0], x) for x in sigs))
    res["global_batch"] = Bg
    res["cols_per_rank"] = Bg // world
    return res


def run_actor_pipeline(args):
    """BASELINE.json configs[2]: `--actors 48` synthetic actor threads feed pinned [T+1, B, ...] slots; full slots travel the
    learner queue as the reference's nest into polybeast_learner.learn() on `--learner_threads` threads (2 = the reference
    default, polybeast_learner.py:62) sharing one model, optimizer and lock.  Value = frames consumed per second end to end
    (T*B per learn step / wall time, stats["step"] as the reference counts it, pl:372), steady state after a warm-up."""
    from torchbeast_b200 import actors, monobeast, optim, polybeast_learner, staging
    T, B, A = args.T, args.B, args.num_actions
    torch.cuda.set_device(0)
    numa = bind_to_gpu_numa_node(0)
    dev = torch.device("cuda", 0)
    model = monobeast.AtariNet((4, 84, 84), A, bool(args.use_lstm), precision=args.precision)
    actor_model = monobeast.AtariNet((4, 84, 84), A, bool(args.use_lstm), precision=args.precision)
    actor_model.copy_params_from(model)
    opt = optim.RMSprop(model, lr=0.00048, momentum=0, eps=0.01, alpha=0.99)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda e: 1.0)
    flags = flags_ns(T, B)
    flags.cuda_graph = bool(args.graph)
    stager = staging.RolloutStager(staging.spec_for(T, B, A, use_last_action=False), dev, depth=4)
    model._tb_stager = stager
    q = actors.LearnerQueue()
    pool = actors.SyntheticActors(stager, args.actors, T, B, A, q, state_shape=(2, 512 + A + 1) if args.use_lstm else None)
    stats, lock = {}, threading.Lock()
    steps_done = [0]
    t_mark = {}
    total = args.warmup + args.steps

    class Log:
        def log(self, st):
            steps_done[0] += 1
            if steps_done[0] == args.warmup:
                torch.cuda.synchronize(); t_mark["t0"] = time.perf_counter()
            if steps_done[0] == total:
                torch.cuda.synchronize(); t_mark["t1"] = time.perf_counter()
                pool.stop()

    pool.start()
    threads = [threading.Thread(target=polybeast_learner.learn, args=(flags, q, model, actor_model, opt, sched, stats, Log(), lock))
               for _ in range(args.learner_threads)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=600)
    dt = t_mark["t1"] - t_mark["t0"]
    sps = args.steps * T * B / dt
    line = dict(metric="end_to_end_sps", value=sps, unit="frames/s", n_gpus=1, steps=args.steps, warmup=args.warmup,
                ms_per_step=dt / args.steps * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype=DTYPE_NAMES.get(model.precision, model.precision), data="synthetic",
                config=dict(workload="polybeast_learner, %d synthetic host actor threads -> pinned slots -> learner queue -> "
                                     "%d learner threads, AtariNet%s, T=%d B=%d, 1 GPU" % (
                                         args.actors, args.learner_threads, "+LSTM" if args.use_lstm else "", T, B),
                            T=T, B_per_gpu=B, num_actions=A, use_lstm=bool(args.use_lstm), actors=args.actors,
                            learner_threads=args.learner_threads),
                e2e=dict(value=sps, unit="frames/s", h2d_bytes_per_step=stager.h2d_bytes, d2h_bytes_per_step=16,
                         numa_node=numa, rollouts_produced=pool.rollouts, **host_cpu_info()),
                final_total_loss=stats.get("total_loss"), learner_steps=steps_done[0])
    print(json.dumps(line))
    sys.stdout.flush()
    os._exit(0)


def main():
    args = parse()
    if args.actors > 0 and args.impl != "reference":
        return run_actor_pipeline(args)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    T, A = args.T, args.num_actions
    config = make_config(args, world)
    B = config["B_per_gpu"]
    if args.scaling == "strong" and args.B % max(world, 1):
        raise SystemExit("--scaling strong needs --B divisible by the number of GPUs")

    if args.impl == "reference":
        if rank != 0:
            return
        r = run_reference(args, world)
        line = dict(
            impl="reference", metric="learner_frames_per_sec", value=r["value"], unit="frames/s", n_gpus=args.gpus,
            steps=r["steps"], warmup=r["warmup"], ms_per_step=r["ms_per_step"], higher_is_better=True, scaling=args.scaling,
            vs_baseline=None, dtype="f32", data="synthetic", config=config,
            cpu_baseline=dict(value=r["value"], unit="frames/s", cores=r["cores"], kind="port", sample=r["sample"],
                              note="port of the reference's learn step, pinned to reference-generated fixtures "
                                   "(tests/test_oracle_golden.py); functional torch ops at the best of several thread counts - a "
                                   "generous baseline", **host_cpu_info()),
            e2e=dict(value=r["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank)  # before any pinned allocation (first-touch placement)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from torchbeast_b200 import _lib, learner, monobeast, optim, staging

    dev = torch.device("cuda", local_rank)
    if args.net == "resnet":
        from torchbeast_b200 import polybeast_learner
        model = polybeast_learner.Net(A, bool(args.use_lstm), precision=args.precision)
        actor = polybeast_learner.Net(A, bool(args.use_lstm), precision=args.precision)
    else:
        model = monobeast.AtariNet((4, 84, 84), A, bool(args.use_lstm), precision=args.precision)
        actor = monobeast.AtariNet((4, 84, 84), A, bool(args.use_lstm), precision=args.precision)
    lib = _lib.lib()
    dp = None
    if world > 1 and args.net == "atari" and not args.no_dp_check:
        dp = dp_check(args, world, rank, dev, A)
    model.reset_parameters_like_torch(seed=0)  # identical replicas on every rank
    actor.copy_params_from(model)
    opt = optim.RMSprop(model, lr=0.00048, momentum=0, eps=0.01, alpha=0.99)
    total_steps = 30_000_000
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda e: 1 - min(e * T * B * world, total_steps) / total_steps)
    flags = flags_ns(T, B)
    flags.cuda_graph = bool(args.graph)
    state = model.initial_state(B)
    NROT = 4  # distinct input batches: 4 x 73 MB > 126 MB L2
    # N1: the rollouts live in the pinned slots of the package's RolloutStager (what the actors would write in place)
    example = synthetic_host_batch(T, B, A, seed=1000 * rank, pin=False)
    stager = staging.RolloutStager(staging.spec_like(example), dev, depth=NROT)
    model._tb_stager = stager
    for i in range(NROT):
        hb = example if i == 0 else synthetic_host_batch(T, B, A, seed=1000 * rank + i, pin=False)
        for k, v in hb.items():
            stager.host[i][k].copy_(v)
    host = stager.host
    devb = [{k: v.to(dev) for k, v in hb.items()} for hb in host]
    h2d_bytes = stager.h2d_bytes
    h2d_gbs = measure_h2d_gbs(dev)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---- device-resident throughput ----------------------------------------------------
    graphed = None
    if args.graph:
        try:
            graphed = learner.GraphedLearner(flags, model, actor, opt, devb[0], state)
            model.__dict__.setdefault("_tb_graphs", {})[
                (tuple((k, tuple(v.shape)) for k, v in devb[0].items() if k in learner.GraphedLearner.KEYS), id(opt), id(actor))] = graphed
        except Exception as exc:  # capture not possible on this setup: report and run eagerly
            sys.stderr.write("CUDA graph capture failed (%s); running eagerly\n" % (exc,))
            graphed = None
            opt.lr_from_device = False
            flags.cuda_graph = False

    def device_step(i):
        if graphed is not None:
            return graphed.step(devb[i % NROT], state, sched)
        return learner.learn_step(flags, model, actor, devb[i % NROT], state, opt, sched, stats_sync=False)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    for i in range(args.warmup):
        device_step(i)
    barrier()
    t_region0 = time.time()
    launches0 = lib.tb_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = device_step(i)
    e1.record()
    barrier()
    launches = lib.tb_launch_count() - launches0
    ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    clocks = sampler.stop(t_region0, time.time()) if sampler else None
    final_loss = float(out["losses"][3])
    assert np.isfinite(final_loss), "non-finite loss"
    if args.dump_outputs and rank == 0:  # before any further step overwrites the outputs or the parameters
        write_outputs(step_outputs(out, model), args.dump_outputs)
    if graphed is not None:  # launches per step: count one eager step (a graph replay launches the same kernels)
        l0 = lib.tb_launch_count()
        learner.learn_step(flags, model, actor, devb[0], state, opt, None, stats_sync=False)
        torch.cuda.synchronize()
        launches = (lib.tb_launch_count() - l0) * args.steps

    # ---- end to end THROUGH THE PLUGIN CALL: monobeast.learn(host rollout) from two learner threads ----------
    # (the reference's own thread structure, polybeast_learner.py:62,505-521: the host->device copy of one thread overlaps
    #  the other thread's step; monobeast.learn stages the pinned rollout through the RolloutStager, takes the lock,
    #  replays the graphed step and reads the stats back - every step, inside the timed region)
    lock = threading.Lock()
    last_stats = [None]

    def e2e_loop(nsteps):
        nthreads = 2
        errs = []

        def body(k):
            try:
                torch.cuda.set_device(local_rank)
                for i in range(k, nsteps, nthreads):
                    last_stats[0] = monobeast.learn(flags, actor, model, host[i % NROT], state, opt, sched, lock) \
                        if args.net == "atari" else learner.learn(flags, model, actor, host[i % NROT], state, opt, sched, lock)
            except Exception as exc:  # surfaced below
                errs.append(exc)

        # (world > 1: every replay of the step graph issues the same collective sequence, so which learner thread replays
        #  next does not matter - the ranks only have to run the same NUMBER of steps)
        body_threads = [threading.Thread(target=body, args=(k,)) for k in range(nthreads)]
        for t in body_threads:
            t.start()
        for t in body_threads:
            t.join()
        if errs:
            raise errs[0]
        return last_stats[0]

    e2e_loop(max(args.warmup, 2))  # untimed warm-up: first-use kernel loads, graph upload, pinned-page first touch
    barrier()
    e2e_steps = args.steps
    t_e0, t_e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_e0.record()
    stats = e2e_loop(e2e_steps)
    t_e1.record()
    barrier()
    e2e_ms = max_over_ranks(t_e0.elapsed_time(t_e1)) / e2e_steps
    d2h_bytes = 4 * 4 + int(sum(1 for _ in stats["episode_returns"])) * 4

    def finish():
        """Leave without tearing NCCL down: destroy_process_group can hang while a captured CUDA graph still
        references the communicator, and the process is exiting anyway."""
        sys.stdout.flush(); sys.stderr.flush()
        if world > 1:
            import torch.distributed as dist
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            os._exit(0)

    PSTEPS = 3
    if rank != 0:
        if not args.no_profile:  # the profiled steps contain the gradient all-reduce: every rank takes part
            for i in range(PSTEPS):
                learner.learn_step(flags, model, actor, devb[i % NROT], state, opt, sched, stats_sync=False)
        finish()
        return

    pk = peaks()
    frames = T * B * world
    line = dict(
        metric="learner_frames_per_sec", value=frames / (ms * 1e-3), unit="frames/s", n_gpus=world, steps=args.steps,
        warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling=args.scaling, vs_baseline=None,
        dtype=DTYPE_NAMES.get(model.precision, model.precision),
        data="synthetic", config=config,
        l2_policy="4 rotating input batches per rank (%.0f MB) > 126 MB L2; ~2.3 GB of activations written per step" % (
            NROT * h2d_bytes / 1e6),
        e2e=dict(value=frames / (e2e_ms * 1e-3), unit="frames/s", ms_per_step=e2e_ms, h2d_bytes_per_step=h2d_bytes,
                 d2h_bytes_per_step=d2h_bytes, h2d_gbs_measured=h2d_gbs, numa_node=numa, cuda_graph=graphed is not None,
                 learner_threads=2,
                 note="every step: monobeast.learn(flags, actor, model, PINNED HOST rollout, ...) -> RolloutStager (one async "
                      "H2D copy of the slot on the copy stream, issued outside the lock so it overlaps the other learner "
                      "thread's step) -> lock -> %s -> stats read-back; all inside the timed region" % (
                          "one CUDA-graph replay of the step" if graphed is not None else "eager step")),
        gpu_launches=int(launches), clocks=clocks, final_total_loss=final_loss,
        parity="default backend %s: tests/test_learner_baseline_gpu.py holds it to reference-generated T=80,B=32 fixtures "
               "(outputs, vs, pg_advantages, losses <= 1e-5)" % model.precision if args.net == "atari" else
               ("backend %s: tests/test_resnet_gpu.py holds it to the reference-generated T=80,B=8 fixture (one GPU's shard of "
                "configs[3]): outputs, vs, pg_advantages, losses <= 1e-5; gradients relative L2 < 6e-3 per tensor "
                "(profiles/parity_r2_resnet.txt)" % model.precision),
    )
    if dp is not None:
        line["dp_check"] = dp

    # ---- per-op device timing (separate steps; CUDA events around every op on its stream) ---
    if not args.no_profile:
        lib.tb_profile_enable(1)
        for i in range(PSTEPS):
            learner.learn_step(flags, model, actor, devb[i % NROT], state, opt, sched, stats_sync=False)
        recs = _lib.profile_collect()
        lib.tb_profile_enable(0)
        agg = {}
        for name, t in recs:
            a = agg.setdefault(name, [0.0, 0])
            a[0] += t; a[1] += 1
        N = (T + 1) * B
        flops = gemm_flops_table(N, A, "resnet" if args.net == "resnet" else args.use_lstm)
        nbytes = hbm_bytes_table(N, T, B, A, args.use_lstm, model.flat_params.numel())
        gbytes = gemm_bytes_table(N, A, args.use_lstm, model.precision != "fp32") if args.net == "atari" else {}
        if args.net == "resnet" and model.precision == "bf16x3":
            gbytes = resnet_bytes_table(N)
            nbytes = dict(nbytes, **{k: v for k, v in gbytes.items() if k not in flops})
        ops = []
        for name, (tot, cnt) in agg.items():
            per_step = tot / PSTEPS
            o = dict(op=name, ms_per_step=per_step, launches_per_step=cnt / PSTEPS)
            if name in flops:
                tf = flops[name] / (per_step * 1e-3) / 1e12
                o.update(bound="tensor", achieved=tf, peak=pk["tensor"], unit="TFLOP/s")
                if name in gbytes:  # a GEMM whose operands stream once: report the binding roofline
                    gb = gbytes[name] / (per_step * 1e-3) / 1e9
                    o["tensor_frac"], o["hbm_frac"] = tf / pk["tensor"], gb / pk["hbm"]
                    if gb / pk["hbm"] > tf / pk["tensor"]:
                        o.update(bound="hbm", achieved=gb, peak=pk["hbm"], unit="GB/s")
            elif name in nbytes:
                o.update(bound="hbm", achieved=nbytes[name] / (per_step * 1e-3) / 1e9, peak=pk["hbm"], unit="GB/s")
            if "achieved" in o:
                o["frac"] = o["achieved"] / o["peak"]
            ops.append(o)
        ops.sort(key=lambda o: -o["ms_per_step"])
        prof_total = sum(o["ms_per_step"] for o in ops)
        line["roofline_ops"] = [dict(o, share=o["ms_per_step"] / prof_total) for o in ops[:12]]
        dom = next((o for o in ops if "achieved" in o), None)
        try:
            traffic_tab = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")))
        except Exception:
            traffic_tab = {}
        if dom is not None:
            line["roofline"] = dict(kernel=dom["op"], bound=dom["bound"], achieved=dom["achieved"], peak=dom["peak"],
                                    unit=dom["unit"], frac=dom["frac"],
                                    traffic=(traffic_tab.get(dom["op"], {}).get("dram_bytes_per_launch")),
                                    launches_per_step=dom["launches_per_step"], peak_source=pk["source"],
                                    note=("latency-bound recurrence: T+1 dependent time steps, each a hand-off through L2 + tile "
                                          "all-gather + mma.sync products; neither roofline is approached - the algorithmic "
                                          "recurrent-product flops (2*M*N*K, not x3 for the split planes) are reported against the "
                                          "sustained bf16 tensor peak" if dom["op"].startswith("lstm_recurrence")
                                          else ("algorithmic bytes (every tensor once: padded split-bf16 images, fp32 outputs / masks / "
                                                "residuals) against the measured HBM copy bandwidth" if dom["bound"] == "hbm"
                                                else "%s backend against the sustained bf16 tensor-core peak (algorithmic flops: the 3 MMAs "
                                                     "of a split product count once)" % model.precision)))
        # the V-trace kernels on their own (BASELINE.json metric: V-trace GB/s vs HBM peak)
        line["vtrace"] = vtrace_numbers(pk, T, B, A)

    if not args.no_cpu_baseline and world == 1:
        os.environ.setdefault("TB_CPU_BASELINE_BUDGET_S", "20")
        r = run_reference(types.SimpleNamespace(**dict(vars(args), steps=3, warmup=1)), 1)
        line["cpu_baseline"] = dict(value=r["value"], unit="frames/s", cores=r["cores"], kind="port", sample=r["sample"],
                                    **host_cpu_info())
    print(json.dumps(line))
    finish()


def vtrace_numbers(pk, T, B, A):
    """Scan-only and fused-loss kernels: achieved algorithmic GB/s at the bench size (launch-latency
    bound) and on a wide batch (HBM bound).  20 back-to-back launches per event pair."""
    from torchbeast_b200 import _lib
    lib, p, st = _lib.lib(), _lib.ptr, _lib.stream_ptr()
    out = {}
    g = torch.Generator(device="cuda").manual_seed(0)
    flush = torch.zeros(64 * 1024 * 1024, device="cuda")
    for tag, (t, b) in (("bench_size", (T, B)), ("config5_T600_B128", (600, 128)), ("wide", (T, 1 << 20))):
        lr = 0.5 * torch.randn(t, b, device="cuda", generator=g)
        dc = 0.99 * (torch.rand(t, b, device="cuda", generator=g) > 0.01).float()
        rw = torch.randn(t, b, device="cuda", generator=g).clamp(-1, 1)
        va = torch.randn(t, b, device="cuda", generator=g); bs = torch.randn(b, device="cuda", generator=g)
        vs = torch.empty_like(va); pg = torch.empty_like(va)
        reps = 20 if tag != "wide" else 3

        def launch_all():
            for _ in range(reps):
                lib.tb_vtrace_from_importance_weights_f32(p(lr), p(dc), p(rw), p(va), p(bs), t, b, 1.0, 1.0, p(vs), p(pg), _lib.stream_ptr())

        graph = None
        if tag != "wide":
            # 20 launches replayed as ONE CUDA graph: the event pair then measures kernel time on the device
            # (launch-to-launch), not the host's ctypes launch rate
            try:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    launch_all()
                torch.cuda.current_stream().wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    launch_all()
            except Exception:
                graph = None
        times = []
        for it in range(6):
            if tag == "wide":
                flush.add_(1)
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if graph is not None:
                graph.replay()
            else:
                launch_all()
            z.record(); torch.cuda.synchronize()
            times.append(a.elapsed_time(z) / reps)
        us = sorted(times[1:])[len(times[1:]) // 2] * 1e3
        nbytes = 24 * t * b + 4 * b
        out[tag] = dict(T=t, B=b, us=us, bytes=nbytes, gbs=nbytes / us / 1e3, frac=nbytes / us / 1e3 / pk["hbm"], peak=pk["hbm"],
                        timing=("%d launches per CUDA-graph replay" % reps) if graph is not None else "%d back-to-back launches" % reps)
        del lr, dc, rw, va, vs, pg
    return out


if __name__ == "__main__":
    main()

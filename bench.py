#!/usr/bin/env python
"""bench.py -- images/sec of VQVAE.forward (enc + VQ + dec) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one VQVAE.forward over one batch of synthetic images per GPU.  Prints ONE JSON line (rank 0).
--dump-outputs DIR writes what the last timed step of the headline returned (see dump_outputs) so that two builds
can be compared output for output: the weights and images are seeded, so the same arguments give the same inputs.

  headline   BASELINE.json configs[1] (cfg2: B=256 per GPU, 3x32x32, K=512, D=64), per-GPU batch fixed as N grows
             (weak scaling, batch-sharded, no data-path collective).  Convs = tcgen05 kind::tf32 on fp32 activations
             (what the reference itself computes on a GPU), VQ bit-exact fp32; the all-FFMA fp32 numbers ride along.
    value      whole-job images/sec, inputs resident in HBM, device time (CUDA events per step, L2 flushed between
               steps, max over ranks)
    e2e        same metric through the package's host-buffer API (vqvae_b200.HostPipeline): every step's pinned
               host -> device copy of x, the forward and the device -> host copy of x_hat + scalars inside the timed
               region, three steps in flight
    kernels    every C-ABI call of the step with its live CUDA-event time and its roofline fraction
    roofline   the dominant kernel of the step
    flips      index flips of the timed mode against the C oracle on the same images
  cfg3       BASELINE.json configs[2] (B=128, 3x256x256, K=1024, bf16 pipeline) on one GPU: images/sec, per-kernel
             roofline, index flips
  cfg5       BASELINE.json configs[4] (GLOBAL batch 1024 at 256x256, K=1024, bf16) split over the N GPUs: strong scaling
  vq_sweep   BASELINE.json configs[3]: the VQ kernel alone, K in {512, 1024, 8192} x D in {64, 256}, N = 2^20 rows
  cpu_baseline / --impl reference   the reference's CPU forward on the host cores (the unmodified reference from
             oracle/_ref when present, else oracle/torch_port.py)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # name: per-GPU batch (global for cfg5), image size, K, D
    "cfg2": dict(batch=256, size=32, K=512, D=64,
                 desc="VQVAE.forward bs=256 3x32x32 K=512 D=64 (BASELINE configs[1])"),
    "cfg3": dict(batch=128, size=256, K=1024, D=64,
                 desc="VQVAE.forward bs=128 3x256x256 K=1024 D=64 bf16 (BASELINE configs[2])"),
    "cfg5": dict(batch=1024, size=256, K=1024, D=64,
                 desc="VQVAE.forward GLOBAL bs=1024 3x256x256 K=1024 D=64 bf16, batch-sharded (BASELINE configs[4])"),
}
HP = dict(h_dim=128, res_h_dim=32, n_res_layers=2)
METRIC = "images/sec VQVAE fwd (enc+VQ+dec)"
DUMP_BYTES = 64 << 20          # what --dump-outputs writes in all


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), bf16=float(d["bf16_tflops"]),
                    bf16_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


# --------------------------------------------------------------------------- synthetic weights / images (no oracle import)
def synth(wl, seed_w=0, seed_x=1, batch=None):
    from vqvae_b200.synth import make_images, make_state_dict
    sd = make_state_dict(seed=seed_w, n_embeddings=wl["K"], embedding_dim=wl["D"], **HP)
    x = make_images(batch or wl["batch"], wl["size"], seed=seed_x)
    return sd, x


# --------------------------------------------------------------------------- CPU arm
def _cpu_forward_fn(wl, batch):
    """A callable running the reference's forward once on the host, and what it is ("reference" | "port")."""
    import oracle
    sd, x = synth(wl, batch=batch)
    xt = torch.from_numpy(x)
    ref_dir = oracle.ref_path()
    if ref_dir:
        # the UNMODIFIED reference (verbatim copy made by oracle.build_ref() in the authoring container); its module-level
        # `device` is pointed at the CPU (SURVEY Q5: it is computed at import time and breaks the CPU path on a GPU box)
        sys.path.insert(0, ref_dir)
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            del sys.modules[k]
        import models.quantizer as Q
        Q.device = torch.device("cpu")
        from models.vqvae import VQVAE as RefVQVAE
        sys.path.remove(ref_dir)
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            del sys.modules[k]                       # (the product's own `models` package must stay importable)
        m = RefVQVAE(HP["h_dim"], HP["res_h_dim"], HP["n_res_layers"], wl["K"], wl["D"], 0.25).eval()
        m.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})

        def fn():
            with torch.no_grad():
                return m(xt)
        return fn, "reference"
    from oracle import torch_port
    tsd = {k: torch.from_numpy(np.array(v)) for k, v in sd.items()}
    return (lambda: torch_port.vqvae_forward(xt, tsd, HP["n_res_layers"])), "port"


def best_cpu_threads(fn):
    """torch's intra-op pool oversubscribes small convs on big hosts (128 threads were 2x slower than 32 on the GPU
    box): time one forward at a few thread counts and keep the fastest, so the CPU baseline is the reference at its
    best on this host."""
    total = os.cpu_count() or 1
    cands = sorted({total, max(1, total // 2), max(1, total // 4), min(total, 32), min(total, 16), min(total, 8)})
    best, best_t = total, None
    for c in cands:
        torch.set_num_threads(c)
        fn()
        t0 = time.perf_counter()
        fn()
        t = time.perf_counter() - t0
        if best_t is None or t < best_t:
            best, best_t = c, t
    return best


def cpu_sample_batch(wl):
    return min(wl["batch"], 256 if wl["size"] <= 32 else 4)     # bounded sample: 256x256 costs seconds per image on a CPU


def cpu_baseline(wl, budget_s, min_iters=3, max_iters=50):
    sb = cpu_sample_batch(wl)
    fn, kind = _cpu_forward_fn(wl, sb)
    cores = best_cpu_threads(fn)
    torch.set_num_threads(cores)
    for _ in range(2):
        fn()
    n, t0 = 0, time.perf_counter()
    while True:
        fn()
        n += 1
        el = time.perf_counter() - t0
        if n >= max_iters or (n >= min_iters and el >= budget_s):
            break
    what = "the unmodified reference (oracle/_ref)" if kind == "reference" else "oracle/torch_port.py = reference forward on torch CPU ops"
    return {"value": sb * n / el, "unit": "images/sec", "cores": cores, "kind": kind,
            "sample": f"{n} forwards of B={sb} 3x{wl['size']}x{wl['size']} in {el:.1f}s ({what}; {cores} threads = fastest of "
                      f"several counts on this {os.cpu_count()}-thread host)"}


def common_config(wl, world, extra=None):
    cfg = {"workload": wl["desc"], "per_gpu_batch": wl["batch"], "global_batch": wl["batch"] * world,
           "parallelism": f"batch-shard x{world}",
           "weights": "synthetic seeded (vqvae_b200/synth.py), reference architecture h=128 res_h=32 n_res=2"}
    cfg.update(extra or {})
    return cfg


def run_reference_arm(args, wl, rank, world):
    if rank != 0:
        return
    sb = cpu_sample_batch(wl)
    fn, kind = _cpu_forward_fn(wl, sb)
    cores = best_cpu_threads(fn)
    torch.set_num_threads(cores)
    for _ in range(args.warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    el = time.perf_counter() - t0
    val = sb * args.steps / el
    sample = (f"{args.steps} forwards of B={sb} 3x{wl['size']}x{wl['size']} "
              f"({'unmodified reference from oracle/_ref' if kind == 'reference' else 'oracle/torch_port.py'}, torch CPU ops, best of "
              f"several thread counts = {cores} of {os.cpu_count()} host threads)")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/sec", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "tf32",
        "dtype_note": "the CPU arm computes in fp32", "data": "synthetic",
        "config": common_config(wl, world, {"l2": "n/a (CPU)", "launch": "n/a (CPU)", "cpu_sample_batch": sb}),
        "cpu_baseline": {"value": val, "unit": "images/sec", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- GPU arm helpers
class ClockSampler:
    """SM clock / throttle-reason samples every 20 ms from a separate light NVML process (tools/clock_sampler.py;
    `nvidia-smi --query-gpu -lms 20` as the fallback: its full query cost the pipelined host loop ~8 %)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p, self.kind = None, None
        if gpu_index < 0:
            return
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")      # NVML indexes physical devices
        try:
            phys = int(vis.split(",")[gpu_index]) if vis else gpu_index
        except (ValueError, IndexError):
            phys = gpu_index
        sampler = os.path.join(ROOT, "tools", "clock_sampler.py")
        try:
            import pynvml  # noqa: F401  (only to know the light sampler can run)
            self.p = subprocess.Popen([sys.executable, sampler, str(phys), "20"], stdout=self.f, stderr=subprocess.DEVNULL)
            self.kind = "nvml"
        except Exception:
            try:
                self.p = subprocess.Popen(["nvidia-smi", "-i", str(phys), f"--query-gpu={self.QUERY}",
                                           "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
                self.kind = "smi"
            except OSError:
                self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        lines = [r.strip() for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for ln in lines:
            try:
                if self.kind == "nvml":                     # "sm,max,reason|reason"
                    a, b, c = ln.split(",", 2)
                    sm.append(float(a)); mx.append(float(b))
                    reasons.update(x for x in c.split("|") if x)
                else:
                    r = ln.split(", ")
                    if len(r) < 9:
                        continue
                    sm.append(float(r[1])); mx.append(float(r[2]))
                    for n, v in zip(self.NAMES, r[5:9]):
                        if v.strip().lower().startswith("active"):
                            reasons.add(n)
            except ValueError:
                continue
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm), sampler=self.kind)
        return out


def layer_model(label, B, K, D):
    """Algorithmic work of one C-ABI call from its label: (flops, bytes, tensor dtype) -- SURVEY 8d's per-unit figures
    times the units of the launch.  Activation bytes: 2 per element in the bf16 pipeline, 4 otherwise; the module boundary
    (x, x_hat) and z_e are fp32 in both."""
    bf = label.startswith("bf16 ")
    parts = (label[5:] if bf else label).split()
    esz = 2 if bf else 4
    if parts[0] == "vq":
        kv = dict(p.split("=") for p in parts[1:4])
        N, K_, D_ = int(kv["N"]), int(kv["K"]), int(kv["D"])
        zq = 2 if "(bf16" in label else 4
        return 2.0 * N * K_ * D_, N * (D_ * 4 + D_ * zq + 8) + K_ * D_ * 4, "tf32"
    if parts[0] == "res":
        napp = 1
        if parts[1].startswith("x"):
            napp = int(parts[1][1:])
            parts = [parts[0]] + parts[2:]
        c, cm, _ = (int(v) for v in parts[1].split("->"))
        h, w = (int(v) for v in parts[2].split("x"))
        # a fused stack reads / writes the activation once; separate applications once each
        return 2.0 * napp * B * h * w * (9 * c * cm + cm * c), 2.0 * B * h * w * c * esz, ("bf16" if bf else "tf32")
    transposed = parts[0] == "convT"
    cin, cout = (int(v) for v in parts[1].split("->"))
    k = int(parts[2][1:parts[2].index("s")])
    s = int(parts[2][parts[2].index("s") + 1:])
    h, w = (int(v) for v in parts[3].split("x"))
    if transposed:
        oh, ow = h * s, w * s
        macs = B * h * w * cin * cout * k * k
    else:
        oh, ow = (h // s, w // s) if k > 1 else (h, w)
        macs = B * oh * ow * cin * cout * k * k
    in_esz = 4 if cin == 3 else esz                         # the image is fp32
    out_esz = 4 if (cout <= 4 or (bf and k == 1)) else esz  # x_hat and (bf16 pipeline) z_e are fp32
    byts = B * h * w * cin * in_esz + B * oh * ow * cout * out_esz + cin * cout * k * k * esz
    return 2.0 * macs, float(byts), ("tf32" if (not bf or cin == 3) else "bf16")


def kernel_entry(label, ms, calls, share, B, K, D, peaks, traffic=None):
    """One row of the `kernels` list: live time + roofline against max(T_hbm, T_tensor)."""
    row = {"kernel": label, "calls": calls, "ms_per_call": ms, "share": share}
    try:
        flops, byts, tdt = layer_model(label, B, K, D)
    except Exception as e:  # pragma: no cover - an unparsable label must not kill the line
        row["error"] = repr(e)[:100]
        return row
    tpeak = peaks["bf16"] * (1.0 if tdt == "bf16" else 0.5)      # TF32 = half the measured bf16 cuBLAS peak
    t_hbm, t_tc = byts / (peaks["hbm"] * 1e9), flops / (tpeak * 1e12)
    if t_tc >= t_hbm:
        ach = flops / (ms * 1e-3) / 1e12
        row.update(bound="tensor", achieved=ach, peak=tpeak, unit="TFLOP/s", frac=ach / tpeak)
    else:
        ach = byts / (ms * 1e-3) / 1e9
        row.update(bound="hbm", achieved=ach, peak=peaks["hbm"], unit="GB/s", frac=ach / peaks["hbm"])
    row["traffic"] = traffic
    return row


def ncu_traffic_table():
    """DRAM bytes (read + write) per launch from this round's committed `ncu --set full` capture, keyed by label."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_step_kernels_traffic.json")) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {}


def build_model(wl, dev):
    from models.vqvae import VQVAE
    sd, _ = synth(wl, batch=1)
    model = VQVAE(HP["h_dim"], HP["res_h_dim"], HP["n_res_layers"], wl["K"], wl["D"], 0.25)
    model.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
    return model.to(dev).eval(), sd


def capture(model, x):
    """(step(), outputs, is_graph): the forward captured in a CUDA graph (eager fallback)."""
    out = model(x)                                      # eager once: packs weights, sizes workspaces
    torch.cuda.synchronize()
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                model(x)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = model(x)
        torch.cuda.synchronize()
        return (lambda: (graph.replay(), out)[1]), out, True
    except Exception as e:  # pragma: no cover - reported in the JSON line
        print(f"[bench] CUDA graph capture failed ({e}); running eagerly", file=sys.stderr)
        return (lambda: model(x)), out, False


def step_outputs(model, out):
    """What a caller of one forward receives, on the host: VQVAE.forward's (loss, x_hat, perplexity) and the model's
    last_min_encoding_indices (as float64, which holds every index exactly)."""
    loss, x_hat, perp = out
    arrays = {"loss": loss, "x_hat": x_hat, "perplexity": perp}
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    arrays["min_encoding_indices"] = model.last_min_encoding_indices.double().cpu().numpy()
    return arrays


def dump_outputs(out_dir, arrays):
    """Write each array as <out_dir>/<name>.npy.  Every array gets an equal share of DUMP_BYTES; one that is larger is
    replaced by a sample of its flattened elements at positions drawn with a fixed seed (the same in every run with the
    same arguments), in increasing order.  Returns what was written, for the JSON line."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    info = {}
    for name, a in arrays.items():
        entry = {"shape": list(a.shape), "dtype": str(a.dtype)}
        keep = share // a.itemsize
        if a.size > keep:
            pos = np.sort(np.random.RandomState(0).choice(a.size, keep, replace=False))
            a = a.reshape(-1)[pos]
            entry["sampled_elements"] = keep
        np.save(os.path.join(out_dir, name + ".npy"), a)
        info[name] = entry
    return info


def oracle_flips(wl, x_np, idx_dev, sd, n_img):
    """Index flips of the timed mode against the C oracle on the first n_img images of the batch (rank 0, untimed)."""
    try:
        from oracle import cref
        o = cref.vqvae_forward(x_np[:n_img], sd, HP["n_res_layers"])
        rows = n_img * (wl["size"] // 4) ** 2
        mine = idx_dev.view(-1)[:rows].cpu().numpy()
        nf = int((mine != o["idx"].ravel()).sum())
        return {"rows_checked": rows, "images_checked": n_img, "flips": nf, "frac": nf / rows,
                "against": "oracle/csrc/oracle.c (fp32-accurate forward of the same images)"}
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3"], help="headline workload (default: BASELINE configs[1])")
    ap.add_argument("--precision", default=None, choices=["fp32", "tf32", "bf16"],
                    help="arithmetic of the headline (default: tf32 for cfg2 -- what the reference computes on a GPU -- and bf16 for cfg3)")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying a CUDA graph")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline only: no fp32 mode, cfg3, cfg5, vq_sweep")
    ap.add_argument("--no-extra-modes", action="store_true", help="alias of --quick")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline's outputs of its last timed step as DIR/<name>.npy (rank 0's shard)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3)
    args.quick = args.quick or args.no_extra_modes
    wl = WORKLOADS[args.workload]
    prec_main = args.precision or ("tf32" if args.workload == "cfg2" else "bf16")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, wl, rank, world)
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    import vqvae_b200
    from vqvae_b200 import ops, _lib
    from vqvae_b200.synth import make_images

    peaks = load_peaks()
    traffic_tab = ncu_traffic_table()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        if dist is None:
            return vals
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def breakdown(model, x, Bx, K, D):
        """Per-kernel CUDA-event times (eager launches behind a spin kernel, L2 flushed) -> `kernels` rows."""
        per = {}
        saved_group, model.process_group = model.process_group, None     # rank-local: no collective here
        reps = 5
        for _ in range(reps):
            flush.zero_()
            ops.PROFILE = []
            torch.cuda._sleep(4_000_000)          # keep the stream busy while the host enqueues
            model(x)
            torch.cuda.synchronize()
            for label, a, b in ops.PROFILE:
                per.setdefault(label, []).append(a.elapsed_time(b))
            ops.PROFILE = None
        model.process_group = saved_group
        tot = {k: float(np.sum(v)) / reps for k, v in per.items()}
        step_ms = sum(tot.values())
        rows = [kernel_entry(k, float(np.mean(v)), len(v) // reps, tot[k] / step_ms, Bx, K, D, peaks, traffic_tab.get(k))
                for k, v in per.items()]
        return sorted(rows, key=lambda r: -r["share"])

    def device_time(step, steps):
        """(device ms of `steps` steps, what the last step returned)."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        out = None
        for s0, s1 in evs:
            flush.zero_()
            s0.record()
            out = step()
            s1.record()
        barrier()
        return sum(a.elapsed_time(b) for a, b in evs), out

    # =============================================================== headline workload
    B, S, K, D = wl["batch"], wl["size"], wl["K"], wl["D"]
    model, sd = build_model(wl, dev)
    if world > 1:
        model.process_group = dist.group.WORLD
        model.sync_scalars = False            # the step returns this shard's scalars; the collective is on demand (below)
    x_np = make_images(B, S, seed=1 + rank)   # every rank gets its own shard of the global batch
    x_host = torch.from_numpy(x_np).pin_memory()
    x_dev = x_host.to(dev)

    def run_mode(prec, full):
        vqvae_b200.set_precision(prec)
        model(x_dev)
        torch.cuda.synchronize()
        l0 = ops.launch_count()
        model(x_dev)
        torch.cuda.synchronize()
        launches_per_step = ops.launch_count() - l0
        static_x = x_dev.clone()
        if args.no_graph:
            step, out, is_graph = (lambda: model(static_x)), model(static_x), False
        else:
            step, out, is_graph = capture(model, static_x)
        for _ in range(args.warmup):
            step()
        barrier()
        clocks = ClockSampler(local_rank if (full and not os.environ.get("VQB_BENCH_NOSAMPLER")) else -1)
        dev_ms, last = device_time(step, args.steps)
        res = dict(launches=int(launches_per_step * args.steps), graph=is_graph)
        if full and args.dump_outputs and rank == 0:
            res["outputs"] = step_outputs(model, last)       # before anything below runs the model again
        if full:
            # ---- end to end: host buffers, copies inside the timed region ----
            xh_host = torch.empty((B, 3, S, S), dtype=torch.float32).pin_memory()
            sc_host = torch.empty((2,), dtype=torch.float32).pin_memory()
            for _ in range(3):
                static_x.copy_(x_host, non_blocking=True); o = step()
                xh_host.copy_(o[1], non_blocking=True)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):           # (1) synchronous caller: copy in, forward, copy out, wait
                static_x.copy_(x_host, non_blocking=True)
                o = step()
                xh_host.copy_(o[1], non_blocking=True)
                sc_host[0:1].copy_(o[0].reshape(1), non_blocking=True)
                sc_host[1:2].copy_(o[2].reshape(1), non_blocking=True)
                torch.cuda.current_stream().synchronize()
            e2e_sync_s = time.perf_counter() - t0
            barrier()
            depth = int(os.environ.get("VQB_BENCH_DEPTH", "3"))      # (2) the package's streaming front end
            pipe = vqvae_b200.HostPipeline(model, (B, 3, S, S), depth=depth, use_graph=is_graph)
            hosts = [x_host] + [torch.from_numpy(make_images(B, S, seed=101 + i + 7 * rank)).pin_memory() for i in range(depth - 1)]
            seen = [0, 0.0]

            def consume(r):
                seen[0] += 1
                seen[1] += float(r.loss)          # the caller reads each step's result on the host

            pipe.run((hosts[i % depth] for i in range(2 * depth)), consume)
            regions = []
            for _ in range(3):                    # three regions of exactly K steps; the median is reported
                barrier()
                seen[0] = 0
                t0 = time.perf_counter()
                pipe.run((hosts[i % depth] for i in range(args.steps)), consume)
                regions.append(time.perf_counter() - t0)
                assert seen[0] == args.steps and np.isfinite(seen[1])
            e2e_s = sorted(regions)[1]
            res.update(h2d=int(pipe.h2d_bytes), d2h=int(pipe.d2h_bytes), depth=depth)
            del pipe
            barrier()
            t_load = time.perf_counter()          # ~0.4 s more of the same step so the clock record has samples under load
            while time.perf_counter() - t_load < 0.4:
                for _ in range(20):
                    step()
                torch.cuda.synchronize()
            res["clocks"] = clocks.stop()
            dev_ms, e2e_s, e2e_sync_s = allmax([dev_ms, e2e_s, e2e_sync_s])
            imgs = B * world * args.steps
            res.update(e2e_value=imgs / e2e_s, e2e_ms=e2e_s / args.steps * 1e3, e2e_sync_value=imgs / e2e_sync_s,
                       e2e_sync_ms=e2e_sync_s / args.steps * 1e3, e2e_regions_ms=[r / args.steps * 1e3 for r in regions])
        else:
            clocks.stop()
            dev_ms, = allmax([dev_ms])
        res.update(value=B * world * args.steps / (dev_ms * 1e-3), ms_per_step=dev_ms / args.steps)
        if rank == 0:
            res["kernels"] = breakdown(model, static_x, B, K, D)
            res["flips"] = oracle_flips(wl, x_np, model.last_min_encoding_indices, sd, min(B, 256 if S <= 32 else 2))
        return res

    main_mode = run_mode(prec_main, True)
    line_extra = {}
    if "outputs" in main_mode:
        line_extra["outputs"] = {"dir": os.path.abspath(args.dump_outputs),
                                 "arrays": dump_outputs(args.dump_outputs, main_mode.pop("outputs"))}
    if not args.quick and prec_main != "fp32" and args.workload == "cfg2":
        m = run_mode("fp32", False)
        line_extra["fp32_mode"] = {"value": m["value"], "unit": "images/sec", "ms_per_step": m["ms_per_step"], "dtype": "f32",
                                   "gpu_launches": m["launches"], "kernels": m.get("kernels", [])[:8], "flips": m.get("flips"),
                                   "note": "same workload with every conv in fp32 FFMA (CUDA cores): the CPU reference's numerics"}
        mb = run_mode("bf16", False)
        line_extra["bf16_mode"] = {"value": mb["value"], "unit": "images/sec", "ms_per_step": mb["ms_per_step"], "dtype": "bf16",
                                   "gpu_launches": mb["launches"], "kernels": mb.get("kernels", [])[:12], "flips": mb.get("flips"),
                                   "note": "same workload through the bf16 pipeline (tcgen05 kind::f16 on bf16 operands, bf16 NHWC "
                                           "activations, exact fp32 VQ): the arithmetic of the reference under torch.autocast(bfloat16)"}
        vqvae_b200.set_precision(prec_main)

    # ---- shard parity (N > 1): rank 0's shard inside the sharded job == the same images through a single-process forward
    shard_parity = None
    if world > 1:
        vqvae_b200.set_precision(prec_main)
        _, xh_s, _ = model(x_dev)
        idx_s = model.last_min_encoding_indices.clone()
        gl, gp = model.reduce_scalars()                     # the on-demand collective (all ranks call it)
        saved, model.process_group = model.process_group, None
        l1, xh_1, p1 = model(x_dev)
        model.process_group = saved
        torch.cuda.synchronize()
        ok = bool(torch.equal(xh_s, xh_1) and torch.equal(idx_s, model.last_min_encoding_indices))
        shard_parity = {"rank0_shard_equals_single_process": ok, "global_loss": float(gl), "rank0_shard_loss": float(l1),
                        "global_perplexity": float(gp),
                        "note": "x_hat and min_encoding_indices bitwise; loss / perplexity of the step are per shard, "
                                "reduce_scalars() gives the whole-batch values"}
    del model
    torch.cuda.empty_cache()

    # =============================================================== cfg3 (one GPU) and cfg5 (global batch split)
    def run_big(name, per_gpu_batch, with_kernels):
        w = WORKLOADS[name]
        vqvae_b200.set_precision("bf16")
        m, sdb = build_model(w, dev)
        xb_np = make_images(per_gpu_batch, w["size"], seed=11 + rank)
        xb = torch.from_numpy(xb_np).to(dev)
        if world > 1:
            m.process_group = dist.group.WORLD
            m.sync_scalars = False
        step, out, is_graph = capture(m, xb)
        for _ in range(3):
            step()
        nsteps = max(3, min(args.steps, 10))
        ms, = allmax([device_time(step, nsteps)[0]])
        o = {"workload": w["desc"], "dtype": "bf16", "per_gpu_batch": per_gpu_batch, "n_gpus": world, "steps": nsteps,
             "value": per_gpu_batch * world * nsteps / (ms * 1e-3), "unit": "images/sec", "ms_per_step": ms / nsteps,
             "launch": "cuda-graph replay" if is_graph else "eager", "l2": "flushed between timed steps"}
        if with_kernels and rank == 0:
            o["kernels"] = breakdown(m, xb, per_gpu_batch, w["K"], w["D"])
            o["flips"] = oracle_flips(w, xb_np, m.last_min_encoding_indices, sdb, 2)
            if o["kernels"]:
                o["limiting_kernel"] = o["kernels"][0]["kernel"]
        del m, xb, step, out
        torch.cuda.empty_cache()
        return o

    cfg3 = cfg5 = None
    if not args.quick:
        if world == 1 and args.workload != "cfg3":
            cfg3 = run_big("cfg3", WORKLOADS["cfg3"]["batch"], True)
        gb = WORKLOADS["cfg5"]["batch"]
        if gb % world == 0:
            cfg5 = run_big("cfg5", gb // world, world > 1)
            cfg5["scaling"] = "strong"
            cfg5["global_batch"] = gb
    vqvae_b200.set_precision(prec_main)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    cpu = None if args.skip_cpu else cpu_baseline(wl, args.cpu_seconds)
    kernels = main_mode.get("kernels", [])
    top = kernels[0] if kernels else None
    roofline = None
    if top and "frac" in top:
        roofline = {k: top[k] for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "traffic")}
        roofline["peak_source"] = peaks["src"]
        roofline["traffic_source"] = "profiles/r02_step_kernels_traffic.json (this round's ncu --set full capture)" if top.get("traffic") else None
        roofline["note"] = "tf32 layers are held against half the measured bf16 cuBLAS peak"
    dtype_note = {"tf32": "fp32 tensors end to end; convs = tcgen05 kind::tf32 with fp32 accumulation (PyTorch/cuDNN's default conv "
                          "arithmetic on this GPU); VQ distances/argmin bit-exact fp32; fp32_mode = all-FFMA numbers",
                  "fp32": "all arithmetic fp32 (FFMA)",
                  "bf16": "bf16 activations and operands between layers (tcgen05 kind::f16), fp32 accumulation, fp32 z_e, "
                          "VQ distances/argmin bit-exact fp32 on that z_e"}[prec_main]
    line = {
        "metric": METRIC, "value": main_mode["value"], "unit": "images/sec", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": main_mode["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "tf32": "tf32", "bf16": "bf16"}[prec_main],
        "data": "synthetic", "dtype_note": dtype_note,
        "config": common_config(wl, world, {"l2": "flushed between timed steps (256 MiB memset)",
                                            "launch": "cuda-graph replay" if main_mode["graph"] else "eager",
                                            "cpu_sample_batch": cpu_sample_batch(wl)}),
        "e2e": {"value": main_mode["e2e_value"], "unit": "images/sec", "h2d_bytes_per_step": main_mode["h2d"],
                "d2h_bytes_per_step": main_mode["d2h"], "ms_per_step": main_mode["e2e_ms"],
                "api": f"vqvae_b200.HostPipeline(depth={main_mode['depth']}): every step copies its pinned host batch to HBM, runs the "
                       f"forward and copies x_hat + loss + perplexity back to pinned host memory, {main_mode['depth']} steps in flight",
                "regions_ms_per_step": main_mode["e2e_regions_ms"],
                "regions_note": "three timed regions of K steps each; value = the median region (max over ranks)",
                "l2": "not flushed between end-to-end steps: every step's input arrives from host memory by DMA",
                "sync_value": main_mode["e2e_sync_value"], "sync_ms_per_step": main_mode["e2e_sync_ms"],
                "sync_note": "same copies with the caller waiting for each step before submitting the next"},
        "gpu_launches": main_mode["launches"],
        "clocks": main_mode["clocks"],
        "roofline": roofline,
        "kernels": kernels,
        "flips": main_mode.get("flips"),
        "cpu_baseline": cpu,
        "peaks": peaks,
        "env_overrides": [],
        "library_build": "diagnostic (-DVQB_DIAG=1)" if _lib.lib().vqb_diag_build() else "release (never reads the environment)",
    }
    if world > 1:
        line["scalars"] = ("per-shard loss / perplexity in the timed step (sync_scalars = False): no collective inside the step; "
                           "reduce_scalars() all-reduces the 4 KB of VQ statistics on demand (checked after the timed region)")
        line["shard_parity"] = shard_parity
    line.update(line_extra)
    if cfg3 is not None:
        line["cfg3"] = cfg3
    if cfg5 is not None:
        line["cfg5"] = cfg5
    if not args.quick:
        line["vq_sweep"] = vq_sweep(ops, peaks, dev)
        line["vq_kernel"] = line["vq_sweep"][0]
    else:
        line["vq_kernel"] = vq_point(ops, peaks, dev, 512, 64)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def vq_point(ops, peaks, dev, K, D, N=1 << 20):
    """The VQ kernel alone at a streaming size (N rows in, N rows + indices out: larger than L2, no flush needed),
    CUDA events around `reps` calls of vqb_vq_forward_f32; algorithmic bytes = (2*D*4 + 8) per row (SURVEY 8d), held
    against max(T_hbm, T_tensor) with the TF32 ceiling = half the measured bf16 peak."""
    try:
        rng = np.random.RandomState(0)
        z = torch.from_numpy(rng.standard_normal((N, D)).astype(np.float32)).to(dev)
        E = torch.from_numpy(rng.standard_normal((K, D)).astype(np.float32)).to(dev)
        for _ in range(2):
            ops.vq_forward(z, E)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5 if K * D <= 1024 * 64 else 2
        e0.record()
        for _ in range(reps):
            ops.vq_forward(z, E)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        byts = N * (2 * D * 4 + 8)
        flops = 2.0 * N * K * D
        t_hbm, t_tc = byts / (peaks["hbm"] * 1e9), flops / (peaks["bf16"] * 0.5 * 1e12)
        bound = "tensor" if t_tc > t_hbm else "hbm"
        out = {"rows": N, "K": K, "D": D, "ms_per_call": ms, "bound": bound,
               "hbm_gbs": byts / (ms * 1e-3) / 1e9, "tensor_tflops": flops / (ms * 1e-3) / 1e12,
               "frac": max(t_hbm, t_tc) / (ms * 1e-3), "algorithmic_bytes_per_row": 2 * D * 4 + 8, "peak_source": peaks["src"],
               "kernel": "tcgen05 (vq2.cu)" if D == 64 and K <= 8192 else "FFMA (vq_exact.cu)",
               "note": "codebook N(0,1), rows N(0,1); idx/z_q bit-exact vs the canonical fp32 order (tests)"}
        if bound == "hbm":
            out.update(achieved=out["hbm_gbs"], peak=peaks["hbm"], unit="GB/s")
        else:
            out.update(achieved=out["tensor_tflops"], peak=peaks["bf16"] * 0.5, unit="TFLOP/s")
        return out
    except Exception as e:  # pragma: no cover - reported, never fatal for the benchmark line
        return {"K": K, "D": D, "error": repr(e)[:200]}


def vq_sweep(ops, peaks, dev):
    return [vq_point(ops, peaks, dev, K, D, N=(1 << 20) if D == 64 else (1 << 18))
            for K, D in ((512, 64), (1024, 64), (8192, 64), (512, 256), (1024, 256), (8192, 256))]


if __name__ == "__main__":
    main()

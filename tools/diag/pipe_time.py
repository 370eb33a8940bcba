"""Diagnostic: HostPipeline throughput, torch copies vs raw stream-ordered copies."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import vqvae_b200
from oracle import weights
sd = weights.make_state_dict(128, 32, 2, 512, 64, seed=5)
m = vqvae_b200.VQVAE(128, 32, 2, 512, 64, 0.25)
m.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
vqvae_b200.set_precision("tf32")
m = m.cuda().eval()
B = 256
hosts = [torch.from_numpy(weights.make_images(B, 32, seed=1 + i)).pin_memory() for i in range(3)]
import subprocess, tempfile
QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
SAMPLERS = {"none": None,
            "smi20": ["nvidia-smi", "-i", "0", f"--query-gpu={QUERY}", "--format=csv,noheader,nounits", "-lms", "20"],
            "smi100": ["nvidia-smi", "-i", "0", f"--query-gpu={QUERY}", "--format=csv,noheader,nounits", "-lms", "100"],
            "nvml20": [sys.executable, "tools/clock_sampler.py", "0", "20"]}
if len(sys.argv) > 1 and sys.argv[1] == "benchlike":
    # what does bench.py do before its pipelined e2e region that a bare loop does not?
    what = sys.argv[2] if len(sys.argv) > 2 else "all"
    x_dev = hosts[0].cuda()
    if what in ("flush", "all"):
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
        for _ in range(20): flush.zero_()
    if what in ("graph", "all"):
        static_x = x_dev.clone()
        side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2): m(static_x)
        torch.cuda.current_stream().wait_stream(side); torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g): out = m(static_x)
        for _ in range(30): g.replay()
        torch.cuda.synchronize()
    if what in ("events", "all"):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(200)]
        for a, b in evs: a.record(); b.record()
        torch.cuda.synchronize()
    pipe = vqvae_b200.HostPipeline(m, (B, 3, 32, 32), depth=3)
    acc = [0.0]
    def consume(r): acc[0] += float(r.loss)
    pipe.run((hosts[i % 3] for i in range(6)), consume)
    torch.cuda.synchronize()
    res = []
    for rep in range(3):
        t0 = time.perf_counter()
        pipe.run((hosts[i % 3] for i in range(200)), consume)
        res.append((time.perf_counter() - t0) / 200 * 1e3)
    print(f"benchlike {what}: ms/step {[round(x, 4) for x in res]}")
    sys.exit(0)
if len(sys.argv) > 1 and sys.argv[1] == "samplers":
    pipe = vqvae_b200.HostPipeline(m, (B, 3, 32, 32), depth=3)
    acc = [0.0]
    def consume(r): acc[0] += float(r.loss)
    pipe.run((hosts[i % 3] for i in range(12)), consume)
    for name, cmd in SAMPLERS.items():
        f = tempfile.NamedTemporaryFile("w+", suffix=".csv")
        pr = subprocess.Popen(cmd, stdout=f, stderr=subprocess.DEVNULL) if cmd else None
        time.sleep(0.5)
        res = []
        for rep in range(3):
            t0 = time.perf_counter()
            pipe.run((hosts[i % 3] for i in range(300)), consume)
            res.append((time.perf_counter() - t0) / 300 * 1e3)
        if pr: pr.terminate(); pr.wait()
        f.flush(); nl = len(open(f.name).read().splitlines())
        print(f"sampler {name}: ms/step {[round(x, 4) for x in res]}  ({nl} sample lines)")
    sys.exit(0)
for raw in (False, True):
    pipe = vqvae_b200.HostPipeline(m, (B, 3, 32, 32), depth=3, raw_copies=raw)
    acc = [0.0]
    def consume(r): acc[0] += float(r.loss)
    pipe.run((hosts[i % 3] for i in range(12)), consume)
    torch.cuda.synchronize()
    for rep in range(2):
        t0 = time.perf_counter()
        pipe.run((hosts[i % 3] for i in range(200)), consume)
        dt = time.perf_counter() - t0
        print(f"raw={raw}: {dt/200*1e3:.3f} ms/step  {200*B/dt/1e6:.3f} M img/s")
    # host-side cost of push alone (GPU idle): time 50 pushes then drain
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(3): pipe.push(hosts[i])
    t1 = time.perf_counter()
    pipe.drain()
    print(f"   3 pushes took {(t1-t0)*1e6/3:.1f} us each (host side)")
    del pipe

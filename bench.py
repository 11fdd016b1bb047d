#!/usr/bin/env python3
"""bench.py — tuples/s of the tree-walk hot path on BASELINE.json's headline configuration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR (ours): after the timed steps, rank 0 writes what its last step returned for a fixed, seeded
  sample of DUMP_TUPLES tuples (all of them when fewer are requested): DIR/scores.npy (float32), DIR/labels.npy
  (0/1 as float32) and DIR/tuple_index.npy (float64, the sampled tuple indices).  The inputs depend only on the
  arguments, so two builds run with the same arguments can be compared file for file.

ours: one "step" = one pass of the walk kernel (through the C ABI, libdte.so) over one batch of
  synthetic tuples already resident in HBM.  N=1 workload = BASELINE configs[2]
  ("1024 trees, depth 12, 256 features, 50M tuples, HBM-bound node walk").  N>1 = the data-sharded
  configuration (configs[4]): ensemble replicated, a fresh 50M-tuple shard per GPU, no collective,
  weak scaling; the ensemble-sharded configuration (configs[3]) is measured in the same run under
  "ensemble_sharded" (ring-order peer-read combine = bit-exact, and one NCCL reduce), and rank 0 also
  drives all GPUs from ONE process through the multi-device C-ABI handle ("c_abi_multi").
reference: the reference has no CPU (or any software) implementation of this path — the RTL is the
  only definition — so the reference arm times the RTL-faithful oracle port (oracle/dte_oracle.c,
  tree-blocked loop) on the usable host cores, on a bounded sample of the same workload.

One JSON line on stdout (rank 0).  Nothing here reads /root/reference.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tuples/s at 1024 trees, depth 12, 256 feats"
T_TREES, DEPTH, FEATS, CLUSTERS = 1024, 12, 256, 8
N_FULL = 50_000_000
MISSING_PPM = 10000
SEED_TUPLES = 0x7091E5
SM_COUNT = 148
DUMP_TUPLES = 1 << 20           # --dump-outputs sample: 16 MiB of .npy files
DUMP_SEED = 0xD0


def algorithmic_bytes_per_tuple(T, D, F):
    """SURVEY.md §8(d) byte model (B): every node visit reads threshold (4) + index (2) + feature (4),
    every tree one leaf (4), plus the tuple in and the score out."""
    return T * (D * 10 + 4) + 4 * F + 4


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("hbm_gbs"), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_profile_json(name):
    p = os.path.join(ROOT, "profiles", name)
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi samples during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def bind_to_gpu_numa(local_gpu):
    """Pin this process (and therefore the first-touch placement of its pinned buffers) to the CPUs of the NUMA node
    the GPU hangs off: with 8 ranks the e2e path is bound by host DRAM / PCIe-root locality (VERDICT r1 weak item 9).
    Returns {"node": n, "cpus": k} or None when the topology cannot be read."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local_gpu), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return None
        dev = "/sys/bus/pci/devices/" + bus[-12:]              # 00000000:19:00.0 -> 0000:19:00.0
        node = int(open(dev + "/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus)}
    except Exception:
        return None


def load_oracle():
    from oracle import oracle as O
    return O


def build_ensemble(T, D, F, seed=None):
    import ddt_b200 as ddt
    W, FI = ddt.layout.synth_ensemble(T, D, F) if seed is None else ddt.layout.synth_ensemble(T, D, F, seed=seed)
    return ddt.layout.pack_streams(W, FI, D)


def oracle_throughput(T, D, F, K, S, seconds_target, threads, first_tuple=0, fixed_n=None, blocked=True):
    """tuples/s of the oracle port on `threads` host threads over a bounded sample."""
    import ddt_b200 as ddt
    O = load_oracle()
    L = ddt.layout
    wl, fl = build_ensemble(T, D, F)
    w_cls, f_cls = L.tree_cls(D)
    cfg = O.make_cfg(D, K, S, L.MISSING_DEFAULT, w_cls, f_cls, F // 4, T)
    run = (lambda xx: O.scores_blocked(cfg, wl, fl, xx, threads=threads)) if blocked else (lambda xx: O.scores(cfg, wl, fl, xx, threads=threads))
    if fixed_n is None:
        n0 = max(threads * 64, 256)
        x = L.synth_tuples(first_tuple, n0, F, seed=SEED_TUPLES, missing_ppm=MISSING_PPM)
        t = time.perf_counter(); run(x); dt = time.perf_counter() - t
        n = int(min(max(n0, seconds_target * n0 / max(dt, 1e-6)), 4_000_000))
        n = max(64 * threads, n // (64 * threads) * (64 * threads))
    else:
        n = fixed_n
    x = L.synth_tuples(first_tuple, n, F, seed=SEED_TUPLES, missing_ppm=MISSING_PPM)
    t = time.perf_counter(); s = run(x); dt = time.perf_counter() - t
    return n / dt, n, dt, (cfg, wl, fl, x, s)


def run_reference(args):
    """--impl reference: the oracle port (tree-blocked loop) on the usable host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    O = load_oracle()
    threads = O.max_threads()
    S = T_TREES // (8 * CLUSTERS)
    seconds = float(os.environ.get("DTE_BENCH_REF_SECONDS", "8"))       # CPU work per step (tests shrink it)
    _, n, _, pack = oracle_throughput(T_TREES, DEPTH, FEATS, CLUSTERS, S, seconds, threads)
    cfg, wl, fl, x, _ = pack
    for _ in range(min(args.warmup, 1)):
        O.scores_blocked(cfg, wl, fl, x, threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.scores_blocked(cfg, wl, fl, x, threads=threads)
    dt = time.perf_counter() - t0
    val = n * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "tuples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg3: 1024 trees, D=12 comparison levels, 256 fp32 features; bounded sample of %d tuples per step" % n,
                   "trees": T_TREES, "depth_levels": DEPTH, "features": FEATS, "tuples_per_step": n},
        "cpu_baseline": {"value": val, "unit": "tuples/s", "cores": threads, "online_cpus": O.online_cpus(), "kind": "port",
                         "loop": "tree-blocked (64 tuples x one tree8 group), bit-identical to the per-tuple loop",
                         "sample": "%d tuples of the cfg3 synthetic set per step, %d steps" % (n, args.steps)},
        "e2e": {"value": val, "unit": "tuples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference ships no software implementation of this path (RTL only, not simulable here); "
                "this arm is the RTL-faithful oracle port on the host cores this process may use (affinity and cgroup quota honoured)",
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, warnings) was sent to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)            # libraries that print to fd 1 (e.g. "NCCL version ...") now land on stderr


def oracle_sample(T, D, F, K, S, wl, fl, idx, first=0, ring_chunks=None):
    """Oracle words for the tuples `idx` of the synthetic set (regenerated on the host).  ring_chunks = G: the
    ensemble-sharded reference — per-chunk partials combined in ring order (host first)."""
    import ddt_b200 as ddt
    O = load_oracle()
    L = ddt.layout
    xs = np.stack([L.synth_tuples(first + int(i), 1, F, seed=SEED_TUPLES, missing_ppm=MISSING_PPM)[0] for i in idx])
    w_cls, f_cls = L.tree_cls(D)
    th = O.max_threads()
    if not ring_chunks:
        return O.scores_blocked(O.make_cfg(D, K, S, L.MISSING_DEFAULT, w_cls, f_cls, F // 4, T), wl, fl, xs, threads=th)
    parts = []
    wl2, fl2 = wl.reshape(T, -1), fl.reshape(T, -1)
    for g in range(ring_chunks):
        first_t, count = ddt.sharding.ensemble_chunk(T, g, ring_chunks)
        cw = np.ascontiguousarray(wl2[first_t:first_t + count]).reshape(-1, 4)
        cf = np.ascontiguousarray(fl2[first_t:first_t + count]).reshape(-1, 8)
        parts.append(O.scores_blocked(O.make_cfg(D, K, S, L.MISSING_DEFAULT, w_cls, f_cls, F // 4, count), cw, cf, xs, threads=th))
    return O.ring_combine(parts)


def sample_indices(n, k):
    return np.unique(np.concatenate([np.arange(min(64, n)), np.arange(0, n, max(1, n // max(1, k - 64)))]))[:k]


def dump_outputs(out_dir, d_scores, d_labels, n, n_requested):
    """Scores and labels of the last timed step for a fixed, seeded sample of its n tuples (see --dump-outputs).  The
    sample is drawn from the requested tuple count, so a step shortened for lack of device memory keeps the sampled
    tuples that it still holds."""
    import torch
    if n_requested <= DUMP_TUPLES:
        idx = np.arange(n)
    else:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n_requested, DUMP_TUPLES, replace=False))
        idx = idx[idx < n]
    sel = torch.from_numpy(idx).to(d_scores.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scores.npy"), d_scores[sel].cpu().numpy())
    np.save(os.path.join(out_dir, "labels.npy"), d_labels[sel].cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "tuple_index.npy"), idx.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tuples", type=int, default=0, help="tuples per GPU per step (default: 50M, reduced only if a step would take > 30 s)")
    ap.add_argument("--e2e-tuples", type=int, default=4_000_000)
    ap.add_argument("--variant", type=int, default=0, help="force a kernel variant (dte_kernel_variant)")
    ap.add_argument("--no-ensemble-mode", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip cfg2 / cfg4-shard / stream-path / full-output equality legs")
    ap.add_argument("--trees", type=int, default=T_TREES)
    ap.add_argument("--depth", type=int, default=DEPTH)
    ap.add_argument("--features", type=int, default=FEATS)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's scores and labels as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs dumps the GPU path; the reference arm times a CPU sample sized by the clock")
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    affinity0 = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local) if os.environ.get("DTE_BENCH_NUMA", "1") != "0" else None

    import torch
    import ddt_b200 as ddt
    from ddt_b200 import engine as E

    if not torch.cuda.is_available():
        emit({"error": "no CUDA device; the engine has no CPU fallback"})
        return 1
    torch.cuda.set_device(local)
    dist = None
    host_group = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout = the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")                 # host-only barrier: an NCCL barrier spins ON the GPUs

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def max_over_ranks(v):
        if dist is None:
            return float(v)
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    T, D, F, K = args.trees, args.depth, args.features, CLUSTERS
    S = -(-T // (8 * K))
    L = ddt.layout
    wl, fl = build_ensemble(T, D, F)
    e = ddt.Engine(local)
    e.configure(T, D, 4 * F, clusters=K, missing_value=L.MISSING_DEFAULT, n_tuples=N_FULL)
    e.load_ensemble(wl, fl)
    if args.variant:
        e.set_kernel_variant(args.variant)
    kernel_name = e.kernel_name()
    st = torch.cuda.current_stream().cuda_stream      # 0 = the legacy default stream; the wrapper names it explicitly

    # ---- size the step: calibrate on 1M tuples ----
    n_cal = 1 << 20
    d_cal = torch.empty((n_cal, F), dtype=torch.int32, device="cuda")
    s_cal = torch.empty(n_cal, dtype=torch.float32, device="cuda")
    e.synth_tuples_device(d_cal, 0, n_cal, F, SEED_TUPLES, MISSING_PPM, L.MISSING_DEFAULT, stream=st)
    e.infer_device(d_cal, n_cal, s_cal, None, stream=st)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(); e.infer_device(d_cal, n_cal, s_cal, None, stream=st); ev1.record(); torch.cuda.synchronize()
    cal_rate = n_cal / (ev0.elapsed_time(ev1) * 1e-3)
    n = args.tuples or N_FULL
    free_b, _ = torch.cuda.mem_get_info()
    n = min(n, int((free_b - (12 << 30)) // (F * 4 + 8)))
    if not args.tuples and n / cal_rate > 30.0:
        n = max(1 << 22, int(cal_rate * 30.0))
    if dist is not None:                                   # every rank must time the same shard size
        tn = torch.tensor([n], dtype=torch.int64, device="cuda")
        dist.all_reduce(tn, op=dist.ReduceOp.MIN)
        n = int(tn.item())
    del d_cal, s_cal

    # ---- resident inputs: this rank's shard of the synthetic set (rank r owns tuples [r*n, (r+1)*n)) ----
    d_x = torch.empty((n, F), dtype=torch.int32, device="cuda")
    d_s = torch.empty(n, dtype=torch.float32, device="cuda")
    d_l = torch.empty(n, dtype=torch.uint8, device="cuda")
    e.synth_tuples_device(d_x, rank * n, n, F, SEED_TUPLES, MISSING_PPM, L.MISSING_DEFAULT, stream=st)
    torch.cuda.synchronize()

    def step():
        e.infer_device(d_x, n, d_s, d_l, stream=st)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    launches0 = e.info()["kernel_launches"]
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    evs[0].record()
    for i in range(args.steps):
        step()
        evs[i + 1].record()
    barrier()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:                    # before any later leg reuses d_s / d_l
        dump_outputs(args.dump_outputs, d_s, d_l, n, args.tuples or N_FULL)
    total_ms = evs[0].elapsed_time(evs[-1])
    per_launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    launches = e.info()["kernel_launches"] - launches0
    total_ms = max_over_ranks(total_ms)
    value = world * n * args.steps / (total_ms * 1e-3)

    # ---- parity of the timed output against the oracle (rank 0): >= 4096 sampled tuples, raw words and labels ----
    parity = None
    if rank == 0 and not args.no_cpu:
        O = load_oracle()
        idx = sample_indices(n, 4096)
        want = oracle_sample(T, D, F, K, S, wl, fl, idx, first=rank * n)
        sel = torch.from_numpy(idx).cuda()
        got = d_s[sel].cpu().numpy().view(np.uint32)
        lab = d_l[sel].cpu().numpy()
        parity = {"sampled": int(idx.size), "score_words_equal": int((got == want).sum()), "labels_equal": int((lab == O.labels(want)).sum())}

    # ---- full-output equality across kernel variants: all n scores of the shipped staged kernel vs the
    #      independent global-memory tile kernel (and the generic kernel on a slice) ----
    variants_equal = None
    if rank == 0 and not args.no_extras and not args.variant:
        d_s2 = torch.empty(n, dtype=torch.float32, device="cuda")
        e.set_kernel_variant(E.DTE_KERNEL_TILE)
        e.infer_device(d_x, n, d_s2, None, stream=st)
        torch.cuda.synchronize()
        eq_tile = bool(torch.equal(d_s2.view(torch.int32), d_s.view(torch.int32)))
        n_g = min(n, 2_000_000)
        e.set_kernel_variant(E.DTE_KERNEL_GENERIC)
        e.infer_device(d_x, n_g, d_s2, None, stream=st)
        torch.cuda.synchronize()
        eq_gen = bool(torch.equal(d_s2[:n_g].view(torch.int32), d_s[:n_g].view(torch.int32)))
        e.set_kernel_variant(E.DTE_KERNEL_AUTO)
        variants_equal = {"tile_vs_tile_staged": {"tuples": int(n), "all_score_words_equal": eq_tile,
                                                  "sum_of_words": int(d_s.view(torch.int32).to(torch.int64).sum().item())},
                          "generic_vs_tile_staged": {"tuples": int(n_g), "all_score_words_equal": eq_gen}}
        del d_s2

    # ---- e2e: host buffers through dte_infer_host (H2D + walk + D2H inside the timed region) ----
    n_e = min(args.e2e_tuples, n)
    h_x = torch.empty((n_e, F), dtype=torch.int32, pin_memory=True)
    h_x.copy_(d_x[:n_e])
    h_s = torch.empty(n_e, dtype=torch.float32, pin_memory=True)
    h_l = torch.empty(n_e, dtype=torch.uint8, pin_memory=True)
    for _ in range(2):
        e.infer_host(h_x, out_scores=h_s, out_labels=h_l)
    barrier()
    e2e_steps = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e.infer_host(h_x, out_scores=h_s, out_labels=h_l)
    torch.cuda.synchronize()
    e2e_mine = time.perf_counter() - t0
    e2e_dt = max_over_ranks(e2e_mine)
    e2e_val = world * n_e * e2e_steps / e2e_dt
    e2e_ok = bool(torch.equal(h_s.view(torch.int32), d_s[:n_e].cpu().view(torch.int32)))
    per_rank_h2d = None
    if dist is not None:
        lst = [None] * world
        dist.all_gather_object(lst, n_e * F * 4 * e2e_steps / e2e_mine / 1e9)
        per_rank_h2d = [round(v, 2) for v in lst]

    # ---- e2e through the REFERENCE-SHAPED path: registers -> start -> ONE line stream -> result packets ----
    e2e_stream = None
    if rank == 0 and not args.no_extras:
        n_s = min(n_e, 2_000_000)
        n_s -= n_s % 4
        es = ddt.Engine(local)
        regs = es.configure(T, D, 4 * F, clusters=K, missing_value=L.MISSING_DEFAULT, n_tuples=n_s)
        out_lines = np.empty((n_s // 4, 4), dtype=np.float32)
        last = np.zeros(n_s // 4, dtype=np.uint8)
        trees = np.concatenate([wl.view(np.uint8).reshape(-1, 16), fl.view(np.uint8).reshape(-1, 16)])

        def stream_run(tuple_lines, write_lines):
            es.start()
            es.stream_write(trees)
            t0 = time.perf_counter()
            got = 0
            for lo in range(0, tuple_lines.shape[0], write_lines):
                es.stream_write(tuple_lines[lo:lo + write_lines])
            while got < n_s // 4:
                k = es.stream_read_into(out_lines, last, got)       # result lines land in the caller's buffer, no extra copy
                got += k
                if k == 0:
                    break
            return time.perf_counter() - t0, got

        hx_lines = h_x[:n_s].numpy().view(np.uint8).reshape(-1, 16)          # pinned
        pg_lines = np.array(hx_lines, copy=True)                                # pageable copy of the same lines
        res = {}
        for label, buf in (("pinned", hx_lines), ("pageable", pg_lines)):
            stream_run(buf, 1 << 24)
            dt_s, got = stream_run(buf, 1 << 24)
            ok = got == n_s // 4 and bool((out_lines.reshape(-1).view(np.uint32) == d_s[:n_s].cpu().numpy().view(np.uint32)).all())
            res[label] = {"tuples_per_s": n_s / dt_s, "bit_equal_to_device_path": ok}
        # the fast path on the same inputs, for the ratio
        es.load_ensemble(wl, fl)
        ref = {}
        for label, buf in (("pinned", h_x[:n_s]), ("pageable", pg_lines.view(np.uint32).reshape(n_s, F))):
            es.infer_host(buf, out_scores=h_s[:n_s] if label == "pinned" else None, want_labels=False)
            t0 = time.perf_counter(); es.infer_host(buf, out_scores=h_s[:n_s] if label == "pinned" else None, want_labels=False)
            ref[label] = n_s / (time.perf_counter() - t0)
        e2e_stream = {"api": "dte_softreg_write(201..208), start, dte_stream_write (trees, then tuple lines in 256 MiB writes), dte_stream_read_packets",
                      "tuples_per_step": int(n_s), "value": res["pinned"]["tuples_per_s"], "unit": "tuples/s",
                      "pinned_input": res["pinned"], "pageable_input": res["pageable"],
                      "infer_host_same_input": ref,
                      "ratio_vs_infer_host": {k: res[k]["tuples_per_s"] / ref[k] for k in ref},
                      "last_flags_every": int(np.diff(np.nonzero(last)[0]).max()) if last.sum() > 1 else None,
                      "exec_ns_reg223": es.softreg_read(223), "process_done": es.process_done()}
        es.close()
        del pg_lines

    # ---- other BASELINE configurations on this GPU (so the driver records them): cfg2 and one cfg4 shard ----
    extras = None
    if rank == 0 and not args.no_extras:
        extras = {}
        for tag, (Tx, Dx, Fx, nx) in (("cfg2", (512, 8, 128, min(10_000_000, n * F // 128))), ("cfg4_shard", (1024, 10, 256, min(n, 20_000_000)))):
            ex = ddt.Engine(local)
            ex.configure(Tx, Dx, 4 * Fx, clusters=K, missing_value=L.MISSING_DEFAULT)
            wx, fx = build_ensemble(Tx, Dx, Fx, seed=0xE5E if tag == "cfg4_shard" else None)
            ex.load_ensemble(wx, fx)
            dxx = d_x.view(-1)[: nx * Fx].view(nx, Fx)          # the same random words, re-read with Fx features per tuple
            sx = torch.empty(nx, dtype=torch.float32, device="cuda")
            for _ in range(2):
                ex.infer_device(dxx, nx, sx, None, stream=st)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                ex.infer_device(dxx, nx, sx, None, stream=st)
            b.record(); torch.cuda.synchronize()
            ms = a.elapsed_time(b) / 3
            bytes_x = algorithmic_bytes_per_tuple(Tx, Dx, Fx)
            pk, _ = measured_peaks()
            ok = None
            if not args.no_cpu:
                O = load_oracle()
                idx = sample_indices(nx, 512)
                xs = dxx[torch.from_numpy(idx).cuda()].cpu().numpy().view(np.uint32)
                w_cls, f_cls = L.tree_cls(Dx)
                want = O.scores_blocked(O.make_cfg(Dx, K, -(-Tx // (8 * K)), L.MISSING_DEFAULT, w_cls, f_cls, Fx // 4, Tx), wx, fx, xs, threads=O.max_threads())
                ok = int((sx[torch.from_numpy(idx).cuda()].cpu().numpy().view(np.uint32) == want).sum())
            extras[tag] = {"workload": "%d trees, D=%d, %d features, %d tuples resident" % (Tx, Dx, Fx, nx), "ms_per_step": ms,
                           "tuples_per_s": nx / (ms * 1e-3), "kernel": ex.kernel_name(),
                           "roofline_frac_model_B": nx * bytes_x / (ms * 1e-3) / 1e9 / pk, "oracle_words_equal_of_512": ok}
            ex.close()
            del sx

    # ---- ensemble-sharded configuration (BASELINE configs[3]): 1024 trees per GPU, D=10 ----
    ens = None
    if world > 1 and not args.no_ensemble_mode:
        ens = ensemble_sharded(args, ddt, E, dist, torch, rank, world, local, d_x, d_s, d_l, n, F, K, st, barrier, max_over_ranks)

    # ---- ONE process driving every GPU through the multi-device C-ABI handle (rank 0; the others wait) ----
    multi = None
    if world > 1 and not args.no_ensemble_mode:
        barrier()
        if rank == 0:
            try:
                multi = c_abi_multi(ddt, E, torch, world, F, K, wl, fl, T, D, h_x, n_e)
            except Exception as ex:                               # noqa: BLE001
                multi = {"error": str(ex)}
        dist.barrier(group=host_group)         # the idle ranks wait on the host, their GPUs stay free for rank 0's handle
        barrier()

    if rank == 0:
        bytes_b = algorithmic_bytes_per_tuple(T, D, F)
        peak, peak_src = measured_peaks()
        launch_ms = float(np.mean(per_launch_ms))
        achieved = (n * bytes_b / (launch_ms * 1e-3)) / 1e9
        tr = load_profile_json("ncu_traffic.json") or {}
        dram_per_tuple = tr.get("dram_bytes_per_tuple")
        traffic = dram_per_tuple * n if dram_per_tuple else None
        pipe = load_profile_json("ncu_pipe.json") or {}
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        roofline_pipe = None
        if pipe.get("pipe_wavefronts_per_tuple"):
            wpt = pipe["pipe_wavefronts_per_tuple"]
            ach = wpt * n / (launch_ms * 1e-3)
            pk_pipe = SM_COUNT * sm_mhz * 1e6
            roofline_pipe = {"bound": "l1_shared_data_pipe", "unit": "wavefronts/s", "achieved": ach, "peak": pk_pipe, "frac": ach / pk_pipe,
                             "peak_is": "%d SMs x %.0f MHz (sampled under load) x 1 wavefront (128 B) per cycle — the shared-memory/L1 data pipe" % (SM_COUNT, sm_mhz),
                             "wavefronts_per_tuple": wpt, "wavefronts_per_warp_tree": wpt * 32.0 / T if T else None,
                             "breakdown_per_warp_tree": pipe.get("per_warp_tree"), "source": "profiles/ncu_pipe.json (from %s)" % pipe.get("from", "?"),
                             "note": "wavefronts per tuple are MEASURED by ncu on this kernel (LSU data-pipe wavefronts + TMA ring-fill bytes / 128) "
                                     "at the profiled geometry; they scale with trees x levels, so the figure is valid for cfg3 only"}
        info = e.info()
        cpu = None
        if not args.no_cpu and world == 1:
            os.sched_setaffinity(0, affinity0)             # the CPU arm may use every core the job owns, not one NUMA node
            O = load_oracle()
            th = O.max_threads()
            v, ns, dt, _ = oracle_throughput(T, D, F, K, S, 12.0, th)
            v1, ns1, dt1, _ = oracle_throughput(T, D, F, K, S, 4.0, 1)
            vp, nsp, dtp, _ = oracle_throughput(T, D, F, K, S, 3.0, th, blocked=False)
            # BASELINE configs[0]: 16 trees, depth 4, 32 features, 10k tuples, ONE host thread, median of 21 runs
            W1, FI1 = L.synth_ensemble(16, 4, 32)
            wl1, fl1 = L.pack_streams(W1, FI1, 4)
            x1 = L.synth_tuples(0, 10000, 32)
            w1c, f1c = L.tree_cls(4)
            c1 = O.make_cfg(4, 2, 1, L.MISSING_DEFAULT, w1c, f1c, 8, 16)
            t_cfg1 = []
            for _ in range(21):
                t0 = time.perf_counter(); O.scores_blocked(c1, wl1, fl1, x1, threads=1); t_cfg1.append(time.perf_counter() - t0)
            cfg1_rate = 10000 / float(np.median(t_cfg1))
            cpu = {"value": v, "unit": "tuples/s", "cores": th, "online_cpus": O.online_cpus(), "kind": "port",
                   "loop": "tree-blocked (64 tuples x one tree8 group at a time; same adds in the same per-tuple order, asserted bit-identical in tests/)",
                   "parallel_speedup": v / v1 if v1 else None,
                   "per_tuple_loop_value": vp,
                   "cfg1_single_thread": {"value": cfg1_rate, "unit": "tuples/s", "what": "BASELINE configs[0]: 16 trees, D=4, 32 features, 10k tuples, 1 thread, median of 21 runs"},
                   "sample": "%d tuples of the same synthetic set in %.1f s on %d threads (oracle/dte_oracle.c); single thread: %.0f tuples/s on %d tuples; "
                             "per-tuple (cache-hostile) loop on %d threads: %.0f tuples/s" % (ns, dt, th, v1, ns1, th, vp),
                   "single_thread_value": v1,
                   "reference_model_fpga": {"value": 150e6 * 8 * 8 / (D * T), "unit": "tuples/s",
                                            "what": "the reference's own analytical law f*Ncu*Npe/(depth*Ntrees) at 150 MHz, 8x8 PEs (profiler/profiler.cpp:97-102); modelled, Catapult v1.2"}}
        line = {
            "metric": METRIC, "value": value, "unit": "tuples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": ("cfg3" if world == 1 else "cfg5 (data-sharded, ensemble replicated, no collective)") +
                                   ": %d trees, D=%d comparison levels, %d fp32 features, %d tuples per GPU per step" % (T, D, F, n),
                       "trees": T, "depth_levels": D, "features": F, "tuples_per_gpu": n, "clusters": K, "trees_per_pu": S,
                       "missing_ppm": MISSING_PPM, "l2": "inputs (%.1f GB per GPU) far larger than L2; no flush needed" % (n * F * 4 / 1e9),
                       "kernel": kernel_name, "tuples_per_cta": info["tuples_per_cta"],
                       "tune": os.environ.get("DTE_TUNE", ""), "numa_binding": numa},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_tuple": bytes_b,
                         "kernel": "dt_walk_tile" if info["kernel_variant"] != 1 else "dt_walk_generic",
                         "launch_ms": launch_ms, "tuples_per_launch": n,
                         "dram_frac": (dram_per_tuple * n / (launch_ms * 1e-3) / 1e9 / peak) if dram_per_tuple else None,
                         "note": "byte model (B) of SURVEY 8d charges every node visit (10 B) and leaf (4 B) as HBM traffic; the engine serves "
                                 "them from shared memory / L2, so frac exceeds 1 and is NOT a physical bound — `traffic`/`dram_frac` are the DRAM "
                                 "bytes ncu measured (profiles/ncu_traffic.json) and `roofline_pipe` is the physical roofline of this kernel"},
            "roofline_pipe": roofline_pipe,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_val, "unit": "tuples/s", "h2d_bytes_per_step": int(n_e * F * 4 * world),
                    "d2h_bytes_per_step": int(n_e * 5 * world), "tuples_per_step": int(n_e * world), "steps": e2e_steps,
                    "bit_equal_to_device_path": e2e_ok, "per_rank_h2d_gbs": per_rank_h2d,
                    "api": "dte_infer_host (pinned host buffers; H2D, walk, D2H pipelined inside the call)"},
            "e2e_stream": e2e_stream,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "parity_spot_check": parity,
            "variants_full_output": variants_equal,
            "extra": extras,
            "calibration_tuples_per_s": cal_rate,
        }
        if ens:
            line["ensemble_sharded"] = ens
        if multi:
            line["c_abi_multi"] = multi
        emit(line)
    e.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def ensemble_sharded(args, ddt, E, dist, torch, rank, world, local, d_x, d_s, d_l, n, F, K, st, barrier, max_over_ranks):
    """BASELINE configs[3]: 1024 trees per GPU (8192 at 8 GPUs), D = 10, every GPU walks every tuple.
    Combine A: ring order, ONE kernel on rank 0 reading every rank's partials over NVLink (CUDA IPC) — bit-exact with
    the reference ring.  Combine B: ONE ncclReduce(SUM) (north_star's wording; order free).  Both checked against the
    oracle ring on a >= 4096-tuple sample.  e2e: each rank uploads 1/G of the tuples over its own PCIe link, an
    NCCL all-gather over NVLink replaces the reference's ring broadcast (InputDistributor.sv:199-204)."""
    L = ddt.layout
    De, Te = 10, 1024 * world
    wle, fle = build_ensemble(Te, De, F, seed=0xE5E)
    first, count = ddt.sharding.ensemble_chunk(Te, rank, world)
    Ke, Se = ddt.sharding.shard_geometry(Te, De, K, world)
    ee = ddt.Engine(local)
    ee.configure(count, De, 4 * F, clusters=Ke, missing_value=L.MISSING_DEFAULT)
    ee.softreg_write(205, (L.MISSING_DEFAULT) | (De << 32) | (Se << 36) | (Ke << 44))
    ee.load_ensemble(wle, fle, first_tree=first, num_local_trees=count)
    ne = min(n, 20_000_000)
    ne -= ne % 4
    # every device sees every tuple: same seed/window on all ranks (the broadcast itself is timed in the e2e leg)
    ee.synth_tuples_device(d_x, 0, ne, F, SEED_TUPLES, MISSING_PPM, L.MISSING_DEFAULT, stream=st)
    part = d_s[:ne]
    steps = 3

    def timed(fn):
        for _ in range(2):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / steps * 1e3
        return max_over_ranks(a.elapsed_time(b) / steps), max_over_ranks(wall)

    # --- B: one NCCL reduce; everything on the default stream, so the reduce, the labels and the next walk are ordered ---
    def estep():
        ee.infer_device(d_x, ne, part, None, stream=st)
        dist.reduce(part, dst=0, op=dist.ReduceOp.SUM)          # ONE collective: ResultsCombiner ring -> NCCL reduce
        if rank == 0:
            ee.labels_device(part, ne, d_l, stream=st)

    nccl_ms, _ = timed(estep)
    idx = sample_indices(ne, 4096)
    sel = torch.from_numpy(idx).cuda()
    nccl_scores = part[sel].cpu().numpy() if rank == 0 else None
    nccl_labels = d_l[sel].cpu().numpy() if rank == 0 else None

    # --- A: ring-order combine, one peer-read kernel ---
    ring_ms = ring_wall = None
    combine_ms = None
    ring_err = None
    ring_scores = ring_labels = None
    try:
        rc = ddt.sharding.RingCombine(ee, dist, ne)
        out = torch.empty(ne, dtype=torch.float32, device="cuda") if rank == 0 else None
        ring_ms, ring_wall = timed(lambda: rc.step(d_x, ne, st, out, d_l if rank == 0 else None))
        if rank == 0:
            ring_scores = out[sel].cpu().numpy().view(np.uint32)
            ring_labels = d_l[sel].cpu().numpy()
        # the combine kernel alone (the partials are in place, the peers idle at the barrier): its roofline is the NVLink
        # read of world-1 peer vectors, against the 770 GB/s peer-copy figure of B200_PROFILING.md
        barrier()
        if rank == 0:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ee.ring_combine_device(rc.ptrs, ne, out, d_l, stream=st)
            a.record()
            for _ in range(5):
                ee.ring_combine_device(rc.ptrs, ne, out, d_l, stream=st)
            b.record(); torch.cuda.synchronize()
            combine_ms = a.elapsed_time(b) / 5
        barrier()
    except Exception as ex:                                        # noqa: BLE001  (IPC not permitted etc.)
        ring_err = str(ex)
        rc = None

    # --- one GPU holding ALL trees: full ne tuples, averaged over 3 launches ---
    one_ms = None
    if rank == 0:
        e1 = ddt.Engine(local)
        e1.configure(Te, De, 4 * F, clusters=K, missing_value=L.MISSING_DEFAULT)
        e1.load_ensemble(wle, fle)
        tmp = torch.empty(ne, dtype=torch.float32, device="cuda")
        e1.infer_device(d_x, ne, tmp, None, stream=st); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            e1.infer_device(d_x, ne, tmp, None, stream=st)
        b.record(); torch.cuda.synchronize()
        one_ms = a.elapsed_time(b) / 3
        e1.close()
        del tmp
    barrier()

    # --- parity against the oracle ring (rank 0) ---
    parity = None
    nccl_rel = None
    if rank == 0 and not args.no_cpu:
        O = load_oracle()
        want = oracle_sample(Te, De, F, Ke, Se, wle, fle, idx, ring_chunks=world)
        wf = want.view(np.float32)
        nccl_rel = float(np.max(np.abs(nccl_scores - wf) / np.maximum(np.abs(wf), 1e-30)))
        parity = {"sampled": int(idx.size),
                  "nccl_labels_equal": int((nccl_labels == O.labels(want)).sum())}
        if ring_scores is not None:
            parity.update(score_words_equal=int((ring_scores == want).sum()), labels_equal=int((ring_labels == O.labels(want)).sum()))

    # --- e2e: 1/G of the tuples over each PCIe link, all-gather over NVLink, walk, ring combine, scores to the host ---
    e2e = None
    try:
        n_e2e = min(ne, 4_000_000)
        n_e2e -= n_e2e % (4 * world)
        per = n_e2e // world
        h_slice = torch.empty((per, F), dtype=torch.int32, pin_memory=True)
        h_slice.copy_(d_x[rank * per:(rank + 1) * per])
        h_out = torch.empty(n_e2e, dtype=torch.float32, pin_memory=True) if rank == 0 else None
        d_full = d_x[:n_e2e]
        d_mine = torch.empty((per, F), dtype=torch.int32, device="cuda")
        out = torch.empty(n_e2e, dtype=torch.float32, device="cuda") if rank == 0 else None
        rc2 = ddt.sharding.RingCombine(ee, dist, n_e2e)

        def e2e_step():
            d_mine.copy_(h_slice, non_blocking=True)                         # own PCIe link
            dist.all_gather_into_tensor(d_full.view(-1), d_mine.view(-1))    # NVLink broadcast of every slice
            rc2.step(d_full, n_e2e, st, out, None)
            if rank == 0:
                h_out.copy_(out, non_blocking=True)
            torch.cuda.synchronize()

        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            e2e_step()
        dt = max_over_ranks((time.perf_counter() - t0) / 3)
        ok = None
        if rank == 0 and ring_scores is not None:
            ok = bool(torch.equal(h_out.view(torch.int32), out.cpu().view(torch.int32)))
        e2e = {"value": n_e2e / dt, "unit": "tuples/s", "tuples_per_step": int(n_e2e), "h2d_bytes_per_step": int(n_e2e * F * 4),
               "h2d_bytes_per_gpu_per_step": int(per * F * 4), "d2h_bytes_per_step": int(n_e2e * 4), "nvlink_allgather_bytes_per_gpu": int((n_e2e - per) * F * 4),
               "scores_reach_host": ok,
               "what": "pinned host slices -> H2D (1/G per GPU, own PCIe link) -> ncclAllGather over NVLink -> walk (all tuples, 1024 trees/GPU) -> ring combine -> D2H"}
        rc2.close()
    except Exception as ex:                                        # noqa: BLE001
        e2e = {"error": str(ex)}

    # --- the older fused-epilogue combine (red.add over NVLink into rank 0's buffer), kept for comparison ---
    fused_ms = None
    try:
        fc = ddt.sharding.FusedCombine(ee, dist, ne, dst=0)
        fused_ms, _ = timed(lambda: fc.step(d_x, ne, st))
        fc.close()
    except Exception:                                              # noqa: BLE001
        fused_ms = None
    if rc is not None:
        rc.close()
    ee.close()
    return {"workload": "cfg4: %d trees split %d/GPU, D=10, 256 features, %d tuples on every GPU" % (Te, count, ne),
            "ms_per_step": ring_ms if ring_ms else nccl_ms, "tuples_per_s": ne / ((ring_ms if ring_ms else nccl_ms) * 1e-3),
            "combine": "ring-order peer-read kernel (bit-exact)" if ring_ms else "ncclReduce",
            "ring": {"ms_per_step": ring_ms, "wall_ms_per_step": ring_wall, "error": ring_err,
                     "combine_kernel": None if not combine_ms else {
                         "ms": combine_ms, "nvlink_bytes": int((world - 1) * 4 * ne), "nvlink_gbs": (world - 1) * 4 * ne / (combine_ms * 1e-3) / 1e9,
                         "roofline": {"bound": "nvlink", "peak": 770.0, "unit": "GB/s", "frac": (world - 1) * 4 * ne / (combine_ms * 1e-3) / 1e9 / 770.0,
                                      "peak_source": "measured peer copy per direction per GPU, B200_PROFILING.md"},
                         "what": "ring_combine_kernel on rank 0: reads %d peer vectors of fp32[%d] over NVLink, adds them in ring order, writes scores + labels" % (world - 1, ne)},
                     "what": "walk -> host barrier -> ONE ring_combine_kernel on rank 0 reading %d peer buffers over NVLink (CUDA IPC) + labels -> host barrier" % (world - 1)},
            "nccl": {"ms_per_step": nccl_ms, "what": "walk -> ONE ncclReduce(SUM) of fp32[%d] to rank 0 -> labels" % ne},
            "ring_vs_nccl_ms": (ring_ms / nccl_ms) if ring_ms else None,
            "one_gpu_all_trees_ms": one_ms, "one_gpu_note": "all %d trees on one GPU, the same %d tuples, mean of 3 launches (measured, not extrapolated)" % (Te, ne),
            "speedup_vs_one_gpu": (one_ms / (ring_ms if ring_ms else nccl_ms)) if one_ms else None,
            "speedup_vs_one_gpu_nccl": (one_ms / nccl_ms) if one_ms else None,
            "parity": parity, "nccl_vs_oracle_max_rel": nccl_rel,
            "e2e": e2e,
            "fused_epilogue_ms_per_step": fused_ms}


def c_abi_multi(ddt, E, torch, world, F, K, wl, fl, T, D, h_x, n_e):
    """Rank 0 only: ONE process, ONE handle (dte_create_multi) over all GPUs of the box — the configuration a C/C++
    host uses.  Host buffers in, host buffers out, through dte_infer_host; both partitions of SURVEY 8(e)."""
    L = ddt.layout
    out = {}
    n = int(n_e)
    h_s = torch.empty(n, dtype=torch.float32, pin_memory=True)
    h_l = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    O = load_oracle()
    idx = sample_indices(n, 1024)
    xs = h_x[torch.from_numpy(idx)].numpy().view(np.uint32)
    w_cls, f_cls = L.tree_cls(D)
    for mode in ("data", "ensemble"):
        eng = ddt.Engine(list(range(world)))
        if mode == "data":
            Tm, Dm, wm, fm = T, D, wl, fl
            flags = 0x2 | 0x20 | 0x40 | 0x8
            Sm = -(-Tm // (8 * K))
        else:
            Tm, Dm = 1024 * world, 10
            wm, fm = build_ensemble(Tm, Dm, F, seed=0xE5E)
            flags = 0x2 | 0x20 | 0x40 | 0x4 | 0x10
            Sm = -(-1024 // (8 * K))
        regs = E.csr_from_profile(Tm, Dm, 4 * F, K, L.MISSING_DEFAULT, n)
        regs[201] = flags | ((4096 * (F // 4)) << 32)
        regs[203] = world << 32          # numDevs; chunk fields 0 = "cut the trees evenly" (1024 trees/GPU do not fit the 16-bit line counts)
        regs[205] = (regs[205] & ~(0xFF << 36)) | (Sm << 36)
        for a, v in sorted(regs.items()):
            eng.softreg_write(a, v)
        eng.load_ensemble(wm, fm)
        for _ in range(2):
            eng.infer_host(h_x, out_scores=h_s, out_labels=h_l)
        t0 = time.perf_counter()
        for _ in range(3):
            eng.infer_host(h_x, out_scores=h_s, out_labels=h_l)
        dt = (time.perf_counter() - t0) / 3
        wcm, fcm = L.tree_cls(Dm)
        if mode == "data":
            want = O.scores_blocked(O.make_cfg(Dm, K, Sm, L.MISSING_DEFAULT, wcm, fcm, F // 4, Tm), wm, fm, xs, threads=O.max_threads())
        else:
            parts = []
            w2, f2 = wm.reshape(Tm, -1), fm.reshape(Tm, -1)
            for g in range(world):
                lo = g * 1024
                cw = np.ascontiguousarray(w2[lo:lo + 1024]).reshape(-1, 4)
                cf = np.ascontiguousarray(f2[lo:lo + 1024]).reshape(-1, 8)
                parts.append(O.scores_blocked(O.make_cfg(Dm, K, Sm, L.MISSING_DEFAULT, wcm, fcm, F // 4, 1024), cw, cf, xs, threads=O.max_threads()))
            want = O.ring_combine(parts)
        got = h_s.numpy()[idx].view(np.uint32)
        out[mode] = {"tuples_per_s": n / dt, "tuples_per_step": n, "h2d_bytes_per_step": int(n * F * 4),
                     "workload": "%d trees D=%d, %s" % (Tm, Dm, "replicated, chunks of tuples round-robin over the GPUs" if mode == "data"
                                                         else "1024 trees per GPU, every tuple on every GPU (1/G uploaded per PCIe link + NVLink peer copies), ring combine"),
                     "parity": {"sampled": int(idx.size), "score_words_equal": int((got == want).sum()),
                                "labels_equal": int((h_l.numpy()[idx] == O.labels(want)).sum())},
                     "info": {k: eng.info()[k] for k in ("num_devices", "partition", "num_trees")}}
        eng.close()
    out["api"] = "dte_create_multi over %d GPUs, registers 201/203 select the partition, dte_load_ensemble + dte_infer_host (pinned host buffers)" % world
    return out


if __name__ == "__main__":
    sys.exit(main())

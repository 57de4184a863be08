#!/usr/bin/env python
"""bench.py — UTF-8 MB/s segmented (bit-exact i32 scores) for the Predictor::predict hot path.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
    python bench.py --impl reference --gpus N --steps K ...  # reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/*.npy

Workload (BASELINE.json configs[1] / SURVEY.md §8d): bccwj-suw-shaped synthetic model (W=3/3, 300 000 char
1-3-gram patterns, 258 type n-grams, no dictionary, no tags) over synthetic 40-char Japanese sentences,
1 000 000 sentences per GPU (weak scaling; sentences shard trivially, the only collective is the one-time
NCCL broadcast of the flat model blob from rank 0).  A "step" is one pass of the hot path over the batch:
one k_fused launch (validation, counts, output offsets, scoring) through vpt_predict_batch_dev with inputs resident in HBM (`value`),
and through vpt_predict_batch with pinned HOST buffers, copies inside the timed region (`e2e`).
The batch (115 MB in, 195 MB out) is larger than L2 (126 MB), so no L2 flush is needed between steps.
"""
from __future__ import annotations

import argparse
import ctypes as C
import functools
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

# Generated models are cached outside the source tree (which may be read-only), per user.  The file name carries a hash
# of the generator's source, so two builds of the project never read each other's model.
CACHE = os.path.join(tempfile.gettempdir(), f"vaporetto_b200_bench_cache_{os.getuid()}")
METRIC = "UTF-8 MB/s segmented (bit-exact i32 scores)"
DUMP_BYTES = 64_000_000
DUMP_SEED = 0x5EED0D0


def log(*a):
    print(*a, file=sys.stderr, flush=True)


@functools.lru_cache(maxsize=None)
def get_model(n_patterns: int, sample: int, config: int = 2) -> bytes:
    from vpt_testlib import synth
    tag = {2: "bccwj_shaped", 3: "bccwj_tags_shaped", 4: "kytea_shaped"}[config]
    src = hashlib.sha256(open(synth.__file__, "rb").read()).hexdigest()[:16]
    fn = os.path.join(CACHE, f"{tag}_{n_patterns}_{sample}_{src}.bin")
    if os.path.exists(fn):
        return open(fn, "rb").read()
    t = time.time()
    m = synth.gen_model_bccwj_shaped(n_patterns=n_patterns, sample_sentences=sample,
                                     dict_words=500_000 if config == 4 else 0, tag_models=20_000 if config == 3 else 0)
    log(f"[bench] generated model ({len(m)} bytes) in {time.time() - t:.1f}s")
    try:
        os.makedirs(CACHE, exist_ok=True)
        with open(fn + ".tmp", "wb") as f:
            f.write(m)
        os.replace(fn + ".tmp", fn)
    except OSError:
        pass
    return m


def dump_outputs(out_dir: str, arrays, budget: int = DUMP_BYTES, prefix: str = "") -> None:
    """Writes the outputs of one step as <out_dir>/<prefix><name>.npy in float64, exact for every i32 / u32 value and for
    offsets below 2^53.  `arrays`: {name: (tensor, numpy dtype its elements are read as)}.  An array larger than its share
    of `budget` bytes is written as its values at a fixed, seeded sample of positions (ascending), the positions beside it
    as <name>_index.npy; the same arguments give the same positions, so two builds can be compared output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = budget // len(arrays)
    for name, (t, dtype) in arrays.items():
        t = t.reshape(-1)
        n = t.numel()
        if 8 * n + 128 > share:   # (128: the .npy header)
            k = (share - 256) // 16
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))
            np.save(os.path.join(out_dir, f"{prefix}{name}_index.npy"), idx.astype(np.float64))
            t = t[torch.from_numpy(idx).to(t.device)]
        v = t.cpu().numpy().view(dtype).astype(np.float64)
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), v)


def get_text(n_sent: int, rank: int, ragged: bool):
    from vpt_testlib import synth
    t = time.time()
    text, offs, lens = synth.gen_text(n_sent, 40, seed=synth.TEXT_SEED + 7919 * rank, ragged=ragged)
    log(f"[bench] rank {rank}: generated {n_sent} sentences, {len(text)} bytes in {time.time() - t:.1f}s")
    return text, offs, lens


TILE_SENTENCES = 1_000_000


def get_text_shard(n_per_gpu: int, rank: int, world: int, ragged: bool):
    """BASELINE configs[4]: ONE global batch of n_per_gpu x world sentences, sharded over the ranks by bytes
    (vaporetto_b200.shard_by_bytes).  The global batch is a 1 M-sentence synthetic block repeated; the shard
    boundaries are computed on the block boundaries (every block boundary is a sentence boundary), and a rank
    materialises only its own blocks."""
    import vaporetto_b200 as vb
    if n_per_gpu <= TILE_SENTENCES or n_per_gpu % TILE_SENTENCES:
        return get_text(n_per_gpu, rank, ragged)
    base_text, base_offs, _ = get_text(TILE_SENTENCES, 0, ragged)
    ntiles = n_per_gpu // TILE_SENTENCES * world
    tile_bytes = int(base_offs[-1])
    lo, hi = vb.shard_by_bytes(np.arange(ntiles + 1, dtype=np.uint64) * np.uint64(tile_bytes), rank, world)
    k = hi - lo
    text = np.tile(base_text[:tile_bytes], k)
    offs = (np.arange(k, dtype=np.uint64)[:, None] * np.uint64(tile_bytes) + base_offs[None, :-1].astype(np.uint64)).reshape(-1)
    offs = np.concatenate([offs, np.array([k * tile_bytes], np.uint64)])
    log(f"[bench] rank {rank}: blocks [{lo}, {hi}) of {ntiles}: {len(offs) - 1} sentences, {len(text)} bytes")
    return text, offs, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


CPU_NOTE = ("C++ restatement of the reference algorithm (oracle/vaporetto_oracle.cpp: parse_raw + predict per sentence, "
            "Aho-Corasick automaton walked as a double array with a code-point mapper -- the layout of the reference's "
            "daachorse CharwiseDoubleArrayAhoCorasick: 16-byte states, child = base XOR code --, merged weights, type "
            "table), text pre-loaded; one pinned thread pool for the whole measurement, sentences handed out in blocks of "
            "256.  The Rust reference cannot be built here (no cargo/rustc): a port, not the reference binary")


def usable_cpus():
    """CPUs this process can really use: the affinity mask, capped by the cgroup CPU quota (cpu.max) if there is one."""
    n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = max(1, int(float(q) / float(per) + 0.5))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = max(1, int(q / per + 0.5))
        except Exception:
            pass
    return n, quota


def cpu_thread_counts(ncpu, quota):
    """Thread counts to try: powers of four up to the CPUs, the cgroup quota if there is one, and all CPUs."""
    c = {1, ncpu}
    t = 4
    while t < ncpu:
        c.add(t)
        t *= 4
    if quota:
        c.add(min(quota, ncpu))
        c.add(min(2 * quota, ncpu))
    return sorted(c)


def cpu_scaling(o, text, offs, budget_s):
    """MB/s of the CPU port per thread count on bounded samples (about budget_s seconds in total).  On a box whose
    container has a CPU quota below its CPU count, more threads than the quota run SLOWER (they are throttled): the
    best count is what the CPU arm uses."""
    n = len(offs) - 1
    ncpu, quota = usable_cpus()
    counts = cpu_thread_counts(ncpu, quota)
    out = {}
    n1 = min(n, 20_000)
    o.bench_batch(text, offs[: n1 + 1], nthreads=1, reps=1)  # warm the tables
    t1 = min(o.bench_batch(text, offs[: n1 + 1], nthreads=1, reps=3))
    mb1 = float(offs[n1] - offs[0]) / t1 / 1e6
    out["1"] = round(mb1, 2)
    per = budget_s / max(len(counts) - 1, 1)
    for nt in counts[1:]:
        nn = int(min(n, max(n1, mb1 * min(nt, quota or nt) * 0.8 * 1e6 * per / 2.0 / 115.0)))   # ~per/2 seconds per repetition
        secs = o.bench_batch(text, offs[: nn + 1], nthreads=nt, reps=2)
        out[str(nt)] = round(float(offs[nn] - offs[0]) / min(secs) / 1e6, 2)
    best = max(out, key=lambda k: out[k])
    return out, int(best), ncpu, quota


def cpu_baseline(model_bytes: bytes, text, offs, budget_s: float = 16.0, predict_tags: bool = False):
    """Reference algorithm (C++ restatement, oracle/) on the host cores over a bounded sample of the workload."""
    from vpt_testlib.oracle import OraclePredictor
    t = time.time()
    o = OraclePredictor(model_bytes, predict_tags=predict_tags)
    build_s = time.time() - t
    n = len(offs) - 1
    scal, best, ncpu, quota = cpu_scaling(o, text, offs, budget_s * 0.5)
    # the best thread count: repetitions of >= 2 s each (>= 1 M sentences when the step has them), best of 3
    nall = int(min(n, max(1_000_000, scal[str(best)] * 1e6 * 2.0 / 115.0)))
    reps = 3
    nbytes = float(offs[nall] - offs[0])
    # (a repetition is at least 2 s: several passes of the pool over the sample when one pass is shorter)
    passes = int(min(64, max(1, np.ceil(2.0 / max(nbytes / (scal[str(best)] * 1e6), 1e-3)))))
    allsecs = o.bench_batch(text, offs[: nall + 1], nthreads=best, reps=reps * passes)
    secs = [float(sum(allsecs[i * passes:(i + 1) * passes])) for i in range(reps)]
    nbytes *= passes
    mba = nbytes / min(secs) / 1e6
    eff = mba / (scal["1"] * best)
    return {"value": round(mba, 2), "unit": "MB/s", "cores": best, "kind": "port",
            "sample": f"{passes} passes over {nall} of the step's sentences x {reps} repetitions on {best} threads ({min(secs):.2f}-{max(secs):.2f} s each; "
                      f"the fastest of the thread counts tried: the box shows {ncpu} CPUs, cgroup CPU quota "
                      f"{quota if quota else 'none'}); " + CPU_NOTE,
            "single_thread_MBps": scal["1"], "threads_MBps": scal, "parallel_efficiency": round(eff, 3),
            "cpus_visible": ncpu, "cgroup_cpu_quota": quota, "oracle_build_s": round(build_s, 1)}, o


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm on the host cores, rank 0 only.  A step is one pass of the pinned
    thread pool -- as many passes as make 2 s -- over a bounded sample (>= 1 M sentences when the workload has them), with the
    thread count that is fastest on this box (a container's CPU quota can be far below its CPU count)."""
    if rank != 0:
        return
    model_bytes = get_model(args.patterns, args.model_sample, args.config)
    text, offs, _ = get_text(min(args.sentences, 4_000_000), 0, args.ragged)
    from vpt_testlib.oracle import OraclePredictor
    o = OraclePredictor(model_bytes, predict_tags=False)
    scal, best, ncpu, quota = cpu_scaling(o, text, offs, 8.0)
    n = len(offs) - 1
    rate = scal[str(best)] * 1e6
    # a step must also fit the driver's clock: steps x 2 s
    nstep = int(min(n, max(min(n, 1_000_000), rate * 2.0 / 115.0)))
    sub = offs[: nstep + 1]
    nbytes = float(sub[-1] - sub[0])
    # a step is at least 2 s of wall time: `passes` passes of the thread pool over the sample (a box whose best thread
    # count does 1 M sentences in 0.1 s would otherwise time thread wake-ups)
    passes = int(min(64, max(1, np.ceil(2.0 / max(nbytes / rate, 1e-3)))))
    allsecs = o.bench_batch(text, sub, nthreads=best, reps=(args.warmup + args.steps) * passes)
    secs = [float(sum(allsecs[i * passes:(i + 1) * passes])) for i in range(args.warmup, args.warmup + args.steps)]
    dt = float(sum(secs))
    nbytes *= passes
    v = nbytes * args.steps / dt / 1e6
    out = {"impl": "reference", "metric": METRIC, "value": round(v, 2), "unit": "MB/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32", "data": "synthetic",
           "config": workload_config(args, args.sentences),
           "cpu_baseline": {"value": round(v, 2), "unit": "MB/s", "cores": best, "kind": "port",
                            "sample": f"{passes} passes over {nstep} sentences per step, {best} pinned host threads (fastest of {scal}; {ncpu} CPUs "
                                      f"visible, cgroup CPU quota {quota if quota else 'none'}), step times "
                                      f"{min(secs):.2f}-{max(secs):.2f} s; " + CPU_NOTE,
                            "threads_MBps": scal},
           "e2e": {"value": round(v, 2), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def bind_to_gpu_numa(gpu_index: int):
    """Pins this process (and the pinned host buffers it allocates afterwards: first touch) to the CPUs of the NUMA
    node the GPU hangs off.  Without it the ranks of a multi-GPU run stage through whatever node torchrun started
    them on, and half of them cross the socket interconnect on every copy.  Returns a description for the JSON line."""
    try:
        import vaporetto_b200 as vb
        buf = C.create_string_buffer(32)
        L = vb.lib()
        L.vpt_device_pci_bus_id.argtypes = [C.c_int, C.c_char_p, C.c_size_t]
        if L.vpt_device_pci_bus_id(gpu_index, buf, 32):  # the CUDA device of this rank (CUDA_VISIBLE_DEVICES applied)
            raise RuntimeError(L.vpt_last_error().decode())
        bus = buf.value.decode().lower()
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA information for the GPU"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus_bound": len(allowed)}
    except Exception as e:  # no NVML / sysfs: run unbound
        return {"numa_node": None, "note": f"unbound ({type(e).__name__})"}


def workload_config(args, n_sent):
    extra = {2: "no dict, no tags", 3: "no dict, 20000 tag models, predict_tags (pattern-id states emitted)",
             4: "500000-word KyTea-shaped dictionary, no tags"}[args.config]
    cfg_index = 4 if (args.config == 2 and n_sent > TILE_SENTENCES) else args.config - 1
    shard = ("; one global batch of %d sentences sharded by bytes over %d GPUs" % (n_sent * args.gpus, args.gpus)
             if cfg_index == 4 else "")
    return {"workload": "BASELINE configs[%d]: bccwj-suw-shaped model (W=3/3, %d char 1-3-gram patterns, 258 type "
                        "n-grams, %s), synthetic JP sentences%s%s" %
                        (cfg_index, args.patterns, extra, " (ragged lognormal lengths)" if args.ragged else " of 40 chars", shard),
            "sentences_per_gpu": n_sent, "parallelism": "dp%d (sentences sharded, NCCL model broadcast only)" % args.gpus,
            "l2": "batch (%d MB in + %d MB out per GPU) exceeds L2; no flush needed" % (round(n_sent * 114.8e-6),
                                                                                            round(n_sent * 195e-6))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sentences", type=int, default=0,
                    help="sentences per GPU (default: 1 000 000 on one GPU = BASELINE configs[1]; 8 000 000 on several "
                         "= configs[4], the 64 M-sentence batch of an 8-GPU box sharded by bytes)")
    ap.add_argument("--patterns", type=int, default=300_000)
    ap.add_argument("--model-sample", type=int, default=2_000_000)
    ap.add_argument("--ragged", action="store_true")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4],
                    help="BASELINE.json config: 2 bccwj-suw-shaped (default, the headline), 3 + tag models (states "
                         "emitted), 4 KyTea-shaped (+ 500K-word dictionary)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (scores, boundaries, offsets, status; "
                         "config 3: also the pattern-id states) as DIR/<name>.npy, float64, at most 64 MB in all "
                         "(a fixed, seeded sample of each larger array)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.sentences <= 0:
        args.sentences = 8_000_000 if (world > 1 or args.gpus > 1) and args.config == 2 else 1_000_000

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import vaporetto_b200 as vb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    numa = bind_to_gpu_numa(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- model: rank 0 parses/builds, the flat blob is broadcast once over NCCL -------------------------
    L = vb.lib()
    if rank == 0:
        model_bytes = get_model(args.patterns, args.model_sample, args.config)
        t = time.time()
        pred = vb.Predictor(vb.Model.read(model_bytes), predict_tags=args.config == 3, device=local_rank)
        log(f"[bench] predictor built in {time.time() - t:.1f}s: {pred.info}")
        blob = pred.export_blob()
    if world > 1:
        size = torch.tensor([len(blob) if rank == 0 else 0], dtype=torch.int64, device=dev)
        dist.broadcast(size, 0)
        tb = torch.empty(int(size.item()), dtype=torch.uint8, device=dev)
        if rank == 0:
            tb.copy_(torch.from_numpy(blob))
        dist.broadcast(tb, 0)
        if rank != 0:
            pred = vb.Predictor.from_blob(tb.cpu().numpy(), device=local_rank)
    assert args.config != 2 or pred.info["fast_path"] == 1, "config-2 model must take the fast kernel"

    # ---- data ------------------------------------------------------------------------------------------
    text, offs, _ = get_text_shard(args.sentences, rank, world, args.ragged)
    n = len(offs) - 1
    nbytes = int(offs[-1])
    d_text = torch.zeros(nbytes + 64, dtype=torch.uint8, device=dev)
    d_text[:nbytes] = torch.from_numpy(text).to(dev)
    d_off = torch.from_numpy(offs.astype(np.int64)).to(dev)
    ws = torch.empty(L.vpt_workspace_size(n), dtype=torch.uint8, device=dev)
    d_scores = torch.empty(nbytes, dtype=torch.int32, device=dev)
    d_bounds = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_boff = torch.empty(n + 1, dtype=torch.int64, device=dev)
    d_status = torch.empty(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)
    want_states = args.config == 3  # config 3: pattern-id states are part of the output (tag prediction input)
    d_cst = torch.empty(nbytes, dtype=torch.int32, device=dev) if want_states else None
    d_tst = torch.empty(nbytes, dtype=torch.int32, device=dev) if want_states else None
    d_coff = torch.empty(n + 1, dtype=torch.int64, device=dev) if want_states else None
    p_cst = d_cst.data_ptr() if want_states else None
    p_tst = d_tst.data_ptr() if want_states else None
    p_coff = d_coff.data_ptr() if want_states else None

    def step_dev():
        rc = L.vpt_predict_batch_dev(pred._h, d_text.data_ptr(), d_off.data_ptr(), n, ws.data_ptr(), ws.numel(),
                                     d_scores.data_ptr(), d_bounds.data_ptr(), d_boff.data_ptr(), d_status.data_ptr(),
                                     p_cst, p_tst, p_coff, sp)
        if rc:
            raise RuntimeError(L.vpt_last_error().decode())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_dev()
    barrier()
    n_bound = int(d_boff[-1].item())
    assert int(d_status.abs().sum().item()) == 0
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_dev()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs:   # before the profiled leg below overwrites the buffers
        outs = {"scores": (d_scores[:n_bound], np.int32), "boundaries": (d_bounds[:n_bound], np.uint8),
                "bound_offsets": (d_boff, np.int64), "status": (d_status, np.int32)}
        if want_states:
            n_chars = int(d_coff[-1].item())
            outs.update(char_states=(d_cst[:n_chars], np.uint32), type_states=(d_tst[:n_chars], np.uint32),
                        char_offsets=(d_coff, np.int64))
        dump_outputs(args.dump_outputs, outs, DUMP_BYTES // world, f"rank{rank}_" if world > 1 else "")
        log(f"[bench] rank {rank}: outputs of the last timed step written to {args.dump_outputs}")
    # stage timing of the dominant kernel (CUDA events inside the library, same stream)
    stage = (C.c_float * 3)()
    stage_acc = np.zeros(3)
    reps = max(3, min(args.steps, 10))
    for _ in range(reps):
        rc = L.vpt_predict_batch_dev_profiled(pred._h, d_text.data_ptr(), d_off.data_ptr(), n, ws.data_ptr(), ws.numel(),
                                              d_scores.data_ptr(), d_bounds.data_ptr(), d_boff.data_ptr(),
                                              d_status.data_ptr(), p_cst, p_tst, p_coff, sp, stage)
        if rc:
            raise RuntimeError(L.vpt_last_error().decode())
        stage_acc += np.array(list(stage))
    stage_ms = stage_acc / reps
    clocks = sampler.stop() if rank == 0 else None
    # config 3: the tag prediction kernel alone, on the device-resident states / boundaries of the step above
    k_tags_ms = None
    if want_states and pred.info.get("predict_tags"):
        d_tagtok = torch.empty(n_bound + n, dtype=torch.int32, device=dev)
        d_tagcand = torch.empty((n_bound + n) * max(int(pred.n_tags), 1), dtype=torch.int32, device=dev)
        d_uns = torch.zeros(1, dtype=torch.int32, device=dev)

        def step_ktags():
            rc = L.vpt_predict_tags_batch_dev(pred._h, d_text.data_ptr(), d_off.data_ptr(), n, d_status.data_ptr(),
                                              d_bounds.data_ptr(), d_boff.data_ptr(), p_coff, p_cst, p_tst,
                                              d_tagtok.data_ptr(), d_tagcand.data_ptr(), d_uns.data_ptr(), sp)
            if rc:
                raise RuntimeError(L.vpt_last_error().decode())

        step_ktags()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record(stream)
        for _ in range(5):
            step_ktags()
        t1e.record(stream)
        torch.cuda.synchronize()
        k_tags_ms = t0e.elapsed_time(t1e) / 5

    tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(nbytes)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_all = float(tmax.item())
    total_bytes = float(tot.item())
    value = total_bytes * args.steps / (ms_all / 1e3) / 1e6

    # ---- end to end through the host-buffer C ABI (pinned host memory, copies inside the timed region) ----
    h_text = torch.from_numpy(text).pin_memory()
    h_off = torch.from_numpy(offs.astype(np.int64)).pin_memory()
    h_scores = torch.empty(n_bound, dtype=torch.int32).pin_memory()
    h_bounds = torch.empty(n_bound, dtype=torch.uint8).pin_memory()
    h_boff = torch.empty(n + 1, dtype=torch.int64).pin_memory()
    h_status = torch.empty(n, dtype=torch.int32).pin_memory()
    nb_out, nc_out = C.c_uint64(), C.c_uint64()
    n_chars_total = n_bound + n  # every sentence is non-empty
    h_cst = torch.empty(n_chars_total, dtype=torch.int32).pin_memory() if want_states else None
    h_tst = torch.empty(n_chars_total, dtype=torch.int32).pin_memory() if want_states else None
    h_coff = torch.empty(n + 1, dtype=torch.int64).pin_memory() if want_states else None

    def step_e2e():
        rc = L.vpt_predict_batch(pred._h, h_text.data_ptr(), h_off.data_ptr(), n, h_scores.data_ptr(),
                                 h_bounds.data_ptr(), n_bound, h_boff.data_ptr(), h_status.data_ptr(),
                                 h_cst.data_ptr() if want_states else None, h_tst.data_ptr() if want_states else None,
                                 n_chars_total if want_states else 0, h_coff.data_ptr() if want_states else None,
                                 C.byref(nb_out), C.byref(nc_out))
        if rc:
            raise RuntimeError(L.vpt_last_error().decode())

    step_e2e()
    step_e2e()
    assert np.array_equal(h_bounds.numpy(), d_bounds[:n_bound].cpu().numpy())
    assert np.array_equal(h_scores.numpy(), d_scores[:n_bound].cpu().numpy())
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = total_bytes * args.e2e_steps / float(te.item()) / 1e6
    # same call without the i32 scores in the D2H copy (boundaries + offsets only): what a tokenizer front-end needs
    def step_e2e_nb():
        rc = L.vpt_predict_batch(pred._h, h_text.data_ptr(), h_off.data_ptr(), n, None, h_bounds.data_ptr(), n_bound,
                                 h_boff.data_ptr(), h_status.data_ptr(), None, None, 0, None, C.byref(nb_out), C.byref(nc_out))
        if rc:
            raise RuntimeError(L.vpt_last_error().decode())

    step_e2e_nb()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        step_e2e_nb()
    torch.cuda.synchronize()
    tnb = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tnb, op=dist.ReduceOp.MAX)
    e2e_nb_value = total_bytes * args.e2e_steps / float(tnb.item()) / 1e6
    # compact results (vpt_predict_batch_compact): one bit per boundary, n_chars / status per sentence -- and, for a
    # predictor with tags, one record per token (token id + one byte per tag slot) with the tag prediction on the device
    h_bits = torch.zeros((n_bound + 31) // 32 + 1, dtype=torch.int32).pin_memory()
    h_nch = torch.empty(n, dtype=torch.int32).pin_memory()
    h_st8 = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_ntok = torch.empty(n, dtype=torch.int32).pin_memory()
    n_tags = int(pred.n_tags) if want_states else 0
    h_tokid = torch.empty(n_chars_total, dtype=torch.int32).pin_memory() if want_states else None
    h_tokcand = torch.empty(n_chars_total * max(n_tags, 1), dtype=torch.uint8).pin_memory() if want_states else None
    ntok_out, nuns_out = C.c_uint64(), C.c_uint64()

    def step_compact():
        rc = L.vpt_predict_batch_compact(pred._h, h_text.data_ptr(), h_off.data_ptr(), n, h_bits.data_ptr(), h_bits.numel(),
                                         h_nch.data_ptr(), h_st8.data_ptr(), h_ntok.data_ptr(),
                                         h_tokid.data_ptr() if want_states else None,
                                         h_tokcand.data_ptr() if want_states else None,
                                         n_chars_total if want_states else 0, C.byref(nb_out), C.byref(ntok_out), C.byref(nuns_out))
        if rc:
            raise RuntimeError(L.vpt_last_error().decode())

    step_compact()
    step_compact()
    assert nb_out.value == n_bound
    bits_np = np.unpackbits(h_bits.numpy().view(np.uint8), bitorder="little")[:n_bound]
    assert np.array_equal(bits_np, h_bounds.numpy()), "compact boundary bits"
    assert int(h_ntok.numpy().sum()) == int(np.count_nonzero(h_bounds.numpy() == 1)) + n
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        step_compact()
    torch.cuda.synchronize()
    tcp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tcp, op=dist.ReduceOp.MAX)
    e2e_compact_value = total_bytes * args.e2e_steps / float(tcp.item()) / 1e6
    compact_d2h = 4 * ((n_bound + 31) // 32) + 4 * n + n + 4 * n + (int(ntok_out.value) * (4 + n_tags) if want_states else 0)
    compact_known = int(np.count_nonzero(h_tokid.numpy()[: ntok_out.value] >= 0)) if want_states else None
    # the reference CLI loop on the device (vpt_tokenize_lines): raw lines in, space-separated tokens out; line
    # splitting and output materialisation run on the GPU, so no offsets / scores cross PCIe
    starts = offs[:-1].astype(np.int64) + np.arange(n, dtype=np.int64)
    lines_np = np.full(nbytes + n, 10, np.uint8)
    keep = np.ones(nbytes + n, bool)
    keep[starts[1:] - 1] = False
    keep[-1] = False
    lines_np[keep] = text[:nbytes]
    h_lines = torch.from_numpy(lines_np).pin_memory()
    h_tok = torch.empty(3 * (nbytes + n), dtype=torch.uint8).pin_memory()
    tok_len, tok_lines = C.c_uint64(), C.c_uint64()

    def step_lines():
        rc = L.vpt_tokenize_lines(pred._h, h_lines.data_ptr(), nbytes + n, 1, 0, h_tok.data_ptr(), h_tok.numel(),
                                  C.byref(tok_len), C.byref(tok_lines))
        if rc:
            raise RuntimeError(L.vpt_last_error().decode())

    step_lines()
    step_lines()
    assert tok_lines.value == n
    # spaces in the output = word boundaries + escaped spaces of the input (the synthetic text has no '/' or '\\')
    tok_np = h_tok.numpy()[: tok_len.value]
    n_wb = int(np.count_nonzero(h_bounds.numpy() == 1))
    assert tok_len.value == nbytes + n + n_wb + int(np.count_nonzero(text[:nbytes] == 0x20)), "tokenize_lines size"
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        step_lines()
    torch.cuda.synchronize()
    tl = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tl, op=dist.ReduceOp.MAX)
    e2e_lines_value = total_bytes * args.e2e_steps / float(tl.item()) / 1e6
    lines_d2h = int(tok_len.value)
    # the same with the CLI's --predict-tags (config 3): tagged output text materialised on the device
    e2e_lines_tags = None
    if want_states and pred.info.get("predict_tags"):
        h_tok2 = torch.empty(8 * (nbytes + n), dtype=torch.uint8).pin_memory()
        tl_len, tl_lines = C.c_uint64(), C.c_uint64()

        def step_lines_tags():
            rc = L.vpt_tokenize_lines_tags(pred._h, h_lines.data_ptr(), nbytes + n, 1, 0, h_tok2.data_ptr(), h_tok2.numel(),
                                           C.byref(tl_len), C.byref(tl_lines))
            if rc:
                raise RuntimeError(L.vpt_last_error().decode())

        step_lines_tags()
        step_lines_tags()
        assert tl_lines.value == n
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            step_lines_tags()
        torch.cuda.synchronize()
        tlt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tlt, op=dist.ReduceOp.MAX)
        e2e_lines_tags = {"value": round(total_bytes * args.e2e_steps / float(tlt.item()) / 1e6, 1), "unit": "MB/s",
                          "api": "vpt_tokenize_lines_tags, no_norm = 1 (raw lines in, tokens with /tag suffixes out)",
                          "h2d_bytes_per_step": nbytes + n, "d2h_bytes_per_step": int(tl_len.value)}
    # the literal drop-in call: Predictor::predict for ONE sentence (vpt_predict: one pinned round trip, one launch)
    one = bytes(text[int(offs[0]):int(offs[1])])
    one_sc = np.empty(len(one), np.int32)
    one_bd = np.empty(len(one), np.uint8)
    one_n = C.c_uint64()

    def step_single():
        rc = L.vpt_predict(pred._h, one, len(one), one_sc.ctypes.data, one_bd.ctypes.data, len(one), None, None, 0, C.byref(one_n))
        if rc:
            raise RuntimeError(L.vpt_last_error().decode())

    for _ in range(200):
        step_single()
    t0 = time.perf_counter()
    n_single = 3000
    for _ in range(n_single):
        step_single()
    single_us = (time.perf_counter() - t0) / n_single * 1e6
    assert one_sc[: one_n.value - 1].tolist() == d_scores[: one_n.value - 1].cpu().numpy().tolist()
    # config 3: predict + predict_tags with the tag prediction on the device (the states never cross PCIe)
    e2e_tags_value = None
    if want_states:
        h_tok = torch.empty(n_chars_total, dtype=torch.int32).pin_memory()
        h_cand = torch.empty(n_chars_total * max(pred.n_tags, 1), dtype=torch.int32).pin_memory()
        nu_out = C.c_uint64()

        def step_tags():
            rc = L.vpt_predict_batch_tags(pred._h, h_text.data_ptr(), h_off.data_ptr(), n, h_scores.data_ptr(), h_bounds.data_ptr(),
                                          n_bound, h_boff.data_ptr(), h_status.data_ptr(), h_tok.data_ptr(), h_cand.data_ptr(),
                                          n_chars_total, h_coff.data_ptr(), C.byref(nb_out), C.byref(nc_out), C.byref(nu_out))
            if rc:
                raise RuntimeError(L.vpt_last_error().decode())

        step_tags()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            step_tags()
        torch.cuda.synchronize()
        tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_tags_value = total_bytes * args.e2e_steps / float(tt.item()) / 1e6
    h2d = nbytes + 8 * (n + 1)
    d2h = 4 * n_bound + n_bound + 8 * (n + 1) + 4 * n + 16 + (8 * n_chars_total + 8 * (n + 1) if want_states else 0)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (burst copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        alg_bytes = nbytes + 8 * n + 5 * n_bound  # SURVEY §8d: read B+8 per sentence, write 4(n-1)+(n-1)
        if want_states:
            alg_bytes += 8 * n_chars_total + 8 * (n + 1)  # config 3 also writes two u32 states per character + offsets
        fused = pred.info["kernel_launches_per_batch"] == 1
        kernel_name = "k_fused" if fused else ("k_tile_fast" if pred.info["fast_path"] else "k_score_general")
        # one launch per step when fused: the kernel time IS the device-timed step (the profiled leg below, with a
        # synchronize per call, is kept as a cross-check); otherwise the scoring stage of the profiled leg
        step_ms = ms_all / args.steps
        score_ms = step_ms if fused else float(stage_ms[2])
        achieved = alg_bytes / (score_ms / 1e3) / 1e9
        traffic = None
        try:
            if args.config == 2 and args.sentences == 1_000_000:
                traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(kernel_name + "_bytes_per_launch")
        except Exception:
            pass
        stage = ({kernel_name: round(score_ms, 4), "profiled_leg_ms": round(float(stage_ms[2]), 4)} if fused else
                 {"k_count": round(float(stage_ms[0]), 4), "k_scan_groups": round(float(stage_ms[1]), 4),
                  kernel_name: round(score_ms, 4)})
        # second roofline: the kernel is bound by random 32-byte record loads (node-table probes), whose rate is set
        # by the L1 tag stage: one 128-byte line per clock per SM, measured by profiles/tools/l2_probe_bench.cu
        roof2 = None
        try:
            from vpt_testlib import probe_model
            lines_peak = None
            for ln in open(os.path.join(ROOT, "profiles", "r02_l1_probe_bench.jsonl")):
                d = json.loads(ln)
                if d.get("test") == "record32" and d.get("variant") == "ilp4" and d.get("table_mb") == 23:
                    lines_peak = float(d["gprobes_s"])
            ns = min(n, 4000)
            sents = [bytes(text[int(offs[i]):int(offs[i + 1])]).decode() for i in range(ns)]
            pm = probe_model.probes_per_char(get_model(args.patterns, args.model_sample, args.config), sents)
            probes = pm["per_char"] * (n_bound + n)
            ach2 = probes / (score_ms / 1e3) / 1e9
            roof2 = {"bound": "l1_lines", "kernel": kernel_name, "achieved": round(ach2, 1), "peak": lines_peak,
                     "unit": "G record loads/s", "frac": round(ach2 / lines_peak, 4) if lines_peak else None,
                     "probes_per_char": round(pm["per_char"], 3),
                     "peak_source": "profiles/r02_l1_probe_bench.jsonl (random 32-byte loads from a 23 MB L2-resident table, "
                                    "0.95 lines/clk/SM: the rate does not change for an L1-resident table or narrower loads)",
                     "note": "host-side count on a 4000-sentence sample (vpt_testlib/probe_model.py); backward-walk "
                             "probes of patterns longer than 3 characters are not counted"}
        except Exception as e:  # the second entry is informative: never fail the bench on it
            roof2 = {"bound": "l1_lines", "error": str(e)}
        out = {
            "metric": METRIC, "value": round(value, 1), "unit": "MB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_all / args.steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "i32", "data": "synthetic",
            "config": workload_config(args, n),
            "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": round(achieved, 1), "peak": peak,
                         "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": round(score_ms, 4),
                         "stage_ms": stage,
                         "read_only_GBps": round((nbytes + 8 * n) / (score_ms / 1e3) / 1e9, 1),
                         "whole_step_frac": round(alg_bytes / (ms_all / args.steps / 1e3) / 1e9 / peak, 4)},
            "roofline_l1_lines": roof2,
            "e2e": {"value": round(e2e_value, 1), "unit": "MB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.e2e_steps, "api": "vpt_predict_batch (pinned host buffers; scores+boundaries returned)",
                    "boundaries_only_value": round(e2e_nb_value, 1),
                    "single_call_us": round(single_us, 1),
                    "single_call": "vpt_predict on one 40-character sentence (host buffers, one launch, one pinned round trip)",
                    "predict_tags_on_device_value": None if e2e_tags_value is None else round(e2e_tags_value, 1),
                    "k_tags_ms": None if k_tags_ms is None else round(k_tags_ms, 4),
                    "compact": {"value": round(e2e_compact_value, 1), "unit": "MB/s",
                                "api": "vpt_predict_batch_compact (1 bit per boundary, n_chars/status/n_tokens per sentence"
                                       + (", token id + %d candidate bytes per token: tag prediction on the device)" % n_tags
                                          if want_states else "; no scores, no tags)"),
                                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": compact_d2h,
                                "tokens": int(ntok_out.value), "tokens_with_tag_model": compact_known},
                    "tokenize_lines_tags": e2e_lines_tags,
                    "tokenize_lines": {"value": round(e2e_lines_value, 1), "unit": "MB/s",
                                       "api": "vpt_tokenize_lines, no_norm = 1 (raw lines in, tokenised text out; split + "
                                              "materialisation on the device)",
                                       "h2d_bytes_per_step": nbytes + n, "d2h_bytes_per_step": lines_d2h}},
            "gpu_launches": args.steps * pred.info["kernel_launches_per_batch"],
            "clocks": clocks,
            "host_binding": numa,
            "bit_exact_checked": True,
        }
        if world == 1 and not args.no_cpu_baseline:
            model_bytes = get_model(args.patterns, args.model_sample, args.config)
            # (config 3: the oracle restates the reference's build-time tag merge literally, which takes minutes on
            #  20 000 tag models; the CPU arm therefore scores boundaries with predict_tags = false)
            cb, oracle = cpu_baseline(model_bytes, text, offs, predict_tags=False)
            if args.config == 3:
                cb["sample"] += "; predict_tags = false on the CPU arm (boundary scores are identical)"
            out["cpu_baseline"] = cb
            # parity spot check of this very run against the oracle
            idx = np.arange(0, n, max(1, n // 200))[:200]
            hb = h_boff.numpy()
            hs = h_scores.numpy()
            for i in idx:
                s = bytes(text[int(offs[i]):int(offs[i + 1])]).decode()
                assert hs[int(hb[i]):int(hb[i + 1])].tolist() == oracle.predict(s)[0].tolist(), "parity failure"
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

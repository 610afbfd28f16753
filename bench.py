#!/usr/bin/env python
"""bench.py — decode MP/s of lossy VarDCT 12 MP 8-bit images (BASELINE.json metric) on N B200s of one node.

A step = one pass of the hot path (LoadImage-equivalent decode) over one batch of 256 synthetic 4000x3000 RGB8 VarDCT d=1.0
files (BASELINE config 3). With --gpus N the 256 files are sharded across the ranks (file i -> rank i mod N, strong scaling, no
data-path collective); --scaling weak gives every rank its own 256 files.
  value : whole-job MP/s with the compressed files already resident in HBM and the decoded pixels left in HBM
  e2e   : the same through the C ABI with HOST buffers (pinned), H2D of the files and D2H of the pixels inside the timed region
  roofline       : the kernel with the largest share of a decode, algorithmic bytes / CUDA-event duration vs measured HBM peak
  stage_rooflines: the HBM-bound stage kernels (dequant+IDCT, gaborish+EPF+colour) — the stages north_star sets the 50 % bar on
  workloads      : the headline files are DCT8-only (what the engine's own low-effort encoder produces); "mixed" is the same images
                   encoded with variable block sizes + chroma-from-luma + adaptive quantisation, measured beside it
  verified       : pixels of one timed batch compared with the CPU oracle outside the timed region
  cpu_baseline   : the CPU oracle (scalar port, NOT libjxl — libjxl is unavailable offline) on a bounded sample, all host cores
The input files of both arms come from the CPU oracle's encoder (test infrastructure, deterministic, no GPU): `--impl reference`
therefore never loads the engine's library. It times the oracle's decoder on the host cores (the reference's libjxl path cannot be
built here: N/vcpkg.json:6-9 is un-vendored).
"""
import argparse
import json
import os

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # one hardware queue per in-flight stream where possible (default 8 serialises streams)
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "decode MP/s (lossy VarDCT, 12 MP 8-bit)"
UNIT = "MP/s"

# What the files really contain (VERDICT r01: the label must say so). Both are single-pass, ANS-coded, XYB, d=1.0, gaborish + one EPF
# iteration, LF coded with a fixed gradient-predictor MA tree (one context property), written by the CPU oracle's encoder.
WORKLOADS = {
    "dct8": dict(enc=dict(effort=7, distance=1.0, varblocks=0, cfl=0, adaptive_quant=0),
                 label="DCT8-only VarDCT d=1.0 (every block 8x8, no chroma-from-luma, one quantiser), gaborish + EPFx1, fixed gradient MA tree for LF, ANS, one pass"),
    "mixed": dict(enc=dict(effort=7, distance=1.0, varblock_scale=4.0, varblock_pattern=1),
                  label="VarDCT d=1.0 with variable blocks (DCT8 / DCT8x16 / DCT16x16 / DCT32x32 in a fixed mix per 64x64 tile; measured area shares in workloads.mixed.block_mix), "
                        "chroma-from-luma and adaptive quantisation, gaborish + EPFx1, fixed gradient MA tree for LF, ANS, one pass"),
}


BLOCK_MIX = {}   # workload -> share of the frame area per AC strategy, measured by the encoder that wrote the files


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--width", type=int, default=4000)
    ap.add_argument("--height", type=int, default=3000)
    ap.add_argument("--batch", type=int, default=256, help="images per step (whole job with --scaling strong, per GPU with weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic images (seeds 0..distinct-1), repeated to fill the batch")
    ap.add_argument("--in-flight", type=int, default=128)
    ap.add_argument("--e2e-depth", type=int, default=1, help="batches in flight in the end-to-end measurement (JxlB200DecodeBatchSubmit / Wait); 1 = synchronous calls")
    ap.add_argument("--cpu-sample", type=int, default=2, help="images in the bounded CPU-baseline sample")
    ap.add_argument("--no-mixed", action="store_true", help="skip the second (variable-block) workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the pixels decoded in the last timed step of each timed path to DIR/<path>.npy "
                    "(float32, one row per file of the step, the same seeded byte positions of every image; DIR/sample_index.npy holds them)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def describe(args, world):
    per = "%d files per step sharded over %d rank(s)" % (args.batch, world) if args.scaling == "strong" else "%d files per step per GPU" % args.batch
    return "batch of synthetic %dx%d RGB8 files, %s (%d distinct images repeated), decoded to interleaved RGB8, no collective; " % (args.width, args.height, per, args.distinct)


DUMP_PATHS = 3                   # timed paths dumped: dct8 device, dct8 e2e, mixed device
DUMP_BYTES = 48 << 20            # the samples of every path plus their index: the dump stays under 64 MB with the .npy headers


def dump_sample_index(n_bytes, n_files):
    """Byte offsets sampled from every decoded image: one seeded offset in each of K equal stripes of the image, K sized so that the
    samples of every path over the whole job's files (float32) and the index itself (float64) fit DUMP_BYTES. Depends only on the arguments."""
    import numpy as np
    k = max(1, min(n_bytes, DUMP_BYTES // (4 * DUMP_PATHS * n_files + 8)))
    stripe = n_bytes // k
    return np.arange(k, dtype=np.int64) * stripe + np.random.default_rng(0).integers(0, stripe, k)


# ------------------------------------------------------------------------------------------------ input files (CPU, deterministic)
def _make_one(job):
    seed, w, h, encs = job
    import oracle_py as O
    from synth import synthetic_image
    img = synthetic_image(w, h, seed=seed)
    files, mixes = [], []
    for enc in encs:
        files.append(O.encode(img, threads=2, **enc))
        mixes.append(O.last_encode_strategy_cells())   # cells per AC strategy: says what the file really contains
    return seed, files, mixes


def make_files(args, seeds, names):
    """-> {name: {seed: bytes}} for the workloads in `names`; synthetic image -> .jxl with the CPU oracle's encoder, in worker processes."""
    import multiprocessing as mp
    import oracle_py as O
    O.lib()   # build the oracle library once, before forking
    jobs = [(s, args.width, args.height, [WORKLOADS[n]["enc"] for n in names]) for s in seeds]
    nproc = max(1, min(len(jobs), (os.cpu_count() or 2) // 2))
    if nproc > 1:
        with mp.get_context("fork").Pool(nproc) as pool:
            res = pool.map(_make_one, jobs)
    else:
        res = [_make_one(j) for j in jobs]
    names_s = {0: "DCT8", 4: "DCT16x16", 5: "DCT32x32", 6: "DCT16x8", 7: "DCT8x16"}
    for k, n in enumerate(names):
        tot = [sum(m[k][i] for _, _, m in res) for i in range(27)]
        BLOCK_MIX[n] = {names_s.get(i, "strategy%d" % i): round(v / max(sum(tot), 1), 3) for i, v in enumerate(tot) if v}
    return {n: {seed: files[k] for seed, files, _ in res} for k, n in enumerate(names)}


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        # In-process NVML when available (a clock read costs microseconds); spawning nvidia-smi five times a second would steal
        # host time from the enqueue threads being measured. Falls back to nvidia-smi.
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self._stop_evt.is_set():
                r = int(get_reasons(h))
                act = lambda bit: "Active" if r & bit else "Not Active"
                self.rows.append([str(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), str(mx), act(0x8), act(0x40), act(0x20), act(0x4)])
                self._stop_evt.wait(0.1)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def cpu_decode_rate(files, args, sample):
    """CPU oracle (tests/oracle_py -> oracle/_build/liboracle.so) on a bounded sample with every host core."""
    import oracle_py as O
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    for i in range(sample):
        O.decode(files[i % len(files)], threads=cores)
    dt = time.perf_counter() - t0
    mp = sample * args.width * args.height / 1e6
    return {"value": mp / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d images of %dx%d decoded by the scalar CPU oracle (own restatement, NOT libjxl) with %d threads over groups" % (sample, args.width, args.height, cores)}


def run_reference(args):
    """The reference arm: the CPU path on the host cores, same files (oracle encoder, same seeds), rank 0 only. Loads no engine code."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    import oracle_py as O
    seeds = list(range(min(args.distinct, max(2, args.cpu_sample))))
    files = [make_files(args, seeds, ["dct8"])["dct8"][s] for s in seeds]
    cores = os.cpu_count() or 1
    O.decode(files[0], threads=cores)   # page in the library and the cosine tables
    per_step = args.cpu_sample
    for _ in range(args.warmup):
        cpu_decode_rate(files, args, 1)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        base = cpu_decode_rate(files, args, per_step)
    dt = time.perf_counter() - t0
    mp_step = per_step * args.width * args.height / 1e6
    value = mp_step * args.steps / dt
    base["value"] = value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": describe(args, world) + WORKLOADS["dct8"]["label"], "mp_per_step": mp_step,
                       "sample": "the same files decoded on the host CPU; each step a bounded sample of %d images" % per_step},
            "cpu_baseline": base, "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def bind_to_gpu_numa_node(torch, local):
    """Pins this rank to the CPUs local to its GPU (what `numactl` would do), so that its page-locked buffers and its enqueue threads
    sit on the GPU's NUMA node. Silently does nothing where sysfs does not expose the topology."""
    if os.environ.get("JXLB200_BENCH_NOBIND"):
        return
    try:
        pr = torch.cuda.get_device_properties(local)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/local_cpulist" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        cpus = set()
        for part in open(path).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    W, H = args.width, args.height
    # this rank's share of the step: file i of the step is distinct image (i mod D), and goes to rank (i mod world) under strong scaling
    if args.scaling == "strong":
        mine = [i for i in range(args.batch) if i % world == rank]
        seed_of = lambda i: i % args.distinct
    else:
        mine = list(range(args.batch))
        seed_of = lambda i: (i % args.distinct) + 1000 * rank
    names = ["dct8"] + ([] if args.no_mixed else ["mixed"])
    seeds = sorted({seed_of(i) for i in mine})
    t_gen = time.perf_counter()
    made = make_files(args, seeds, names)    # CPU work, before the CUDA context exists (worker processes are forked)
    t_gen = time.perf_counter() - t_gen

    import numpy as np
    import torch
    dist = None
    torch.cuda.set_device(local)
    bind_to_gpu_numa_node(torch, local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import pkgload
    P = pkgload.load(build_if_missing=True)
    ok, why = P.cuda_available()
    if not ok:
        raise SystemExit("bench.py needs a GPU: " + why)
    B = len(mine)
    out_bytes_one = W * H * 3
    files_per_step = args.batch if args.scaling == "strong" else args.batch * world
    total_mp_step = files_per_step * W * H / 1e6
    dev_out = [torch.empty(out_bytes_one, dtype=torch.uint8, device="cuda") for _ in range(B)]
    # --e2e-depth N > 1: the end-to-end steps are submitted asynchronously with N batches in flight, each writing its own set of host buffers
    # (measured in r02: two batches in flight are SLOWER than synchronous calls, 378 vs 260 ms per step — profiles/r02_e2e_pipeline.md)
    E2E_DEPTH = max(1, args.e2e_depth)
    try:
        host_out = [torch.empty(out_bytes_one, dtype=torch.uint8).pin_memory() for _ in range(B * E2E_DEPTH)]
        host_pinned = True
    except RuntimeError:   # the box cannot page-lock that much per rank: pageable buffers (the engine then stages through its own pinned pool)
        host_out = [torch.empty(out_bytes_one, dtype=torch.uint8) for _ in range(B * E2E_DEPTH)]
        host_pinned = False
    host_out_sets = [[t.numpy() for t in host_out[k * B:(k + 1) * B]] for k in range(E2E_DEPTH)]
    host_out_np = host_out_sets[0]
    dump_index = dump_sample_index(out_bytes_one, files_per_step) if args.dump_outputs else None

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, drain=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if drain is not None:
            drain()          # every step submitted above has delivered its pixels before the clock stops
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        barrier()
        return float(t.item())

    def measure(name, steps, warmup, with_host):
        files = [made[name][seed_of(i)] for i in mine]
        dev_in = [torch.frombuffer(bytearray(f), dtype=torch.uint8).cuda() for f in files]
        torch.cuda.synchronize()

        def step_device():
            st = P.decode_batch(None, device=local, max_in_flight=args.in_flight, device_inputs=[t.data_ptr() for t in dev_in], device_outputs=[t.data_ptr() for t in dev_out],
                                sizes=[t.numel() for t in dev_in], out_sizes=[out_bytes_one] * B)
            assert all(s == 0 for s in st)

        pending = []
        submitted = [0]

        def step_host():   # JxlB200DecodeBatchSubmit / Wait with E2E_DEPTH batches in flight; step k writes output set k mod depth
            outs = host_out_sets[submitted[0] % E2E_DEPTH]
            submitted[0] += 1
            pending.append(P.decode_batch_submit(files, outs, device=local, max_in_flight=args.in_flight))
            while len(pending) >= E2E_DEPTH:
                assert all(s == 0 for s in pending.pop(0).wait())

        def drain_host():
            while pending:
                assert all(s == 0 for s in pending.pop(0).wait())

        for _ in range(warmup):
            step_device()
        sampler = ClockSampler(local)
        sampler.start()
        launches0 = P.kernel_launch_count()
        ms_dev = timed(step_device, steps)
        launches = P.kernel_launch_count() - launches0
        clocks = sampler.stop()
        r = {"files": files, "ms_dev": ms_dev, "launches": launches, "clocks": clocks, "comp_bytes": sum(len(f) for f in files), "value": total_mp_step * steps / (ms_dev / 1e3)}
        if dump_index is not None:   # dev_out is reused by the next workload: sample it now, outside the timed region
            idx = torch.from_numpy(dump_index).cuda()
            r["dump_device"] = torch.stack([t[idx] for t in dev_out]).float().cpu().numpy()
        if with_host:
            for _ in range(max(1, warmup // 2)):
                step_host()
            drain_host()
            r["ms_host"] = timed(step_host, steps, drain_host)
            r["last_host_set"] = (submitted[0] - 1) % E2E_DEPTH
            r["e2e"] = total_mp_step * steps / (r["ms_host"] / 1e3)
            if dump_index is not None:
                r["dump_e2e"] = np.stack([o[dump_index] for o in host_out_sets[r["last_host_set"]]]).astype(np.float32)
        return r

    head = measure("dct8", args.steps, args.warmup, True)
    # pixels of the last timed e2e batch against the CPU oracle (outside the timed region; rank 0, a bounded number of distinct files)
    verified, max_err, checked = None, None, 0
    if rank == 0:
        try:
            import oracle_py as O
            seen, max_err = set(), 0
            for k, i in enumerate(mine):
                s = seed_of(i)
                if s in seen or len(seen) >= 3:
                    continue
                seen.add(s)
                ref = O.decode(head["files"][k], threads=os.cpu_count() or 1).pixels
                got = host_out_sets[head.get("last_host_set", 0)][k].reshape(H, W, 3)
                max_err = max(max_err, int(np.abs(got.astype(np.int16) - ref.astype(np.int16)).max()))
            checked = len(seen)
            verified = bool(max_err <= 1)
        except Exception as e:   # the oracle library may be absent
            verified, max_err = None, "unavailable: %s" % e
    mixed = None
    if not args.no_mixed:
        mixed = measure("mixed", args.steps, 2, False)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        suffix = ".rank%d" % rank if world > 1 else ""
        dumps = {"dct8_device": head["dump_device"], "dct8_e2e": head["dump_e2e"]}
        if mixed is not None:
            dumps["mixed_device"] = mixed["dump_device"]
        for name, arr in dumps.items():
            np.save(os.path.join(args.dump_outputs, name + suffix + ".npy"), arr)
        if rank == 0:
            np.save(os.path.join(args.dump_outputs, "sample_index.npy"), dump_index.astype(np.float64))

    launches = head["launches"]
    if dist is not None:
        lt = torch.tensor([launches], dtype=torch.float64, device="cuda")
        dist.all_reduce(lt)
        launches = int(lt.item())
    comp_bytes, files = head["comp_bytes"], head["files"]
    line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_dev"] / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": describe(args, world) + WORKLOADS["dct8"]["label"],
                       "mp_per_step": total_mp_step, "files_per_rank_per_step": B, "bpp": 8.0 * comp_bytes / (B * W * H), "in_flight": args.in_flight,
                       "input_files": "CPU oracle encoder (test infrastructure), %.1f s to generate" % t_gen,
                       "l2": "inputs+outputs per step and rank (%.0f MB) exceed the 126 MB L2" % ((comp_bytes + B * out_bytes_one) / 1e6)},
            "e2e": {"value": head["e2e"], "unit": UNIT, "h2d_bytes_per_step": None, "d2h_bytes_per_step": None, "ms_per_step": head["ms_host"] / args.steps, "host_buffers": "page-locked" if host_pinned else "pageable",
                    "pipeline": "%d batch(es) in flight (JxlB200DecodeBatchSubmit / Wait), every step's pixels delivered inside the timed region; image starts paced to the D2H rate" % E2E_DEPTH},
            "gpu_launches": launches, "clocks": head["clocks"],
            "verified": verified, "max_err_lsb": max_err, "verified_files": checked}
    # bytes crossing PCIe per step, whole job (every rank moves its own share)
    tb = torch.tensor([float(comp_bytes), float(B * out_bytes_one)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tb)
    line["e2e"]["h2d_bytes_per_step"], line["e2e"]["d2h_bytes_per_step"] = int(tb[0].item()), int(tb[1].item())
    if mixed is not None:
        line["workloads"] = {"dct8": {"value": head["value"], "bpp": 8.0 * comp_bytes / (B * W * H), "what": WORKLOADS["dct8"]["label"]},
                             "mixed": {"value": mixed["value"], "bpp": 8.0 * mixed["comp_bytes"] / (B * W * H), "ms_per_step": mixed["ms_dev"] / args.steps,
                                       "ratio_to_dct8": mixed["value"] / head["value"], "what": WORKLOADS["mixed"]["label"], "block_mix": BLOCK_MIX.get("mixed")}}
        line["workloads"]["dct8"]["block_mix"] = BLOCK_MIX.get("dct8")

    if rank == 0:
        # per-kernel durations of one decode, CUDA events on the stream the kernels are launched on (engine StageTimes)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

        def single_image(f):
            acc, reps = {}, 5
            for i in range(reps + 1):
                img = P.DecoderImage()
                P.JpegXLNative.LoadImage(f, img)
                if i:   # first one is a warm-up
                    for k, v in P.last_stage_times().items():
                        acc[k] = acc.get(k, 0.0) + v / reps
            return acc
        acc = single_image(files[0])
        px = W * H
        comp_px = len(files[0]) / px
        stage_bytes = {"lf": (comp_px * 0.12 + (12 + 3) / 64.0), "ac": (comp_px * 0.88 + 6.0), "recon": 18.0, "filters": 24.0 * 2, "output": 15.0}
        names_k = {"lf": "k_lf_group (LF coefficients + HF metadata entropy decode; latency-bound serial streams)", "ac": "k_ac_vardct (AC coefficient entropy decode; latency-bound serial streams)",
                   "recon": "k_reconstruct_dct8 (dequant + CfL + IDCT)", "filters": "k_gaborish + k_epf<1>", "output": "k_output (XYB->sRGB + interleave)"}
        if acc.get("output", 0.0) < 0.02 and acc.get("filters", 0.0) > 0:   # fused path: one kernel reads XYB once and writes RGB8 once
            stage_bytes["filters"] = 15.0
            acc["filters"] += acc.get("output", 0.0)
            acc["output"] = 0.0
            names_k["filters"] = "k_render<GAB,EPF> (gaborish + EPF + XYB->sRGB + interleave fused; XYB read once, RGB8 written once)"
        stages = {}
        for k in ("lf", "ac", "recon", "filters", "output"):
            ms = acc.get(k, 0.0)
            if ms > 0:
                ach = stage_bytes[k] * px / (ms * 1e-3) / 1e9
                stages[k] = {"kernel": names_k[k], "ms": ms, "bytes_per_px": stage_bytes[k], "achieved": ach, "frac": ach / peak, "traffic": None}
        dom = max(stages, key=lambda k: stages[k]["ms"]) if stages else None
        if dom:
            d = stages[dom]
            line["roofline"] = {"bound": "hbm", "kernel": d["kernel"], "achieved": d["achieved"], "peak": peak, "unit": "GB/s", "frac": d["frac"], "traffic": None,
                                "peak_source": peak_src, "share_of_decode": d["ms"] / max(acc.get("total", 1e-9), 1e-9),
                                "note": "dominant kernel of a single-image decode; entropy decode is a serial bit stream per section, so its HBM fraction is tiny by nature — ns/symbol is the relevant figure (DESIGN.md)"}
        # DRAM bytes per launch come from an `ncu --set full` capture, which cannot run inside this process: they are read from the
        # committed capture summary when it matches this frame size, and are null otherwise (never a hard-coded constant here).
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            if tr.get("width") == W and tr.get("height") == H:
                for k in ("recon", "filters"):
                    if k in stages and k in tr.get("kernels", {}):
                        stages[k]["traffic"] = tr["kernels"][k]["dram_bytes"]
                        stages[k]["traffic_source"] = tr["source"]
        except Exception:
            pass
        line["stage_rooflines"] = {k: v for k, v in stages.items() if k in ("recon", "filters", "output")}
        line["single_image_ms"] = acc
        if mixed is not None:
            line["workloads"]["mixed"]["single_image_ms"] = single_image(mixed["files"][0])
        try:
            import oracle_py as O
            O.decode(files[0], threads=os.cpu_count() or 1)
            line["cpu_baseline"] = cpu_decode_rate(files, args, args.cpu_sample)
        except Exception as e:   # the oracle library may be absent; the GPU numbers stand on their own
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": "unavailable: %s" % e}
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

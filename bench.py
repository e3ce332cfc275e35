#!/usr/bin/env python
"""Driver benchmark for the B200-native quantized-linear hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--no-extras] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  The default workload is the configuration
BASELINE.json's metric is quoted on (configs[1]): the bf16 x int4 QLinear GEMM M=4096, K=4096, N=14336 (Llama-3-8B FFN
gate/up projection) -- `qlinear_bf16_int4_m4096`.  Because the driver only ever runs the default command, the default
run appends the other BASELINE configurations to the same JSON line under `"extra"` (each with value / roofline):
`decode_m1|m8|m32` (HBM-bound int4 decode, replayed from CUDA graphs), `int8_m4096` (int8 x int8 qbytes_mm),
`llama3_8b_decode_b1|b8|b32` (the 224 qint4 linears of one decode step, one CUDA graph), and under `"compare"` the
kernels the reference would dispatch to on this GPU (torch.matmul bf16, torch._int_mm + epilogue,
torch._weight_int4pack_mm) timed on the same shapes in the same process.  `--workload NAME` runs one of them as the
headline instead.

At N > 1 (torchrun, one rank per GPU) the layer is column-sharded over out_features and every rank ends up with the
full output.  int4: the all-gather and the rank synchronisation are fused into the kernel (peer stores from the epilogue,
in-kernel flags; `parallel.FusedGather`); `--gather nccl` selects kernel + NCCL all-gather instead.  Strong scaling: the
total work is fixed.  Outside the timed region every rank checks the gathered output bit for bit against the single-rank
linear on the full weight and the line carries `"parity_ok"`.

One JSON line is printed by rank 0 (see the keys in DESIGN.md "Measurement").

`--dump-outputs DIR` also writes what the last timed step of every measured workload returned, as DIR/<workload>.npy in
float32 (for M > 32 a fixed, seeded sample of rows; about 32 MB for the default run).  Every input comes from a fixed
seed, so two builds run with the same arguments can be compared output for output.
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
sys.path.insert(0, os.path.join(ROOT, "optimum-quanto_b200"))

import torch  # noqa: E402

K_DIM, N_DIM, GROUP = 4096, 14336, 128

LLAMA3_8B_LAYER = [("q", 4096, 4096), ("k", 1024, 4096), ("v", 1024, 4096), ("o", 4096, 4096),
                   ("gate", 14336, 4096), ("up", 14336, 4096), ("down", 4096, 14336)]  # (name, N, K), 32 layers

WORKLOADS = {
    "qlinear_bf16_int4_m4096": dict(kind="int4", M=4096, bound="tensor"),
    "llama3_8b_decode_b1": dict(kind="llama", M=1, bound="hbm"),
    "llama3_8b_decode_b8": dict(kind="llama", M=8, bound="hbm"),
    "llama3_8b_decode_b32": dict(kind="llama", M=32, bound="hbm"),
    "decode_m1": dict(kind="int4", M=1, bound="hbm"),
    "decode_m8": dict(kind="int4", M=8, bound="hbm"),
    "decode_m32": dict(kind="int4", M=32, bound="hbm"),
    "int8_m4096": dict(kind="int8", M=4096, bound="tensor"),
}
DEFAULT_WORKLOAD = "qlinear_bf16_int4_m4096"
EXTRA_WORKLOADS = ["decode_m1", "decode_m8", "decode_m32", "int8_m4096", "llama3_8b_decode_b1", "llama3_8b_decode_b8",
                   "llama3_8b_decode_b32"]
EXTRA_WORKLOADS_MULTI = ["decode_m1", "decode_m8", "llama3_8b_decode_b1", "llama3_8b_decode_b8"]


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tensor=p["bf16_tflops"], tensor_sustained=p.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json, burst)")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def algorithmic(kind, M, N, K):
    """Algorithmic flops and bytes of one launch (SURVEY 8d / DESIGN.md)."""
    flops = 2.0 * M * N * K
    if kind == "int4":
        byts = M * K * 2 + N * K // 2 + 2 * (N * K // GROUP) * 2 + M * N * 2
    else:
        byts = M * K + N * K + N * 2 + M * N * 2
    return flops, byts


DUMP_LIMIT_BYTES = 64 << 20


def dump_rows(M):
    """Rows of an [M, N] result that --dump-outputs writes: all of them up to M = 32, else two rows of every 32-row band
    picked with a fixed seed (every M tile of every kernel is represented: 256 rows of M = 4096)."""
    import numpy as np
    if M <= 32:
        return np.arange(M)
    rng = np.random.default_rng(0)
    return np.concatenate([b0 + np.sort(rng.choice(min(32, M - b0), size=min(2, M - b0), replace=False))
                           for b0 in range(0, M, 32)])


def write_outputs(directory, outputs):
    """DIR/<workload>.npy, float32, for every workload the run timed (at most DUMP_LIMIT_BYTES in all)."""
    import numpy as np
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, arr in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), arr)


def llama_weight_bytes():
    return 32 * sum(N * K // 2 + 2 * (N * K // GROUP) * 2 for _, N, K in LLAMA3_8B_LAYER)


def metric_name(workload):
    if workload.startswith("llama3_8b_decode"):
        return "llama3_8b_qint4_decode_tokens_per_s"
    return {"qlinear_bf16_int4_m4096": "qlinear_bf16xint4_tflops", "int8_m4096": "qbytes_mm_int8_tops"}.get(
        workload, "qlinear_bf16xint4_decode_gbs")


class ClockSampler:
    """Samples SM clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).

    NVML is read in-process from a thread (pynvml, ~0.1 ms per sample, every 2 ms); the timed regions of the default
    workload last only a few milliseconds, less than `nvidia-smi -lms` needs to print its first line.  Falls back to
    the `nvidia-smi` query loop when pynvml is unavailable.  Samples are only kept while `self.active` is set.
    """

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    # nvmlClocksEventReason* bit masks (nvml.h)
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.samples, self.proc, self.nvml, self.handle = index, [], None, None, None
        self.sm, self.max_mhz, self.reasons, self.stop_flag, self.source = [], None, set(), False, None
        self.active = False  # samples are kept only while a timed region (or the load loop) is running

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            try:
                handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except TypeError:
                handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        return pynvml, handle

    def start(self):
        try:
            self.nvml, self.handle = self._nvml_handle()
            self.max_mhz = float(self.nvml.nvmlDeviceGetMaxClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
            self.source = "nvml"
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.t = threading.Thread(target=self._read_smi, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.samples and time.time() - t0 < 5.0:  # wait for the first line before timing anything
                time.sleep(0.02)
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(
            n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            if not self.active:
                time.sleep(0.001)
                continue
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                mask = int(get_reasons(self.handle))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def _read_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            self.samples.append(line.strip())
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7 or not self.active:
                continue
            try:
                self.sm.append(float(f[0]))
                self.max_mhz = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    self.reasons.add(nm)

    def n_samples(self):
        return len(self.sm)

    def snapshot(self, since=0):
        """Summary of the samples taken since index `since` (one timed workload)."""
        sm = sorted(self.sm[since:])
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": self.source}

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            time.sleep(0.1)
            self.proc.terminate()
        elif self.nvml is not None:
            self.t.join(timeout=1.0)


def make_int4(N, K, device, seed, dtype=torch.bfloat16):
    """Synthetic canonical int4 weight (uniform nibbles, MaxOptimizer-shaped scale/shift), generated on `device`."""
    import quanto_b200 as q
    g = torch.Generator(device=device).manual_seed(seed)
    rows = N * K // GROUP
    packed = torch.randint(0, 256, (rows // 2, GROUP), dtype=torch.uint8, device=device, generator=g)
    scale = (torch.rand(rows, 1, device=device, generator=g) * 0.01 + 0.002).to(dtype)
    shift = (scale.float() * (7.0 + 2 * torch.rand(rows, 1, device=device, generator=g))).to(dtype)
    return q.WeightQBitsTensor(q.qint4, 0, GROUP, torch.Size([N, K]), (K, 1),
                               q.PackedTensor(packed, 4, torch.Size([rows, GROUP]), (GROUP, 1)), scale, shift)


# ---------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU `library/python` path (oracle port), all host threads, SAME workload size
# ---------------------------------------------------------------------------------------------------------------------
THREAD_CANDIDATES = (None, 64, 32, 16)  # None = every host core


def pick_threads(step, cores):
    """Fixed policy: one step at each of {all cores, 64, 32, 16} threads, keep the fastest.  (The reference's CPU path
    mixes a bf16 GEMM, which wants every core, with elementwise bf16 passes that run several times SLOWER with 128 threads
    than with 32 on the GPU box's host.)"""
    best, best_t = cores, None
    for n in THREAD_CANDIDATES:
        n = cores if n is None else n
        if n > cores:
            continue
        torch.set_num_threads(n)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_problem(kind, M, seed=0):
    """(step, flops, bytes) of the oracle port on CPU tensors for `M` rows of the workload (full N and K)."""
    from oracle import torch_port as P
    g = torch.Generator().manual_seed(seed)
    if kind == "int4":
        rows = N_DIM * K_DIM // GROUP
        packed = torch.randint(0, 256, (rows // 2, GROUP), dtype=torch.uint8, generator=g)
        scale = (torch.rand(rows, 1, generator=g) * 0.01 + 0.002).to(torch.bfloat16)
        shift = (scale.float() * 8).to(torch.bfloat16)
        x = torch.randn(M, K_DIM, generator=g).to(torch.bfloat16)
        step = lambda: P.qbits_linear(x, packed, scale, shift, None, N_DIM, GROUP)  # noqa: E731
    else:
        a = torch.randint(-127, 127, (M, K_DIM), dtype=torch.int8, generator=g)
        w = torch.randint(-127, 127, (N_DIM, K_DIM), dtype=torch.int8, generator=g)
        s = (torch.rand(N_DIM, 1, generator=g) / 1e3).to(torch.bfloat16)
        step = lambda: P.qbytes_mm(a, w, s)  # noqa: E731
    flops, byts = algorithmic(kind, M, N_DIM, K_DIM)
    return step, flops, byts


def run_reference(args, wl):
    """The reference's own CPU implementation of the path (oracle port; torch CPU ops on the host cores) on the SAME
    workload as the GPU arm: full M, N, K.  A step of the default workload is ~1-2 s of CPU time."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    host_cores = os.cpu_count() or 1
    kind, M = wl["kind"], wl["M"]
    step, flops, byts = cpu_problem(kind, M)
    cores = pick_threads(step, host_cores)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    hbm = wl["bound"] == "hbm"
    value = (byts / dt / 1e9) if hbm else (flops / dt / 1e12)
    unit = "GB/s" if hbm else "TFLOP/s"
    sample = (f"the full workload (M={M}, N={N_DIM}, K={K_DIM}) per step; oracle/torch_port.py, torch {torch.__version__} "
              f"CPU, {cores} threads (fastest of all/64/32/16 on {host_cores} host cores)")
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": value, "unit": unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "bf16" if kind == "int4" else "int8", "data": "synthetic",
        "config": {"workload": args.workload, "M": M, "N": N_DIM, "K": K_DIM, "group_size": GROUP,
                   "sample": sample, "sample_fraction": 1.0},
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def run_reference_llama(args, wl):
    """CPU arm of the Llama-3-8B decode workloads, same metric and unit (tokens/s): a step is the 7 qint4 linears of ONE
    layer (the bounded sample; the 32 layers are identical in shape), tokens/s = batch / (32 x layer time)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import torch_port as P
    host_cores = os.cpu_count() or 1
    M = wl["M"]
    g = torch.Generator().manual_seed(0)
    layer = []
    for _, N, K in LLAMA3_8B_LAYER:
        rows = N * K // GROUP
        packed = torch.randint(0, 256, (rows // 2, GROUP), dtype=torch.uint8, generator=g)
        scale = (torch.rand(rows, 1, generator=g) * 0.01 + 0.002).to(torch.bfloat16)
        shift = (scale.float() * 8).to(torch.bfloat16)
        layer.append((torch.randn(M, K, generator=g).to(torch.bfloat16), packed, scale, shift, N))

    def step():
        for x, packed, scale, shift, N in layer:
            P.qbits_linear(x, packed, scale, shift, None, N, GROUP)

    cores = pick_threads(step, host_cores)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt_layer = (time.perf_counter() - t0) / args.steps
    value = M / (32 * dt_layer)
    sample = (f"one of 32 identical layers per step (7 qint4 linears, batch {M}), rate scaled by 1/32; oracle/torch_port.py, "
              f"torch {torch.__version__} CPU, {cores} threads (fastest of all/64/32/16 on {host_cores} host cores)")
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": value, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 32 * dt_layer * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": args.workload, "batch": M, "layers": 32, "linears_per_step": 224,
                   "weights": "qint4 canonical packing, group 128", "sample": sample, "sample_fraction": 1.0 / 32},
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def cpu_baseline_sample(kind, M):
    """Rank-0, N=1 only: the oracle port on a bounded sample of the same workload (about 10-20 s of CPU work)."""
    host_cores = os.cpu_count() or 1
    prev = torch.get_num_threads()
    m_sample = min(M, 512)
    step, flops, byts = cpu_problem(kind, m_sample)
    cores = pick_threads(step, host_cores)
    step()
    t0 = time.perf_counter()
    n = 0
    while n < 3 or (time.perf_counter() - t0 < 8.0 and n < 40):
        step()
        n += 1
    dt = (time.perf_counter() - t0) / n
    torch.set_num_threads(prev)
    note = "" if m_sample == M else (
        f" -- a RATE on a {m_sample}/{M} row slice: the CPU path dequantises the whole weight once per call (~60 ms), "
        "amortised over fewer rows here than at the full M, so this understates the CPU's full-M rate; "
        "`bench.py --impl reference` runs the full M")
    return dt, flops, byts, cores, (f"M={m_sample} rows of the workload's {M}, full N={N_DIM} K={K_DIM}, {n} repeats, "
                                    f"{cores} threads (fastest of all/64/32/16 on {host_cores} host cores){note}")


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
class Bench:
    def __init__(self, args):
        import torch.distributed as dist

        import quanto_b200 as q
        from quanto_b200 import _native

        self.args, self.dist, self.q, self.native = args, dist, q, _native
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torchrun --nproc-per-node {args.gpus}")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        lib = _native.load()  # fail loudly if the native library is missing
        assert lib.qb200_debug_flags() == 0 and lib.qb200_developer_build() == 0, "bench.py needs the release library"
        self.lib = lib
        self.peaks = load_peaks()
        self.sampler = ClockSampler(self.local_rank)
        self.sampler.start()
        self.warm = max(args.warmup, 3)
        self.fused_note = None
        self._llama = None
        self.last_out = None
        self.outputs = {} if args.dump_outputs else None  # workload -> float32 array for --dump-outputs

    def keep_output(self, name, y):
        """--dump-outputs: a float32 host copy of the [M, N] result of workload `name`'s last timed step (the rows of
        dump_rows(M)), taken right after its timed region."""
        if self.outputs is None or self.rank != 0:
            return
        rows = torch.from_numpy(dump_rows(y.shape[0])).to(y.device)
        self.outputs[name] = y.index_select(0, rows).float().cpu().numpy()

    # ---- timing -------------------------------------------------------------------------------------------------
    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, step_fn, steps, warmup):
        """`steps` calls of step_fn(i) on the current stream between two CUDA events, bracketed by barrier +
        synchronize; max over ranks.  Returns ms per step; what the last call returned is kept in `self.last_out`."""
        for i in range(warmup):
            step_fn(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.sampler.active = True
        e0.record()
        for i in range(steps - 1):
            step_fn(warmup + i)
        self.last_out = step_fn(warmup + steps - 1)
        e1.record()
        self.barrier()
        self.sampler.active = False
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps

    def load_for_clocks(self, step_fn, mark, min_samples=25, max_seconds=1.5):
        """The timed regions of a sub-millisecond step end before enough clock samples exist: keep running the same
        step (untimed) until the sampler has seen the GPU under this workload's load.  With several ranks every rank
        runs the same fixed count (the step contains cross-rank synchronisation)."""
        self.sampler.active = True
        if self.world > 1:
            for i in range(100):
                step_fn(i)
            torch.cuda.synchronize()
        else:
            t0, i = time.time(), 0
            while self.sampler.n_samples() - mark < min_samples and time.time() - t0 < max_seconds:
                for _ in range(10):
                    step_fn(i)
                    i += 1
                torch.cuda.synchronize()
        self.sampler.active = False

    def all_ranks_ok(self, ok):
        if self.world == 1:
            return bool(ok)
        flag = torch.tensor([1 if ok else 0], device=self.dev)
        self.dist.all_reduce(flag, op=self.dist.ReduceOp.MIN)
        return bool(int(flag.item()))

    # ---- column-parallel plumbing -------------------------------------------------------------------------------
    def make_gather(self, n_local):
        """FusedGather for this shard width, or None (then kernel + NCCL all-gather)."""
        if self.world == 1 or self.args.gather != "fused":
            return None
        from quanto_b200.parallel import FusedGather
        ok, fg = True, None
        try:
            fg = FusedGather(n_local)
        except Exception as e:  # noqa: BLE001
            ok, self.fused_note = False, f"{type(e).__name__}: {e}"[:200]
        return fg if self.all_ranks_ok(ok) else None

    def sharded(self, w_full):
        from quanto_b200.parallel import shard_weight
        return shard_weight(w_full, self.rank, self.world) if self.world > 1 else w_full

    def gathered_linear(self, fg, x, w, wait_input=False, wait_output=True):
        from quanto_b200.parallel import gather_columns
        if fg is not None:
            return fg.forward(x, w, None, wait_input=wait_input, wait_output=wait_output)
        y = torch.nn.functional.linear(x, w)
        return gather_columns(y) if self.world > 1 else y

    def parallelism_note(self, fused):
        if self.world == 1:
            return "1 GPU"
        how = ("all-gather + rank synchronisation fused into the kernel (TMA stores into the peers' buffers, in-kernel "
               "flags; no collective launch)" if fused else
               "NCCL all-gather" + (f" (fused set-up failed: {self.fused_note})" if self.fused_note else ""))
        return f"column-sharded out_features over {self.world} GPUs, {how}"

    # ---- bf16 x int4 (and int8) single-layer workloads ------------------------------------------------------------
    def run_layer(self, name, with_cpu_baseline):
        wl = WORKLOADS[name]
        kind, M, hbm = wl["kind"], wl["M"], wl["bound"] == "hbm"
        q, dev, world, args = self.q, self.dev, self.world, self.args
        n_local = N_DIM // world
        mark = self.sampler.n_samples()
        # resident state: the local weight shard; several rotated copies for the HBM-bound decode shapes so that the
        # packed weights are re-read from HBM, not from the 126 MB L2
        n_copies = 1 if not hbm else max(2, int(160e6 // (n_local * K_DIM // 2)) + 1)
        if kind == "int4":
            fulls = [make_int4(N_DIM, K_DIM, dev, seed=1000 + c) for c in range(n_copies)]  # same on every rank
            weights = [self.sharded(w) for w in fulls]
            x_host = torch.randn(M, K_DIM, dtype=torch.float32, generator=torch.Generator().manual_seed(7)).to(
                torch.bfloat16).pin_memory()  # the activation is replicated: same seed on every rank
            fwd = lambda x, w: torch.nn.functional.linear(x, w)  # noqa: E731  -> quanto::qbits_mm (one launch)
            fg = self.make_gather(n_local)
        else:
            g = torch.Generator(device=dev).manual_seed(5)
            fulls, weights = [], []
            for c in range(n_copies):
                wd = torch.randint(-127, 127, (N_DIM, K_DIM), dtype=torch.int8, device=dev, generator=g)
                sc = (torch.rand(N_DIM, 1, device=dev, generator=g) / 1e3).to(torch.bfloat16)
                full = q.WeightQBytesTensor(q.qint8, 0, wd.size(), wd.stride(), wd, sc, q.qint8)
                fulls.append(full)
                weights.append(self.sharded(full))
            x_host = torch.randint(-127, 127, (M, K_DIM), dtype=torch.int8,
                                   generator=torch.Generator().manual_seed(7)).pin_memory()
            act_scale = torch.tensor(0.01, dtype=torch.bfloat16, device=dev)
            fwd = lambda x, w: torch.nn.functional.linear(  # noqa: E731  -> quanto::qbytes_mm (one launch)
                q.ActivationQBytesTensor(q.qint8, x.size(), x.stride(), x, act_scale), w)
            fg = None  # 8-bit weights: kernel + NCCL all-gather
        x_dev = x_host.to(dev)
        y_host = torch.empty((M, N_DIM), dtype=torch.bfloat16).pin_memory()

        def gathered(x, w):
            if world == 1:
                return fwd(x, w)
            if fg is not None:
                return fg.forward(x, w, None)
            from quanto_b200.parallel import gather_columns
            return gather_columns(fwd(x, w))

        # ---- parity, outside the timed regions: the gathered result of this rank against the single-rank linear on the
        # FULL weight, bit for bit (same operands, same k order per output element)
        parity_ok = None
        if world > 1:
            y_g = gathered(x_dev, weights[0]).clone()
            y_1 = fwd(x_dev, fulls[0])
            torch.cuda.synchronize()
            parity_ok = self.all_ranks_ok(torch.equal(y_g, y_1))
            del y_g, y_1
        if world > 1:
            fulls = None  # only the shards stay resident
            torch.cuda.empty_cache()

        # HBM-bound decode shapes: the kernel takes 5-20 us, less than the Python dispatch of one QTensor F.linear call
        # (~50 us), so the step is replayed from CUDA graphs (as a serving loop would): one graph per rotated weight copy
        # for the end-to-end step, one graph holding a full rotation for the device-timed steps.
        graphs, graph_outs, rotation = None, None, None
        if hbm:
            for c in range(n_copies):
                gathered(x_dev, weights[c])
            self.barrier()
            graphs, graph_outs = [], []
            for c in range(n_copies):
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr):
                    graph_outs.append(gathered(x_dev, weights[c]))
                graphs.append(gr)
            rotation = torch.cuda.CUDAGraph()
            with torch.cuda.graph(rotation):
                for c in range(n_copies - 1):
                    gathered(x_dev, weights[c])
                rotation_out = gathered(x_dev, weights[n_copies - 1])

        def step_device(i):
            if graphs is not None:
                graphs[i % n_copies].replay()
                return graph_outs[i % n_copies]
            return gathered(x_dev, weights[i % n_copies])

        pipe = None
        if not hbm and world == 1:
            pipe = q.HostPipelinedLinear(weights[0], None, slabs=4, linear_fn=lambda x: fwd(x, weights[0]))

        def step_e2e(i):
            if graphs is not None:
                x_dev.copy_(x_host, non_blocking=True)  # H2D of this step's input into the graph's static input
                graphs[i % n_copies].replay()
                y_host.copy_(graph_outs[i % n_copies], non_blocking=True)  # D2H of the step's result
                return
            if pipe is not None:  # host buffers in, host buffers out: slabs of M pipelined over three streams
                pipe.forward(x_host, y_host, dev)
                return
            xd = x_host.to(dev, non_blocking=True)  # H2D of this step's input from pinned host memory
            y = gathered(xd, weights[i % n_copies])
            y_host.copy_(y, non_blocking=True)  # D2H of the step's result

        steps = args.steps
        if rotation is not None:
            # exactly `steps` steps are timed: whole rotations from one graph, the remainder from single-step graphs
            full, rest = divmod(steps, n_copies)

            def run_steps(_):
                for _r in range(full):
                    rotation.replay()
                for c in range(rest):
                    graphs[c].replay()
                return graph_outs[rest - 1] if rest else rotation_out
            ms_dev = self.timed(run_steps, 1, self.warm) / steps
        else:
            ms_dev = self.timed(step_device, steps, self.warm)
        self.keep_output(name, self.last_out)
        self.last_out = None  # not held through the next timed regions
        ms_e2e = self.timed(step_e2e, steps, self.warm)
        # roofline of the dominant kernel: the local shard's kernel alone (no gather), CUDA events on the launching stream
        if world == 1:
            ms_kernel = ms_dev
        elif hbm:  # graph replay of the local kernels (an eager loop would time the interpreter)
            local = torch.cuda.CUDAGraph()
            with torch.cuda.graph(local):
                for c in range(n_copies):
                    fwd(x_dev, weights[c])
            ms_kernel = self.timed(lambda i: local.replay(), max(1, steps // n_copies), self.warm) / n_copies
            del local
        else:
            ms_kernel = self.timed(lambda i: fwd(x_dev, weights[i % n_copies]), steps, self.warm)
        self.load_for_clocks(step_device, mark)
        clocks = self.sampler.snapshot(mark)

        flops, byts = algorithmic(kind, M, N_DIM, K_DIM)
        flops_l, byts_l = algorithmic(kind, M, n_local, K_DIM)
        unit = "GB/s" if hbm else "TFLOP/s"
        scale_f = (lambda ms: byts / (ms * 1e-3) / 1e9) if hbm else (lambda ms: flops / (ms * 1e-3) / 1e12)
        if hbm:
            achieved, peak, peak_src = byts_l / (ms_kernel * 1e-3) / 1e9, self.peaks["hbm"], self.peaks["source"]
        else:
            achieved, peak, peak_src = flops_l / (ms_kernel * 1e-3) / 1e12, self.peaks["tensor"], self.peaks["source"]
            if kind == "int8":
                peak, peak_src = self.int8_peak()
        traffic = None
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        if world == 1 and os.path.exists(prof):  # measured once under ncu for the single-GPU kernel; meaningless per shard
            traffic = json.load(open(prof)).get(name)
        res = {
            "metric": metric_name(name), "value": scale_f(ms_dev), "unit": unit, "ms_per_step": ms_dev,
            "dtype": "bf16" if kind == "int4" else "int8",
            "config": {"workload": name, "M": M, "N": N_DIM, "K": K_DIM, "group_size": GROUP,
                       "weights": "qint4 canonical packing" if kind == "int4" else "qint8",
                       "parallelism": self.parallelism_note(fg is not None),
                       "l2": ("inputs larger than L2 (A+W+out = %.0f MB > 126 MB)" % (byts / 1e6)) if not hbm else
                             f"{n_copies} rotated weight copies ({n_copies * n_local * K_DIM // 2 / 1e6:.0f} MB > L2)",
                       **({"launch": "CUDA graph replay (one kernel per step)"} if graphs is not None else {}),
                       **({"e2e_path": "HostPipelinedLinear: 4 slabs of M, H2D / GEMM / D2H on three streams"}
                          if pipe is not None else {})},
            "roofline": {"bound": wl["bound"], "achieved": achieved, "peak": peak, "unit": unit,
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "kernel_ms": ms_kernel},
            "e2e": {"value": scale_f(ms_e2e), "unit": unit, "h2d_bytes_per_step": x_host.numel() * x_host.element_size(),
                    "d2h_bytes_per_step": y_host.numel() * y_host.element_size(), "ms_per_step": ms_e2e},
            "gpu_launches": steps * (1 if (world == 1 or fg is not None) else 2),
            "clocks": clocks,
        }
        if parity_ok is not None:
            res["parity_ok"] = parity_ok
        if with_cpu_baseline and self.rank == 0 and world == 1:
            dt, fl, by, cores, sample = cpu_baseline_sample(kind, M)
            res["cpu_baseline"] = {"value": (by / dt / 1e9) if hbm else (fl / dt / 1e12), "unit": unit,
                                   "cores": cores, "kind": "port", "sample": sample}
        del weights, graphs, rotation
        torch.cuda.empty_cache()
        return res

    def int8_peak(self):
        """Measured dense int8 peak on this GPU: torch._int_mm (cuBLASLt) at 8192^3, best of 10 -- the same recipe the
        driver uses for the bf16 figure in MEASURED_PEAKS.json."""
        if getattr(self, "_int8_peak", None) is None:
            try:
                a = torch.randint(-127, 127, (8192, 8192), dtype=torch.int8, device=self.dev)
                b = torch.randint(-127, 127, (8192, 8192), dtype=torch.int8, device=self.dev).t()
                best = None
                for _ in range(12):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    torch._int_mm(a, b)
                    e1.record()
                    torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1)
                    best = ms if best is None else min(best, ms)
                self._int8_peak = (2.0 * 8192 ** 3 / (best * 1e-3) / 1e12, "measured in this run: torch._int_mm 8192^3, best of 12 (burst)")
            except Exception as e:  # noqa: BLE001
                self._int8_peak = (2 * self.peaks["tensor"], f"2 x measured bf16 (torch._int_mm unavailable: {type(e).__name__})")
        return self._int8_peak

    # ---- Llama-3-8B decode step -------------------------------------------------------------------------------------
    def llama_state(self):
        """The 224 qint4 weights of the step (random packed bytes, generated on the device): full tensors on one GPU,
        column shards at N > 1 (only the last layer keeps its full tensors, for the parity check)."""
        if self._llama is not None:
            return self._llama
        dev, world = self.dev, self.world
        layers, last_full = [], None
        for li in range(32):
            ws, fulls = {}, {}
            for idx, (name, N, K) in enumerate(LLAMA3_8B_LAYER):
                full = make_int4(N, K, dev, seed=10000 + 16 * li + idx)
                fulls[name] = full
                ws[name] = self.sharded(full)
            layers.append(ws)
            if li == 31:
                last_full = fulls
            del fulls
        torch.cuda.empty_cache()
        self._llama = (layers, last_full)
        return self._llama

    def run_llama(self, name):
        """BASELINE configs[3] / [4]: the 7 x 32 qint4 QLinear calls of one Llama-3-8B decode step (lm_head excluded, as
        in the reference's bench), batch = M tokens, replayed as one CUDA graph.  Attention / norms are not part of the
        quantized linear path and are not executed; the activation chain between the linears is the one of the model
        (q/k/v read the layer input, o reads q's output, gate/up read o's output, the next layer reads down's output),
        down reads a fixed [M, 14336] activation."""
        M = WORKLOADS[name]["M"]
        dev, world, args = self.dev, self.world, self.args
        mark = self.sampler.n_samples()
        layers, last_full = self.llama_state()
        w_bytes = llama_weight_bytes()
        x_host = torch.randn(M, 4096, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16).pin_memory()
        x = x_host.to(dev)
        h14 = torch.randn(M, 14336, device=dev, generator=torch.Generator(device=dev).manual_seed(4)).to(torch.bfloat16)
        lin = torch.nn.functional.linear
        fgs = None
        if world > 1:
            fgs = {nm: self.make_gather(N // world) for nm, N, _ in LLAMA3_8B_LAYER}
            if any(v is None for v in fgs.values()):
                fgs = None

        def glin(nm, xin, ws, wait_input, wait_output=False):
            if world == 1:
                return lin(xin, ws[nm])
            if fgs is not None:
                return fgs[nm].forward(xin, ws[nm], None, wait_input=wait_input, wait_output=wait_output)
            from quanto_b200.parallel import gather_columns
            return gather_columns(lin(xin, ws[nm]))

        def step(xin, keep=None):
            h = xin
            for li, ws in enumerate(layers):
                last = li == len(layers) - 1
                if keep is not None and last:
                    # (parity step only: the previous layer's down projection was issued with wait_output, so every
                    # rank's slab of `h` has landed before this ATen copy reads it)
                    keep["h_in"] = h.clone()
                # a kernel waits (in-kernel) for the peers' slabs of its INPUT only if the previous gathered kernel
                # produced it; k and v read what q already waited for
                qv = glin("q", h, ws, wait_input=True)
                glin("k", h, ws, wait_input=False)
                glin("v", h, ws, wait_input=False)
                o = glin("o", qv, ws, wait_input=True)
                glin("gate", o, ws, wait_input=True)
                glin("up", o, ws, wait_input=False)
                h = glin("down", h14, ws, wait_input=True, wait_output=last or keep is not None)  # the step's result is complete on exit
                if keep is not None and last:
                    keep["o"] = o.clone()
            return h

        for _ in range(2):
            out = step(x)
        self.barrier()
        parity_ok = None
        if world > 1:
            keep = {}
            out = step(x, keep)
            # single-rank linears on the FULL weights of the last layer, fed with the gathered activations
            o_ref = lin(lin(keep["h_in"], last_full["q"]), last_full["o"])
            h_ref = lin(h14, last_full["down"])
            torch.cuda.synchronize()
            parity_ok = self.all_ranks_ok(torch.equal(out, h_ref) and torch.equal(keep["o"], o_ref))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out_g = step(x)
        y_host = torch.empty_like(out_g, device="cpu").pin_memory()

        def e2e_step(_):
            x.copy_(x_host, non_blocking=True)
            graph.replay()
            y_host.copy_(out_g, non_blocking=True)

        ms_dev = self.timed(lambda i: graph.replay(), args.steps, self.warm)
        self.keep_output(name, out_g)  # the graph's output buffer holds the last replay's result
        ms_e2e = self.timed(e2e_step, args.steps, self.warm)
        self.load_for_clocks(lambda i: graph.replay(), mark, max_seconds=1.0)
        clocks = self.sampler.snapshot(mark)
        achieved = (w_bytes / world) / (ms_dev * 1e-3) / 1e9  # per GPU: each streams its shard of every weight
        res = {
            "metric": metric_name(name), "value": M / (ms_dev * 1e-3), "unit": "tokens/s", "ms_per_step": ms_dev,
            "dtype": "bf16",
            "config": {"workload": name, "batch": M, "layers": 32, "linears_per_step": 224,
                       "weights": "qint4 canonical packing, group 128", "weight_bytes_per_step": w_bytes,
                       "parallelism": self.parallelism_note(fgs is not None),
                       "l2": "3.7 GB of weights per step >> L2", "launch": "one CUDA graph per step",
                       "note": "quantized linears only (lm_head, attention, norms excluded)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": self.peaks["hbm"], "unit": "GB/s",
                         "frac": achieved / self.peaks["hbm"], "traffic": None, "peak_source": self.peaks["source"],
                         "per_gpu": True},
            "e2e": {"value": M / (ms_e2e * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": x_host.numel() * 2,
                    "d2h_bytes_per_step": y_host.numel() * 2, "ms_per_step": ms_e2e},
            "gpu_launches": args.steps * 224 * (1 if (world == 1 or fgs is not None) else 2),
            "clocks": clocks,
        }
        if parity_ok is not None:
            res["parity_ok"] = parity_ok
        del graph
        return res

    # ---- the kernels the reference would dispatch to on this GPU, same shapes, same process ---------------------------
    def compare_set(self):
        """SURVEY 2.2 / BASELINE.md 5: what optimum-quanto itself runs on a B200 for these layers -- library kernels, timed
        here so that the comparison is same-box, same-run.  (The reference's own AWQ / Marlin CUDA sources JIT-compile
        only from its package; tools/compare_reference_kernels.py times them when oracle/_ref carries it.)"""
        dev = self.dev
        out = {}
        M, N, K = 4096, N_DIM, K_DIM

        def best_ms(fn, reps=10):
            fn()
            torch.cuda.synchronize()
            best = None
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                best = ms if best is None else min(best, ms)
            return best

        try:
            a = torch.randn(M, K, device=dev, dtype=torch.bfloat16)
            w = torch.randn(N, K, device=dev, dtype=torch.bfloat16)
            ms = best_ms(lambda: torch.matmul(a, w.t()))
            out["torch_matmul_bf16_m4096"] = {"ms": ms, "tflops": 2.0 * M * N * K / (ms * 1e-3) / 1e12,
                                              "role": "dense bf16 cuBLAS GEMM on the dequantised weight (reference base path, weights pre-dequantised)"}
            del w
        except Exception as e:  # noqa: BLE001
            out["torch_matmul_bf16_m4096"] = {"error": f"{type(e).__name__}: {e}"[:160]}
        try:
            ai = torch.randint(-127, 127, (M, K), dtype=torch.int8, device=dev)
            wi = torch.randint(-127, 127, (N, K), dtype=torch.int8, device=dev)
            sc = (torch.rand(N, 1, device=dev) / 1e3).to(torch.bfloat16)

            def ref_int():  # optimum/quanto/library/qbytes_mm.py:36-50
                acc = torch._int_mm(ai, wi.t())
                return (acc.to(torch.float32) * sc.t()).to(torch.bfloat16)
            ms = best_ms(ref_int)
            ms_mm = best_ms(lambda: torch._int_mm(ai, wi.t()))
            out["torch_int_mm_plus_epilogue_m4096"] = {"ms": ms, "tops": 2.0 * M * N * K / (ms * 1e-3) / 1e12,
                                                       "int_mm_only_ms": ms_mm,
                                                       "int_mm_only_tops": 2.0 * M * N * K / (ms_mm * 1e-3) / 1e12,
                                                       "role": "reference CUDA route for int8 x int8 (library/qbytes_mm.py:36-50,73-88)"}
            del wi
        except Exception as e:  # noqa: BLE001
            out["torch_int_mm_plus_epilogue_m4096"] = {"error": f"{type(e).__name__}: {e}"[:160]}
        try:  # tinygemm: the reference's bf16 int4 route (tensor/weights/tinygemm/qbits.py:42-62)
            wu = torch.randint(0, 256, (N, K // 2), dtype=torch.uint8, device=dev)
            wp = torch._convert_weight_to_int4pack(wu, 2)
            sz = torch.rand(K // GROUP, N, 2, device=dev).to(torch.bfloat16)
            for m in (4096, 1, 8, 32):
                xa = torch.randn(m, K, device=dev, dtype=torch.bfloat16)
                ms = best_ms(lambda: torch._weight_int4pack_mm(xa, wp, GROUP, sz), reps=10 if m > 32 else 30)
                fl, by = algorithmic("int4", m, N, K)
                out[f"torch_weight_int4pack_mm_m{m}"] = {"ms": ms, "tflops": fl / (ms * 1e-3) / 1e12,
                                                         "gbs": by / (ms * 1e-3) / 1e9,
                                                         "role": "reference CUDA route for bf16 x int4 (TinyGemm); L2-warm for small m"}
        except Exception as e:  # noqa: BLE001
            out["torch_weight_int4pack_mm"] = {"error": f"{type(e).__name__}: {e}"[:160]}
        torch.cuda.empty_cache()
        return out

    # ---- top level --------------------------------------------------------------------------------------------------
    def run(self):
        args = self.args
        name = args.workload
        wl = WORKLOADS[name]
        t_start = time.time()
        if wl["kind"] == "llama":
            head = self.run_llama(name)
        else:
            head = self.run_layer(name, with_cpu_baseline=True)
        line = {
            "metric": head["metric"], "value": head["value"], "unit": head["unit"], "n_gpus": self.world,
            "steps": args.steps, "warmup": self.warm, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": head["dtype"], "data": "synthetic",
            "config": head["config"], "roofline": head["roofline"], "e2e": head["e2e"],
            "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
        }
        for k in ("parity_ok", "cpu_baseline"):
            if k in head:
                line[k] = head[k]
        if name == DEFAULT_WORKLOAD and not args.no_extras:
            extra = {}
            for nm in (EXTRA_WORKLOADS if self.world == 1 else EXTRA_WORKLOADS_MULTI):
                try:
                    r = self.run_llama(nm) if WORKLOADS[nm]["kind"] == "llama" else self.run_layer(nm, False)
                    extra[nm] = {k: r[k] for k in ("metric", "value", "unit", "ms_per_step", "roofline", "e2e", "clocks",
                                                   "parity_ok", "gpu_launches") if k in r}
                    extra[nm]["config"] = {k: v for k, v in r["config"].items() if k in ("parallelism", "l2", "launch", "batch")}
                except Exception as e:  # noqa: BLE001  (an extra must never cost the headline)
                    extra[nm] = {"error": f"{type(e).__name__}: {e}"[:300]}
                    if self.world > 1:
                        raise
            line["extra"] = extra
            if self.world == 1:
                line["compare"] = self.compare_set()
            line["bench_seconds"] = round(time.time() - t_start, 1)
        self.sampler.stop()
        if self.outputs is not None and self.rank == 0:
            write_outputs(args.dump_outputs, self.outputs)
        if self.rank == 0:
            print(json.dumps(line))
        if self.world > 1:
            self.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--gather", default="fused", choices=["fused", "nccl"],
                    help="multi-GPU int4: all-gather fused into the kernel (default) or kernel + NCCL all-gather")
    ap.add_argument("--no-extras", action="store_true", help="default workload only: skip the extra / compare sections")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result of each timed workload's last step to "
                         "DIR/<workload>.npy (float32; for M > 32 two seeded rows of every 32-row band)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        if wl["kind"] == "llama":
            run_reference_llama(args, wl)
        else:
            run_reference(args, wl)
    else:
        Bench(args).run()


if __name__ == "__main__":
    main()

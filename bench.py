#!/usr/bin/env python
"""bench.py -- the hot path of the physics layer on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--dtype f64] [--dump-outputs DIR]
    python bench.py --impl reference ...          # the reference's CPU arithmetic (oracle port), host cores

A "step" is one pass of the physics layer over one batch of synthetic log-normal fields (SURVEY.md section 8d):
    unit 1  coarse-grained model forward (logX, F -> u) and its adjoint (gbar_u -> dL/dlogX); exp(.)+1e-8 inside,
            as ReducedOrderModelOperator.forward does (components.py:298);
    unit 2  virtual-observable residual r = V^T (K_fom(a) y~ - f) for the same samples, a = exp(x) the fine
            conductivity field (the reference evaluates exp(x) once per data point when it assembles and caches K,
            VirtualObservables.py:52-59, so the per-step input is the conductivity; the log-input timing is reported
            beside it in ``components``).
``value`` = samples/s with inputs resident in HBM (each sample = 1 CGM fwd+adjoint solve + 1 VO residual evaluation).
``e2e`` is the same pass through the public module API from pinned HOST buffers, copies included (chunked, copies
overlapped with compute).  ``configs`` holds the other BASELINE.json configurations measured in the same run (config 3,
config 4 strong-scaled over the ranks, FP32 I/O).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "CGM fwd+adjoint solves/s & VO residual evals/s"
UNIT = "samples/s (1 CGM fwd+adjoint solve + 1 VO residual eval per sample)"
FP64_PEAK_TFLOPS = 37.0   # DMMA/DFMA rate measured on this pool (profiles/r1_fp64_peak.txt); MEASURED_PEAKS.json has no FP64 entry


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON record: everything libraries print there (NCCL's version banner, ...)
    is sent to stderr for the whole run; ``emit`` writes the record to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the records of the other configurations (configs 3, 4, FP32)")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replays")
    ap.add_argument("--no-overlap", action="store_true", help="keep the ROM and VO kernels on one stream")
    ap.add_argument("--e2e-stream-fields", action="store_true",
                    help="e2e: copy the VO data points' conductivity fields from the host every step too (default: resident)")
    ap.add_argument("--sm-reserve", type=int, default=-1,
                    help="SMs the VO kernel leaves to the ROM kernels of the overlapped step (-1 = calibrate during warm-up)")
    ap.add_argument("--log-input", action="store_true", help="VO residual from the log-field (exp inside the kernel) in the step")
    ap.add_argument("--e2e-chunks", type=int, default=4)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (u, dL/dlogX, VO residual of rank 0's "
                         "batch) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "b200" or args.workload == "cfg5"):
        ap.error("--dump-outputs writes the outputs of the physics-layer step: --impl b200, workloads cfg1 - cfg4")
    return args


def workload_config(w):
    """The ``config`` object: identical in both arms (the driver compares them)."""
    return dict(w.describe(), vo_input="conductivity a = exp(x) (SURVEY 8d unit 2)", rom_input="log-conductivity (exp inside)",
                l2="inputs larger than L2: %.0f MB streamed per step per GPU"
                   % ((w.vo_bytes_per_eval(8) + w.cgm_bytes_per_solve(8)) * w.B / 1e6))


# ------------------------------------------------------------------------------- CPU arm (oracle port)
class CpuReference(object):
    """The reference's own arithmetic on the host cores (oracle port, ``kind: port``: FEniCS is not installable here):
      CGM   bottleneck/ROM.py ops through torch autograd (oracle/rom_ref.py), all torch threads;
      VO    (a) ``cached_gamma``: r_n = Gamma_n y_n - alpha_n in a Python loop over data points with Gamma_n = V^T K_n and
                alpha_n cached, exactly what LinearQuerry / VirtualObservable.update do every step for a constant sampler
                (VirtualObservables.py:61-69 once, :662 per step) -- the HEADLINE variant;
            (b) ``assemble``: K_n re-assembled and Gamma_n re-formed per data point per step (what a resample() of a
                non-constant sampler costs; FEniCS' assemble replaced by a precomputed-pattern CSR assembly);
            (c) ``vectorised``: (K_n y_n - f_n) V with the cached CSR K_n (SURVEY 8d's fair variant).
    Works on the first ``n`` samples of the workload."""

    def __init__(self, w, n):
        import numpy as np
        import torch
        from oracle import rom_ref, vo_ref
        self.np, self.torch, self.rom_ref, self.vo_ref = np, torch, rom_ref, vo_ref
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.w, self.n = w, int(min(n, w.B))
        rom, fom = w.physics["rom"], w.physics["fom"]
        self.M = torch.tensor(rom.mesh.dense_element_tensor())
        self.bc = torch.tensor(rom.constrained_dofs)
        self.asm = vo_ref.CsrAssembler(fom.mesh.coords, fom.mesh.cells, fom.constrained_dofs, fom.free_dofs,
                                       Ke=fom.mesh.element_stiffness())
        self.pix = fom.mesh.pixel_of_cell()
        # setup (not timed): K_n, f_n, Gamma_n, alpha_n of the sampled data points, cached as the reference caches them
        self.K, self.f, self.Gamma, self.alpha = [], [], [], []
        for b in range(self.n):
            K, f = self.asm.assemble(np.exp(w.log_image[b][self.pix]), w.g_fom[b])
            G, al = vo_ref.construct_querry_weak_galerkin(K, f, w.V)
            self.K.append(K); self.f.append(f); self.Gamma.append(np.ascontiguousarray(G)); self.alpha.append(al)
        self.tX, self.tF, self.tg = (torch.tensor(t[:self.n]) for t in (w.logX, w.F, w.gbar_u))

    def cgm(self):
        t0 = time.perf_counter()
        self.rom_ref.rom_fwd_adjoint(self.M, self.bc, self.tX, self.tF, self.tg)
        return time.perf_counter() - t0

    def vo_cached_gamma(self):
        w = self.w
        t0 = time.perf_counter()
        for b in range(self.n):   # Python loop over data points, as VirtualObservables.py:895 / :985
            _ = self.Gamma[b] @ w.y[b] - self.alpha[b]
        return time.perf_counter() - t0

    def vo_assemble(self, n):
        np_, w = self.np, self.w
        t0 = time.perf_counter()
        for b in range(n):
            K, f = self.asm.assemble(np_.exp(w.log_image[b][self.pix]), w.g_fom[b])
            Gamma, alpha = self.vo_ref.construct_querry_weak_galerkin(K, f, w.V)
            _ = Gamma @ w.y[b] - alpha
        return (time.perf_counter() - t0) / n

    def vo_vectorised(self):
        w = self.w
        t0 = time.perf_counter()
        for b in range(self.n):
            _ = (self.K[b] @ w.y[b] - self.f[b]) @ w.V
        return (time.perf_counter() - t0) / self.n

    def step(self):
        """One step of the arm = the n sampled samples through both units (cached-Gamma VO): seconds."""
        return self.cgm() + self.vo_cached_gamma()


def reference_sample_size(w):
    return 512 if w.d <= 4095 else 64       # Gamma cache: n * m * d doubles (430 MB at config 2, 2.1 GB / 64 at config 3)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import gpde_b200  # noqa: F401
    from gpde_b200.workloads import Workload
    from gpde_b200.workloads import CONFIGS
    full = Workload(args.workload, B=int(args.batch or min(CONFIGS[args.workload]["B"], 4096)), seed=0)
    n = reference_sample_size(full)
    ref = CpuReference(full, n)
    for _ in range(max(3, args.warmup)):      # the first calls pay torch's thread-pool start-up (2 s, 0.6 s, 0.04 s measured)
        ref.step()
    steps, acc, acc_c, acc_v = args.steps, 0.0, 0.0, 0.0
    for _ in range(steps):
        c, v = ref.cgm(), ref.vo_cached_gamma()
        acc += c + v; acc_c += c; acc_v += v
    value = steps * ref.n / acc
    t_asm = ref.vo_assemble(min(ref.n, 32))
    t_vec = ref.vo_vectorised()
    sample_desc = ("each step = the first %d samples of the workload batch (%d): CGM fwd+adjoint (torch autograd, %d threads) + "
                   "VO r = Gamma y - alpha per data point with cached Gamma" % (ref.n, full.B, ref.cores))
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * acc / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "impl": "reference",
        "config": workload_config(full),
        "samples_per_step": ref.n,
        "extrapolated_from": "none: value = samples_per_step / (ms_per_step / 1000); the step is a bounded sample (%d of %d samples)"
                             % (ref.n, full.B),
        "components": {"cgm_solves_per_s": steps * ref.n / acc_c, "vo_evals_per_s": steps * ref.n / acc_v,
                       "vo_evals_per_s_assemble_each_step": 1.0 / t_asm, "vo_evals_per_s_vectorised_cached_K": 1.0 / t_vec},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores, "kind": "port", "sample": sample_desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------- clocks sampler
class ClockSampler(threading.Thread):
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt, self.proc = index, [], threading.Event(), None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for ln in self.proc.stdout:
                self.samples.append((time.perf_counter(), ln.strip()))
                if self._stop_evt.is_set():
                    break
        except Exception:
            pass

    def stop(self):
        self._stop_evt.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self, t0, t1):
        rows = [s for (t, s) in self.samples if t0 <= t <= t1] or [s for (_, s) in self.samples]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            p = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except Exception:
                continue
            for nm, val in zip(names, p[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------- B200 arm
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_traffic(workload, dtype):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
            return json.load(fh).get("%s_%s" % (workload, dtype))
    except Exception:
        return None


def bind_near_gpu(index):
    """Pins this process (and the pinned host buffers it allocates next: first touch) to the CPU cores nvidia-smi reports as
    local to GPU ``index`` -- with 8 ranks each streaming 270 MB per step from host memory, buffers on the far socket halve
    the per-GPU copy rate.  Returns the affinity string or None."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
                             timeout=20).stdout
        header = None
        for ln in out.splitlines():
            cells = [c.strip() for c in ln.split("\t")]
            if header is None and any("CPU Affinity" in c for c in cells):
                header = [c for c in cells if c]
                continue
            if header and cells and cells[0].replace("\x1b[4m", "").replace("\x1b[0m", "").strip() == "GPU%d" % index:
                vals = [c for c in cells if c]
                aff = vals[1 + [h for h in header].index("CPU Affinity")] if "CPU Affinity" in header else None
                cores = set()
                for part in (aff or "").split(","):
                    if "-" in part:
                        lo, hi = part.split("-")
                        cores.update(range(int(lo), int(hi) + 1))
                    elif part.strip().isdigit():
                        cores.add(int(part))
                cores &= set(os.sched_getaffinity(0))
                if cores:
                    os.sched_setaffinity(0, cores)
                    return aff
    except Exception:
        pass
    return None


class HotPath(object):
    """Plans, resident inputs and the launch sequence of one workload on one device."""

    def __init__(self, torch, dev, w, tdt, host_inputs, log_input=False):
        from gpde_b200 import ROM as rom_mod
        from gpde_b200.components import ReducedOrderModelOperator
        from gpde_b200.VirtualObservables import VoPlan
        self.torch, self.dev, self.w, self.tdt, self.rom_mod, self.log_input = torch, dev, w, tdt, rom_mod, log_input
        self.op = ReducedOrderModelOperator.FromPhysics(w.physics, dtype=tdt, device=dev)
        self.rom = self.op.rom
        self.rom.deferred_checks = True
        self.plan = self.rom._get_plan()
        self.vplan = VoPlan.cached(w.physics["fom"], dev, pixel_input=True)
        self.d = host_inputs
        self.B = int(self.d["logX"].shape[0])
        self.path = self.vplan.kernel_path(w.m, tdt)
        self.vo_stream = torch.cuda.Stream(device=dev)
        self.packed, self.ev_packed = None, torch.cuda.Event()
        self.split_pack = self.path == 2
        self.sm_reserve = 0      # SMs the VO kernel leaves to the ROM kernels of the overlapped step (run_b200 calibrates it)

    def vo(self, log_input=None):
        d = self.d
        log_input = self.log_input if log_input is None else log_input
        return self.vplan.residual(d["a_log"] if log_input else d["a"], d["y"], d["g"], d["V"], a_is_log=log_input)

    def vo_prepacked(self):
        """The residual call as VirtualObservablesEnsemble.residuals makes it between two resample() calls: V = W of the
        coarse-grained-residual sampler packed once (VirtualObservables.py:297-321 keeps it constant), no packing launch."""
        d = self.d
        if getattr(self, "packed_once", None) is None:
            pw = self.vplan.pack_weights(d["V"], self.B)
            self.packed_once = pw if hasattr(pw, "buf") else False
        if not self.packed_once:
            return None
        return self.vplan.residual(d["a_log"] if self.log_input else d["a"], d["y"], d["g"], self.packed_once, a_is_log=self.log_input)

    def rom_forward(self):
        d = self.d
        return self.rom_mod._launch_forward(self.plan, d["logX"], d["F"], True, want_factor=True, info=self.rom._info_word(self.dev))

    def rom_adjoint(self, u, factor):
        return self.rom_mod._launch_adjoint(self.plan, self.d["logX"], u, factor, self.d["gbar"], True, want_gradF=False)

    def step(self, overlap=False):
        """One pass of the physics layer.  The coarse-grained model (forward -> adjoint) and the VO residual are independent:
        with ``overlap`` the VO kernels go to a second stream (fork / join by events), so the small ROM kernels fill the SMs
        the VO grid leaves idle."""
        torch, d = self.torch, self.d
        cur = torch.cuda.current_stream(self.dev)
        if overlap:
            self.vo_stream.wait_stream(cur)
            with torch.cuda.stream(self.vo_stream):
                if self.split_pack:
                    # V packed by its own call; the ROM kernels are held back until the packing has run, so that the VO
                    # kernel's CTAs (one whole SM each) are placed first and the ROM CTAs take the SMs left
                    pw = self.vplan.pack_weights(d["V"], self.B, out=self.packed)
                    if self.packed is None and hasattr(pw, "buf"):
                        self.packed = pw
                    self.ev_packed.record(self.vo_stream)
                    r = self.vplan.residual(d["a_log"] if self.log_input else d["a"], d["y"], d["g"], pw, a_is_log=self.log_input,
                                            sm_reserve=self.sm_reserve)
                else:
                    r = self.vo()
            if self.split_pack:
                cur.wait_event(self.ev_packed)
        u, factor = self.rom_forward()
        gX, _ = self.rom_adjoint(u, factor)
        if overlap:
            cur.wait_stream(self.vo_stream)
        else:
            r = self.vo()
        return u, gX, r

    def launches_per_step(self):
        return 1 + 1 + self.vplan.launches_per_residual(self.w.m, self.tdt)


def calibrate_sm_reserve(torch, hp, K, candidates):
    """The VO kernel's CTAs own a whole SM each and its last wave is sized for the SMs it may use; the ROM kernels of the
    overlapped step need a few SMs beside it.  Times one graph of the step per candidate number of SMs left to them
    (untimed warm-up work), keeps the fastest in ``hp.sm_reserve`` and returns {candidate: ms per step}."""
    ms = {}
    if hp.split_pack:
        for cand in candidates:
            hp.sm_reserve = cand
            ms[cand] = graph_timed(torch, lambda: hp.step(overlap=True), K)[0]
        hp.sm_reserve = min(ms, key=ms.get)
    return ms


def graph_timed(torch, fn, K):
    """Average device milliseconds of ``fn`` over K replays of its CUDA graph (eager launches if capture is refused)."""
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            keep = fn()
        gr.replay()
        torch.cuda.synchronize()
        run, mode = gr.replay, "cuda_graph"
    except Exception as exc:   # noqa: BLE001
        sys.stderr.write("bench: CUDA graph capture failed (%s); timing eager launches\n" % (exc,))
        keep, run, mode = None, fn, "eager"
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(K):
        run()
    a1.record()
    torch.cuda.synchronize()
    return a0.elapsed_time(a1) / K, keep, run, mode


def device_inputs(torch, dev, w, B, tdt, seed):
    """Device-generated stand-ins of the workload's inputs for the secondary records (same shapes and value ranges as the
    workload generator's fields, without the spatial correlation: generating 131072 correlated 64 x 64 fields on the host
    would take longer than the whole bench; kernel time does not depend on the values)."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=gen, device=dev, dtype=torch.float64)
    a_log = (0.4 + 0.8 * rn(B, w.P)).to(tdt)
    d = dict(a_log=a_log, a=torch.exp(a_log.double()).to(tdt), logX=(0.4 + 0.5 * rn(B, w.E)).to(tdt),
             F=torch.tensor(w.F[0], device=dev, dtype=tdt).expand(B, -1).contiguous(), gbar=rn(B, w.n).to(tdt),
             y=(torch.tensor(w.y[0], device=dev).expand(B, -1) + 0.01 * rn(B, w.d)).to(tdt),
             g=torch.tensor(w.g_fom[0], device=dev, dtype=tdt), V=torch.tensor(w.V, device=dev, dtype=tdt))
    return d


DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, outputs):
    """Writes each array of ``outputs`` (name -> [B, ...] device tensor) as out_dir/<name>.npy in its own float dtype.  Above
    DUMP_MAX_BYTES in all, every array keeps the same fixed, seeded sample of batch rows (in increasing order)."""
    import numpy as np
    arrays = {k: t.detach().cpu().numpy() for k, t in outputs.items()}
    B = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    if B * row_bytes > DUMP_MAX_BYTES:
        keep = (DUMP_MAX_BYTES - 4096) // row_bytes         # 4096: room for the .npy headers
        rows = np.sort(np.random.RandomState(0).choice(B, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def nonzero_tile_fraction(w):
    """Fraction of the (16 consecutive nodes of a node row) x (8 columns) blocks of V with a non-zero entry: the blocks
    vo_gridgemm.cuh does not skip."""
    import numpy as np
    mesh = w.physics["fom"].mesh
    nx, ny = mesh.nx, mesh.ny
    ncol = nx - 1
    V = np.asarray(w.V).reshape(ny + 1, ncol, w.m)
    cp, mp = -(-nx // 16) * 16, -(-w.m // 8) * 8
    Z = np.zeros((ny + 1, cp, mp), dtype=bool)
    Z[:, :ncol, :w.m] = V != 0
    blocks = Z.reshape(ny + 1, cp // 16, 16, mp // 8, 8).any(axis=(2, 4))
    return float(blocks.mean())


def roofline_record(w, B, s, t_vo, path, workload, dtype, peak, peak_src, t_kernel=None):
    """t_vo: device time of the residual call (packing launch + kernel); t_kernel: the dominant kernel alone, measured as the
    call with the weights packed beforehand (exactly one launch: vo_grid2_kernel) -- the duration the roofline is taken on."""
    vo_bytes = w.vo_bytes_per_eval(s) * B
    t_call = t_vo
    if t_kernel is not None and path == 2:
        t_vo = t_kernel
    achieved = vo_bytes / (t_vo * 1e-3) / 1e9
    # FP64 work of one VO evaluation (DESIGN.md section 4): fluxes 10 + contraction m per free node (FMA = 2 flop)
    vo_flops = 2.0 * w.d * (10 + w.m) * B
    if path in (0, 3) and w.m > 32:
        rec = {"kernel": "vo_gridgemm_kernel (fine residual produced inside the FP64 DMMA contraction)" if path == 3
               else "vo_matvec_kernel + vo_gemm_kernel (FP64 DMMA contraction dominates)", "bound": "tensor",
               "achieved": vo_flops / (t_vo * 1e-3) / 1e12, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
               "frac": vo_flops / (t_vo * 1e-3) / 1e12 / FP64_PEAK_TFLOPS, "traffic": recorded_traffic(workload, dtype),
               "peak_source": "measured FP64 mma.sync rate (profiles/r1_fp64_peak.txt); MEASURED_PEAKS.json has no FP64 entry",
               "algorithmic_flops_per_launch": vo_flops, "hbm_frac": achieved / peak}
        if path == 3:
            # the kernel skips the 16-node x 8-column blocks of V that are all zero (exact); what the tensor pipe really executes
            fill = nonzero_tile_fraction(w)
            ex = 2.0 * w.d * (10 + fill * w.m) * B
            rec.update({"nonzero_tile_fraction_of_V": fill, "executed_flops_per_launch": ex,
                        "executed_frac_of_peak": ex / (t_vo * 1e-3) / 1e12 / FP64_PEAK_TFLOPS})
        return rec
    return {"kernel": {2: "vo_grid2_kernel", 1: "vo_fused_kernel"}.get(path, "vo_matvec_kernel + vo_gemm_kernel"),
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": recorded_traffic(workload, dtype), "peak_source": peak_src, "algorithmic_bytes_per_launch": vo_bytes,
            "fp64_pipe_frac": vo_flops / (t_vo * 1e-3) / 1e12 / FP64_PEAK_TFLOPS,
            "ms_kernel": t_vo, "ms_call_with_packing_launch": t_call, "frac_of_call_with_packing_launch": vo_bytes / (t_call * 1e-3) / 1e9 / peak}


def sub_record(torch, dist, dev, name, B_total, tdt, K, rank, world, peak, peak_src, strong):
    """One secondary record: ROM forward + adjoint + VO residual on device-generated inputs, graph-replayed, max over ranks."""
    from gpde_b200.sharding import shard_range
    from gpde_b200.workloads import Workload
    lo, hi = shard_range(B_total, rank, world) if strong else (0, B_total)
    B = hi - lo
    w = Workload(name, B=8, seed=0)
    hp = HotPath(torch, dev, w, tdt, device_inputs(torch, dev, w, B, tdt, 100 + rank))
    for _ in range(2):
        hp.step()
    torch.cuda.synchronize()
    t_fwd, keep, _, _ = graph_timed(torch, hp.rom_forward, K)
    t_adj, _, _, _ = graph_timed(torch, lambda: hp.rom_adjoint(*keep), K)
    t_vo, _, _, _ = graph_timed(torch, hp.vo, K)
    t_vo_log, _, _, _ = graph_timed(torch, lambda: hp.vo(True), K)
    t_vo_pre = None
    if hp.split_pack and hp.vo_prepacked() is not None:
        t_vo_pre, _, _, _ = graph_timed(torch, hp.vo_prepacked, K)
    calibrate_sm_reserve(torch, hp, max(5, K), [0, 8, 11, 16])
    _, _, run, mode = graph_timed(torch, lambda: hp.step(overlap=True), 2)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    hp.rom.check()
    if world > 1:
        tt = torch.tensor([ms, t_fwd, t_adj, t_vo, t_vo_log, t_vo_pre or 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, t_fwd, t_adj, t_vo, t_vo_log, t_pre_max = (float(x) for x in tt.tolist())
        t_vo_pre = t_pre_max if t_vo_pre is not None else None
    s = 8 if tdt == torch.float64 else 4
    total = B_total if strong else world * B
    rec = {"workload": name, "desc": w.cfg["desc"], "dtype": "f64" if s == 8 else "f32", "scaling": "strong" if strong else "weak",
           "global_batch": total, "per_gpu_batch": B, "value": total / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": K,
           "launch_mode": mode, "data": "synthetic, device-generated (uncorrelated N(0.4, 0.8^2) log-fields of the workload's shapes)",
           "ms_rom_forward": t_fwd, "ms_rom_adjoint": t_adj, "ms_vo_residual": t_vo, "ms_vo_residual_log_input": t_vo_log,
           "cgm_solves_per_s": total / ((t_fwd + t_adj) * 1e-3), "vo_evals_per_s": total / (t_vo * 1e-3),
           "cgm_hbm_frac": w.cgm_bytes_per_solve(s) * B / ((t_fwd + t_adj) * 1e-3) / 1e9 / peak,
           "vo_kernel_path": hp.path, "sms_left_to_rom_kernels": hp.sm_reserve,
           "roofline": roofline_record(w, B, s, t_vo, hp.path, name, "f64" if s == 8 else "f32", peak, peak_src, t_kernel=t_vo_pre)}
    del hp
    torch.cuda.empty_cache()
    return rec


def svi_record(torch, dist, dev, K, rank, world, peak_unused=None):
    """BASELINE config 5: the semi-supervised SVI ELBO step around the physics layer, data-parallel over the ranks
    (owner-sharded per-sample tables, ONE flat NCCL all-reduce of the shared gradients), FP32 modules (the reference's model
    dtype).  Every rank owns N_s = 128 supervised + N_vo = 128 virtual-observable data points and an unsupervised batch of
    64 (weak scaling).  Times the eager step, the CUDA-graph replay of the whole step, the all-reduce alone and the batched
    virtual-observable update; max over ranks."""
    from gpde_b200 import svi
    from gpde_b200.svi_workload import SviWorkload
    wl = SviWorkload(dev, torch.float32, seed=100 + rank)
    wl.build_virtual_observables()
    wl.update_virtual_observables(N_mc=64, step=0)
    dp = svi.DataParallelSVI(wl.shared_parameters(), wl.local_parameters(), wl.elbo, lr=1e-3, capturable=True)

    def timed(fn, n):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    for _ in range(3):
        dp.step()
    t_eager = timed(dp.step, K)
    t_ar = timed(dp.bucket.allreduce_, K) if world > 1 else 0.0
    for _ in range(2):      # untimed: the first update past iteration 0 builds the precision update's plans and scratch
        wl.update_virtual_observables(N_mc=64, step=1)
    t_vo = timed(lambda: wl.update_virtual_observables(N_mc=64, step=1), max(5, K))
    mode = "cuda_graph"
    try:
        gs = svi.GraphedStep(dp)
        t_graph = timed(gs.replay, K)
    except Exception as exc:   # noqa: BLE001
        sys.stderr.write("bench: cfg5 graph capture failed (%s)\n" % (exc,))
        t_graph, mode = t_eager, "eager"
    wl.g.rom.check()
    elbo = float(dp.global_elbo().item())
    if world > 1:
        tt = torch.tensor([t_eager, t_graph, t_ar, t_vo], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_eager, t_graph, t_ar, t_vo = (float(x) for x in tt.tolist())
    return {"workload": "cfg5", "desc": "semi-supervised SVI ELBO step (stand-in CNN encoder / decoder + ROM + VO term), data-parallel, "
                                        "one flat NCCL all-reduce of the shared gradients", "dtype": "f32", "scaling": "weak",
            "per_gpu": {"N_supervised": wl.N_s, "N_vo": wl.N_vo, "bs_unsupervised": wl.bs_u}, "n_gpus": world,
            "value": world * wl.samples_per_step() / (t_graph * 1e-3), "unit": "data points/s through the SVI step",
            "ms_per_step": t_graph, "launch_mode": mode, "ms_per_step_eager": t_eager, "steps": K,
            "cgm_solves_per_s": world * wl.cgm_solves_per_step() / (t_graph * 1e-3),
            "shared_parameters": dp.bucket.numel, "allreduce_bytes": dp.bucket.nbytes, "ms_allreduce_alone": t_ar,
            "ms_vo_update_N_mc64": t_vo, "fused_log_likelihood": wl.fused, "elbo_sum_over_ranks": elbo,
            "batchnorm": "none in the stand-in CNNs", "data": "synthetic, random-init weights"}


def run_cfg5(args):
    import torch
    import torch.distributed as dist
    import gpde_b200  # noqa: F401
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    t0 = time.perf_counter()
    rec = svi_record(torch, dist, dev, args.steps, rank, world)
    t1 = time.perf_counter()
    if sampler:
        sampler.stop()
    if rank == 0:
        line = {"metric": METRIC, "value": rec["value"], "unit": rec["unit"], "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": "cfg5", "desc": rec["desc"]},
                "components": rec, "gpu_launches": None, "clocks": sampler.summary(t0, t1) if sampler else None}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_b200(args):
    import numpy as np  # noqa: F401
    import torch
    import torch.distributed as dist
    import gpde_b200  # noqa: F401
    from gpde_b200.workloads import Workload
    if args.workload == "cfg5":
        return run_cfg5(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    affinity = bind_near_gpu(local)      # before the pinned buffers are allocated
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    tdt = torch.float64 if args.dtype == "f64" else torch.float32
    s = 8 if args.dtype == "f64" else 4
    peak, peak_src = measured_peaks()

    # per-GPU shard of the sample-sharded batch.  Default: weak scaling, every rank owns a full workload batch.
    # cfg4 (BASELINE config 4): ONE batch of 131072 cut into contiguous shards (gpde_b200.sharding), strong scaling.
    from gpde_b200.sharding import shard_range
    strong = args.workload == "cfg4"
    if strong:
        from gpde_b200.workloads import CONFIGS
        total = int(args.batch if args.batch is not None else CONFIGS["cfg4"]["B"])
        lo, hi = shard_range(total, rank, world)
        w = Workload(args.workload, B=hi - lo, seed=rank)
    else:
        w = Workload(args.workload, B=args.batch, seed=rank)
    B = w.B

    host = dict(logX=w.logX, F=w.F, gbar=w.gbar_u, a_log=w.log_image, y=w.y,
                g=(w.g_fom[0] if w.ptype == "ND" else w.g_fom), V=w.V)
    pinned = {k: torch.tensor(v, dtype=tdt).pin_memory() for k, v in host.items()}
    pinned["a"] = torch.exp(torch.tensor(w.log_image)).to(tdt).pin_memory()     # conductivities, computed once at setup
    d = {k: v.to(dev, non_blocking=True) for k, v in pinned.items()}
    torch.cuda.synchronize()
    hp = HotPath(torch, dev, w, tdt, d, log_input=args.log_input)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        hp.step()
    torch.cuda.synchronize()
    K = args.steps

    # ---- (1) eager launches: host enqueue cost and the eager step time (events on the launching stream)
    e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    e_start.record()
    for k in range(K):
        hp.step()
    e_end.record()
    t_host1 = time.perf_counter()
    torch.cuda.synchronize()
    hp.rom.check()
    eager_ms = e_start.elapsed_time(e_end) / K
    host_enqueue_ms = (t_host1 - t_host0) * 1e3 / K

    # ---- (1b) per-kernel-group device times, free of host launch gaps (each group in its own CUDA graph)
    t_fwd, keep, _, _ = graph_timed(torch, hp.rom_forward, K)
    t_adj, _, _, _ = graph_timed(torch, lambda: hp.rom_adjoint(*keep), K)
    t_vo, _, _, _ = graph_timed(torch, hp.vo, K)
    t_vo_other, _, _, _ = graph_timed(torch, lambda: hp.vo(not hp.log_input), K)
    t_vo_pre = None
    if hp.split_pack and hp.vo_prepacked() is not None:
        t_vo_pre, _, _, _ = graph_timed(torch, hp.vo_prepacked, K)
    # the transposed application q = K_ff(a) (V s) = Gamma^T s, the residual's gradient w.r.t. y (VirtualObservables.py:663)
    t_vo_T = None
    if w.m <= 32:
        s_T = torch.randn(B, w.m, dtype=tdt, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
        t_vo_T, _, _, _ = graph_timed(torch, lambda: hp.vplan.residual_T(d["a"], d["V"], s_T, a_is_log=False), K)
    hp.rom.check()

    # ---- (2) the timed region: K steps, each step = the same launches replayed from one CUDA graph (the step is
    # launch-bound from Python at this batch); eager launches if capture is refused or --no-graph
    # The VO kernel's CTAs own a whole SM each and its last wave is sized for the SMs it may use; the ROM kernels of the
    # overlapped step need a few SMs beside it: the number left to them is calibrated here (untimed), one graph per candidate
    reserve_ms = {}
    if args.sm_reserve >= 0:
        hp.sm_reserve = args.sm_reserve
    elif not args.no_overlap and not args.no_graph:
        reserve_ms = calibrate_sm_reserve(torch, hp, max(10, min(K, 30)), [0, 8, 11, 16, 20])
    if args.no_graph:
        run, keep, mode = (lambda: hp.step(overlap=not args.no_overlap)), None, "eager"
    else:
        _, keep, run, mode = graph_timed(torch, lambda: hp.step(overlap=not args.no_overlap), 3)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    start.record()
    for k in range(K):
        out = run()      # eager: the step's (u, dL/dlogX, r); a graph replay returns None and refills ``keep``
    end.record()
    torch.cuda.synchronize()
    t_wall1 = time.perf_counter()
    hp.rom.check()
    if args.dump_outputs is not None and rank == 0:
        u, gX, r = keep if out is None else out
        dump_outputs(args.dump_outputs, {"u": u, "grad_logX": gX, "vo_residual": r})
    elapsed_ms = start.elapsed_time(end)
    if world > 1:
        tt = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        elapsed_ms = float(tt.item())
    ms_per_step = elapsed_ms / K

    # ---- end to end through the public module API from pinned host buffers: the batch is cut into chunks; the copies of
    # chunk c+1 (copy stream) overlap the kernels of chunk c (compute stream) and the read-back of chunk c-1
    e2e = None
    if not args.no_e2e:
        from gpde_b200.VirtualObservables import VoPlan  # noqa: F401
        a_key = "a_log" if hp.log_input else "a"
        outs = dict(u=torch.empty((B, w.n), dtype=tdt).pin_memory(), gX=torch.empty((B, w.E), dtype=tdt).pin_memory(),
                    r=torch.empty((B, w.m), dtype=tdt).pin_memory())
        # Per-step inputs: what changes from step to step in the reference's loop -- the coarse-grained model's (logX, F) with
        # the incoming gradient, and the fine-scale output y the residuals are evaluated at.  The conductivity fields of the VO
        # data points are STATE of the ensemble (QuerryPoint.x, VirtualObservables.py:52-59: assembled once per data point;
        # the reference arm accordingly runs with its Gamma_n cached), resident on the device like the weighting functions;
        # ``fields_streamed`` below is the same step with the fields copied from the host every step as well.
        names_step = ["logX", "F", "gbar", "y"] + (["g"] if pinned["g"].dim() == 2 else [])
        names_all = names_step + [a_key]
        names_in = names_all if args.e2e_stream_fields else names_step
        bytes_in = sum(pinned[k].numel() * pinned[k].element_size() for k in names_in)
        bytes_out = sum(t.numel() * t.element_size() for t in outs.values())
        nch = max(1, min(args.e2e_chunks, B // 256))
        bounds = [(c * B // nch, (c + 1) * B // nch) for c in range(nch)]
        copy_stream = torch.cuda.Stream(device=dev)
        g_shared = d["g"] if pinned["g"].dim() == 1 else None
        # device-side landing buffers of the copies, allocated once (the caller's staging memory: a fresh allocation per
        # copy goes through the caching allocator with cross-stream reuse rules and showed up as steps of 6 - 45 ms among
        # steps of 2.6 ms).  Two sets, used alternately: the copies of step k + 1 run while step k computes, and wait only for
        # the kernels of step k - 1 (the last user of their set) -- the host-to-device link never idles between steps
        landing2 = [{k: torch.empty_like(d[k]) for k in names_all} for _ in range(2)]
        evs2 = [[torch.cuda.Event() for _ in bounds] for _ in range(2)]
        set_free = [torch.cuda.Event() for _ in range(2)]
        state = {"n": 0}

        def step_e2e():
            cur = torch.cuda.current_stream(dev)
            which = state["n"] & 1
            landing, evs = landing2[which], evs2[which]
            if state["n"] >= 2:
                copy_stream.wait_event(set_free[which])
            else:
                copy_stream.wait_stream(cur)
            state["n"] += 1
            staged = []
            with torch.cuda.stream(copy_stream):         # all H2D copies are enqueued first, on the copy stream
                for (lo, hi), ev in zip(bounds, evs):
                    dd = {}
                    for k in names_in:
                        dd[k] = landing[k][lo:hi]
                        dd[k].copy_(pinned[k][lo:hi], non_blocking=True)
                    if a_key not in dd:
                        dd[a_key] = d[a_key][lo:hi]          # resident field rows of this chunk's data points
                    ev.record(copy_stream)
                    staged.append((dd, ev))
            for (lo, hi), (dd, ev) in zip(bounds, staged):
                cur.wait_event(ev)
                lX = dd["logX"].detach().requires_grad_(True)
                uu = hp.rom.solve_log(lX, dd["F"])            # public API: autograd.Function forward
                uu.backward(dd["gbar"])                        # ... and its adjoint
                rr = hp.vplan.residual(dd[a_key], dd["y"], dd["g"] if g_shared is None else g_shared, d["V"], a_is_log=hp.log_input)
                # results back to pinned host memory on the compute stream itself (2.7 MB per step against 137 MB in: a third
                # stream with record_stream() on the API's freshly allocated outputs kept the caching allocator growing its
                # pools for tens of steps -- timed blocks of 10, 5, 3.6 ms before settling at 2.6 ms)
                outs["u"][lo:hi].copy_(uu.detach(), non_blocking=True)
                outs["gX"][lo:hi].copy_(lX.grad, non_blocking=True)
                outs["r"][lo:hi].copy_(rr, non_blocking=True)
            set_free[which].record(cur)

        Ke = max(3, min(K, 10))
        for _ in range(8):                 # untimed: the allocator's pools of the per-chunk outputs settle
            step_e2e()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        # five timed blocks of Ke steps; the MEDIAN block is reported and all five are listed: the copies share the host's
        # memory system and PCIe root with whatever else runs on the box
        def timed_blocks(n_blocks):
            blocks = []
            for _ in range(n_blocks):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(Ke):
                    step_e2e()
                e1.record()
                torch.cuda.synchronize()
                b_ms = e0.elapsed_time(e1) / Ke
                if world > 1:
                    tt = torch.tensor([b_ms], dtype=torch.float64, device=dev)
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                    b_ms = float(tt.item())
                blocks.append(b_ms)
            return blocks

        blocks = timed_blocks(5)
        e_ms = sorted(blocks)[len(blocks) // 2]
        e2e = {"value": world * B / (e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(bytes_in),
               "d2h_bytes_per_step": int(bytes_out), "ms_per_step": e_ms, "steps": Ke, "chunks": nch,
               "ms_per_step_blocks": blocks,
               "h2d_gbs_per_gpu": bytes_in / (e_ms * 1e-3) / 1e9, "cpu_affinity": affinity,
               "inputs_copied_per_step": names_in,
               "resident": [] if args.e2e_stream_fields else
               ["conductivity fields of the VO data points (ensemble state, as the reference arm's cached Gamma_n)", "V"],
               "bound": "host-to-device copy (PCIe): compute is %.1f %% of the step" % (100.0 * ms_per_step / e_ms)}
        if not args.e2e_stream_fields:
            # the same step with the fields copied every step too (the round-1 definition of this number)
            names_in = names_all
            bytes_all = sum(pinned[k].numel() * pinned[k].element_size() for k in names_in)
            step_e2e()
            torch.cuda.synchronize()
            blocks_all = timed_blocks(3)
            f_ms = sorted(blocks_all)[1]
            e2e["fields_streamed"] = {"value": world * B / (f_ms * 1e-3), "ms_per_step": f_ms, "ms_per_step_blocks": blocks_all,
                                      "h2d_bytes_per_step": int(bytes_all), "h2d_gbs_per_gpu": bytes_all / (f_ms * 1e-3) / 1e9}

    # ---- the other BASELINE configurations, same run (rank 0 prints them under "configs")
    subs = {}
    if not args.no_sub and args.workload == "cfg2" and args.batch is None:
        Ks = max(3, min(K, 10))
        try:
            subs["cfg4_strong_b131072"] = sub_record(torch, dist, dev, "cfg4", 131072, torch.float64, Ks, rank, world, peak, peak_src, True)
            subs["cfg3_b16384"] = sub_record(torch, dist, dev, "cfg3", 16384, torch.float64, max(3, Ks // 2), rank, world, peak, peak_src, False)
            subs["cfg2_f32"] = sub_record(torch, dist, dev, "cfg2", 4096, torch.float32, Ks, rank, world, peak, peak_src, False)
            subs["cfg5_svi_step"] = svi_record(torch, dist, dev, max(10, Ks), rank, world)
        except Exception as exc:   # noqa: BLE001 -- the headline record must survive a failing secondary record
            subs["error"] = "%s: %s" % (type(exc).__name__, exc)
    if sampler:
        sampler.stop()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cgm_bytes = w.cgm_bytes_per_solve(s) * B
    other = "ms_vo_residual_conductivity_input" if hp.log_input else "ms_vo_residual_log_input"
    line = {
        "metric": METRIC, "value": (total if strong else world * B) / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": workload_config(w),
        "run": {"per_gpu_batch": B, "global_batch": (total if strong else world * B),
                "parallelism": "sample-sharded x%d, no data-path collective" % world,
                "vo_input_in_step": "log-field (exp inside the kernel)" if hp.log_input else "conductivity",
                "sms_left_to_rom_kernels": hp.sm_reserve,
                "ms_per_step_by_sms_left": {str(k): v for k, v in reserve_ms.items()}},
        "components": {
            "cgm_solves_per_s": world * B / ((t_fwd + t_adj) * 1e-3), "vo_evals_per_s": world * B / (t_vo * 1e-3),
            "ms_rom_forward": t_fwd, "ms_rom_adjoint": t_adj, "ms_vo_residual": t_vo, other: t_vo_other,
            "launch_mode": mode + ("" if args.no_overlap else " + ROM/VO on two streams"), "ms_per_step_eager": eager_ms,
            "ms_host_enqueue_per_step": host_enqueue_ms,
            "cgm_hbm_frac": cgm_bytes / ((t_fwd + t_adj) * 1e-3) / 1e9 / peak,
            "vo_hbm_frac_log_input": w.vo_bytes_per_eval(s) * B / ((t_vo if hp.log_input else t_vo_other) * 1e-3) / 1e9 / peak,
            "ms_vo_residual_weights_packed_once": t_vo_pre,     # informational: the step and the roofline use ms_vo_residual
            "ms_vo_residual_T": t_vo_T,
            "vo_residual_T_hbm_frac": None if t_vo_T is None else
            s * (w.P + w.d + w.m) * B / (t_vo_T * 1e-3) / 1e9 / peak,      # a read, q written, s read: w = s V^T stays on the SM
        },
        "roofline": roofline_record(w, B, s, t_vo, hp.path, args.workload, args.dtype, peak, peak_src, t_kernel=t_vo_pre),
        "gpu_launches": hp.launches_per_step() * K,
        "clocks": sampler.summary(t_wall0, t_wall1) if sampler else None,
        "e2e": e2e,
        "configs": subs,
    }
    if world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(w, reference_sample_size(w))
        for _ in range(3):
            ref.step()
        t0, n, acc = time.perf_counter(), 0, 0.0
        while n < 3 or (time.perf_counter() - t0 < 10.0 and n < 50):
            acc += ref.step()
            n += 1
        line["cpu_baseline"] = {
            "value": n * ref.n / acc, "unit": UNIT, "cores": ref.cores, "kind": "port",
            "sample": "%d x (CGM fwd+adjoint via torch autograd + VO r = Gamma y - alpha with cached Gamma, Python loop over data "
                      "points) on the first %d samples of the batch" % (n, ref.n),
            "vo_evals_per_s_assemble_each_step": 1.0 / ref.vo_assemble(min(ref.n, 32)),
            "vo_evals_per_s_vectorised_cached_K": 1.0 / ref.vo_vectorised()}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

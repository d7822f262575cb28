"""bench.py -- asymptotic Wilcoxon rank-sum throughput on B200 at the BASELINE.json shapes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...        # the reference's CPU algorithm (oracle port) on the host cores
    python bench.py --dump-outputs DIR ...      # also write what the last timed step computed, as DIR/<name>.npy

A "step" is one pass of the hot path over the whole workload (all genes x all groups).  `value` is gene x group tests
per second with the input resident in HBM; `e2e` is the same metric through the public `asymptotic_wilcoxon` call with
HOST input (H2D and D2H inside the timed region).  Genes shard across ranks with no data-path collective: `value` is the
weak-scaling figure (every rank ranks its own full-size gene shard), the `strong` block splits ONE workload's genes
across the ranks.  The default line is BASELINE configs[1] (K562-shape dense OVO) and carries an `other_workloads`
block with one short measurement of every other BASELINE workload and of the data variants that do not take the
count-data fast path.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (which may be read-only)

DUMP_MAX_TESTS = 1 << 20         # --dump-outputs: at most this many tests (32 MB with the index), a fixed sample beyond
DUMP_SEED = 0

# name: format, test, data kind, description (BASELINE.json config it belongs to)
WORKLOADS = {
    "dense_ovo": dict(fmt="dense", test="ovo", data="counts", what="configs[1]: K562-shape dense OVO"),
    "dense_ovr": dict(fmt="dense", test="ovr", data="counts", what="K562-shape dense OVR"),
    "csr_ovo": dict(fmt="csr", test="ovo", data="counts", what="configs[2]: K562-shape CSR OVO"),
    "csr_ovr": dict(fmt="csr", test="ovr", data="counts", what="configs[2]: K562-shape CSR OVR"),
    "dense_ovo_continuous": dict(fmt="dense", test="ovo", data="continuous",
                                 what="K562-shape dense OVO, log1p of library-normalised counts (no ties among non-zeros)"),
    "dense_ovr_continuous": dict(fmt="dense", test="ovr", data="continuous", what="K562-shape dense OVR, continuous values"),
    "dense_ovo_unique": dict(fmt="dense", test="ovo", data="unique",
                             what="K562-shape dense OVO, log1p of counts normalised by library sizes spread over a decade "
                                  "(every non-zero value of a gene distinct)"),
    "dense_ovr_unique": dict(fmt="dense", test="ovr", data="unique",
                             what="K562-shape dense OVR, every non-zero value of a gene distinct"),
    "csr_ovo_continuous": dict(fmt="csr", test="ovo", data="continuous", what="K562-shape CSR OVO, continuous values"),
    "dense_ovo_highcount": dict(fmt="dense", test="ovo", data="highcount",
                                what="K562-shape dense OVO, 20 % of the genes (scattered) dense Poisson(30) counts"),
    "dense_ovo_lambda": dict(fmt="dense", test="ovo", data="lambda",
                             what="K562-shape dense OVO, Poisson(lambda_gene ~ U(0.1, 15)) counts, 50 % masked "
                                  "(the reference's own fixture distribution, tests/conftest.py:82-100)"),
    "backed_csc_ovr": dict(fmt="csc", test="ovr", data="counts", clusters=50, backed=True,
                           what="configs[3]: K562 shape as on-disk CSC, OVR with 50 clusters, streamed in 256-gene batches"),
    "c5_shard": dict(fmt="csr", test="ovo", data="counts", cells=2_000_000, genes=2_500, perts=10_000,
                     what="configs[4]: one GPU's gene shard (20000 / 8 genes) of the 2M-cell CSR, 10000 perturbations OVO"),
}
OTHERS_DEFAULT = ["dense_ovr", "csr_ovo", "csr_ovr", "dense_ovo_continuous", "dense_ovr_continuous", "dense_ovo_unique",
                  "dense_ovr_unique", "dense_ovo_highcount", "dense_ovo_lambda", "backed_csc_ovr", "c5_shard"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="dense_ovo", choices=list(WORKLOADS))
    ap.add_argument("--cells", type=int, default=0, help="override the workload's cell count (0 = the BASELINE shape)")
    ap.add_argument("--genes", type=int, default=0)
    ap.add_argument("--perts", type=int, default=0)
    ap.add_argument("--cpu-sample-genes", type=int, default=0, help="genes of the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--others", default="auto",
                    help="'auto' (the default line at N=1 carries every other workload), 'none', or a comma list")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last one as DIR/p_value.npy, statistic.npy, "
                         "fold_change.npy (float64) and test_index.npy (the flat index group * genes + gene of each "
                         f"entry, float64): every test, or a fixed seeded sample of {DUMP_MAX_TESTS} of them (rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 path")
    return a


def shape_of(a, spec):
    cells = a.cells or spec.get("cells", 300_000)
    genes = a.genes or spec.get("genes", 8_000)
    perts = a.perts or spec.get("perts", 2_000)
    return cells, genes, perts


def config_for(name, spec, cells, genes, G):
    """The `config` object -- identical in the b200 and the reference arm (measured quantities live elsewhere)."""
    fmt, test = spec["fmt"], spec["test"]
    return {"workload": f"{name}: {spec['what']}; {cells} cells x {genes} genes x {G} groups per GPU"
                        + (", reference=non-targeting" if test == "ovo" else ""),
            "format": fmt, "test": test, "data_kind": spec["data"], "cells": cells, "genes_per_gpu": genes, "groups": G,
            "l2": "inputs larger than L2 (the matrix is streamed from HBM every step), no explicit flush",
            "sharding": "genes sharded across ranks, no collective in the data path"}


# ---------------------------------------------------------------------------------------------------------
def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows: list = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class Ad:
    def __init__(self, X, labels, n_genes):
        import pandas as pd

        self.X, self.layers = X, {}
        self.obs = pd.DataFrame({"pert": pd.Categorical(labels)})   # AnnData keeps obs columns categorical
        self.var_names = pd.Index([f"g{i:05d}" for i in range(n_genes)])


def make_labels(seed, n_cells, n_perts, spec):
    from illico_b200 import synth

    if "clusters" in spec:
        return synth.cluster_labels(seed, n_cells, spec["clusters"]), None
    rng = np.random.RandomState(seed)
    labels, _ = synth.perturbation_labels(rng, n_cells, n_perts)
    return labels, (synth.CONTROL if spec["test"] == "ovo" else None)


# ---------------------------------------------------------------------------------------------------------
# synthetic data (device side; SURVEY.md 8d)
def gen_dense(kind, seed, cells, genes, dev):
    import torch

    from illico_b200 import synth

    if kind == "lambda":
        g = torch.Generator(device=dev)
        g.manual_seed(seed)
        lam = torch.rand(genes, device=dev, generator=g) * 14.9 + 0.1
        X = torch.empty((cells, genes), dtype=torch.float32, device=dev)
        for r0 in range(0, cells, 16384):
            r1 = min(cells, r0 + 16384)
            x = torch.poisson(lam.expand(r1 - r0, genes), generator=g)
            X[r0:r1] = x * (torch.rand((r1 - r0, genes), device=dev, generator=g) >= 0.5)
        return X
    X = synth.k562_like_torch(seed, cells, genes, device=dev)
    if kind == "highcount":
        g = torch.Generator(device=dev).manual_seed(7)
        gsel = torch.randperm(genes, device=dev, generator=g)[: max(1, int(genes * 0.2))]
        for r0 in range(0, cells, 16384):
            blk = X[r0:r0 + 16384]
            blk[:, gsel] = torch.poisson(torch.full((blk.shape[0], gsel.numel()), 30.0, device=dev))
    elif kind in ("continuous", "unique"):
        g = torch.Generator(device=dev).manual_seed(11)
        for r0 in range(0, cells, 16384):   # in place, chunked: log1p(x / library size * 1e4)
            blk = X[r0:r0 + 16384]
            lib = blk.sum(dim=1, keepdim=True) + 1.0
            if kind == "unique":            # library sizes spread over a decade, as in real data: (almost) every value is unique
                lib = lib * torch.exp(2.3 * torch.rand(lib.shape, device=dev, generator=g))
            blk.copy_(torch.log1p(blk / lib * 1.0e4))
    return X


def gen_csr(kind, seed, cells, genes, dev, chunk_rows=32768):
    """CSR triplet (values f32, col indices i32, indptr i64) built chunk by chunk on the device, so that a 2M-cell
    shard never exists as one dense matrix."""
    import torch

    vals, cols, counts = [], [], []
    for r0 in range(0, cells, chunk_rows):
        r1 = min(cells, r0 + chunk_rows)
        blk = gen_dense(kind, seed + 7919 * (r0 // chunk_rows), r1 - r0, genes, dev)
        nz = blk != 0
        counts.append(nz.sum(dim=1))
        idx = nz.nonzero(as_tuple=False)
        cols.append(idx[:, 1].to(torch.int32))
        vals.append(blk[nz])
        del blk, nz, idx
    counts = torch.cat(counts)
    indptr = torch.zeros(cells + 1, dtype=torch.int64, device=dev)
    indptr[1:] = torch.cumsum(counts, 0)
    return torch.cat(vals).contiguous(), torch.cat(cols).contiguous(), indptr


# ---------------------------------------------------------------------------------------------------------
KERNEL_BYTES_NOTE = ("algorithmic bytes: pass/stage kernels = every input element read once (+ one 24-byte record per test "
                     "for the fused passes); rank kernels = staged non-zeros + counts read once, results written once; "
                     "epilogue = record read + result written")


def kernel_bytes(name, fmt, test, cells, genes, G, nnz, n_ref, S):
    """ALGORITHMIC bytes one step gives kernel `name` (DESIGN.md section 2)."""
    Gt = G - (1 if test == "ovo" else 0)
    dense_in = cells * genes * 4
    sparse_in = nnz * 8 + (cells + 1) * 8
    rank = nnz * 4 + S * genes * 4 + 24 * G * genes
    table = {
        "fused_pass_kernel": (cells - n_ref) * genes * 4 + 24 * Gt * genes,
        "fused_wide_pass_kernel": (cells - n_ref) * genes * 4 + 24 * Gt * genes,
        "fused_csr_pass_kernel": sparse_in + 24 * Gt * genes,
        "fused_epilogue_kernel": 48 * G * genes,
        "stage_dense_tma_kernel": dense_in, "stage_dense_kernel": dense_in,
        "stage_csr_kernel": sparse_in, "stage_csc_kernel": nnz * 8 + (genes + 1) * 8,
        "ovo_kernel": rank, "ovr_kernel": rank, "ovr_table_kernel": rank,
    }
    return table.get(name)


class Workload:
    """One workload on this rank's GPU: data, engine, device-resident and end-to-end measurements."""

    def __init__(self, name, a, dev, rank, world, genes_override=None):
        import torch

        from illico_b200 import _lib
        from illico_b200.engine import DeviceMatrix, Engine, make_flags
        from illico_b200.groups import encode_and_count_groups

        self.name, self.spec, self.dev, self.rank, self.world = name, WORKLOADS[name], dev, rank, world
        spec = self.spec
        self.cells, self.genes, self.perts = shape_of(a, spec)
        if genes_override:
            self.genes = genes_override
        self.fmt, self.test = spec["fmt"], spec["test"]
        self.labels, self.reference = make_labels(a.seed, self.cells, self.perts, spec)
        seed = a.seed + 1000 * rank + 17
        if self.fmt == "dense":
            self.Xdev = gen_dense(spec["data"], seed, self.cells, self.genes, dev)
            self.nnz = int((self.Xdev != 0).sum().item())
            self.M = DeviceMatrix("dense", (self.cells, self.genes), self.Xdev)
        else:
            v, c, p = gen_csr(spec["data"], seed, self.cells, self.genes, dev)
            self.nnz = int(v.numel())
            if self.fmt == "csc":   # transpose once on the device (plumbing: the bench needs a CSC-format input)
                order = torch.argsort(c.to(torch.int64), stable=True)
                rows = torch.repeat_interleave(torch.arange(self.cells, device=dev, dtype=torch.int32), p[1:] - p[:-1])
                cp = torch.zeros(self.genes + 1, dtype=torch.int64, device=dev)
                cp[1:] = torch.cumsum(torch.bincount(c.to(torch.int64), minlength=self.genes), 0)
                v, c, p = v[order].contiguous(), rows[order].contiguous(), cp
                del order, rows
            self.M = DeviceMatrix(self.fmt, (self.cells, self.genes), v, c, p)
        uniq, self.grpc = encode_and_count_groups(self.labels, self.reference)
        self.G = int(self.grpc.counts.size)
        self.n_ref = int(self.grpc.counts[self.grpc.encoded_ref_group]) if self.test == "ovo" else 0
        self.eng = Engine(self.grpc, dev)
        self.flags = make_flags(False, True, True, "two-sided", self.fmt)
        self.results = torch.empty((self.G, self.genes, 3), dtype=torch.float64, device=dev)
        bmax = self.eng.max_batch_genes(self.genes)
        bounds = list(range(0, self.genes, bmax)) + [self.genes]
        self.batches = list(zip(bounds[:-1], bounds[1:]))
        self.n_tests = self.G * self.genes
        self._lib = _lib

    def step(self):
        for lb, ub in self.batches:
            self.eng.run_batch(self.M, lb, ub, self.flags, self.results, lb)

    def barrier(self):
        import torch
        import torch.distributed as dist

        torch.cuda.synchronize(self.dev)
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize(self.dev)

    def timed(self, steps, warmup, min_load_s=0.6, post_load_s=0.3, keep=None):
        """K timed steps (CUDA events, max over ranks) inside a longer stretch of the same load: a step takes a few
        milliseconds, far below nvidia-smi's sampling period, and the SM clock needs tens of milliseconds of load to
        reach its boost state.  ``keep`` (flat test indices on the device): those rows of the last timed step's
        results are copied to ``self.kept`` before the steps after the timed window overwrite them."""
        import torch
        import torch.distributed as dist

        t_load, n_warm = time.perf_counter(), 0
        while n_warm < max(warmup, 3) or time.perf_counter() - t_load < min_load_s:
            self.step()
            n_warm += 1
            if n_warm % 8 == 0:
                torch.cuda.synchronize(self.dev)
        l0 = self._lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(steps):
            self.step()
        e1.record()
        launches = self._lib.launch_count() - l0
        if keep is not None:
            self.kept = self.results.view(-1, 3).index_select(0, keep)
        t_post = time.perf_counter()
        while time.perf_counter() - t_post < post_load_s:
            self.step()
        self.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, int(launches), n_warm

    def kernel_profile(self, reps=3):
        """Per-kernel durations of one step: the library brackets every launch with CUDA events on the launching
        stream (ILLICO_PROFILE=1); median over `reps` steps."""
        import torch

        os.environ["ILLICO_PROFILE"] = "1"
        try:
            self.step()
            torch.cuda.synchronize(self.dev)
            self._lib.profile_report()
            runs = []
            for _ in range(reps):
                self.step()
                torch.cuda.synchronize(self.dev)
                runs.append(self._lib.profile_report())
        finally:
            os.environ.pop("ILLICO_PROFILE", None)
        names = list(runs[-1])
        return {k: (float(np.median([r.get(k, (0.0, 0))[0] for r in runs])), runs[-1][k][1]) for k in names}

    def roofline(self, ms_step, prof):
        peak, peak_src = load_peaks()
        S = self.eng.host_plan.n_segments
        dom = max(prof, key=lambda k: prof[k][0])
        dom_ms, dom_n = prof[dom]
        dom_bytes = kernel_bytes(dom, self.fmt, self.test, self.cells, self.genes, self.G, self.nnz, self.n_ref, S)
        in_bytes = self.cells * self.genes * 4 if self.fmt == "dense" else self.nnz * 8 + (self.cells + 1) * 8
        path_bytes = in_bytes + 24 * self.G * self.genes + 4 * self.cells
        traffic = None
        try:
            if (self.cells, self.genes, self.G) == (300_000, 8_000, 2_001) and len(self.batches) == 1:
                with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
                    traffic = json.load(f)["bytes_per_launch"].get(dom)
        except Exception:
            traffic = None
        achieved = None if not dom_bytes else dom_bytes / (dom_ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": dom, "achieved": None if achieved is None else round(achieved, 1), "peak": peak,
                "unit": "GB/s", "frac": None if achieved is None else round(achieved / peak, 4), "traffic": traffic,
                "traffic_source": "profiles/r2_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full "
                                  "capture of this kernel at this shape" if traffic else None,
                "peak_source": peak_src, "launches_per_step": dom_n, "ms_per_launch": round(dom_ms / max(dom_n, 1), 4),
                "algorithmic_bytes_per_launch": None if not dom_bytes else int(dom_bytes / max(dom_n, 1)),
                "kernels_ms": {k: round(v[0], 4) for k, v in prof.items()},
                "kernel_share_of_step": round(dom_ms / ms_step, 3),
                "path_achieved_GBps": round(path_bytes / (ms_step * 1e-3) / 1e9, 1),
                "path_frac": round(path_bytes / (ms_step * 1e-3) / 1e9 / peak, 4), "note": KERNEL_BYTES_NOTE}

    # ---- end to end through the public API ------------------------------------------------------------------
    def host_input(self, pinned=True):
        """Host copy of the input (pinned unless asked otherwise) + the bytes one call uploads."""
        import torch
        from scipy import sparse

        extra = {}

        def host_buffer(t):
            if pinned:
                try:
                    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                    h.copy_(t)
                    return h
                except RuntimeError:  # not enough lockable memory on this host
                    extra["host_memory"] = "pageable"
            return t.cpu()

        if self.fmt == "dense":
            h = host_buffer(self.Xdev)
            return h.numpy(), h.numel() * 4, extra, h
        M = self.M
        hs = [host_buffer(t) for t in (M.data, M.indices, M.indptr)]
        cls = sparse.csr_matrix if self.fmt == "csr" else sparse.csc_matrix
        Xh = cls((hs[0].numpy(), hs[1].numpy(), hs[2].numpy()), shape=(self.cells, self.genes))
        return Xh, Xh.data.nbytes + Xh.indices.nbytes + Xh.indptr.nbytes, extra, hs

    def e2e(self, Xh, h2d, reps=5, warm=2, frame=False, **kw):
        import torch
        import torch.distributed as dist

        from illico_b200 import asymptotic_wilcoxon

        from illico_b200 import hostio

        ad = Ad(Xh, self.labels, self.genes)
        times = []
        hostio.LAST_UPLOAD.clear()
        for i in range(warm + reps):
            self.barrier()
            t0 = time.perf_counter()
            out = asymptotic_wilcoxon(ad, is_log1p=False, group_keys="pert", reference=self.reference,
                                      return_array=not frame, device=self.dev, **kw)
            torch.cuda.synchronize(self.dev)
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
            del out
        upload = None
        if hostio.LAST_UPLOAD:      # the dense matrix went up packed (hostio._h2d_2d_packed): bytes that crossed the link
            st = dict(hostio.LAST_UPLOAD)
            upload = {"mode": "packed on the host (bit mask + non-zero values), rebuilt in HBM", "host_matrix_bytes": int(h2d),
                      "chunks_packed": int(st.get("packed", 0)), "chunks_sent_as_they_are": int(st.get("raw", 0)),
                      "host_threads": hostio.pack_threads()}
            h2d = st.get("bytes", h2d)
        tt = torch.tensor([float(np.median(times))], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        s = float(tt.item())
        out = {"value": round(self.n_tests * self.world / s, 1), "unit": "tests/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(self.G * self.genes * 24), "s_per_step": round(s, 4),
               "returns": "DataFrame" if frame else "result array (return_array=True)",
               "timing": f"median of {reps} calls after {warm} warm-ups, max over ranks"}
        if upload:
            out["upload"] = upload
        return out

    def backed_e2e(self, reps=3, warm=1):
        """configs[3]: the matrix lives on disk as a CSC triplet (np.memmap behind the `[:, lb:ub]` protocol; h5py /
        anndata are not installed on this image), streamed in 256-gene batches through the pinned ring."""
        import torch

        from illico_b200 import asymptotic_wilcoxon
        from illico_b200.backed import MemmapCSC, save_csc

        d = tempfile.mkdtemp(prefix="illico_c4_")
        try:
            M = self.M
            save_csc(d, M.data.cpu().numpy(), M.indices.cpu().numpy(), M.indptr.cpu().numpy(), (self.cells, self.genes))
            Xb = MemmapCSC(d)
            ad = Ad(Xb, self.labels, self.genes)
            times = []
            for i in range(warm + reps):
                self.barrier()
                t0 = time.perf_counter()
                out = asymptotic_wilcoxon(ad, is_log1p=False, group_keys="pert", reference=self.reference, return_array=True,
                                          device=self.dev, batch_size=256, n_threads=4)
                torch.cuda.synchronize(self.dev)
                if i >= warm:
                    times.append(time.perf_counter() - t0)
                del out
            s = float(np.median(times))
            nbytes = Xb.nbytes
            return {"value": round(self.n_tests / s, 1), "unit": "tests/s", "h2d_bytes_per_step": int(nbytes),
                    "d2h_bytes_per_step": int(self.G * self.genes * 24), "s_per_step": round(s, 4),
                    "source": "np.memmap CSC triplet on local disk (page cache warm after the first call), batch_size=256, "
                              "4 reader threads, pinned ring + copy stream",
                    "disk_read_GBps": round(nbytes / s / 1e9, 2)}
        finally:
            shutil.rmtree(d, ignore_errors=True)

    def close(self):
        import torch

        for k in ("Xdev", "M", "results", "eng"):
            if hasattr(self, k):
                delattr(self, k)
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------
def numba_reference():
    """The unmodified reference (numba kernels), importable from baseline/_ref on the GPU box or /root/reference in the
    build container -- None when it is not there or numba cannot run it."""
    try:
        from oracle import reference_import as R

        if R.reference_root() is None:
            return None
        R.import_reference()
        return R
    except Exception:
        return None


def reference_run(R, Xhost, labels, reference, sample, threads):
    """Times the reference's own `illico.asymptotic_wilcoxon` (its settings: batch_size=256, all threads,
    tests/test_asymptotic_wilcoxon.py:296-303) on `sample` genes.  The numba JIT is excluded by the caller's warm-up."""
    Xs = Xhost[:, :sample]
    t0 = time.perf_counter()
    groups, p, U, fc = R.ref_run(Xs, labels, reference, batch_size=256, n_threads=threads)
    dt = time.perf_counter() - t0
    return len(groups) * sample / dt, dt


def cpu_run(Xhost, labels, reference, sample, threads):
    """Times the oracle port (the reference's algorithm, oracle/wilcoxon_oracle.c) on `sample` genes."""
    import oracle

    P = oracle.Prepared(Xhost, labels, reference)
    bs = max(1, -(-sample // max(threads, 1)))
    bs = min(bs, 256)  # the reference's own benchmark batch size is 256 (tests/test_asymptotic_wilcoxon.py:302)
    t0 = time.perf_counter()
    oracle.run_prepared(P, batch_size=bs, n_threads=threads, gene_lb=0, gene_ub=sample)
    dt = time.perf_counter() - t0
    return P.counts.size * sample / dt, dt


def dump_sample(n_tests):
    """Flat test indices (group * genes + gene) that --dump-outputs writes: all of them, or a fixed seeded sample."""
    if n_tests <= DUMP_MAX_TESTS:
        return np.arange(n_tests, dtype=np.int64)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n_tests, DUMP_MAX_TESTS, replace=False)).astype(np.int64)


def dump_outputs(directory, kept, index):
    """``kept[i]`` = (p_value, statistic, fold_change) of test ``index[i]``: one float64 .npy file per column."""
    os.makedirs(directory, exist_ok=True)
    for k, name in enumerate(("p_value", "statistic", "fold_change")):
        np.save(os.path.join(directory, f"{name}.npy"), np.ascontiguousarray(kept[:, k], dtype=np.float64))
    np.save(os.path.join(directory, "test_index.npy"), index.astype(np.float64))


def cpu_sample_size(a, fmt, genes, threads):
    return a.cpu_sample_genes or min(genes, (32 if fmt == "dense" else 256) * threads)


def short_entry(w: Workload, a, e2e=True):
    """One `other_workloads` entry: a short device-resident measurement + one end-to-end figure."""
    ms, launches, n_warm = w.timed(steps=3, warmup=3, min_load_s=0.15, post_load_s=0.0)
    prof = w.kernel_profile(reps=2)
    roof = w.roofline(ms, prof)
    ent = {"workload": w.name, "what": w.spec["what"], "cells": w.cells, "genes": w.genes, "groups": w.G,
           "nnz_fraction": round(w.nnz / (w.cells * w.genes), 4), "ms_per_step": round(ms, 4),
           "value": round(w.n_tests / (ms * 1e-3), 1), "unit": "tests/s", "steps": 3, "gpu_launches": launches,
           "dominant_kernel": roof["kernel"], "dominant_ms": roof["ms_per_launch"] * roof["launches_per_step"],
           "frac": roof["frac"], "path_frac": roof["path_frac"], "kernels_ms": roof["kernels_ms"]}
    if e2e and not a.no_e2e:
        if w.spec.get("backed"):
            ent["e2e"] = w.backed_e2e()
        else:
            Xh, h2d, extra, keep = w.host_input()
            ent["e2e"] = w.e2e(Xh, h2d, reps=2, warm=1)
            ent["e2e"].update(extra)
            del Xh, keep
    return ent


def main():
    a = parse()
    spec = WORKLOADS[a.workload]
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if a.impl == "reference":
        return reference_arm(a, spec, rank, world)

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        from illico_b200 import hostio

        hostio.bind_thread_to_device_node(local)   # pinned host buffers are then first-touched next to this rank's GPU
        dist.init_process_group("nccl", device_id=dev)

    # ---- headline workload: weak scaling, every rank owns a full-size gene shard
    w = Workload(a.workload, a, dev, rank, world)
    dump_index = dump_sample(w.n_tests) if a.dump_outputs and rank == 0 else None
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_step, launches, n_warm = w.timed(a.steps, a.warmup, keep=None if dump_index is None else
                                        torch.from_numpy(dump_index).to(dev))
    clocks = sampler.stop() if rank == 0 else None
    if dump_index is not None:
        dump_outputs(a.dump_outputs, w.kept.cpu().numpy(), dump_index)
        del w.kept
    if clocks is not None:
        clocks["window"] = (f"{n_warm} warm-up steps (>= 0.6 s of the same load) + the {a.steps} timed steps + 0.3 s of the "
                            "same load")
    prof = w.kernel_profile()
    roofline = w.roofline(ms_step, prof)

    e2e, e2e_pageable, extra = None, None, {}
    if not a.no_e2e:
        if spec.get("backed"):
            e2e = w.backed_e2e()
        else:
            Xh, h2d, extra, keep = w.host_input()
            e2e = w.e2e(Xh, h2d)
            e2e["host_memory"] = extra.pop("host_memory", "pinned")
            if world == 1 and w.fmt == "dense":
                # what a user's `adata.X` is: a pageable ndarray in, the DataFrame out
                Xp = np.array(Xh, copy=True)
                del Xh, keep
                e2e_pageable = w.e2e(Xp, h2d, reps=3, warm=1, frame=True)
                e2e_pageable["host_memory"] = "pageable ndarray (np.array copy), chunked pinned staging inside the call"
                del Xp
            else:
                del Xh, keep

    # ---- strong scaling: ONE workload's genes split across the ranks (rank r ranks genes/world genes)
    strong = None
    if world > 1 and not spec.get("backed"):
        w.close()
        gs = w.genes // world
        ws = Workload(a.workload, a, dev, rank, world, genes_override=gs)
        ms_s, _, _ = ws.timed(a.steps, a.warmup, min_load_s=0.3, post_load_s=0.0)
        strong = {"workload_genes": gs * world, "genes_per_gpu": gs, "ms_per_step": round(ms_s, 4),
                  "value": round(ws.G * gs * world / (ms_s * 1e-3), 1), "unit": "tests/s", "scaling": "strong",
                  "what": f"the {gs * world}-gene workload split into {world} contiguous gene shards, one per GPU; "
                          "time = max over ranks"}
        if not a.no_e2e:
            Xh, h2d, ex, keep = ws.host_input()
            es = ws.e2e(Xh, h2d, reps=3, warm=1)
            strong["e2e"] = {"value": es["value"], "unit": "tests/s", "s_per_step": es["s_per_step"],
                             "h2d_bytes_per_step": es["h2d_bytes_per_step"] * world,
                             "d2h_bytes_per_step": es["d2h_bytes_per_step"] * world,
                             "aggregate_h2d_GBps": round(es["h2d_bytes_per_step"] * world / es["s_per_step"] / 1e9, 1)}
            del Xh, keep
        ws.close()

    # ---- CPU baseline beside it (rank 0, N == 1 only): the oracle port on a bounded sample
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        import oracle
        from scipy import sparse

        threads = oracle.max_threads()
        sample = cpu_sample_size(a, w.fmt, w.genes, threads)
        if w.fmt == "dense":
            Xs = w.Xdev[:, :sample].contiguous().cpu().numpy()
        else:
            Xs = gen_dense(spec["data"], a.seed + 17, w.cells, sample, dev).cpu().numpy()
            Xs = sparse.csr_matrix(Xs) if w.fmt == "csr" else sparse.csc_matrix(Xs)
        R = numba_reference()
        kind = "reference" if R is not None else "port"
        if R is not None:
            try:   # numba JIT warm-up on a tiny problem of the same format / test (excluded, like the reference's own benchmark)
                tiny_l = list(w.labels[:3000])
                if w.reference is not None and w.reference not in tiny_l:
                    tiny_l[0] = w.reference
                R.ref_run(Xs[:3000, :8], tiny_l, w.reference, batch_size=8, n_threads=threads)
            except Exception as e:
                sys.stderr.write(f"reference not runnable here ({type(e).__name__}: {e}); timing the C port instead\n")
                R, kind = None, "port"
        if R is not None:
            v, dt = reference_run(R, Xs, w.labels, w.reference, sample, threads)
        else:
            cpu_run(Xs[:, : min(sample, 4)], w.labels, w.reference, min(sample, 4), threads)  # page cache / thread pool
            v, dt = cpu_run(Xs, w.labels, w.reference, sample, threads)
        cpu = {"value": round(v, 1), "unit": "tests/s", "cores": threads, "kind": kind,
               "what": "the unmodified reference (numba kernels, batch_size=256, joblib threads) imported from baseline/_ref"
                       if kind == "reference" else "the C port of the reference's algorithm (oracle/wilcoxon_oracle.c, pthreads)",
               "sample": f"first {sample} of {w.genes} genes, all {w.G} groups, {dt:.2f} s wall", "seconds": round(dt, 3),
               "calibration": "profiles/r2_port_vs_numba.json: the C port against the unmodified numba reference on the same "
                              "sample and cores (build container)"}
        del Xs

    line = None
    if rank == 0:
        line = {
            "metric": "gene_x_group_tests_per_s", "value": round(w.n_tests * world / (ms_step * 1e-3), 1), "unit": "tests/s",
            "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "warmup_steps_run": n_warm,
            "ms_per_step": round(ms_step, 4), "wall_s_per_step": round(ms_step * 1e-3, 6),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 keys / int64 ranks / f64 epilogue",
            "data": "synthetic", "impl": "b200",
            "config": config_for(a.workload, spec, w.cells, w.genes, w.G),
            "measured": {"nnz_fraction": round(w.nnz / (w.cells * w.genes), 4), "gene_batches": len(w.batches)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_pageable_dataframe": e2e_pageable, "strong": strong,
            "gpu_launches": int(launches), "clocks": clocks,
        }
        line.update(extra)
    if world == 1 or strong is None:
        w.close()

    # ---- every other BASELINE workload / data variant, one short measurement each (N == 1 only)
    others = []
    names = [] if a.others == "none" else (OTHERS_DEFAULT if a.others == "auto" else [s for s in a.others.split(",") if s])
    if a.others == "auto" and (world > 1 or a.workload != "dense_ovo" or a.cells or a.genes or a.perts):
        names = []
    for nm in names:
        t0 = time.perf_counter()
        try:
            wo = Workload(nm, a, dev, rank, world)
            ent = short_entry(wo, a)
            wo.close()
        except Exception as e:  # one failing variant must not cost the headline line
            ent = {"workload": nm, "error": f"{type(e).__name__}: {e}"[:300]}
        ent["bench_seconds"] = round(time.perf_counter() - t0, 1)
        others.append(ent)
    if rank == 0:
        line["other_workloads"] = others or None
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def reference_arm(a, spec, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port: the reference is Python + numba and does
    not travel to the GPU box) on all host cores, each step a bounded sample of the same workload."""
    if rank != 0:
        return 0
    import oracle
    from scipy import sparse

    fmt, test = spec["fmt"], spec["test"]
    cells, genes, perts = shape_of(a, spec)
    threads = oracle.max_threads()
    sample = cpu_sample_size(a, fmt, genes, threads)
    labels, reference = make_labels(a.seed, cells, perts, spec)
    Xs = None
    try:
        import torch

        if torch.cuda.is_available():
            Xs = gen_dense(spec["data"], a.seed + 17, cells, sample, torch.device("cuda", 0)).cpu().numpy()
    except Exception:
        Xs = None
    if Xs is None:
        from illico_b200 import synth

        Xs, _ = synth.k562_like(a.seed, cells, sample, perts, continuous=spec["data"] == "continuous")
    if fmt != "dense":
        Xs = sparse.csr_matrix(Xs) if fmt == "csr" else sparse.csc_matrix(Xs)
    G = len(set(labels))
    R = numba_reference()
    kind = "reference" if R is not None else "port"
    if R is not None:
        try:   # JIT warm-up on a tiny problem of the same format / test (excluded, as the reference's own benchmark does)
            tiny_l = list(labels[:3000])
            if reference is not None and reference not in tiny_l:
                tiny_l[0] = reference
            R.ref_run(Xs[:3000, :8], tiny_l, reference, batch_size=8, n_threads=threads)
        except Exception as e:
            sys.stderr.write(f"reference not runnable here ({type(e).__name__}: {e}); timing the C port instead\n")
            R, kind = None, "port"
    vals, secs = [], []
    for i in range(a.warmup + a.steps):
        v, dt = reference_run(R, Xs, labels, reference, sample, threads) if R is not None else cpu_run(Xs, labels, reference, sample, threads)
        if i >= a.warmup:
            vals.append(v); secs.append(dt)
    v = float(np.mean(vals))
    what = ("the unmodified reference (illico.asymptotic_wilcoxon, numba kernels, batch_size=256, joblib threads) imported from "
            "baseline/_ref" if kind == "reference" else "the C port of the reference's algorithm (oracle/wilcoxon_oracle.c, pthreads)")
    line = {"metric": "gene_x_group_tests_per_s", "value": round(v, 1), "unit": "tests/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(float(np.mean(secs)) * 1e3, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 (CPU)", "data": "synthetic",
            "impl": "reference", "config": config_for(a.workload, spec, cells, genes, G),
            "cpu_baseline": {"value": round(v, 1), "unit": "tests/s", "cores": threads, "kind": kind, "what": what,
                             "sample": f"each step = the first {sample} of {genes} genes, all {G} groups "
                                       "(tests/s is per test, so the sample size does not bias it)",
                             "calibration": "profiles/r2_port_vs_numba.json"},
            "e2e": {"value": round(v, 1), "unit": "tests/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())

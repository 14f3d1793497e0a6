#!/usr/bin/env python
"""bench.py -- tiles/sec of the HoVer-Net tile hot path (infer_step + post_proc.process per patch).

    python bench.py --gpus N --steps K --warmup W                 # this repo (libhvn, sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...       # the reference path on the same box
    python bench.py --workload fast64|tile4k|wsi40k ...           # the other BASELINE.json configs

Default workload = BASELINE.json configs[2], the configuration the metric is quoted on (SURVEY.md 8d, unit U1):
a step = one batch of 256 synthetic 270x270x3 uint8 patches, `original` mode, nr_types=5, each patch through the
CNN (-> 80x80x4 float map) and the instance post-processing (-> inst_map + instance table).  `fast64` =
configs[1] (64 patches of 256x256, `fast` mode cannot ingest 270x270), `tile4k` = configs[3] (one 4096x4096 image
through the tile driver, patch grid sharded over the ranks), `wsi40k` = configs[4] (synthetic slide through the WSI
driver).  Weights: seeded synthetic checkpoint (hover_net_b200.synth).  One process per GPU; patch workloads give
every rank its own batch (weak scaling) and rank 0 receives the packed instance tables over NCCL.

`value`   : device-timed (CUDA events on the library's stream), inputs resident in HBM, gather included at N > 1.
`e2e`     : same metric through the host-buffer C-ABI call (`hvn_forward_postproc`): pinned host uint8 in,
            inst_map + instance table out, copies (and at N > 1 the gather) inside the timed region.
`roofline`: dominant kernel class = the tcgen05 convolution; algorithmic 2*MACs of the reference graph per launch /
            its measured launch time (per-launch CUDA events, kernels serialised) vs MEASURED_PEAKS.json.
`roofline_postproc`: the post-processing half of the metric: algorithmic bytes (C*4 B read + 4 B written per pixel)
            / device time vs the measured HBM copy bandwidth, on the CNN's own output maps and on nuclei-like maps.
`--impl reference` (default arm = what north_star names): the unmodified reference graph restated in torch
            (oracle/hovernet_torch.py, pinned bit-for-bit against the reference) on PyTorch-CUDA with stock settings,
            overlapped with the reference-faithful CPU post-processing in a pool of os.cpu_count() processes
            (infer/tile.py:232-234).  `--ref-forward cpu` times the all-CPU arm instead.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as build() left it (it may be read-only)

CLOCK_Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
           "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
           "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

WORKLOADS = {
    "orig256": {"mode": "original", "nr_types": 5, "batch": 256, "config": 2},
    "fast64": {"mode": "fast", "nr_types": 6, "batch": 64, "config": 1},
    "tile4k": {"mode": "fast", "nr_types": 6, "batch": 125, "config": 3},
    "wsi40k": {"mode": "fast", "nr_types": 6, "batch": 128, "config": 4},
}


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks/throttle reasons for one GPU while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        try:
            p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + CLOCK_Q,
                                  "--format=csv,noheader,nounits", "-lms", "200"],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        try:
            while not self.stop_flag.is_set():
                line = p.stdout.readline()
                if not line:
                    break
                self.rows.append([c.strip() for c in line.split(",")])
        finally:
            p.terminate()
            p.wait()    # reaped here, so no exited nvidia-smi outlives the benchmark

    def summary(self):
        sm, mx, reasons, pw = [], 0, set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                pw.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx or None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def measured_traffic(kernel_class, mode):
    """dram__bytes_read+write per launch of the dominant kernel from the committed ncu capture of this workload's
    mode (profiles/*_traffic*.json, newest first); null when no capture of that mode is committed."""
    try:
        import glob
        for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*traffic*.json")), reverse=True):
            t = json.load(open(path))
            if t.get("mode", "fast") != mode:
                continue
            # the tcgen05 convolution class = k_conv_tc + its A-resident (k_conv_ar) and row-stacked (k_conv_rs) variants
            names = ("k_conv_tc", "k_conv_ar", "k_conv_rs") if kernel_class == "conv_tc" else ("k_conv_ref",)
            ks = [t["kernels"][n] for n in names if n in t["kernels"]]
            k = {"dram_bytes": sum(x["dram_bytes"] for x in ks), "launches": sum(x["launches"] for x in ks)}
            return {"dram_bytes_per_launch": k["dram_bytes"] / k["launches"], "launches": k["launches"],
                    "batch": t["batch"], "source": "profiles/" + os.path.basename(path) + " (" + t["command"] + ")"}
    except Exception:
        pass
    return None


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def np_from_addr(addr, shape, dtype):
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    buf = (ctypes.c_char * n).from_address(addr)
    return np.frombuffer(buf, dtype=dtype).reshape(shape)


def make_batch(B, S, seed):
    """B distinct synthetic patches: up to 64 generated blob images (synth.make_patches) and their dihedral variants."""
    from hover_net_b200 import synth
    base = synth.make_patches(min(B, 64), S, seed=seed)
    outs = [base]
    k = 1
    while sum(o.shape[0] for o in outs) < B:
        v = np.rot90(base, k % 4, axes=(1, 2))
        if k >= 4:
            v = v[:, :, ::-1]
        outs.append(np.ascontiguousarray(v))
        k += 1
    return np.ascontiguousarray(np.concatenate(outs)[:B])


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays, sampled):
    """Writes {name: array} as out_dir/<name>.npy, float32 arrays as float32 and everything else as float64 (exact for
    the integer outputs).  When they would come to more than DUMP_LIMIT bytes, the arrays named in `sampled` (those
    whose leading axis is a patch or an image row) keep the same share of that axis, drawn by a fixed seed, so equal
    shapes give equal positions and two runs stay comparable; the other arrays are written whole."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v.astype(np.float32 if v.dtype in (np.float16, np.float32) else np.float64) for k, v in arrays.items()}
    whole = sum(a.nbytes for k, a in arrays.items() if k not in sampled)
    part = sum(arrays[k].nbytes for k in sampled)
    share = min(1.0, (DUMP_LIMIT * 15 // 16 - whole) / max(1, part))
    assert share > 0, "outputs beyond the %d MB dump limit" % (DUMP_LIMIT >> 20)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if name in sampled and share < 1.0:
            keep = max(1, int(a.shape[0] * share))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def info_arrays(info):
    """The tile driver's inst_info_dict as arrays, in instance-id order; contour r = contour[offsets[r]:offsets[r+1]]."""
    ids = sorted(info)
    cnt = [np.asarray(info[i]["contour"]).reshape(-1, 2) for i in ids]
    out = {"inst_id": np.array(ids, np.int64),
           "inst_bbox": np.array([info[i]["bbox"] for i in ids], np.int64).reshape(-1, 4),
           "inst_centroid": np.array([info[i]["centroid"] for i in ids], np.float64).reshape(-1, 2),
           "inst_contour": np.concatenate(cnt) if cnt else np.zeros((0, 2), np.int32),
           "inst_contour_offsets": np.cumsum([0] + [c.shape[0] for c in cnt])}
    if ids and info[ids[0]]["type"] is not None:
        out["inst_type"] = np.array([info[i]["type"] for i in ids], np.int64)
        out["inst_type_prob"] = np.array([info[i]["type_prob"] for i in ids], np.float64)
    return out


def workload_config(args, world, note=None):
    out = 164 if args.mode == "fast" else 80
    cfg = {"workload": "BASELINE configs[%d]%s: batch=%d synthetic %s-mode patches %dx%dx3 uint8, nr_types=%s, forward + "
                       "instance post-processing per patch (output %dx%d)" % (
                           args.config, "" if args.stock else " (modified by flags)", args.batch, args.mode, args.patch,
                           args.patch, args.nr_types, out, out),
           "name": args.workload, "mode": args.mode, "nr_types": args.nr_types, "batch_per_gpu": args.batch,
           "patch": args.patch,
           "parallelism": "tiles sharded per rank (dp%d), end-of-batch NCCL gather of the packed instance tables" % world,
           "l2": "per-step activations (%.0f GB at %.2f GB/patch) exceed the 126 MB L2; a 256 MB buffer is also written "
                 "between timed steps" % (0.5 * args.batch, 0.5)}
    if note:
        cfg["note"] = note
    return cfg


# ------------------------------------------------------------------------------------------------
# reference arm
def _pp_worker(args):
    from oracle import postproc_oracle as P
    return P.process_table(args[0], args[1])


_FWD = {}


def _cpu_fwd_init(mode, nt, threads):
    """Pool initialiser of the all-CPU arm: import torch and build the checkpoint once per process (untimed)."""
    import torch
    from hover_net_b200 import synth
    from oracle import hovernet_torch as O
    torch.set_num_threads(threads)
    _FWD.update(O=O, sd=O.to_torch_state_dict(synth.make_state_dict(mode, nt, seed=0)), mode=mode, nt=nt)


def _cpu_fwd_worker(x):
    """One process of the all-CPU arm: torch fp32 forward of its share of the patches."""
    return _FWD["O"].infer_step(x, _FWD["sd"], _FWD["mode"], _FWD["nt"])


class CpuArm(object):
    """All-CPU reference-style path: torch forward in `procs` processes x `threads` threads (torch's CPU convolution
    stops scaling near 32 threads: measured 8 -> 1.56, 32 -> 1.27, 64 -> 2.30, 128 -> 16.5 s/patch on the 128-core
    box), then the pooled post-processing (one process per core, infer/tile.py:232-234)."""

    def __init__(self, mode, nt, patch, threads):
        import multiprocessing as mp
        self.cores = os.cpu_count() or 1
        self.threads = max(1, min(threads, self.cores))
        self.procs = max(1, self.cores // self.threads)
        self.mode, self.nt, self.patch = mode, nt, patch
        ctx = mp.get_context("spawn")
        self.fwd = ctx.Pool(self.procs, initializer=_cpu_fwd_init, initargs=(mode, nt, self.threads))
        self.pp = ctx.Pool(self.cores)
        self.pp.map(_pp_worker, [(np.zeros((16, 16, 3 if nt is None else 4), np.float32), nt)] * self.cores)
        self.fwd.map(_cpu_fwd_worker, [make_batch(1, patch, seed=5)] * self.procs)   # warm-up: imports, first convs

    def run(self, n):
        """n patches -> (tiles/s, forward s, post-proc s, single-core post-proc ms/tile)."""
        x = make_batch(n, self.patch, seed=1)
        shares = [s for s in np.array_split(x, self.procs) if s.shape[0]]
        t0 = time.perf_counter()
        pred = np.concatenate(self.fwd.map(_cpu_fwd_worker, shares))
        t1 = time.perf_counter()
        self.pp.map(_pp_worker, [(pred[i], self.nt) for i in range(n)])
        t2 = time.perf_counter()
        from oracle import postproc_oracle as P
        k = min(n, 8)
        t3 = time.perf_counter()
        for i in range(k):
            P.process_table(pred[i], self.nt)
        pp1 = (time.perf_counter() - t3) / k
        return n / (t2 - t0), t1 - t0, t2 - t1, pp1 * 1e3

    def close(self):
        self.fwd.close()
        self.pp.close()


def run_reference(args):
    """Reference arm (rank 0 only).  Default = the north-star arm: reference graph on PyTorch-CUDA (fp32, stock
    cuDNN settings incl. TF32 convolutions) in sub-batches, each sub-batch's maps handed to a pool of
    os.cpu_count() post-processing workers while the next sub-batch runs (infer/tile.py:232-234, 353-363)."""
    rank, world, local = dist_env()
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    use_cuda_arm = args.ref_forward == "cuda"
    from oracle import postproc_oracle as P
    P.lib()                         # libhvo.so as build() left it: no make run inside the tree
    pool = None
    if use_cuda_arm:
        pool = mp.get_context("fork").Pool(cores)  # forked before CUDA is initialised in this process
        pool.map(_pp_worker, [(np.zeros((16, 16, 3 if args.nr_types is None else 4), np.float32), args.nr_types)] * cores)
    import torch
    from hover_net_b200 import synth
    from oracle import hovernet_torch as O
    mode, nt = args.mode, args.nr_types
    use_cuda = args.ref_forward == "cuda" and torch.cuda.is_available()
    if not use_cuda:
        arm = CpuArm(mode, nt, args.patch, args.cpu_threads)
        n = args.ref_sample or max(2 * arm.procs, 8)
        for _ in range(max(1, args.warmup // 3)):
            arm.run(max(arm.procs, 2))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            arm.run(n)
        dt = (time.perf_counter() - t0) / args.steps
        arm.close()
        val = n / dt
        sample = ("%d patches/step (bounded sample of the %d-patch batch): torch fp32 CPU forward in %d processes x %d "
                  "threads, then oracle post-proc in a %d-process pool" % (n, args.batch, arm.procs, arm.threads, cores))
        same, h2d, d2h = False, 0, 0
    else:
        dev = torch.device("cuda", local)
        sd = {k: v.to(dev) for k, v in O.to_torch_state_dict(synth.make_state_dict(mode, nt, seed=0)).items()}
        B = args.batch
        x = make_batch(B, args.patch, seed=1)
        sub = min(B, args.ref_sub_batch)

        def step():
            pending = []
            for b0 in range(0, B, sub):
                pred = O.infer_step(x[b0:b0 + sub], sd, mode, nt, device=dev)      # H2D, forward, D2H (run_desc.py:171-197)
                pending.append(pool.map_async(_pp_worker, [(pred[i], nt) for i in range(pred.shape[0])],
                                              chunksize=max(1, pred.shape[0] // cores)))
            return [r.get() for r in pending]

        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = step()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / args.steps
        val = B / dt
        # forward alone / post-proc alone, for the record (untimed region)
        torch.cuda.synchronize(); t1 = time.perf_counter()
        preds = [O.infer_step(x[b0:b0 + sub], sd, mode, nt, device=dev) for b0 in range(0, B, sub)]
        torch.cuda.synchronize(); t2 = time.perf_counter()
        pred = np.concatenate(preds)
        pool.map(_pp_worker, [(pred[i], nt) for i in range(B)], chunksize=max(1, B // cores)); t3 = time.perf_counter()
        oh = pred.shape[1]
        sample = ("whole %d-patch batch per step in sub-batches of %d: torch fp32 forward on cuda (stock cuDNN settings, "
                  "allow_tf32=%s) overlapped with oracle post-proc in a %d-process pool; alone: forward %.3f s, pooled "
                  "post-proc %.3f s" % (B, sub, torch.backends.cudnn.allow_tf32, cores, t2 - t1, t3 - t2))
        same, h2d, d2h = True, int(x.nbytes), int(B * oh * oh * pred.shape[-1] * 4)
        n = B
    if pool is not None:
        pool.close()
    line = {
        "impl": "reference", "metric": "tiles/sec", "value": val, "unit": "tiles/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" + (" (cuDNN TF32 convolutions)" if use_cuda else ""),
        "data": "synthetic", "config": workload_config(args, 1, note=sample), "same_config": same,
        "arm": "north-star: reference graph on PyTorch-CUDA + pooled CPU post-proc" if use_cuda else "all-CPU",
        "cpu_baseline": {"value": val, "unit": "tiles/s", "cores": cores, "host_cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "tiles/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
    }
    print(json.dumps(line))


def cpu_baseline(args):
    """All-CPU arm (oracle port of the reference path on every host core), bounded sample -- reported, not the target."""
    from oracle import postproc_oracle as P
    P.lib()                         # libhvo.so as build() left it: no make run inside the tree
    arm = CpuArm(args.mode, args.nr_types, args.patch, args.cpu_threads)
    try:
        n = args.cpu_sample or max(2 * arm.procs, 8)
        v, tf, tp, pp1 = arm.run(n)
    finally:
        arm.close()
    return {"value": v, "unit": "tiles/s", "cores": arm.cores, "host_cores": arm.cores, "kind": "port",
            "sample": "%d patches: torch fp32 CPU forward in %d processes x %d threads %.2f s + oracle post-proc in a "
                      "%d-process pool %.3f s; single-core post-proc %.2f ms/tile" % (
                          n, arm.procs, arm.threads, tf, arm.cores, tp, pp1),
            "forward_s_per_tile": tf / n, "postproc_ms_per_tile_1core": pp1,
            "postproc_ms_per_tile_allcores": pp1 / arm.cores}


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    rank, world, local = dist_env()
    import torch
    from hover_net_b200 import _lib, synth
    from hover_net_b200.dist import PackedGather
    from hover_net_b200.models.hovernet.net_desc import create_model

    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    mode, nt, B, S = args.mode, args.nr_types, args.batch, args.patch
    net = create_model(mode=mode, input_ch=3, nr_types=nt, device=local)
    net.load_state_dict(synth.make_state_dict(mode, nt, seed=0), strict=True)
    ctx = net.ctx
    if args.chunk:
        ctx.set_option("chunk", args.chunk)
    if args.conv_path is not None:
        ctx.set_option("conv_path", args.conv_path)
    for kv in args.opt or []:
        k, v = kv.split("=")
        ctx.set_option(k, int(v))
    oh, ow, oc = ctx.out_shape(S, S)
    max_rows = max(16, oh * ow // 64)
    cap_rows = B * max(8, max_rows // 4)          # packed gather payload (rows); a fuller batch fails loudly below
    x = make_batch(B, S, seed=1 + rank)
    in_bytes = x.nbytes

    # device-resident buffers are torch tensors (so NCCL can gather them); libhvn gets raw pointers
    d_img = torch.from_numpy(x).to(dev)
    d_inst = torch.empty((B, oh, ow), dtype=torch.int32, device=dev)
    d_tab = torch.zeros((B, max_rows, 10), dtype=torch.int64, device=dev)
    d_nr = torch.zeros((B,), dtype=torch.int32, device=dev)
    # the network's map is written here instead of the library's scratch arena (same kernels, same writes) so that
    # --dump-outputs can return it as well
    d_pred = torch.empty((B, oh, ow, oc), dtype=torch.float32, device=dev) if args.dump_outputs else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    pg = PackedGather(ctx, B, max_rows, cap_rows, world, dev)
    torch.cuda.synchronize()

    def step_resident():
        ctx.forward_postproc_dev(d_img.data_ptr(), B, S, S, None if d_pred is None else d_pred.data_ptr(),
                                 d_inst.data_ptr(), d_tab.data_ptr(), max_rows, d_nr.data_ptr())
        return pg.launch(d_tab, d_nr)     # pack on the library stream + async all_gather (overlaps the next step)

    def barrier():
        pg.wait()
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_resident()
    barrier()
    launches0 = ctx.counter("kernel_launches")
    sampler = ClockSampler(local)
    sampler.start()
    # ---- timed: exactly K steps between two barriers.  Device time = CUDA events on the library's stream around each
    # step (the L2 flush between steps is outside the events); the last gather is joined inside the last event pair.
    step_ms = []
    t_wall = time.perf_counter()
    for i in range(args.steps):
        with torch.cuda.stream(pg.stream):     # L2 flush on the library's stream, outside the event pair; no host or
            flush.fill_(1)                     # device-wide sync between steps, so gather i really overlaps step i+1
        ctx.timer_start()
        k = step_resident()
        if i == args.steps - 1 or not args.overlap_gather:
            pg.wait()                      # library stream waits for the collective(s) still in flight
        step_ms.append(ctx.timer_stop())
    barrier()
    wall = time.perf_counter() - t_wall
    launches = ctx.counter("kernel_launches") - launches0
    total_ms = float(np.sum(step_ms))
    got = pg.rows(k)
    assert len(got) == world and all(int(o[-1]) <= cap_rows for o, _ in got), "packed gather payload overflow"
    rows_gathered = int(sum(p.shape[0] for _, p in got))
    # the last timed step's results on rank 0 as the forward + post-processing call returns them: per patch the
    # prediction map, the instance map and the instance table padded to max_rows (its first inst_count[b] rows are
    # the instances), so every shape is fixed by the arguments; the passes below reuse these buffers
    last = {"pred_map": d_pred.cpu().numpy(), "inst_map": d_inst.cpu().numpy(), "inst_table": d_tab.cpu().numpy(),
            "inst_count": d_nr.cpu().numpy()} if args.dump_outputs and rank == 0 else None

    # ---- e2e through the host-buffer entry point (pinned host buffers), gather included
    h_in = ctx.malloc_host(in_bytes)
    h_inst = ctx.malloc_host(B * oh * ow * 4)
    h_tab = ctx.malloc_host(B * max_rows * 10 * 8)
    h_nr = ctx.malloc_host(B * 4)
    np_from_addr(h_in, x.shape, np.uint8)[...] = x
    L = _lib.lib()
    h_tab_t = torch.from_numpy(np_from_addr(h_tab, (B, max_rows, 10), np.int64))
    h_nr_t = torch.from_numpy(np_from_addr(h_nr, (B,), np.int32))

    def step_e2e():
        _lib.check(L.hvn_forward_postproc(ctx._h, ctypes.c_void_p(h_in), B, S, S, None, ctypes.c_void_p(h_inst),
                                          ctypes.c_void_p(h_tab), max_rows, ctypes.c_void_p(h_nr)))
        if world > 1:   # the host-buffer caller's gather: tables back to the device, packed, all_gather, joined
            d_tab.copy_(h_tab_t, non_blocking=True)
            d_nr.copy_(h_nr_t, non_blocking=True)
            torch.cuda.synchronize()
            pg.wait(pg.launch(d_tab, d_nr))
            ctx.sync()

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    e2e_ms = []
    for _ in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step_e2e()
        torch.cuda.synchronize()
        e2e_ms.append((time.perf_counter() - t0) * 1e3)
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    e2e_total = float(np.sum(e2e_ms))
    inst_e2e = np_from_addr(h_inst, (B, oh, ow), np.int32).copy()
    nr_e2e = np_from_addr(h_nr, (B,), np.int32).copy()
    same = bool(np.array_equal(d_inst.cpu().numpy(), inst_e2e)) and bool(np.array_equal(d_nr.cpu().numpy(), nr_e2e))

    # ---- per-kernel-class profile pass (untimed): per-launch CUDA events, kernels serialised
    ctx.set_option("branch_streams", 0)  # isolated kernels: per-launch event times must not overlap
    ctx.set_option("profile", 2)
    for _ in range(2):
        ctx.forward_postproc_dev(d_img.data_ptr(), B, S, S, None, d_inst.data_ptr(), d_tab.data_ptr(), max_rows, d_nr.data_ptr())
    ctx.sync()
    prof = {}
    for cls in ("conv_tc", "conv_ref", "conv0", "bnrelu", "head"):
        prof[cls] = {"ms": ctx.stage_ms(cls), "launches": ctx.counter("launches:" + cls),
                     "gflop": ctx.counter("flops:" + cls) / 1e9}
    prof["postproc"] = {"ms": ctx.stage_ms("postproc"), "launches": ctx.counter("pp_launches")}
    prof["cnn_total_ms"] = ctx.stage_ms("cnn")
    flops_step = float(ctx.counter("last_flops"))
    pp_cnn_ms = ctx.stage_ms("postproc")
    # post-processing alone on nuclei-like maps (synth_pred_map): the per-instance work of post_proc.py:120-181
    # depends on the map content, and the synthetic-weight CNN output is not nuclei-like
    nm = min(B, 64)
    maps = np.stack([synth.synth_pred_map(oh, ow, nt, s) for s in range(nm)])
    maps = np.ascontiguousarray(np.concatenate([maps] * ((B + nm - 1) // nm))[:B])
    d_maps = torch.from_numpy(maps).to(dev)
    ctx.set_option("profile", 1)
    for _ in range(3):
        ctx.postproc_dev(d_maps.data_ptr(), B, oh, ow, oc, nt, d_inst.data_ptr(), d_tab.data_ptr(), max_rows, d_nr.data_ptr())
    ctx.sync()
    pp_nuc_ms = ctx.stage_ms("postproc")
    nuc_inst = int(d_nr.sum().item())
    ctx.set_option("profile", 0)
    ctx.set_option("branch_streams", 1)

    # max over ranks
    t = torch.tensor([total_ms, e2e_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_total = float(t[0]), float(t[1])

    if rank == 0:
        pk, pk_kind = peaks()
        dom = "conv_tc" if prof["conv_tc"]["launches"] > 0 else "conv_ref"
        d = prof[dom]
        ach = (d["gflop"] / 1e3) / (d["ms"] / 1e3) if d["ms"] > 0 else 0.0  # TFLOP/s
        peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
        value = world * B * args.steps / (total_ms / 1e3)
        e2e_v = world * B * args.steps / (e2e_total / 1e3)
        pp_bytes = B * oh * ow * (oc * 4 + 4)
        hbm = pk["hbm_gbs"]
        line = {
            "metric": "tiles/sec", "value": value, "unit": "tiles/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16x3-split (fp32-equivalent products, fp32 accumulate); "
                                                              "post-proc int32/f64",
            "data": "synthetic", "config": workload_config(args, world),
            "e2e": {"value": e2e_v, "unit": "tiles/s", "h2d_bytes_per_step": int(in_bytes),
                    "d2h_bytes_per_step": int(B * oh * ow * 4 + B * max_rows * 80 + B * 4),
                    "ms_per_step": e2e_total / args.steps, "matches_resident_path": same,
                    "gather_in_timed_region": world > 1},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                         "frac": ach / peak if peak else None, "peak_source": pk_kind + " bf16_tflops_sustained",
                         "algorithmic_gflop_per_launch": d["gflop"] / max(1, d["launches"]),
                         "avg_launch_ms": d["ms"] / max(1, d["launches"]), "launches_per_step": d["launches"],
                         "traffic": measured_traffic(dom, mode),
                         "note": "algorithmic 2*MACs of the reference graph; every product is formed three times in "
                                 "fp16 (hi*hi+hi*lo+lo*hi, issued as two or three MMA instructions per K-step), so frac <= 1/3 "
                                 "by construction"},
            "roofline_postproc": {"bound": "hbm", "unit": "GB/s", "peak": hbm, "peak_source": pk_kind + " hbm_gbs",
                                  "algorithmic_bytes_per_step": pp_bytes,
                                  "on_cnn_output": {"ms_per_step": pp_cnn_ms, "ms_per_tile": pp_cnn_ms / B,
                                                    "achieved": pp_bytes / 1e9 / (pp_cnn_ms / 1e3) if pp_cnn_ms > 0 else None},
                                  "on_nuclei_maps": {"ms_per_step": pp_nuc_ms, "ms_per_tile": pp_nuc_ms / B, "instances": nuc_inst,
                                                     "achieved": pp_bytes / 1e9 / (pp_nuc_ms / 1e3) if pp_nuc_ms > 0 else None},
                                  "achieved": pp_bytes / 1e9 / (pp_nuc_ms / 1e3) if pp_nuc_ms > 0 else None,
                                  "frac": pp_bytes / 1e9 / (pp_nuc_ms / 1e3) / hbm if pp_nuc_ms > 0 else None,
                                  "note": "latency-bound, not bandwidth-bound: the sequential per-blob priority flood "
                                          "dominates (DESIGN.md 4.2)"},
            "kernel_classes": prof,
            "algorithmic_gflop_per_tile": flops_step / B / 1e9,
            "postproc_ms_per_tile": pp_cnn_ms / B,
            "gather": {"rows": rows_gathered, "payload_bytes_per_rank": int((cap_rows * 10 + B + 1) * 8),
                       "overlapped_with_next_step": bool(args.overlap_gather)},
            "wall_s_timed_region": wall,
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(args)
        if last is not None:
            dump_outputs(args.dump_outputs, last, sampled=tuple(last))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    for p in (h_in, h_inst, h_tab, h_nr):
        ctx.free_host(p)
    ctx.close()


# ------------------------------------------------------------------------------------------------
def synth_image(size, seed=90):
    """size x size RGB image assembled from synthetic 256x256 blob patches."""
    from hover_net_b200 import synth
    base = synth.make_patches(8, 256, seed=seed)
    rng = np.random.default_rng(seed)
    n = (size + 255) // 256
    rows = [np.concatenate([base[rng.integers(0, 8)] for _ in range(n)], 1) for _ in range(n)]
    return np.ascontiguousarray(np.concatenate(rows, 0)[:size, :size])


def run_tile(args):
    """configs[3]: one size x size image through the tile driver (infer/tile.py), patch grid sharded over the ranks,
    ONE whole-map post-processing on rank 0.  Strong scaling: the image is fixed as N grows."""
    rank, world, local = dist_env()
    import torch
    from hover_net_b200 import synth
    from hover_net_b200.infer.tile import InferManager
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    mode, nt = args.mode, args.nr_types
    img = synth_image(args.size)
    mgr = InferManager(method={"model_args": {"nr_types": nt, "mode": mode, "device": local},
                               "model_path": synth.make_state_dict(mode, nt, seed=0)}, type_info_path=None)
    win = 256 if mode == "fast" else 270
    mgr.patch_input_shape, mgr.patch_output_shape, mgr.batch_size = win, (164 if mode == "fast" else 80), args.batch
    rows, cols = mgr.net.ctx.tile_grid(args.size, args.size, win)
    sampler = ClockSampler(local)
    res = None
    for _ in range(args.warmup):
        res = mgr.infer_image(img)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    times = []
    for _ in range(args.steps):
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        res = mgr.infer_image(img)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    t = torch.tensor([float(np.sum(times))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total = float(t[0])
    if rank == 0:
        pred, inst, info = res
        npatch = rows * cols
        import hashlib
        line = {"metric": "tiles/sec", "value": npatch * args.steps / total, "unit": "tiles/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / args.steps * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16x3-split; post-proc int32/f64",
                "data": "synthetic",
                "config": {"workload": "BASELINE configs[3]: one %dx%d synthetic image through the tile driver, %s mode, "
                                       "%dx%d = %d patches sharded over %d rank(s), maps reduced to rank 0, one whole-map "
                                       "post-processing" % (args.size, args.size, mode, rows, cols, npatch, world),
                           "name": "tile4k", "mode": mode, "nr_types": nt, "patches": npatch, "batch": args.batch},
                "e2e": {"value": npatch * args.steps / total, "unit": "tiles/s", "h2d_bytes_per_step": int(img.nbytes),
                        "d2h_bytes_per_step": int(inst.nbytes + (pred.nbytes if pred is not None else 0)),
                        "note": "host image in, host maps + instance dict out (wall clock, max over ranks)"},
                "gpu_launches": int(mgr.net.ctx.counter("kernel_launches")), "clocks": sampler.summary(),
                "instances": len(info), "inst_map_sha1": hashlib.sha1(np.ascontiguousarray(inst).tobytes()).hexdigest()}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dict(pred_map=pred, inst_map=inst, **info_arrays(info)),
                         sampled=("pred_map", "inst_map"))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    mgr.net.ctx.close()


def run_wsi(args):
    """configs[4]: a size x size synthetic slide (.npy, all-tissue mask) through the WSI driver (infer/wsi.py):
    patches of every chunk and tiles of every merge phase sharded over the ranks, JSON written by rank 0."""
    rank, world, local = dist_env()
    import hashlib
    import shutil
    import tempfile
    import cv2
    import torch
    from hover_net_b200 import synth
    from hover_net_b200.infer.wsi import InferManager
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    mode, nt = args.mode, args.nr_types
    # one slide file for all ranks (a 40000^2 slide is 4.8 GB): rank 0 writes it, the others wait at the barrier
    work = os.path.join(tempfile.gettempdir(), "hvn_wsi_bench_%s" % os.environ.get("MASTER_PORT", "0"))
    if rank == 0:
        shutil.rmtree(work, ignore_errors=True)
        os.makedirs(work + "/in"); os.makedirs(work + "/msk"); os.makedirs(work + "/out")
        np.save(work + "/in/slide.npy", synth_image(args.size))
        cv2.imwrite(work + "/msk/slide.png", np.full((max(8, args.size // 32),) * 2, 255, np.uint8))
    if world > 1:
        dist.barrier()
    win, out = (256, 164) if mode == "fast" else (270, 80)
    mgr = InferManager(method={"model_args": {"nr_types": nt, "mode": mode, "device": local},
                               "model_path": synth.make_state_dict(mode, nt, seed=0)}, type_info_path=None)
    run_args = {"batch_size": args.batch, "nr_inference_workers": 0, "nr_post_proc_workers": 0, "patch_input_shape": win,
                "patch_output_shape": out, "input_dir": work + "/in", "output_dir": work + "/out", "input_mask_dir": work + "/msk",
                "proc_mag": 40, "cache_path": work + "/cache%d" % rank, "chunk_shape": 10000, "tile_shape": 2048, "ambiguous_size": 128,
                "save_thumb": False, "save_mask": False}
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    t0 = time.perf_counter()
    mgr.process_wsi_list(run_args)
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total = float(t[0])
    if rank == 0:
        js = open(work + "/out/slide.json", "rb").read()
        n_step = (args.size - (win - out)) // out + 1
        line = {"metric": "tiles/sec", "value": n_step * n_step / total, "unit": "tiles/s", "n_gpus": world, "steps": 1,
                "warmup": 0, "ms_per_step": total * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f16x3-split; post-proc int32/f64", "data": "synthetic",
                "config": {"workload": "BASELINE configs[4]: %dx%d synthetic slide through the WSI driver, %s mode, %d patches, "
                                       "chunks of 10000, 2048 tiles + boundary + cross phases, %d rank(s), JSON on rank 0" % (
                                           args.size, args.size, mode, n_step * n_step, world),
                           "name": "wsi40k", "mode": mode, "nr_types": nt, "patches": n_step * n_step},
                "e2e": {"value": n_step * n_step / total, "unit": "tiles/s", "h2d_bytes_per_step": int(args.size) ** 2 * 3,
                        "d2h_bytes_per_step": len(js), "note": "slide file in, JSON out (wall clock, max over ranks)"},
                "gpu_launches": int(mgr.net.ctx.counter("kernel_launches")), "clocks": sampler.summary(),
                "instances": len(json.loads(js)["nuc"]), "json_sha1": hashlib.sha1(js).hexdigest()}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    mgr.net.ctx.close()
    if rank == 0:
        shutil.rmtree(work, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="orig256", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default=None, choices=["fast", "original"])
    ap.add_argument("--nr-types", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--size", type=int, default=None, help="tile4k / wsi40k: image side in pixels")
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--conv-path", type=int, default=None)
    ap.add_argument("--opt", action="append", help="libhvn option key=value (development)")
    ap.add_argument("--no-overlap-gather", dest="overlap_gather", action="store_false")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--ref-sample", type=int, default=0)
    ap.add_argument("--ref-sub-batch", type=int, default=64)
    ap.add_argument("--cpu-threads", type=int, default=32)
    ap.add_argument("--ref-forward", default="cuda", choices=["cpu", "cuda"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32/float64, <= 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "wsi40k"):
        ap.error("--dump-outputs covers this project's patch and tile4k workloads")
    w = WORKLOADS[args.workload]
    args.stock = args.mode is None and args.nr_types is None and args.batch is None and args.size is None
    args.config = w["config"]
    args.mode = args.mode or w["mode"]
    if args.nr_types is None:
        args.nr_types = w["nr_types"] if args.mode == w["mode"] else {"fast": 6, "original": 5}[args.mode]
    if args.nr_types == 0:
        args.nr_types = None
    args.batch = args.batch or w["batch"]
    args.patch = 256 if args.mode == "fast" else 270
    args.size = args.size or (4096 if args.workload == "tile4k" else 40000)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "tile4k":
        run_tile(args)
    elif args.workload == "wsi40k":
        run_wsi(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

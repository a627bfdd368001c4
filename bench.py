#!/usr/bin/env python
"""bench.py -- throughput of the clip.cpp encode path on N B200s of one node, one JSON line per run.

    python bench.py --gpus 1 --steps 5 --warmup 3                    # headline: image-embeddings/sec, ViT-L/14 q4_0, b=512 per GPU
    python bench.py --config cfg2|cfg3|cfg4|cfg5                     # the other BASELINE.json configs (see CONFIGS)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...      # one rank per GPU
    python bench.py --impl reference ...                             # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                           # also write what the last timed step computed, DIR/<name>.npy

torch.distributed.run is only the LAUNCHER: the rank processes never import torch.  The library builds its own NCCL communicator
from RANK / WORLD_SIZE / LOCAL_RANK / MASTER_PORT (clip_b200_dist_init: ncclCommInitRank, unique id through a rendezvous file), and
the one collective of the path -- an in-place all-gather of the final embeddings, K5 writing into the rank's slot -- is enqueued by
the C++ library on its launch stream (clip_b200_*_all).

A step = one pass of the hot path over one batch of synthetic input per GPU (weak scaling; `--scaling strong` splits a fixed global
batch instead).
  value : whole-job units/s with the inputs already resident in HBM
  e2e   : the same metric through the reference-facing C call with HOST buffers (H2D of the inputs, D2H of the embeddings timed)
Timing: CUDA events on the library's launch stream (clip_b200_mark) around the K steps -- the NCCL all-gather is on that stream too
-- bracketed by a barrier (all-reduce + device sync) on both sides, max over ranks (clip_b200_dist_max_f64).  Inputs per step exceed
the 126 MB L2 for the image configs (308 MB / 154 MB of pixels); cfg4's token ids are tiny, its activations (> 1 GB per pass) are not.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "clip.cpp_b200"))

SEED = 1234
# algorithmic FLOPs per unit (SURVEY.md section 8d): whole tower, and its attention part (everything else but ~0.01 % runs in K1)
FLOPS = {
    ("vit-l14", "image"): (162_025_537_536, 24 * 270_536_704),
    ("vit-b32", "image"): (8_817_623_040, 12 * 7_680_000),
    ("vit-l14", "text"): (13_299_683_328, 12 * 18_213_888),
    ("vit-b32", "text"): (5_959_540_736, 12 * 12_142_592),
}
CONFIGS = {
    # name: kind, geometry, file type, units per GPU, what BASELINE.json calls it
    "headline": dict(kind="image", geom="vit-l14", ftype="q4_0", batch=512,
                     workload="ViT-L/14 q4_0 image encode, b=512 per GPU, 224x224x3 synthetic (BASELINE.json metric config)"),
    "cfg2": dict(kind="image", geom="vit-b32", ftype="q4_0", batch=256,
                 workload="ViT-B/32 q4_0 image encode, b=256 per GPU, 224x224x3 synthetic (BASELINE.json configs[1])"),
    "cfg3": dict(kind="image", geom="vit-l14", ftype="q8_0", batch=512,
                 workload="ViT-L/14 q8_0 image encode, b=512 per GPU, 224x224x3 synthetic (BASELINE.json configs[2])"),
    "cfg4": dict(kind="text", geom="vit-l14", ftype="q4_0", batch=2048, tokens=77,
                 workload="text encoder (ViT-L/14 text tower, h=768, 12 layers) q4_0, 2048 x 77-token sequences per GPU (BASELINE.json configs[3])"),
    "cfg5": dict(kind="zsl", geom="vit-l14", ftype="q4_0", batch=4096, labels=1000, tokens=77,
                 workload="ViT-L/14 q4_0 zero-shot: 4096 images x 1000 labels, images AND labels sharded over the GPUs, label embeddings "
                          "all-gathered, device logits + softmax + top-5 (BASELINE.json configs[4]); global sizes fixed"),
}
FTYPE_ID = {"f32": 0, "f16": 1, "q4_0": 2, "q4_1": 3, "q5_0": 6, "q5_1": 7, "q8_0": 8}

# dram__bytes_read.sum + dram__bytes_write.sum per launch of gemm_dq_kernel from the committed `ncu --set full` captures
# (profiles/): mean over the four layer-GEMM shapes of the configuration's micro-batch; None = not captured for this config.
NCU_GEMM_TRAFFIC = {"headline": (694_300_000, 742_900_000, "profiles/r02_gemm.md")}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def model_for(cfg, rank, quantize_with):
    """(geometry, SEED, ftype) -> file; rank 0 writes it, the others wait.  quantize_with(src, dst, itype) -> bool."""
    import synth_gguf as sg
    geom, ftype = cfg["geom"], cfg["ftype"]
    path = sg.model_path(geom, SEED, ftype)
    if os.path.exists(path):
        return path
    if rank != 0:
        t0 = time.time()
        while not os.path.exists(path):
            time.sleep(1.0)
            if time.time() - t0 > 1800:
                raise RuntimeError("timed out waiting for rank 0 to write " + path)
        return path
    f16 = sg.model_path(geom, SEED, "f16")
    if not os.path.exists(f16):
        t0 = time.time()
        sg.write_model(f16 + ".tmp", sg.GEOMETRIES[geom], SEED, 1)
        os.replace(f16 + ".tmp", f16)
        log("bench: wrote %s in %.1fs" % (f16, time.time() - t0))
    if ftype != "f16":
        t0 = time.time()
        assert quantize_with(f16, path + ".tmp", FTYPE_ID[ftype]), "quantize failed"
        os.replace(path + ".tmp", path)
        log("bench: quantized to %s in %.1fs" % (path, time.time() - t0))
    return path


def quantize_with_reference(src, dst, itype):
    """clip_model_quantize of the UNMODIFIED reference (oracle/_ref), in a subprocess: the reference arm never maps libclip_b200.so"""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import binding as bd, ref_run; "
            "sys.exit(0 if bd.ClipLib(ref_run.REF_LIB).quantize(%r, %r, %d) else 1)"
            % (os.path.join(ROOT, "clip.cpp_b200"), os.path.join(ROOT, "oracle"), src, dst, itype))
    return subprocess.run([sys.executable, "-c", code], stdout=subprocess.DEVNULL).returncode == 0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.th.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 8 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """arrays: name -> what the last timed step handed its caller.  Written as float32 / float64 .npy, at most DUMP_BYTES in all: a larger
    array is cut to a fixed, seeded sample of its rows (the same rows for the same arguments, so two builds compare row for row)."""
    os.makedirs(path, exist_ok=True)
    budget = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a, np.float32 if a.dtype == np.float32 else np.float64)
        if a.nbytes > budget:
            keep = budget // (a.nbytes // len(a))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j.get("bf16_tflops_sustained", j.get("bf16_tflops", 1590.0))), "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
    return 1400.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)"


# ---- CPU side: the reference's own implementation on a bounded sample ---------------------------------------------------
def cpu_reference_sample(cfg, model, n_units, threads):
    """oracle/_ref (the unmodified reference) on n_units of the config's workload; falls back to the oracle port."""
    import synth_gguf as sg
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_run
    kind = "image" if cfg["kind"] in ("image", "zsl") else "text"
    if kind == "image":
        imgs, seqs = sg.synth_images(n_units, 224, 4321), None
    else:
        imgs, seqs = None, list(sg.synth_tokens(n_units, cfg["tokens"], 4321))
    unit = "img/s" if kind == "image" else "seq/s"
    if ref_run.available():
        ref_lib, ref_isa = ref_run.timing_lib()
        r = ref_run.run_reference(model, images=imgs, token_seqs=seqs, n_threads=threads, lib_path=ref_lib)
        secs = float(r["img_s"] if kind == "image" else r["txt_s"])
        what = "single-image clip_image_encode calls (the reference cannot batch ViT-L/14)" if kind == "image" else "clip_text_encode calls (the reference has no text batch)"
        return {"value": n_units / secs, "unit": unit, "cores": int(r["threads"]), "kind": "reference",
                "sample": "%d %s; %s" % (n_units, what, ref_isa)}, (r["img"] if kind == "image" else r["txt"])
    import oracle as orc
    om = orc.OracleModel(model, n_threads=threads)
    t0 = time.perf_counter()
    out = np.stack([om.encode_image(imgs[i]) for i in range(n_units)]) if kind == "image" else np.stack([om.encode_text(s) for s in seqs])
    dt = time.perf_counter() - t0
    return {"value": n_units / dt, "unit": unit, "cores": threads or os.cpu_count(), "kind": "port",
            "sample": "%d units through the CPU oracle restatement (oracle/_ref absent)" % n_units}, out


def pick_threads(cfg, model):
    """ggml's spin-wait pool stops scaling long before 128 threads: take the fastest of a few candidates on a tiny sample."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_run
    n = os.cpu_count() or 8
    if not ref_run.available():
        return n
    best, best_v = None, -1.0
    for t in sorted({min(n, c) for c in (8, 16, 32, 64)}):
        b, _ = cpu_reference_sample(cfg, model, 2, t)
        log("bench(reference): %d threads -> %.2f %s" % (t, b["value"], b["unit"]))
        if b["value"] > best_v:
            best, best_v = t, b["value"]
    return best


def run_reference_arm(args, cfg, rank):
    if rank != 0:
        return
    model = model_for(cfg, 0, quantize_with_reference)
    threads = pick_threads(cfg, model)
    per_step = 4 if cfg["kind"] != "text" else 8
    for _ in range(max(args.warmup - 1, 0)):       # the calibration passes above already warmed the page cache
        cpu_reference_sample(cfg, model, 1, threads)
    vals, base = [], None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        base, emb = cpu_reference_sample(cfg, model, per_step, threads)
        vals.append(base["value"])
    wall = time.perf_counter() - t0
    v = float(np.mean(vals))
    base["value"] = v
    unit = base["unit"]
    metric = "image-embeddings/sec" if cfg["kind"] != "text" else "text-embeddings/sec"
    out = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1000.0 * per_step / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "%s x q8 int8 dot, fp32 accumulate (ggml CPU)" % cfg["ftype"], "data": "synthetic",
           "config": {"workload": cfg["workload"], "name": args.config, "global_batch": cfg["batch"] * args.gpus,
                      "step_sample": "%d units per step" % per_step},
           "cpu_baseline": base, "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": wall}
    print(json.dumps(out), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {("text" if cfg["kind"] == "text" else "image") + "_embeddings": emb})


# ---- GPU side -----------------------------------------------------------------------------------------------------------
class Bench:
    def __init__(self, args, cfg, rank, world, local):
        import binding as bd
        self.bd, self.args, self.cfg, self.rank, self.world = bd, args, cfg, rank, world
        os.environ["CLIP_B200_DEVICE"] = str(local)
        os.environ["CLIP_B200_PROFILE"] = "1"
        self.lib = bd.ClipLib(bd.PRODUCT_LIB)      # raises if the CUDA library is not built: there is no fallback path
        self.L = self.lib.lib
        self.model = model_for(cfg, rank, self.lib.quantize)
        self.ctx = self.lib.load(self.model, 0)
        if world > 1:
            assert self.L.clip_b200_dist_init(self.ctx, rank, world, None), self.lib.last_error()
        assert "torch" not in sys.modules
        self.d = self.lib.vision_hparams(self.ctx).projection_dim

    # barrier (NCCL all-reduce inside the library) + device synchronize
    def sync_all(self):
        assert self.L.clip_b200_dist_barrier(self.ctx), self.lib.last_error()

    def timed(self, fn, steps):
        L, ctx = self.L, self.ctx
        self.sync_all()
        assert L.clip_b200_mark(ctx, 0)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        assert L.clip_b200_mark(ctx, 1)
        ms_dev = L.clip_b200_mark_elapsed_ms(ctx, 0, 1)
        self.sync_all()
        ms_wall = (time.perf_counter() - t0) * 1e3
        v = (C.c_double * 2)(ms_dev, ms_wall)
        assert L.clip_b200_dist_max_f64(ctx, v, 2)                  # max over ranks
        return v[0] / steps, v[1] / steps

    def fetch(self, d_ptr, shape):
        """float32 device buffer -> host array (after timed(), which synchronises)"""
        a = np.empty(shape, np.float32)
        assert self.L.clip_b200_memcpy_d2h(self.ctx, a.ctypes.data, d_ptr, a.nbytes), self.lib.last_error()
        return a

    def drop_profile(self):
        for k in range(4):
            self.L.clip_b200_kernel_ms(self.ctx, k, None)

    def kinds(self, steps):
        kcount, out = C.c_uint64(0), {}
        for k, nm in enumerate(("gemm", "attention", "layernorm", "other")):
            ms = self.L.clip_b200_kernel_ms(self.ctx, k, C.byref(kcount))
            out[nm] = {"ms_per_step": ms / steps, "launches_per_step": kcount.value / steps}
        return out

    def pinned(self, shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = self.L.clip_b200_host_malloc(n)
        assert p
        ct = {np.dtype(np.float32): C.c_float, np.dtype(np.int32): C.c_int32}[np.dtype(dtype)]
        return p, np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), shape=tuple(shape))


def bench_image(b, units):
    """image configs: value = device-resident pixels, e2e = clip_image_batch_encode(_all) from pinned host buffers, plus a pageable leg"""
    import synth_gguf as sg
    L, ctx, lib, d, world, rank, args = b.L, b.ctx, b.lib, b.d, b.world, b.rank, b.args
    B, per = units, 224 * 224 * 3
    h_pix, pix = b.pinned((B, 224, 224, 3), np.float32)
    pix[:] = sg.synth_images(B, 224, 1000 + rank)
    h_out, out_host = b.pinned((B * world, d), np.float32)
    batch, keep = lib.make_image_batch(pix)
    d_pix = L.clip_b200_device_malloc(ctx, B * per * 4)
    d_all = L.clip_b200_device_malloc(ctx, B * world * d * 4)
    assert d_pix and d_all and L.clip_b200_memcpy_h2d(ctx, d_pix, h_pix, B * per * 4)
    fp = C.POINTER(C.c_float)

    def step_device():     # K5 writes this rank's slot of d_all; the library enqueues the in-place NCCL all-gather (N > 1)
        assert L.clip_b200_image_encode_device_all(ctx, d_pix, B, d_all, True), lib.last_error()

    def step_e2e():        # pinned host pixels in, ALL ranks' embeddings out on the host
        assert L.clip_b200_image_batch_encode_all(ctx, 4, C.byref(batch), C.cast(h_out, fp), True), lib.last_error()

    for _ in range(args.warmup):
        step_device()
    b.drop_profile()
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        sampler.start()
    l0 = L.clip_b200_kernel_launches(ctx)
    ms_step, ms_wall = b.timed(step_device, args.steps)
    launches = (L.clip_b200_kernel_launches(ctx) - l0) + (args.steps if world > 1 else 0)
    clocks = sampler.stop() if rank == 0 else None
    kinds = b.kinds(args.steps)
    outputs = {"image_embeddings": b.fetch(d_all, (B * world, d))} if args.dump_outputs else None
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = b.timed(step_e2e, max(2, args.steps // 2))
    b.drop_profile()
    res = {"outputs": outputs, "ms_step": ms_step, "ms_wall": ms_wall, "launches": launches, "clocks": clocks, "kinds": kinds,
           "e2e": {"value": B * world / (ms_e2e / 1e3), "unit": "img/s", "h2d_bytes_per_step": B * per * 4, "d2h_bytes_per_step": B * world * d * 4,
                   "ms_per_step": ms_e2e, "call": "clip_b200_image_batch_encode_all" if world > 1 else "clip_image_batch_encode",
                   "host_buffers": "pinned (cudaMallocHost)"}}
    if not args.quick:
        # pageable leg: every image its own malloc'ed buffer, exactly what clip_image_preprocess hands a reference caller
        imgs_pg = [np.array(pix[i]) for i in range(B)]
        arr = (b.bd.clip_image_f32 * B)()
        for i, a in enumerate(imgs_pg):
            arr[i] = b.bd.clip_image_f32(224, 224, a.ctypes.data_as(fp), per)
        batch_pg = b.bd.clip_image_f32_batch(arr, B)

        def step_pg():
            assert L.clip_b200_image_batch_encode_all(ctx, 4, C.byref(batch_pg), C.cast(h_out, fp), True), lib.last_error()

        for _ in range(2):
            step_pg()
        ms_pg, _ = b.timed(step_pg, max(2, args.steps // 2))
        res["e2e_pageable"] = {"value": B * world / (ms_pg / 1e3), "unit": "img/s", "ms_per_step": ms_pg,
                               "host_buffers": "pageable: %d separate 602 KB new[]-style buffers, gathered into the library's pinned arena by host threads" % B}
        b.drop_profile()
        if world == 1:
            # N1 leg (SURVEY 8f): raw u8 images in, resize + crop + normalise on the GPU, then the same encode
            SRC = 256
            rng8 = np.random.default_rng(7)
            pool = [rng8.integers(0, 256, (SRC, SRC, 3), dtype=np.uint8) for _ in range(16)]
            items = (b.bd.clip_image_u8 * B)()
            for i in range(B):
                a = pool[i % len(pool)]
                items[i] = b.bd.clip_image_u8(SRC, SRC, a.ctypes.data_as(C.POINTER(C.c_uint8)), a.size)
            batch8 = b.bd.clip_image_u8_batch(items, B)

            def step_u8():
                assert L.clip_b200_image_batch_encode_u8(ctx, C.byref(batch8), C.cast(h_out, fp), True), lib.last_error()

            step_u8()
            _, ms_u8 = b.timed(step_u8, 2)
            res["e2e_u8"] = {"value": B / (ms_u8 / 1e3), "unit": "img/s", "ms_per_step": ms_u8, "h2d_bytes_per_step": B * SRC * SRC * 3,
                             "source": "%dx%d u8 RGB per image; resize/crop/normalise on the GPU, bit-identical to clip_image_preprocess; wall "
                                       "clock around clip_b200_image_batch_encode_u8 (includes the host copy into pinned staging)" % (SRC, SRC)}
            b.drop_profile()
    return res


def bench_text(b, units):
    """cfg4: value = device-resident token ids, e2e = clip_text_batch_encode(_all) with HOST clip_tokens arrays"""
    import synth_gguf as sg
    L, ctx, lib, d, world, rank, args = b.L, b.ctx, b.lib, b.d, b.world, b.rank, b.args
    TB, TL = units, b.cfg["tokens"]
    ids = sg.synth_tokens(TB, TL, 2000 + rank)
    d_ids = L.clip_b200_device_malloc(ctx, ids.nbytes)
    d_all = L.clip_b200_device_malloc(ctx, TB * world * d * 4)
    assert d_ids and d_all and L.clip_b200_memcpy_h2d(ctx, d_ids, ids.ctypes.data, ids.nbytes)
    h_out, out_host = b.pinned((TB * world, d), np.float32)
    seqs = [np.ascontiguousarray(ids[i]) for i in range(TB)]
    arr, keep = lib.make_token_array(seqs)
    fp = C.POINTER(C.c_float)

    def step_device():
        assert L.clip_b200_text_encode_device_all(ctx, d_ids, None, TB, TL, d_all, True), lib.last_error()

    def step_e2e():
        assert L.clip_b200_text_batch_encode_all(ctx, 4, arr, TB, C.cast(h_out, fp), True), lib.last_error()

    for _ in range(args.warmup):
        step_device()
    b.drop_profile()
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        sampler.start()
    l0 = L.clip_b200_kernel_launches(ctx)
    ms_step, ms_wall = b.timed(step_device, args.steps)
    launches = (L.clip_b200_kernel_launches(ctx) - l0) + (args.steps if world > 1 else 0)
    clocks = sampler.stop() if rank == 0 else None
    kinds = b.kinds(args.steps)
    outputs = {"text_embeddings": b.fetch(d_all, (TB * world, d))} if args.dump_outputs else None
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = b.timed(step_e2e, max(2, args.steps // 2))
    b.drop_profile()
    T_pad = (TL + 7) // 8 * 8 if TL < 77 else 77
    return {"outputs": outputs, "ms_step": ms_step, "ms_wall": ms_wall, "launches": launches, "clocks": clocks, "kinds": kinds,
            "e2e": {"value": TB * world / (ms_e2e / 1e3), "unit": "seq/s", "h2d_bytes_per_step": TB * T_pad * 4 + TB * 4,
                    "d2h_bytes_per_step": TB * world * d * 4, "ms_per_step": ms_e2e,
                    "call": "clip_b200_text_batch_encode_all" if world > 1 else "clip_text_batch_encode", "host_buffers": "pageable clip_tokens arrays"}}


def bench_zsl(b, n_img_global, n_lab_global):
    """cfg5: value = composition of the device-resident entry points, e2e = ONE clip_b200_zero_shot_images call per rank from host buffers"""
    import synth_gguf as sg
    L, ctx, lib, d, world, rank, args = b.L, b.ctx, b.lib, b.d, b.world, b.rank, b.args
    assert n_img_global % world == 0 and n_lab_global % world == 0, "cfg5 needs a GPU count that divides 4096 and 1000"
    B, NL, TL, K = n_img_global // world, n_lab_global // world, b.cfg["tokens"], 5
    per = 224 * 224 * 3
    h_pix, pix = b.pinned((B, 224, 224, 3), np.float32)
    pix[:] = sg.synth_images(B, 224, 1000 + rank)
    batch, keep = lib.make_image_batch(pix)
    ids = sg.synth_tokens(NL, TL, 3000 + rank)
    seqs = [np.ascontiguousarray(ids[i]) for i in range(NL)]
    arr, keep2 = lib.make_token_array(seqs)
    d_pix = L.clip_b200_device_malloc(ctx, B * per * 4)
    d_img = L.clip_b200_device_malloc(ctx, B * d * 4)
    d_ids = L.clip_b200_device_malloc(ctx, ids.nbytes)
    d_txt = L.clip_b200_device_malloc(ctx, NL * world * d * 4)
    assert d_pix and d_img and d_ids and d_txt
    assert L.clip_b200_memcpy_h2d(ctx, d_pix, h_pix, B * per * 4) and L.clip_b200_memcpy_h2d(ctx, d_ids, ids.ctypes.data, ids.nbytes)
    scores, idx = np.empty((B, K), np.float32), np.empty((B, K), np.int32)
    fp, ipp = C.POINTER(C.c_float), C.POINTER(C.c_int)

    def step_device():
        assert L.clip_b200_image_encode_device(ctx, d_pix, B, d_img, True), lib.last_error()
        assert L.clip_b200_text_encode_device_all(ctx, d_ids, None, NL, TL, d_txt, True), lib.last_error()      # the one all-gather
        assert L.clip_b200_zero_shot_batch(ctx, d_img, B, d_txt, NL * world, scores.ctypes.data_as(fp), idx.ctypes.data_as(ipp), K), lib.last_error()

    def step_e2e():
        assert L.clip_b200_zero_shot_images(ctx, 4, C.byref(batch), arr, NL, True, K, scores.ctypes.data_as(fp), idx.ctypes.data_as(ipp)), lib.last_error()

    for _ in range(args.warmup):
        step_device()
    ref_idx = idx.copy()
    b.drop_profile()
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        sampler.start()
    l0 = L.clip_b200_kernel_launches(ctx)
    ms_step, ms_wall = b.timed(step_device, args.steps)
    launches = (L.clip_b200_kernel_launches(ctx) - l0) + (args.steps if world > 1 else 0)
    clocks = sampler.stop() if rank == 0 else None
    kinds = b.kinds(args.steps)
    outputs = None
    if args.dump_outputs:       # this rank's images; the label embeddings are all ranks' (all-gathered)
        outputs = {"image_embeddings": b.fetch(d_img, (B, d)), "label_embeddings": b.fetch(d_txt, (NL * world, d)),
                   "top5_scores": scores.copy(), "top5_labels": idx.astype(np.float64)}
    for _ in range(2):
        step_e2e()
    same = bool(np.array_equal(idx, ref_idx))
    ms_e2e, _ = b.timed(step_e2e, max(2, args.steps // 2))
    b.drop_profile()
    return {"outputs": outputs, "ms_step": ms_step, "ms_wall": ms_wall, "launches": launches, "clocks": clocks, "kinds": kinds, "units": B,
            "e2e": {"value": B * world / (ms_e2e / 1e3), "unit": "img/s", "h2d_bytes_per_step": B * per * 4 + NL * 80 * 4,
                    "d2h_bytes_per_step": B * K * 8, "ms_per_step": ms_e2e, "call": "clip_b200_zero_shot_images",
                    "top5_identical_to_device_resident_path": same}}


def parity_check(b):
    """this very build against the reference-produced golden vectors (first images / texts of the fixture)"""
    import synth_gguf as sg
    cfg = b.cfg
    gpath = os.path.join(ROOT, "tests", "golden", "%s-s%d.npz" % (cfg["geom"], SEED))
    if not os.path.exists(gpath):
        return None
    g = np.load(gpath)
    ft = cfg["ftype"]
    key = ("txt_" if cfg["kind"] == "text" else "img_") + ft
    if key not in g.files or str(g["sha_" + ft]) != sg.sha256_file(b.model):
        return None
    if cfg["kind"] == "text":
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        lens = [int(x) for x in g["tok_lens"]]
        seqs = [sg.synth_tokens(1, n, int(g["tok_seed"]) + i)[0] for i, n in enumerate(lens)]
        got = b.lib.text_batch_encode(b.ctx, seqs)
    else:
        got = b.lib.image_batch_encode(b.ctx, sg.synth_images(int(g["n_img"]), 224, int(g["img_seed"])))
    ref = g[key]
    c = (got * ref).sum(1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(ref, axis=1))
    return {"one_minus_cos_max": float((1 - c).max()), "n": int(len(ref)), "tolerance": 1e-2 if ft.startswith("q") else 1e-3,
            "against": "reference ggml CPU embeddings (tests/golden, produced by oracle/_ref)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: the config's batch is the GLOBAL batch, split over the GPUs")
    ap.add_argument("--batch", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--no-cpu-baseline", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--quick", action="store_true", help=argparse.SUPPRESS)        # skip the secondary legs (ncu captures, probes)
    ap.add_argument("--no-text", action="store_true", help=argparse.SUPPRESS)       # kept for old command lines: same as --quick
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (rank 0; float32/float64, <= 64 MB)")
    args = ap.parse_args()
    args.quick = args.quick or args.no_text
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = dict(CONFIGS[args.config])
    if args.batch:
        cfg["batch"] = args.batch

    if args.impl == "reference":
        run_reference_arm(args, cfg, rank)
        return

    b = Bench(args, cfg, rank, world, local)
    kind = cfg["kind"]
    scaling = "strong" if (args.scaling == "strong" or kind == "zsl") else "weak"
    if kind == "zsl":
        res = bench_zsl(b, cfg["batch"], cfg["labels"])
        units = res["units"]
    else:
        units = cfg["batch"] // world if scaling == "strong" else cfg["batch"]
        res = bench_image(b, units) if kind == "image" else bench_text(b, units)
    ms_step = res["ms_step"]
    value = units * world / (ms_step / 1e3)

    if rank == 0:
        peak, peak_src = peaks()
        fkey = (cfg["geom"], "image" if kind in ("image", "zsl") else "text")
        f_total, f_attn = FLOPS[fkey]
        f_gemm = f_total - f_attn
        gemm_flops = f_gemm * units
        if kind == "zsl":
            ft_total, ft_attn = FLOPS[(cfg["geom"], "text")]
            gemm_flops += (ft_total - ft_attn) * (cfg["labels"] // world)
        gemm_ms = res["kinds"]["gemm"]["ms_per_step"]
        achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
        traffic = NCU_GEMM_TRAFFIC.get(args.config if not args.batch and scaling == "weak" else None)
        parity = parity_check(b) if kind != "zsl" else None
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                cpu, _ = cpu_reference_sample(cfg, b.model, 8 if kind != "text" else 32, pick_threads(cfg, b.model))
            except Exception as e:           # the baseline leg must never take the GPU number down with it
                cpu = {"value": None, "unit": None, "cores": None, "kind": "unavailable", "sample": str(e)[:200]}
        metric = {"image": "image-embeddings/sec", "text": "text-embeddings/sec", "zsl": "zero-shot images/sec (4096 images x 1000 labels)"}[kind]
        unit = "seq/s" if kind == "text" else "img/s"
        out = {
            "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "bf16 (%s blocks unpacked to bf16 in-kernel, fp32 accumulate in TMEM; fp32 residual stream)" % cfg["ftype"], "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "global_batch": units * world, "per_gpu_batch": units, "parallelism": "dp%d" % world,
                       "l2": "inputs per step exceed the 126 MB L2 (no flush needed)" if kind != "text" else "token ids are tiny; the activations of a pass (> 1 GB) exceed L2",
                       "collective": "1 in-place NCCL all-gather of the final embeddings per step, enqueued by the C++ library (no torch in the rank processes)" if world > 1 else "none (1 GPU)"},
            "clocks": res["clocks"], "e2e": res["e2e"], "gpu_launches": int(res["launches"]),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                         "traffic": traffic[0] if traffic else None,
                         "traffic_unit": ("bytes/launch (dram read+write, mean of the 4 layer GEMM shapes; %s) vs %d algorithmic" % (traffic[2], traffic[1])) if traffic else None,
                         "kernel": "gemm_dq_kernel (all fused-dequant GEMMs of the step)", "flops_per_step": gemm_flops, "kernel_ms_per_step": gemm_ms,
                         "peak_source": peak_src, "whole_step_frac": (f_total * units / (ms_step / 1e3) / 1e12) / peak if kind != "zsl" else None},
            "kernel_time_ms_per_step": res["kinds"], "wall_ms_per_step": res["ms_wall"], "parity": parity, "cpu_baseline": cpu,
            "nccl": L_nccl(b) if world > 1 else None,
        }
        for k in ("e2e_pageable", "e2e_u8"):
            if k in res:
                out[k] = res[k]
        print(json.dumps(out), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, res["outputs"])
    b.sync_all()
    b.lib.free(b.ctx)


def L_nccl(b):
    return {"version": int(b.L.clip_b200_nccl_version()), "ranks": int(b.L.clip_b200_dist_world(b.ctx)), "torch_imported": "torch" in sys.modules}


if __name__ == "__main__":
    main()

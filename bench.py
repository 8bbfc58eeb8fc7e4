#!/usr/bin/env python
"""bench.py -- headline benchmark: Mpixels/s for thumbnail(4K -> 512, lanczos3).

Workload = BASELINE.json configs[1]: vips_thumbnail 4096x4096 uchar RGBA -> 512x512,
a batch of 1024 synthetic frames per GPU (64 GiB resident in HBM, >> the 126 MB L2).  A "step" is
one pass of the fused thumbnail kernel over the whole batch, frames resident in HBM.

  python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1)
  python bench.py ... --dump-outputs DIR                    also write what the last timed step computed, DIR/*.npy
  python bench.py --impl reference ...                      CPU arm (the oracle port
                                                            of the reference algorithm)

torch is used only for device memory, CUDA events/streams and torch.distributed.
The kernels are libvips_b200/libvb200.so, called through its C ABI.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W = H = 4096
BANDS = 4
TARGET = 512
MPIX_PER_FRAME = W * H / 1e6
METRIC = "Mpixels/s for thumbnail(4K->512,lanczos3)"
METRIC_PIPELINE = "Mpixels/s for thumbnail(4K->512,lanczos3) + sharpen + sRGB (BASELINE config 5 stream)"
# dram__bytes_read.sum + dram__bytes_write.sum of the fused kernel per 4096x4096 frame, from the
# committed `ncu --set full` capture (a launch of 148 frames: 10.1220 GB read, 159.4 MB written)
DRAM_BYTES_PER_FRAME = (10.124448e9 + 161.176576e6) / 148
DRAM_SOURCE = "profiles/r2/headline_random_alpha_ncu_summary.txt (ncu --set full, 148 frames: per frame x frames in the launch)"
WORKLOAD = "vips_thumbnail 4K->512 uchar RGBA (premultiply,shrinkv4,reducev13,shrinkh4,reduceh13,unpremultiply), synthetic frames, device-resident"
WORKLOAD_PIPELINE = ("vips_thumbnail 4K->512 uchar RGBA then vips_sharpen (sRGB->LabS, 3-tap integer blur of L, LUT, LabS->sRGB) on the 512x512 "
                     "result, synthetic frames, device-resident")
PIPELINE = False  # set by --workload pipeline: the CPU arm and the GPU arm both append the sharpen stage


DUMP_BYTES = 64_000_000


def dump_outputs(dirname, arrays, budget=DUMP_BYTES):
    """--dump-outputs: each device array as <dirname>/<name>.npy in float32 (float64 data stays float64).  An array over
    its share of the budget is sampled along its first axis by a fixed seed, the indices written beside it as
    <name>_index.npy, so that two builds run with the same arguments write files that compare entry for entry."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    share = budget // len(arrays)
    for name, t in arrays.items():
        dt = np.dtype(np.float64 if t.dtype == torch.float64 else np.float32)
        if t.numel() * dt.itemsize > share:
            if t[0].numel() * dt.itemsize > share:
                t = t.reshape(-1)
            k = max(1, share // (t[0].numel() * dt.itemsize))
            idx = np.sort(np.random.default_rng(0).choice(t.shape[0], k, replace=False))
            np.save(os.path.join(dirname, name + "_index.npy"), idx.astype(np.float64))
            t = t[torch.as_tensor(idx, device=t.device)]
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy().astype(dt))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in self.rows:
            for i, n in enumerate(names):
                if len(r) > 3 + i and r[3 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _ref_worker(i):
    """one frame through the reference's own C sources (oracle/_ref), in a worker process"""
    from oracle import pyref
    t = pyref.thumbnail_image(_REF_FRAMES[i], TARGET)
    if PIPELINE:
        # sharpen.c runs under oracle/_ref for 3-band images only (the shim's colourspace stand-in has no alpha
        # re-attach): the 512x512 RGBA result -- 1.5% of the frame's pixels -- goes through the oracle port, which
        # tests/test_convolution.py pins bit for bit to the reference's sharpen.c
        from oracle import pyconv
        t = pyconv.sharpen(t, "srgb")
    return int(t[0, 0, 0])


_REF_FRAMES = None


class CpuArm:
    """The reference chain on the host cores, one frame per worker (the reference's inter-image threading).

    kind "reference": the reference's OWN sources -- premultiply.c, reducev.cpp, reduceh.cpp, shrinkv.c,
    shrinkh.c, resize.c, unpremultiply.c compiled in place into oracle/_ref/libvipsref.so (scalar C
    paths: Highway is not in this image) under oracle/ref_shim's region engine, one process per frame.
    kind "port": the oracle port (liboracle_fast.so, -O3 -march=native), one thread per frame; used when
    oracle/_ref is not there (it is built from /root/reference, which does not exist on every machine).
    """

    def __init__(self, n_frames, threads):
        import numpy as np
        global _REF_FRAMES
        self.n, self.threads = n_frames, threads
        rng = np.random.default_rng(1234)
        one = rng.integers(0, 256, (H, W, BANDS), dtype=np.uint8)
        self.a = np.stack([np.roll(one, 7 * i, axis=1) for i in range(n_frames)])
        self.kind = "port"
        if os.environ.get("VB200_CPU_ARM") != "port":
            try:
                from oracle import pyref
                if pyref.available():
                    import multiprocessing as mp
                    _REF_FRAMES = self.a                      # inherited by fork: no copies, no pickling
                    self.pool = mp.get_context("fork").Pool(threads)
                    self.kind = "reference"
            except Exception:
                self.kind = "port"
        if self.kind == "port":
            from oracle import pyoracle
            fast = os.path.join(ROOT, "oracle", "liboracle_fast.so")
            if not os.path.exists(fast):
                pyoracle.build()
            self.L = C.CDLL(fast)
            self.out = np.empty((n_frames, TARGET, TARGET, BANDS), np.uint8)

    def describe(self):
        tail = "; then vips_sharpen on the 512x512 result through the oracle port (pinned to the reference's sharpen.c)" if PIPELINE else ""
        if self.kind == "reference":
            return ("the reference's own sources (oracle/_ref: premultiply, shrinkv, reducev, shrinkh, reduceh, unpremultiply; "
                    "scalar C paths, no Highway) under the shim region engine, one frame per process" + tail)
        return "oracle port of the reference chain (liboracle_fast.so), one frame per thread" + tail

    def step(self):
        t = time.perf_counter()
        if self.kind == "reference":
            self.pool.map(_ref_worker, range(self.n), chunksize=1)
        else:
            rc = self.L.orc_thumbnail_image_batch(C.c_void_p(self.a.ctypes.data), self.n, W, H, BANDS, TARGET, TARGET,
                                                  0, 1, C.c_void_p(self.out.ctypes.data), TARGET, TARGET, self.threads)
            assert rc == 0
            if PIPELINE:
                from concurrent.futures import ThreadPoolExecutor
                from oracle import pyconv
                with ThreadPoolExecutor(self.threads) as ex:  # ctypes releases the GIL
                    list(ex.map(lambda f: pyconv.sharpen(f, "srgb"), self.out))
        return time.perf_counter() - t

    def close(self):
        if self.kind == "reference":
            self.pool.terminate()


def host_threads():
    """CPUs this process may really use: the affinity mask, capped by a cgroup CPU quota if there is one
    (a container can see 128 CPUs in its mask and be allowed 8 CPUs' worth of time)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                      # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()
            if q != "max":
                quota = float(q) / float(p)
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:     # cgroup v1
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0 and p > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.999)))
    return n


def numa_cpus(node):
    """CPUs of a NUMA node (sysfs cpulist), or None"""
    try:
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        return cpus or None
    except (OSError, ValueError):
        return None


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    frames = max(threads, 8)
    arm = CpuArm(frames, threads)
    for _ in range(args.warmup):
        arm.step()
    t = time.perf_counter()
    for _ in range(args.steps):
        arm.step()
    dt = time.perf_counter() - t
    arm.close()
    v = frames * args.steps * MPIX_PER_FRAME / dt
    also = None
    if arm.kind == "reference":
        # for transparency, the faster restatement too (same algorithm, -O3 -march=native, threads instead of the shim engine)
        os.environ["VB200_CPU_ARM"] = "port"
        port = CpuArm(frames, threads)
        port.step()
        also = {"kind": "port", "value": frames * MPIX_PER_FRAME / min(port.step() for _ in range(2)), "unit": "Mpixels/s",
                "sample": port.describe()}
    line = {
        "impl": "reference", "metric": METRIC_PIPELINE if PIPELINE else METRIC, "value": v, "unit": "Mpixels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": (WORKLOAD_PIPELINE if PIPELINE else WORKLOAD).replace("device-resident", "host RAM"),
                   "frames_per_step": frames},
        "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": threads, "kind": arm.kind,
                         "sample": "%d 4096x4096 RGBA frames per step: %s" % (frames, arm.describe()), "also": also},
        "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


_JPEG_CPU = None


def _jpeg_cpu_worker(i):
    """one frame the reference's way on the host: libjpeg-turbo shrink-on-load, then the thumbnail chain"""
    import io
    import numpy as np
    from PIL import Image
    from oracle import pyoracle
    distinct, shrink, save = _JPEG_CPU
    im = Image.open(io.BytesIO(distinct[i % len(distinct)]))
    im.draft("RGB", (W // shrink, H // shrink))
    a = np.asarray(im)[: H // shrink, : W // shrink]
    t = pyoracle.thumbnail_image(a, TARGET)
    if save:
        b = io.BytesIO()
        Image.fromarray(t).save(b, "JPEG", quality=75, subsampling=2)
        return len(b.getvalue())
    return int(t[0, 0, 0])


def side_workload(args):
    """BASELINE.json configs 1, 3, 4 on one GPU, device-resident, CUDA events: not the
    headline line, the rows of BASELINE.md's results table."""
    import numpy as np
    import torch

    import libvips_b200 as vb
    from libvips_b200 import CImage, CMask

    vb.init(0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    vb.set_stream(stream.cuda_stream)
    L = vb.lib()
    peak, peak_src = peaks()

    def dimg(t, interp):
        h, w, b = t.shape
        fmt = {torch.uint8: 0, torch.float32: 6, torch.int16: 3}[t.dtype]
        return CImage(w, h, b, fmt, interp, vb.DEVICE, C.c_void_p(t.data_ptr()), w * b * t.element_size())

    def cpu_side(cpu_fn, units, sample):
        """the oracle port of the same op on a bounded sample, one host thread (it is a scalar port)"""
        if args.no_cpu or cpu_fn is None:
            return None
        cpu_fn()
        t = time.perf_counter()
        cpu_fn()
        dt = time.perf_counter() - t
        return {"value": units / dt, "unit": "Mpixels/s", "cores": 1, "kind": "port", "sample": "%s, %.1f s" % (sample, dt)}

    def run(fn, alg_bytes, label, units, unit_name, cpu=None, outputs=None):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = vb.launch_count()
        e0.record(stream)
        for _ in range(args.steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        ms = e0.elapsed_time(e1) / args.steps
        ach = alg_bytes / (ms / 1e3) / 1e9
        print(json.dumps({"metric": label, "value": units / (ms / 1e3), "unit": unit_name, "n_gpus": 1,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                          "dtype": "f32/f64 accumulate" if "conv" in label or "colour" in label or "linear" in label else "u8",
                          "data": "synthetic", "config": {"workload": label, "device_resident": True},
                          "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                                       "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                                       "algorithmic_bytes": alg_bytes},
                          "cpu_baseline": cpu, "gpu_launches": int(vb.launch_count() - n0)}))

    if args.workload == "convsep":
        n = 8192
        a = torch.rand((n, n, 3), device=dev) * 255
        out = torch.empty_like(a)
        m, scale, off = vb.gaussmat(4.0, 0.2, True, "float")
        cm = CMask(m.shape[1], m.shape[0], m.ctypes.data_as(C.POINTER(C.c_double)), scale, off)
        cin = dimg(a, 22)

        def fn():
            cout = dimg(out, 22)
            vb._check(L.vb200_convsep(C.byref(cin), C.byref(cout), C.byref(cm), 1))
        from oracle import pyconv
        ca = (np.random.default_rng(1234).random((2048, 2048, 3), dtype=np.float32) * 255)
        cpu = cpu_side(lambda: pyconv.convsep(ca, m, scale, off, "float"), 2048 * 2048 / 1e6, "2048x2048x3 float32")
        run(fn, 2 * a.numel() * 4, "vips_convsep 15-tap Gaussian float on 8192x8192 RGB float32", n * n / 1e6, "Mpixels/s", cpu, {"out": out})
    elif args.workload == "colour":
        n = 16384
        a = torch.randint(0, 256, (n, n, 3), dtype=torch.uint8, device=dev)
        lab = torch.empty((n, n, 3), dtype=torch.float32, device=dev)
        back = torch.empty_like(a)
        cin = dimg(a, 22)

        def fn():
            clab = dimg(lab, 13)
            vb._check(L.vb200_colourspace(C.byref(cin), C.byref(clab), 13))
            clab = dimg(lab, 13)
            cback = dimg(back, 22)
            vb._check(L.vb200_colourspace(C.byref(clab), C.byref(cback), 22))
        fn()
        torch.cuda.synchronize()
        assert torch.equal(a, back), "sRGB -> Lab -> sRGB must be the identity on 8-bit data"
        from oracle import pyoracle
        ca = np.random.default_rng(1234).integers(0, 256, (2048, 2048, 3), dtype=np.uint8)
        cpu = cpu_side(lambda: pyoracle.colourspace(pyoracle.colourspace(ca, "lab", "srgb"), "srgb", "lab"),
                       2 * 2048 * 2048 / 1e6, "2048x2048x3 uint8, both directions")
        run(fn, 2 * (a.numel() + lab.numel() * 4), "vips_colourspace sRGB->Lab->sRGB round trip on 16384x16384",
            2 * n * n / 1e6, "Mpixels/s", cpu, {"lab": lab, "srgb": back})
    elif args.workload == "reduce49":
        n = 4096
        a = torch.randint(0, 256, (n, n, 4), dtype=torch.uint8, device=dev)
        out = torch.empty((n // 8, n // 8, 4), dtype=torch.uint8, device=dev)
        cin = dimg(a, 22)

        def fn():
            cout = dimg(out, 22)
            vb._check(L.vb200_reduce(C.byref(cin), C.byref(cout), 8.0, 8.0, 5, 0.0))
        from oracle import pyoracle
        ca = np.random.default_rng(1234).integers(0, 256, (n, n, 4), dtype=np.uint8)
        cpu = cpu_side(lambda: pyoracle.reduceh(pyoracle.reducev(ca, 8.0, "lanczos3", 0.0), 8.0, "lanczos3", 0.0),
                       n * n / 1e6, "one 4096x4096 RGBA frame")
        run(fn, a.numel() + out.numel(), "vips_reduce(8, 8) Lanczos3 gap 0 (49 taps) on one 4096x4096 uchar RGBA",
            n * n / 1e6, "Mpixels/s", cpu, {"out": out})
    elif args.workload == "upsize":
        # SURVEY 8(a) a7: vips_resize x2 = vips_affine + bicubic (resize.c:235-305)
        n = 4096
        a = torch.randint(0, 256, (n, n, 4), dtype=torch.uint8, device=dev)
        out = torch.empty((2 * n, 2 * n, 4), dtype=torch.uint8, device=dev)
        cin = dimg(a, 22)

        def fn():
            cout = dimg(out, 22)
            vb._check(L.vb200_resize(C.byref(cin), C.byref(cout), 2.0, 2.0, 5, 2.0))
        from oracle import pyoracle
        ca = np.random.default_rng(1234).integers(0, 256, (1024, 1024, 4), dtype=np.uint8)
        cpu = cpu_side(lambda: pyoracle.resize(ca, 2.0), 4 * 1024 * 1024 / 1e6, "1024x1024 RGBA -> 2048x2048")
        run(fn, a.numel() + out.numel(), "vips_resize x2 (affine + bicubic) 4096x4096 uchar RGBA -> 8192x8192",
            4 * n * n / 1e6, "output Mpixels/s", cpu, {"out": out})
    elif args.workload == "sharpen":
        # SURVEY 8(a) a11: vips_sharpen defaults on an sRGB image (sRGB -> LabS, L blur + LUT, LabS -> sRGB)
        n = 4096
        a = torch.randint(0, 256, (n, n, 3), dtype=torch.uint8, device=dev)
        out = torch.empty_like(a)
        cin = dimg(a, 22)

        def fn():
            cout = dimg(out, 22)
            vb._check(L.vb200_sharpen(C.byref(cin), C.byref(cout), 0.5, 2.0, 10.0, 20.0, 0.0, 3.0))
        from oracle import pyconv
        ca = np.random.default_rng(1234).integers(0, 256, (1024, 1024, 3), dtype=np.uint8)
        cpu = cpu_side(lambda: pyconv.sharpen(ca, "srgb"), 1024 * 1024 / 1e6, "1024x1024 RGB")
        run(fn, 2 * a.numel(), "vips_sharpen defaults on 4096x4096 sRGB uchar", n * n / 1e6, "Mpixels/s", cpu, {"out": out})
    elif args.workload == "thumbnail_linear":
        # north_star's "fused Lanczos3-reduce -> sRGB -> linear" path: vips_thumbnail_image(linear=TRUE), SURVEY 3.1b
        F = max(1, min(args.frames, 128))
        plan = vb.ThumbnailPlan(W, H, BANDS, TARGET, linear=True)
        assert plan.fused, "the two-kernel linear path must be the one under measurement"
        g = torch.Generator(device=dev)
        g.manual_seed(4321)
        frames = torch.randint(0, 256, (F, H, W, BANDS), dtype=torch.uint8, device=dev, generator=g)
        common = np.random.default_rng(1234).integers(0, 256, (H, W, BANDS), dtype=np.uint8)
        frames[0].copy_(torch.from_numpy(common))
        outs = torch.empty((F, TARGET, TARGET, BANDS), dtype=torch.uint8, device=dev)

        def fn():
            plan.run_device(frames.data_ptr(), outs.data_ptr(), F)
        fn()
        torch.cuda.synchronize()
        from oracle import pyoracle
        want = pyoracle.thumbnail_image(common, TARGET, linear=True)
        assert np.array_equal(outs[0].cpu().numpy(), want), "GPU linear thumbnail differs from the oracle"
        ca = np.random.default_rng(7).integers(0, 256, (H, W, BANDS), dtype=np.uint8)
        cpu = cpu_side(lambda: pyoracle.thumbnail_image(ca, TARGET, linear=True), W * H / 1e6, "one 4096x4096 RGBA frame")
        run(fn, plan.bytes_per_frame * F, "vips_thumbnail_image(linear=TRUE) 4K->512 uchar RGBA, %d frames (%s)" % (F, plan.kernel),
            F * W * H / 1e6, "Mpixels/s", cpu, {"thumbnails": outs})
    elif args.workload == "icc":
        # SURVEY 8(a) a20: vips_icc_import then vips_icc_export through an sRGB-like v4 matrix/TRC profile
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import icc_fixtures
        prof = icc_fixtures.rgb_profile("srgb")
        n = 8192
        a = torch.randint(0, 256, (n, n, 3), dtype=torch.uint8, device=dev)
        lab = torch.empty((n, n, 3), dtype=torch.float32, device=dev)
        back = torch.empty_like(a)
        cin = dimg(a, 22)

        def fn():
            clab = dimg(lab, 13)
            vb._check(L.vb200_icc_import(C.byref(cin), C.byref(clab), prof, len(prof), 1, 0))
            clab = dimg(lab, 13)
            cback = dimg(back, 22)
            vb._check(L.vb200_icc_export(C.byref(clab), C.byref(cback), prof, len(prof), 1, 8, 0))
        fn()
        torch.cuda.synchronize()
        assert (a.to(torch.int16) - back.to(torch.int16)).abs().max().item() <= 1, "import then export is the identity to 1 LSB"
        cpu = None
        from oracle import pylcms
        if pylcms.available() and not args.no_cpu:
            ca = np.random.default_rng(1234).integers(0, 256, (2048, 2048, 3), dtype=np.uint8)
            cpu = cpu_side(lambda: pylcms.icc_export(pylcms.icc_import(ca, prof), prof), 2 * 2048 * 2048 / 1e6,
                           "2048x2048x3 uint8 through lcms2 2.18 itself, both directions")
            cpu["kind"] = "reference"
        run(fn, 2 * (a.numel() + lab.numel() * 4), "vips_icc_import + vips_icc_export (sRGB-like v4 profile) on 8192x8192",
            2 * n * n / 1e6, "Mpixels/s", cpu, {"lab": lab, "srgb": back})
    elif args.workload in ("rank", "flatten", "greyscale"):
        # SURVEY 8f ranks 3 / 4 (DESIGN 4.10-4.12): parity-green in round 2, never timed there (the GPU budget was spent)
        n = 4096
        from oracle import pyconv
        rng = np.random.default_rng(1234)
        if args.workload == "rank":
            a = torch.randint(0, 256, (n, n, 3), dtype=torch.uint8, device=dev)
            out = torch.empty_like(a)
            cin = dimg(a, 22)

            def fn():
                cout = dimg(out, 22)
                vb._check(L.vb200_rank(C.byref(cin), C.byref(cout), 3, 3, 4))
            ca = rng.integers(0, 256, (1024, 1024, 3), dtype=np.uint8)
            cpu = cpu_side(lambda: pyconv.median(ca, 3), 1024 * 1024 / 1e6, "1024x1024 RGB")
            run(fn, 2 * a.numel(), "vips_median 3x3 on 4096x4096 sRGB uchar", n * n / 1e6, "Mpixels/s", cpu, {"out": out})
        elif args.workload == "flatten":
            a = torch.randint(0, 256, (n, n, 4), dtype=torch.uint8, device=dev)
            out = torch.empty((n, n, 3), dtype=torch.uint8, device=dev)
            cin = dimg(a, 22)
            bg = (C.c_double * 3)(255.0, 255.0, 255.0)

            def fn():
                cout = dimg(out, 22)
                vb._check(L.vb200_flatten(C.byref(cin), C.byref(cout), bg, 3, 0.0))
            ca = rng.integers(0, 256, (1024, 1024, 4), dtype=np.uint8)
            cpu = cpu_side(lambda: pyconv.flatten(ca, (255, 255, 255)), 1024 * 1024 / 1e6, "1024x1024 RGBA")
            run(fn, a.numel() + out.numel(), "vips_flatten (white background) on 4096x4096 RGBA uchar", n * n / 1e6, "Mpixels/s", cpu,
                {"out": out})
        else:
            from oracle import pyoracle
            a = torch.randint(0, 256, (n, n, 3), dtype=torch.uint8, device=dev)
            out = torch.empty((n, n, 1), dtype=torch.uint8, device=dev)
            cin = dimg(a, 22)

            def fn():
                cout = dimg(out, 1)
                vb._check(L.vb200_colourspace(C.byref(cin), C.byref(cout), 1))
            ca = rng.integers(0, 256, (1024, 1024, 3), dtype=np.uint8)
            cpu = cpu_side(lambda: pyoracle.colourspace(ca, "b-w", "srgb"), 1024 * 1024 / 1e6, "1024x1024 RGB")
            run(fn, a.numel() + out.numel(), "vips_colourspace sRGB -> B_W on 4096x4096 uchar", n * n / 1e6, "Mpixels/s", cpu, {"out": out})
    elif args.workload in ("thumbnail_jpeg", "thumbnail_jpeg_norestart", "thumbnail_jpeg_progressive"):
        # SURVEY 8(f) rank 1: vips_thumbnail_buffer() of JPEG streams.  Host memory holds only the COMPRESSED frames; the
        # shrink-on-load decode (thumbnail.c:489-517 picks 1/4 for 4K -> 512) and the thumbnail run on the device.
        # End to end by construction: every step uploads its streams.  The CPU side is the reference's own recipe:
        # libjpeg-turbo (the one inside Pillow) at scale 1/4, then the thumbnail chain (oracle port), one frame per process.
        import io
        from PIL import Image
        restart = args.workload != "thumbnail_jpeg_norestart"
        progressive = args.workload == "thumbnail_jpeg_progressive"
        F = max(1, min(args.frames, 1024))
        yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
        distinct = []
        for i in range(8):
            rng = np.random.default_rng(100 + i)
            img = np.stack([128 + 100 * np.sin(xx / (37.0 + i) + yy / 91.0), 128 + 90 * np.cos(xx / 53.0 - yy / (29.0 + i)),
                            np.mod(xx * 3 + yy * 5, 256)], -1) + rng.normal(0, 10, (H, W, 3)).astype(np.float32)
            b = io.BytesIO()
            from PIL import ImageFile
            ImageFile.MAXBLOCK = 1 << 26
            Image.fromarray(np.clip(img, 0, 255).astype(np.uint8)).save(b, "JPEG", quality=85, subsampling=2, progressive=progressive,
                                                                     **({"restart_marker_rows": 1} if restart else {}))
            distinct.append(b.getvalue())
        del yy, xx
        streams = [distinct[i % len(distinct)] for i in range(F)]
        batch = vb.JpegBatch(streams)
        shrink = vb.thumbnail_jpegshrink(W, H, TARGET)
        dw, dh, db = vb.jpeg_geometry(batch, shrink)
        plan = vb.ThumbnailPlan(dw, dh, db, TARGET)
        outs = torch.empty((F, plan.out_height, plan.out_width, db), dtype=torch.uint8, device=dev)

        def turbo(data):
            im = Image.open(io.BytesIO(data))
            im.draft("RGB", (W // shrink, H // shrink))
            return np.asarray(im)[: H // shrink, : W // shrink]

        saved = []

        def fn():
            plan.run_jpeg(batch, shrink, out_ptr=outs.data_ptr())
            if args.save:
                saved[:] = vb.jpegsave_batch(None, 75, in_ptr=outs.data_ptr(), shape=tuple(outs.shape), stride=256 * 1024)
        fn()
        from oracle import pyoracle
        want = pyoracle.thumbnail_image(turbo(streams[0]), TARGET)
        assert np.array_equal(outs[0].cpu().numpy(), want), "GPU JPEG thumbnail differs from libjpeg-turbo + the oracle"
        if args.save:
            b = io.BytesIO()
            Image.fromarray(want).save(b, "JPEG", quality=75, subsampling=2)
            assert saved[0] == b.getvalue(), "the encoded thumbnail is not libjpeg-turbo's stream"
        for _ in range(max(0, args.warmup - 1)):
            fn()
        os.environ["VB200_JPEG_TIMING"] = "1"
        fn()
        hm, im = C.c_float(), C.c_float()
        L.vb200_debug_jpeg_times(C.byref(hm), C.byref(im))
        del os.environ["VB200_JPEG_TIMING"]
        torch.cuda.synchronize()
        n0 = vb.launch_count()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / args.steps
        if args.dump_outputs:
            dumped = {"thumbnails": outs}
            if args.save:
                dumped["jpeg_streams"] = torch.frombuffer(bytearray(b"".join(saved)), dtype=torch.uint8)
                dumped["jpeg_stream_lengths"] = torch.tensor([len(x) for x in saved], dtype=torch.float64)
            dump_outputs(args.dump_outputs, dumped)
        cpu = None
        if not args.no_cpu:
            import multiprocessing as mp
            threads = host_threads()
            global _JPEG_CPU
            _JPEG_CPU = (distinct, shrink, args.save)
            with mp.get_context("fork").Pool(threads) as pool:
                pool.map(_jpeg_cpu_worker, range(threads))
                t1 = time.perf_counter()
                pool.map(_jpeg_cpu_worker, range(2 * threads))
                ct = time.perf_counter() - t1
            cpu = {"value": 2 * threads * MPIX_PER_FRAME / ct, "unit": "Mpixels/s", "cores": threads, "kind": "reference + port",
                   "sample": "%d frames: libjpeg-turbo (Pillow's) decode at scale 1/%d, then the oracle port of the thumbnail chain, "
                             "one frame per process" % (2 * threads, shrink)}
        label = ("vips_thumbnail_buffer: 4096x4096 4:2:0 JPEG streams (q85, %s) -> shrink-on-load 1/%d on the device -> 512x512%s, %d frames per step"
                 % (("progressive, " if progressive else "") + ("one restart interval per MCU row" if restart else "no restart markers"), shrink,
                    " -> vips_jpegsave_buffer (Q 75) on the device, streams to the host" if args.save else "", F))
        print(json.dumps({"metric": label, "value": F * MPIX_PER_FRAME / dt, "unit": "Mpixels/s (input pixels)", "n_gpus": 1,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "dtype": "u8",
                          "data": "synthetic", "config": {"workload": label, "device_resident": False, "frames_per_second": F / dt,
                                                          "compressed_bytes_per_frame": batch.nbytes / F},
                          "kernels": {"jpeg_huffman_kernel_ms": hm.value, "jpeg_idct_kernel_ms": im.value,
                                      "note": "CUDA events over one step (chunks serialised for the measurement)"},
                          "e2e": {"value": F * MPIX_PER_FRAME / dt, "unit": "Mpixels/s", "h2d_bytes_per_step": batch.nbytes,
                                  "d2h_bytes_per_step": sum(len(x) for x in saved) if args.save else 0,
                                  "api": "vb200_thumbnail_plan_run_jpeg" + (" + vb200_jpegsave_batch" if args.save else "")},
                          "cpu_baseline": cpu, "gpu_launches": int(vb.launch_count() - n0)}))
    else:
        raise SystemExit("unknown workload %s" % args.workload)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--frames", type=int, default=1024, help="synthetic frames resident per GPU")
    ap.add_argument("--e2e-frames", type=int, default=24, help="host frames per end-to-end step")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--save", action="store_true",
                    help="thumbnail_jpeg workloads: also encode the thumbnails to JPEG on the device (vips_jpegsave_buffer, Q 75) and "
                         "bring the streams to the host -- the thumbnail server's whole loop")
    ap.add_argument("--alpha", default="random", choices=["random", "opaque"],
                    help="alpha band of the synthetic frames: random (the headline) | opaque (255 everywhere, what a PNG without "
                         "transparency decodes to: the kernel's opaque-stage fast path; a second line, never the headline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (float32; outputs over "
                         "64 MB in all are sampled by a fixed seed, the indices in DIR/<name>_index.npy)")
    ap.add_argument("--workload", default="thumbnail",
                    help="thumbnail (the headline, default) | pipeline (BASELINE config 5: thumbnail + sharpen + sRGB, runs under "
                         "--gpus N like the headline) | thumbnail_jpeg | thumbnail_jpeg_norestart | thumbnail_jpeg_progressive (decode staging, SURVEY 8f; --save adds the encoder) | thumbnail_linear | convsep | colour | reduce49 | upsize | sharpen | icc | rank | flatten | greyscale: the other BASELINE.json "
                         "configs, one device-resident JSON line each (1 GPU)")
    args = ap.parse_args()

    global PIPELINE
    PIPELINE = args.workload == "pipeline"
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the device computed: not with --impl reference")
        return reference_arm(args)
    if args.workload not in ("thumbnail", "pipeline"):
        return side_workload(args)

    import numpy as np
    import torch

    import libvips_b200 as vb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    vb.init(local)
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream()
    vb.set_stream(stream.cuda_stream)

    plan = vb.ThumbnailPlan(W, H, BANDS, TARGET)
    assert plan.fused, "the fused kernel must be the path under measurement"
    assert (plan.out_width, plan.out_height) == (TARGET, TARGET)

    # synthetic frames, generated on the device (seeded per rank); frame 0 is the shared
    # numpy-seeded frame used for the cross-rank parity check below
    F = args.frames
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    frames = torch.empty((F, H, W, BANDS), dtype=torch.uint8, device=dev)
    for i in range(0, F, 16):
        n = min(16, F - i)
        frames[i:i + n] = torch.randint(0, 256, (n, H, W, BANDS), dtype=torch.uint8, device=dev, generator=g)
    common = np.random.default_rng(1234).integers(0, 256, (H, W, BANDS), dtype=np.uint8)
    if args.alpha == "opaque":
        frames[..., BANDS - 1] = 255
        common[..., BANDS - 1] = 255
    frames[0].copy_(torch.from_numpy(common))
    outs = torch.empty((F, TARGET, TARGET, BANDS), dtype=torch.uint8, device=dev)
    SHARPEN = (0.5, 2.0, 10.0, 20.0, 0.0, 3.0)  # vips_sharpen's defaults
    Lc = vb.lib()
    mid = torch.empty_like(outs) if PIPELINE else None
    ev_mid = []

    def step():
        if PIPELINE:
            # the two stages of the stream through their public batch entry points, so that an event can sit
            # between the kernels (a plan with set_sharpen() launches the same two kernels: tests/test_pipeline.py)
            plan.run_device(frames.data_ptr(), mid.data_ptr(), F)
            if ev_mid:
                ev_mid[0].record(stream)
            vb._check(Lc.vb200_sharpen_batch_device(mid.data_ptr(), plan.out_frame_bytes, outs.data_ptr(), plan.out_frame_bytes, F,
                                                    TARGET, TARGET, BANDS, *SHARPEN))
        else:
            plan.run_device(frames.data_ptr(), outs.data_ptr(), F)

    # correctness gate before timing: frame 0 against the oracle (rank 0), same checksum on all ranks.  Always run:
    # a tuning build (VB200_LIB, tools/build_variant.sh) that computes wrong pixels is reported as such, never as the metric
    step()
    torch.cuda.synchronize()
    csum = outs[0].to(torch.int64).sum()
    parity = "ok"
    if rank == 0:
        from oracle import pyoracle
        want = pyoracle.thumbnail_image(common, TARGET)
        if PIPELINE:
            from oracle import pyconv
            want = pyconv.sharpen(want, "srgb", *SHARPEN)
        if not np.array_equal(outs[0].cpu().numpy(), want):
            parity = "failed"
            assert os.environ.get("VB200_LIB") is not None, "GPU result differs from the oracle"
    if dist:
        from libvips_b200 import shard
        assert shard.all_agree(dist, csum.reshape(1)), "ranks disagree on the shared frame"

    for _ in range(max(0, args.warmup - 1)):
        step()

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    mids = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = vb.launch_count()
    barrier()
    evs[0].record(stream)
    for i in range(args.steps):
        ev_mid[:] = [mids[i]]
        step()
        evs[i + 1].record(stream)
    barrier()
    ev_mid[:] = []
    launches = vb.launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"thumbnails" + ("" if world == 1 else "_rank%d" % rank): outs}, DUMP_BYTES // world)
    clocks = sampler.stop() if rank == 0 else None
    total_ms = evs[0].elapsed_time(evs[-1])
    per_step = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if dist:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms_max = float(tmax.item())

    value = world * F * args.steps * MPIX_PER_FRAME / (total_ms_max / 1e3)

    # roofline of the dominant (only) kernel: algorithmic bytes / mean launch duration on this rank
    peak, peak_src = peaks()
    kern_ms = sum(per_step) / len(per_step)
    bytes_per_launch = plan.bytes_per_frame * F
    kernels = None
    if PIPELINE:
        # dominant kernel = the fused thumbnail (start -> mid event); the sharpen kernel (mid -> end) beside it
        thumb_ms = sum(evs[i].elapsed_time(mids[i]) for i in range(args.steps)) / args.steps
        sharp_ms = sum(mids[i].elapsed_time(evs[i + 1]) for i in range(args.steps)) / args.steps
        sharp_bytes = 2 * plan.out_frame_bytes * F
        kernels = [{"kernel": plan.kernel, "ms": thumb_ms, "algorithmic_bytes": bytes_per_launch,
                    "frac": bytes_per_launch / (thumb_ms / 1e3) / 1e9 / peak},
                   {"kernel": "sharpen_fused_kernel<4>", "ms": sharp_ms, "algorithmic_bytes": sharp_bytes,
                    "frac": sharp_bytes / (sharp_ms / 1e3) / 1e9 / peak}]
        kern_ms = thumb_ms
    achieved = bytes_per_launch / (kern_ms / 1e3) / 1e9

    # end to end through the C ABI with HOST (pinned) buffers: H2D + kernel + D2H inside the timed region
    e2e = None
    E = args.e2e_frames
    L = vb.lib()
    # the feeder runs on the GPU's NUMA node, its pinned buffers live there (vb200_host_alloc places them):
    # on the 8-GPU boxes GPUs 4-7 hang off node 1
    node = L.vb200_device_numa_node()
    affinity0 = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    local_cpus = numa_cpus(node) if node >= 0 else None
    if affinity0 and local_cpus and (local_cpus & affinity0):
        os.sched_setaffinity(0, local_cpus & affinity0)
    hin = L.vb200_host_alloc(E * plan.in_frame_bytes)
    hout = L.vb200_host_alloc(E * plan.out_frame_bytes)
    if PIPELINE:
        plan.set_sharpen(*SHARPEN)
    if hin and hout:
        src = np.frombuffer((C.c_uint8 * (E * plan.in_frame_bytes)).from_address(hin), dtype=np.uint8)
        one = np.random.default_rng(99 + rank).integers(0, 256, plan.in_frame_bytes, dtype=np.uint8)
        if args.alpha == "opaque":
            one[BANDS - 1::BANDS] = 255
        for i in range(E):
            src[i * plan.in_frame_bytes:(i + 1) * plan.in_frame_bytes] = np.roll(one, 4 * i)
        for _ in range(2):
            plan.run_host_ptr(hin, hout, E)
        barrier()
        n_e2e = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            plan.run_host_ptr(hin, hout, E)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        te = torch.tensor([dt], dtype=torch.float64, device=dev)
        if dist:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": world * E * n_e2e * MPIX_PER_FRAME / float(te.item()), "unit": "Mpixels/s",
               "h2d_bytes_per_step": E * plan.in_frame_bytes, "d2h_bytes_per_step": E * plan.out_frame_bytes,
               "frames_per_step": E, "steps": n_e2e, "host_memory": "pinned (vb200_host_alloc)",
               "api": "vb200_thumbnail_batch_host" + (" (plan with vb200_thumbnail_plan_set_sharpen)" if PIPELINE else ""),
               "numa_node": node}
    if affinity0:
        os.sched_setaffinity(0, affinity0)  # the CPU baseline below gets every core back
    if hin:
        L.vb200_host_free(hin)
    if hout:
        L.vb200_host_free(hout)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # in a child process: the reference arm forks workers, which a process that holds a CUDA context should not
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1",
                                "--workload", args.workload], capture_output=True, text=True, timeout=900)
            cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as e:  # the baseline is a reported number, never a reason to lose the bench line
            cpu = {"value": None, "unit": "Mpixels/s", "cores": host_threads(), "kind": "port", "sample": "failed: %r" % (e,)}

    if rank == 0:
        line = {
            "metric": ("" if parity == "ok" else "UNVERIFIED (pixels differ from the oracle) ") + (METRIC_PIPELINE if PIPELINE else METRIC),
            "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "parity": parity, "lib": vb.library_path(),
            "config": {"workload": (WORKLOAD_PIPELINE if PIPELINE else WORKLOAD) + ("" if args.alpha == "random" else ", alpha band 255 everywhere"),
                       "alpha": args.alpha, "frames_per_gpu": F, "frame": "4096x4096x4 u8",
                       "output": "512x512x4 u8", "l2": "inputs (%.1f GiB per GPU) larger than L2" % (F * plan.in_frame_bytes / 2**30),
                       "sharding": "independent frames per rank, no data-path collective"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": DRAM_BYTES_PER_FRAME * F, "traffic_source": DRAM_SOURCE, "peak_source": peak_src,
                         "kernel": plan.kernel, "bytes_per_launch": bytes_per_launch, "kernel_ms": kern_ms, "kernels": kernels},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        }
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

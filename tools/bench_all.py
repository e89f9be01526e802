"""Times every pipeline of SURVEY.md §8a through the C ABI on device-resident synthetic frames (CUDA events, L2-rotating
buffer sets) and the CPU oracle beside it on a bounded sample; prints one JSON line per pipeline with the HBM / FP32
roofline fraction from the algorithmic bytes / flops of SURVEY.md §8d.   python tools/bench_all.py [--quick]"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from halide_b200 import HalideBuffer, filters  # noqa: E402
from oracle import pyoracle  # noqa: E402

M3200 = [[1.6697, -0.2693, -0.4004, -42.4346], [-0.3576, 1.0615, 1.5949, -37.1158], [-0.2175, -1.8751, 6.9640, -26.6970]]
M7000 = [[2.2997, -0.4478, 0.1706, -39.0923], [-0.3826, 1.5906, -0.2080, -25.4311], [-0.0888, -0.7344, 2.2832, -20.0826]]


def peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0


def u16(shape, dev, g):
    return torch.randint(-32768, 32768, shape, dtype=torch.int16, device=dev, generator=g).view(torch.uint16)


def gpu_info():
    """Card name, power limit and max SM clock (nvidia-smi query, read-only) and the SM count of cuda:0."""
    import subprocess
    name, power, mhz = "unknown", "unknown", 0
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.splitlines()[0]
        name, power, mhz = (v.strip() for v in q.split(","))
        power, mhz = f"{float(power):.0f} W", int(float(mhz))
    except Exception:
        pass
    return {"name": name, "power_limit": power, "max_sm_mhz": mhz or 1965,
            "sms": torch.cuda.get_device_properties(0).multi_processor_count}


LAST_KERNELS = {}


def time_gpu(make_sets, call, steps, warmup=5):
    """Mean seconds per call over `steps` calls (CUDA events), then one event-bracketed pass for the per-kernel split
    (left in LAST_KERNELS for report())."""
    import halide_b200.lib as hlib
    sets = make_sets()
    for i in range(warmup):
        call(*sets[i % len(sets)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        call(*sets[i % len(sets)])
    e1.record()
    torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) / steps * 1e-3
    hlib.profile(True)
    hlib.profile_reset()
    reps = 3
    for i in range(reps):
        call(*sets[i % len(sets)])
    torch.cuda.synchronize()
    rep = hlib.profile_report()
    hlib.profile(False)
    LAST_KERNELS.clear()
    LAST_KERNELS.update({k: {"launches": c / reps, "us": ms / reps * 1e3} for k, (c, ms) in rep.items()})
    return dt


def main():
    quick = "--quick" in sys.argv
    only = sys.argv[sys.argv.index("--only") + 1].split(",") if "--only" in sys.argv else None
    want = lambda name: only is None or name in only
    if os.environ.get("BENCH_ALL_VARIANT"):   # A/B: route stencil_chain / nl_means through the chosen kernel variant (hooks)
        import halide_b200
        _l = halide_b200.load_library()
        _l.halide_b200_stencil_chain_variant(int(os.environ["BENCH_ALL_VARIANT"]))
        _l.halide_b200_nl_means_variant(int(os.environ["BENCH_ALL_VARIANT"]))
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    pk = peak()
    pyoracle.set_threads(min(16, pyoracle.use_all_cores()))
    rows = []

    def report(name, workload, px, alg_bytes, t_gpu, t_cpu, cpu_sample, bound="hbm", flops=None, note=""):
        line = {"pipeline": name, "workload": workload, "us_per_call": t_gpu * 1e6, "Mpixels_per_s": px / 1e6 / t_gpu,
                "algorithmic_bytes": alg_bytes, "achieved_GBps": alg_bytes / t_gpu / 1e9, "hbm_frac_of_measured": alg_bytes / t_gpu / 1e9 / pk,
                "bound": bound, "cpu_oracle_ms": t_cpu * 1e3, "cpu_sample": cpu_sample, "cpu_threads": pyoracle.num_threads(), "note": note,
                "kernels": dict(LAST_KERNELS)}
        if flops:
            line["achieved_TFLOPs"] = flops / t_gpu / 1e12
        rows.append(line)
        print(json.dumps(line), flush=True)

    def cpu_time(fn, reps=2):
        fn()
        t = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            t.append(time.perf_counter() - t0)
        return min(t)

    nsets = 4
    if want("blur"):  # ---- blur, config 1: 1920x1080 u16 (+ an 8K frame so the kernel is not launch-bound)
        for (W, H) in [(1920, 1080), (7680, 4320)]:
            def mk():
                return [(HalideBuffer.from_torch(u16((H + 2, W + 2), dev, g)), HalideBuffer.from_torch(torch.zeros((H, W), dtype=torch.uint16, device=dev)))
                        for _ in range(nsets * (8 if W < 4000 else 1))]
            t = time_gpu(mk, filters.halide_blur, 200 if W < 4000 else 50)
            a = np.random.default_rng(0).integers(0, 65536, (H + 2, W + 2), dtype=np.uint16)
            report("blur", f"{W}x{H} u16", W * H, 4 * W * H, t, cpu_time(lambda: pyoracle.blur(a)), "full frame")
    if want("bilateral_grid"):  # ---- bilateral_grid, config 3: 7680x4320 f32
        W, H = (7680, 4320)
        def mk():
            return [(HalideBuffer.from_torch(torch.rand((H, W), dtype=torch.float32, device=dev, generator=g)),
                     HalideBuffer.from_torch(torch.zeros((H, W), dtype=torch.float32, device=dev))) for _ in range(2)]
        t = time_gpu(mk, lambda i, o: filters.bilateral_grid(i, 0.1, o), 20)
        a = np.random.default_rng(0).random((H // 4, W), dtype=np.float32)
        report("bilateral_grid", f"{W}x{H} f32 r_sigma=0.1", W * H, 8 * W * H, t, cpu_time(lambda: pyoracle.bilateral_grid(a, 0.1)) * 4, "1/4 of the frame x4")
    if want("nl_means"):  # ---- nl_means, config 4 (single GPU here): 3840x2160x3 f32, patch 3 / search 7
        W, H = (3840, 2160)
        def mk():
            return [(HalideBuffer.from_torch(torch.rand((3, H, W), dtype=torch.float32, device=dev, generator=g)),
                     HalideBuffer.from_torch(torch.zeros((3, H, W), dtype=torch.float32, device=dev))) for _ in range(2)]
        t = time_gpu(mk, lambda i, o: filters.nl_means(i, 3, 7, 0.12, o), 5 if quick else 10)
        a = np.random.default_rng(0).random((3, 64, W // 8), dtype=np.float32)
        scale = (H / 64) * 8
        report("nl_means", f"{W}x{H}x3 f32 patch 3 search 7", W * H, 24 * W * H, t, cpu_time(lambda: pyoracle.nl_means(a, 3, 7, 0.12), 1) * scale,
               "480x64 crop scaled by area", bound="fp32", flops=W * H * 49 * (9 * 8 + 30.0))
    if want("stencil_chain"):  # ---- stencil_chain: harness frame 1536x2560 u16
        W, H = (1536, 2560)
        def mk():
            return [(HalideBuffer.from_torch(u16((H, W), dev, g)), HalideBuffer.from_torch(torch.zeros((H, W), dtype=torch.uint16, device=dev)))
                    for _ in range(nsets)]
        t = time_gpu(mk, filters.stencil_chain, 20)
        a = np.random.default_rng(0).integers(0, 65536, (H // 4, W), dtype=np.uint16)
        report("stencil_chain", f"{W}x{H} u16, 32 stages", W * H, 4 * W * H, t, cpu_time(lambda: pyoracle.stencil_chain(a)) * 4, "1/4 of the frame x4",
               bound="int-alu", note="800 MAC/px in the reference formulation (320 after the exact separable rewrite)")
    if want("camera_pipe"):  # ---- camera_pipe: harness frame 2592x1968 raw -> 2560x1920x3
        W, H = (2560, 1920)
        m32 = torch.tensor(M3200, dtype=torch.float32, device=dev)
        m70 = torch.tensor(M7000, dtype=torch.float32, device=dev)
        b32, b70 = HalideBuffer.from_torch(m32), HalideBuffer.from_torch(m70)
        def mk():
            return [(HalideBuffer.from_torch(torch.randint(0, 1024, (H + 48, W + 32), dtype=torch.int16, device=dev, generator=g).view(torch.uint16)),
                     HalideBuffer.from_torch(torch.zeros((3, H, W), dtype=torch.uint8, device=dev))) for _ in range(nsets * 2)]
        t = time_gpu(mk, lambda i, o: filters.camera_pipe(i, b32, b70, 3700.0, 2.0, 50.0, 1.0, 25, 1023, o), 50)
        raw = np.random.default_rng(0).integers(0, 1024, (H + 48, W + 32), dtype=np.uint16)
        t_cpu = cpu_time(lambda: pyoracle.camera_pipe(raw, np.array(M3200, np.float32), np.array(M7000, np.float32), 3700.0, 2.0, 50.0, 1.0, 25,
                                                        1023, (3, H, W)))
        report("camera_pipe", f"{W + 32}x{H + 48} raw -> {W}x{H}x3 u8", W * H, 5 * W * H, t, t_cpu, "full frame")
    if want("conv_layer"):  # ---- conv_layer: fixed shapes
        ti = torch.rand((5, 82, 102, 128), dtype=torch.float32, device=dev, generator=g)
        tf = torch.rand((128, 3, 3, 128), dtype=torch.float32, device=dev, generator=g)
        tb = torch.rand((128,), dtype=torch.float32, device=dev, generator=g)
        bi, bf, bb = (HalideBuffer.from_torch(x) for x in (ti, tf, tb))
        def mk():
            return [(HalideBuffer.from_torch(torch.zeros((5, 80, 100, 128), dtype=torch.float32, device=dev)),) for _ in range(2)]
        t = time_gpu(mk, lambda o: filters.conv_layer(bi, bf, bb, o), 20)
        ci, cf, cb = ti[:1].cpu().numpy(), tf.cpu().numpy(), tb.cpu().numpy()
        report("conv_layer", "N5 CI128 CO128 100x80 3x3 f32", 5 * 80 * 100, 42.5e6, t, cpu_time(lambda: pyoracle.conv_layer(ci, cf, cb), 1) * 5,
               "1 of 5 images x5", bound="tensor (tcgen05 kind::tf32, 3-term split)", flops=11.8e9)
    if want("local_laplacian"):  # ---- local_laplacian (headline; bench.py measures it with the full contract)
        for (W, H) in [(3840, 2160), (16384, 2048)] + ([] if quick else [(16384, 16384)]):
            def mk():
                return [(HalideBuffer.from_torch(u16((3, H, W), dev, g)), HalideBuffer.from_torch(torch.zeros((3, H, W), dtype=torch.uint16, device=dev)))
                        for _ in range(nsets if W * H < 1e8 else 1)]
            t = time_gpu(mk, lambda i, o: filters.local_laplacian(i, 8, 1.0 / 7.0, 1.0, o), 20 if W * H < 1e8 else 5)
            a = np.random.default_rng(0).integers(0, 65536, (3, 1080, 3840), dtype=np.uint16)
            report("local_laplacian", f"{W}x{H}x3 u16 levels 8", W * H, 12 * W * H, t, cpu_time(lambda: pyoracle.local_laplacian(a, 8, 1 / 7, 1.0)) * (W * H / (3840 * 1080)),
                   "3840x1080 band scaled by area")
    if want("harris") or want("unsharp"):  # ---- harris / unsharp: the generators' estimate frame and 8K, f32
        from oracle import pyoracle_apps
        gpu = gpu_info()
        # f32 flops per output pixel from the generators' expressions (apron recomputation not counted)
        fl_gray = 3 + 2                                      # 3 mul, 2 add
        fl_harris = (fl_gray + 2 * 11 + 3                    # gray; Ix, Iy: 6 mul + 5 add each; Ixx, Iyy, Ixy
                     + 3 * 8 + 3 + 1 + 3)                    # three 9-term sums; det; trace; det - 0.04 trace^2
        fl_unsharp = (fl_gray + 2 * 10                       # gray; blur_y, blur_x: 4 mul + 6 add each
                      + 2 + 1 + 3)                           # sharpen; ratio (one divide); ratio * input for 3 channels
        fp32_peak = gpu["sms"] * 128 * 2 * gpu["max_sm_mhz"] * 1e6
        for name, bpp, fpp in (("harris", 16, fl_harris), ("unsharp", 24, fl_unsharp)):
            if not want(name):
                continue
            for (W, H) in [(1536, 2560), (7680, 4320)]:
                fn = getattr(filters, name)
                # enough buffer sets that one rotation exceeds the 126 MB L2
                sets = max(2, int(np.ceil(4 * 126e6 / (bpp * W * H))))
                def mk():
                    out_shape = (H, W) if name == "harris" else (3, H, W)
                    ins = (3, H + 6, W + 6) if name == "harris" else (3, H, W)
                    res = []
                    for _ in range(sets):
                        bo = HalideBuffer.from_torch(torch.zeros(out_shape, dtype=torch.float32, device=dev),
                                                     mins=(3, 3) if name == "harris" else None)
                        res.append((HalideBuffer.from_torch(torch.rand(ins, dtype=torch.float32, device=dev, generator=g)), bo))
                    return res
                t = time_gpu(mk, fn, 200 if W < 4000 else 50)
                frac = 1 if W < 4000 else 4
                pad = 6 if name == "harris" else 0
                a = np.random.default_rng(0).random((3, H // frac + pad, W + pad), dtype=np.float32)
                t_cpu = cpu_time(lambda: getattr(pyoracle_apps, name)(a)) * frac
                bound = "hbm" if bpp / (pk * 1e9) >= fpp / fp32_peak else "fp32"
                report(name, f"{W + 6}x{H + 6}x3 f32 -> {W}x{H} at (3,3)" if name == "harris" else f"{W}x{H}x3 f32", W * H, bpp * W * H, t,
                       t_cpu, "full frame" if frac == 1 else "1/4 of the frame x4", bound=bound, flops=fpp * W * H,
                       note=f"{fpp} flop/px, {bpp} B/px; {sets} buffer sets; fp32 peak {fp32_peak / 1e12:.1f} TFLOP/s from "
                            f"{gpu['sms']} SMs at {gpu['max_sm_mhz']} MHz; {gpu['name']}, power limit {gpu['power_limit']}")
                rows[-1]["fp32_frac"] = fpp * W * H / t / fp32_peak
    json.dump(rows, open(os.path.join(ROOT, "gpurun_out", "bench_all.json"), "w"), indent=1)


if __name__ == "__main__":
    main()

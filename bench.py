"""bench.py -- samples/s of the OccFormer hot path (6-cam 256x704 -> 200x200x16 voxel forward) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" = one connected pass of the hot path (SURVEY.md section 8: ViewTransformerLiftSplatShootVoxel.forward (lift-splat
voxel pooling) -> OccupancyEncoder.forward -> MSDeformAttnPixelDecoder3D.forward -> Mask2FormerNuscOccHead.simple_test,
every module built from the registry and called through its own forward) over one batch of synthetic samples per GPU,
BASELINE.json configs[2] shapes (nuScenes R50: 6 cameras, 16x44 feature maps, D=112, C=128 -> 200x200x16 voxels, 100
queries, 17 classes).  Data parallel over samples, no collective on the data path (weak scaling: fixed batch per GPU).

One JSON line on stdout (rank 0).  `value` = inputs resident in HBM, CUDA-event timed, L2 flushed between steps;
`e2e` = the same metric with pinned HOST inputs copied H2D, the per-voxel class labels (uint8) copied D2H and -- for N > 1
-- the metric all-gather inside the timed region; `roofline` = the dominant kernel, `roofline_extra` = window attention and
voxel pooling (the two kernels BASELINE.json's metric names), all timed live with CUDA events;
`cpu_baseline` = the CPU oracle (port of the reference's PyTorch path) on the host cores, bounded sample, per segment.
`--impl reference` times that CPU path alone (the reference itself is Python under mmcv and cannot travel to the GPU
box; see DESIGN.md).

`--dump-outputs DIR` writes what the timed path returned in its last timed step as .npy files, so that two builds
can be compared output for output (inputs and weights are seeded: the same arguments give the same inputs):
  voxel_index.npy    (n,)    float64, flat indices into the (batch, X, Y, Z) output grid, sorted
  output_voxels.npy  (n, K)  float32, class logits of ``output_voxels`` at those voxels
  output_labels.npy  (n,)    float32, ``output_labels`` (argmax class) at those voxels
n is every voxel when the three arrays fit in 48 MB, else a fixed seeded sample of that size.
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

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "samples/sec (6-cam->200x200x16 voxel fwd)"
UNIT = "samples/s"
DOWNSAMPLE, C_TRANS = 16, 128
PLANES, NUMS, STRIDES = [128, 256, 512, 1024], [2, 2, 2, 2], [1, 2, 2, 2]
EMBED, QUERIES, DEC_LAYERS, HEADS = 192, 100, 9, 6
# the workload (occformer_b200.synth.WORKLOADS): default = BASELINE.json configs[2], the configuration the metric is quoted
# on; --workload kitti = configs[1] (its own metric string says so)
WL = "nusc_200"
WORKLOAD = "nusc_r50_6cam_256x704_to_200x200x16"
N_CAMS, INPUT_SIZE, CLASSES, GRID = 6, (256, 704), 17, "nusc_200"
PC_RANGE = [-40.0, -40.0, -1.0, 40.0, 40.0, 5.4]
OCC_SIZE = [200, 200, 16]
HEAD_TYPE = "Mask2FormerNuscOccHead"


def set_workload(name):
    global WL, WORKLOAD, N_CAMS, INPUT_SIZE, CLASSES, GRID, PC_RANGE, OCC_SIZE, HEAD_TYPE, METRIC
    from occformer_b200 import synth
    w = synth.WORKLOADS[name]
    WL, WORKLOAD, N_CAMS, INPUT_SIZE, CLASSES, GRID = name, w["name"], w["cams"], tuple(w["input_size"]), w["classes"], w["grid"]
    PC_RANGE, OCC_SIZE, HEAD_TYPE = list(w["pc"]), list(w["occ"]), w["head"]
    if name != "nusc_200":
        METRIC = f"samples/sec ({w['name']} voxel fwd)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi in a side thread during the timed region)
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
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
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        # median over the busy samples (upper half): the sampler also sees the idle gaps between steps
        busy = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------------
# workload construction
# ----------------------------------------------------------------------------------------------------------------------
NECK = dict(strides=[2, 4, 8, 16], layers=6, heads=8, levels=3, points=4, ffn=4 * EMBED)
STAGES_ALL = ["view_transformer(lift_splat)", "occupancy_encoder", "msdeform_pixel_decoder_3d", "mask2former_head.simple_test"]


class PassThroughDepthNet(torch.nn.Module):
    """The step starts from post-DepthNet maps on both arms (image backbone + DepthNet are cuDNN-class work in front of
    the hot path, SURVEY.md 8(f)3): ``depth_net(x, mlp_input)`` hands its input through."""

    def forward(self, x, mlp_input=None):
        return x


def build_b200(dev):
    """The registered modules of the B200 path, built through the registries from config-style dicts, with deterministic
    synthetic weights (occformer_b200.synth; the oracle is not imported on this leg)."""
    from occformer_b200 import BACKBONES, HEADS as HEAD_REG, NECKS, synth
    from occformer_b200.head import head_cfg
    from occformer_b200.neck import neck_cfg
    gc = synth.grid_config(GRID)
    vt = NECKS.build(dict(type="ViewTransformerLiftSplatShootVoxel", loss_depth_weight=1.0, grid_config=gc,
                          data_config={"input_size": INPUT_SIZE}, numC_input=112 + C_TRANS, numC_Trans=C_TRANS,
                          downsample=DOWNSAMPLE, depth_net=PassThroughDepthNet())).to(dev)
    enc = BACKBONES.build(dict(type="OccupancyEncoder", in_channels=C_TRANS, num_stage=4, block_numbers=NUMS,
                               block_inplanes=PLANES, block_strides=STRIDES, out_indices=(0, 1, 2, 3),
                               norm_cfg=dict(type="GN", num_groups=32, requires_grad=True), with_cp=True))
    enc.load_state_dict(synth.make_encoder_state(C_TRANS, PLANES, NUMS, STRIDES, seed=0), strict=True)
    neck = NECKS.build(dict(type="MSDeformAttnPixelDecoder3D", **neck_cfg(PLANES, NECK["strides"], EMBED, NECK["layers"],
                                                                          NECK["heads"], NECK["levels"], NECK["points"],
                                                                          NECK["ffn"])))
    neck.load_state_dict(synth.make_neck_state(PLANES, EMBED, NECK["layers"], NECK["heads"], NECK["levels"], NECK["points"],
                                               NECK["ffn"], seed=2), strict=True)
    head = HEAD_REG.build(dict(type=HEAD_TYPE, **head_cfg(EMBED, QUERIES, CLASSES, DEC_LAYERS, HEADS, PC_RANGE)))
    head.load_state_dict(synth.make_head_state(EMBED, QUERIES, CLASSES, DEC_LAYERS, 3, seed=1), strict=True)
    return vt, enc.to(dev).eval(), neck.to(dev).eval(), head.to(dev).eval()


def host_inputs(batch, seed):
    """Pinned host tensors of one step: post-DepthNet maps (B, N, D+C, fH, fW) + the camera matrices."""
    from occformer_b200 import synth
    fH, fW = INPUT_SIZE[0] // DOWNSAMPLE, INPUT_SIZE[1] // DOWNSAMPLE
    D = 112
    dd, feat = synth.lift_inputs(batch, N_CAMS, D, fH, fW, C_TRANS, seed=seed)
    x = torch.cat([dd, feat], dim=1).view(batch, N_CAMS, D + C_TRANS, fH, fW).contiguous()
    cams = synth.workload_cameras(WL, batch)
    out = {"x": x, **cams}
    return {k: (v.pin_memory() if torch.cuda.is_available() else v) for k, v in out.items()}


class Pipeline:
    """One step = the registered modules' own ``forward`` calls, in the order the reference detector issues them
    (OccupancyFormer.extract_img_feat / simple_test, occupancyformer.py:77-80,115-123,211-217)."""

    def __init__(self, dev, batch):
        self.dev, self.batch = dev, batch
        self.vt, self.enc, self.neck, self.head = build_b200(dev)
        self.metas = [dict(occ_size=OCC_SIZE, pc_range=PC_RANGE)] * batch
        self.labels = None

    def stages(self):
        return list(STAGES_ALL)

    @torch.no_grad()
    def run(self, inp):
        mats = [inp[k] for k in ("rots", "trans", "intrins", "post_rots", "post_trans", "bda")]
        voxel, _ = self.vt([inp["x"]] + mats + [None])           # ViewTransformerLiftSplatShootVoxel.forward(input)
        feats = self.enc(voxel)                                   # OccupancyEncoder.forward(x) -> 4 levels
        feats = self.neck(feats)                                  # MSDeformAttnPixelDecoder3D.forward(feats)
        res = self.head.simple_test(feats, self.metas)            # Mask2FormerNuscOccHead.simple_test
        self.labels = res["output_labels"]
        return res["output_voxels"][0]


# ----------------------------------------------------------------------------------------------------------------------
# CPU oracle leg (cpu_baseline / --impl reference)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_sample(threads):
    """One sample of the same connected workload through the CPU oracle (port of the reference's PyTorch path), with a
    timer per segment (BASELINE.md section 2: pooling / encoder / neck / head)."""
    from occformer_b200 import synth
    from oracle import port
    torch.set_num_threads(threads)
    gc = synth.grid_config(GRID)
    frustum = port.create_frustum(INPUT_SIZE, DOWNSAMPLE, gc["dbound"])
    cams = synth.workload_cameras(WL, 1)
    D, fH, fW = frustum.shape[:3]
    dd, feat = synth.lift_inputs(1, N_CAMS, D, fH, fW, C_TRANS, seed=0)
    dx, bx, nx = port.gen_dx_bx(gc["xbound"], gc["ybound"], gc["zbound"])
    sd_e = synth.make_encoder_state(C_TRANS, PLANES, NUMS, STRIDES, seed=0)
    sd_n = synth.make_neck_state(PLANES, EMBED, NECK["layers"], NECK["heads"], NECK["levels"], NECK["points"], NECK["ffn"], seed=2)
    sd_h = synth.make_head_state(EMBED, QUERIES, CLASSES, DEC_LAYERS, 3, seed=1)

    def step():
        seg = {}
        with torch.no_grad():
            t0 = time.perf_counter()
            geom = port.get_geometry(frustum, **cams)
            vol, _ = port.lift(dd, feat, 1, N_CAMS)
            grid, _, _ = port.voxel_pooling(geom, vol, dx, bx, nx)
            del vol
            t1 = time.perf_counter()
            outs = port.occupancy_encoder(grid, sd_e, NUMS, STRIDES, (0, 1, 2, 3))
            t2 = time.perf_counter()
            feats = port.ms_deform_pixel_decoder_3d(outs, sd_n, NECK["strides"], NECK["heads"], NECK["layers"], NECK["levels"],
                                                    NECK["points"])
            t3 = time.perf_counter()
            res = port.head_simple_test(feats, sd_h, HEADS, DEC_LAYERS, OCC_SIZE)
            t4 = time.perf_counter()
        seg.update(voxel_pooling_s=t1 - t0, occupancy_encoder_s=t2 - t1, pixel_decoder_s=t3 - t2, head_simple_test_s=t4 - t3,
                   total_s=t4 - t0)
        return res["output_voxels"][0], seg

    return step


PASSES = 3  # tensor-core passes per contraction of the b200 arm (--precision)


def cpu_threads():
    """Host threads for the CPU oracle: all cores up to 32 -- beyond that torch's fp32 conv / GEMM paths slow down on
    this workload (measured on the 128-core GPU box: 103 s with 128 threads), so this is the reference's best case."""
    return int(os.environ.get("OCC_CPU_THREADS", min(os.cpu_count() or 1, 32)))


def cpu_measure(threads, max_timed, budget_s):
    """1 warm-up + up to max_timed timed samples inside budget_s (exactly max_timed when budget_s is None); returns (median
    seconds per sample, per-segment medians, k)."""
    step = cpu_sample(threads)
    t0 = time.perf_counter()
    _, seg0 = step()
    est = time.perf_counter() - t0
    k = max_timed if budget_s is None else max(1, min(max_timed, int(budget_s / max(est, 1e-3))))
    segs = []
    for _ in range(k):
        _, sg = step()
        segs.append(sg)
    med = lambda key: sorted(sg[key] for sg in segs)[len(segs) // 2]  # noqa: E731
    return med("total_s"), {key: med(key) for key in segs[0]}, k, est


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = cpu_threads()
    per, seg, k, warm = cpu_measure(threads, args.steps, None)
    val = 1.0 / per
    sample = (f"1 sample/step of {WORKLOAD} (connected: {', '.join(STAGES_ALL)}) through the CPU oracle port, fp32, "
              f"{threads} threads of {os.cpu_count()} cores; 1 warm-up ({warm:.1f} s) + median of {k} timed steps")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": k,
            "warmup": 1, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": 1, "stages": STAGES_ALL},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                             "segments_s": seg},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# B200 leg
# ----------------------------------------------------------------------------------------------------------------------
def _time_cuda(fn, dev, iters=5, warm=3, flush=None):
    ts = []
    for i in range(warm + iters):
        if flush is not None:
            flush.fill_(float(i))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        if i >= warm:
            ts.append(a.elapsed_time(b))
    return sum(ts) / len(ts)


def rooflines(pipe, dev, peak):
    """Rooflines of the dominant kernel and of the two kernels BASELINE.json's metric names (window attention: tensor
    pipe; voxel pooling: HBM), each timed live with CUDA events on the current stream, L2 flushed before every launch.
    Algorithmic work per launch = SURVEY.md 8(d) per-unit figures x units per launch (DESIGN.md section 2)."""
    from occformer_b200 import ops, synth
    B = pipe.batch
    C = 128
    X, Y, Z = pipe.vt.grid_size()
    flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    # ---- 1. Conv3d 3x3x3, C = 128, stage-0 grid: the largest FLOP item of the step
    x = ops.to_split(torch.randn(B, X, Y, Z, C, device=dev))
    w2, ks = ops.repack_conv_weight(torch.randn(C, C, 3, 3, 3) * 0.02)
    w2 = w2.to(dev)
    stats = torch.zeros(B, 32, 2, dtype=torch.float64, device=dev)
    ms = _time_cuda(lambda: ops.conv(x, w2, ks, gn_stats=stats, cpg=4), dev, flush=flush)
    flops = 2.0 * 27 * C * C * B * X * Y * Z
    ach = flops / (ms * 1e-3) / 1e12
    conv = {"kernel": f"gemm_bf16x3_kernel<conv3d 3x3x3, C=128, {X}x{Y}x{Z}>", "bound": "tensor", "achieved": ach,
            "peak": peak["tf"], "unit": "TFLOP/s", "frac": ach / peak["tf"], "traffic": None, "passes": PASSES,
            "frac_of_3pass_ceiling": PASSES * ach / peak["tf"], "ms_per_launch": ms,
            "peak_src": f"bf16 dense burst, {peak['src']}",
            "note": f"algorithmic (fp32-problem) FLOPs 2*27*Cin*Cout*V = {flops / 1e9:.1f} GF per launch; the kernel executes "
                    f"3 bf16 tensor-core passes per algorithmic FLOP (split-bf16 operands, fp32-faithful), so its ceiling is "
                    f"peak/3 = {peak['tf'] / 3:.0f} TF/s algorithmic; algorithmic bytes = {2 * B * X * Y * Z * C * 4 / 1e6:.0f} MB"}
    del x
    # ---- 2. window attention core (A7/A8), stage-0 tokens
    heads = C // 32
    rows = B * X * Y * (Z + 1)
    qkv = ops.to_split(torch.randn(rows, 3 * C, device=dev))
    qb = ops.split_weight(torch.randn(1, 3 * C) * 0.1).view(-1).to(dev)
    bias_pad = torch.randn(heads, 2404, device=dev) * 0.1
    ms = _time_cuda(lambda: ops.window_attention(qkv, qb, bias_pad, B, X, Y, Z, C, heads, True, head_major=True), dev, flush=flush)
    nwin = B * (Z + 1) * ((X + 6) // 7) * ((Y + 6) // 7)
    fl = nwin * 4.0 * 49 * 49 * C  # QK^T + PV per window, all heads (SURVEY 8(d): 4*49^2*C)
    by = rows * 4.0 * C * 4       # qkv read + out write
    wattn = {"kernel": f"window_attn_tc_kernel (stage 0, {X}x{Y}x({Z}+1) images)", "bound": "hbm",
             "achieved": by / (ms * 1e-3) / 1e9, "peak": peak["hbm"], "unit": "GB/s", "frac": by / (ms * 1e-3) / 1e9 / peak["hbm"],
             "traffic": None, "ms_per_launch": ms, "algorithmic_tflops": fl / (ms * 1e-3) / 1e12,
             "tensor_frac_algorithmic": fl / (ms * 1e-3) / 1e12 / peak["tf"], "peak_src": peak["src"],
             "note": f"unfused attention core: rows*(3C+C)*4 = {by / 1e9:.2f} GB in/out per launch bound it by HBM; "
                     f"algorithmic QK^T+PV = {fl / 1e9:.1f} GF; tensor-pipe % from ncu: profiles/"}
    del qkv
    # ---- 2b. the kernel the pipeline runs at stage 0: QKV projection + shifted-window attention fused (swin_attn_fused.cu)
    tokn_wl = ops.to_window_layout(ops.to_split(torch.randn(rows, C, device=dev)), B, X, Y, Z, True)
    wq = ops.split_weight(torch.randn(3 * C, C) * C ** -0.5).to(dev)
    bq = torch.randn(3 * C, device=dev) * 0.1
    ms_f = _time_cuda(lambda: ops.swin_qkv_attention(tokn_wl, wq, bq, bias_pad, B, X, Y, Z, C, heads, True), dev, flush=flush)
    fl_f = 2.0 * rows * C * 3 * C + fl          # QKV projection of every token + QK^T + PV per window
    by_f = tokn_wl.numel() * 4.0 + rows * C * 4.0
    ach_f = fl_f / (ms_f * 1e-3) / 1e12
    fused_attn = {"kernel": f"swin_qkv_attn_kernel (stage 0, {X}x{Y}x({Z}+1) images: QKV projection + window attention)", "bound": "tensor",
             "achieved": ach_f, "peak": peak["tf"], "unit": "TFLOP/s", "frac": ach_f / peak["tf"], "passes": PASSES,
             "frac_of_3pass_ceiling": PASSES * ach_f / peak["tf"], "traffic": None, "ms_per_launch": ms_f,
             "hbm_GBps": by_f / (ms_f * 1e-3) / 1e9, "peak_src": f"bf16 dense burst, {peak['src']}",
             "note": f"algorithmic FLOPs 2*rows*C*3C + nwin*4*49^2*C = {fl_f / 1e9:.1f} GF per launch (real tokens only: the kernel "
                     f"pads 98 -> 128 rows per window pair, 1.31x executed); ncu tensor-pipe active 48 % "
                     f"(profiles/r02_ncu_swin_qkv_attn_v7.md); bytes = window-layout tokens in + attention out = {by_f / 1e9:.2f} GB"}
    del tokn_wl
    # ---- 2c. Conv3d 3x3x3 of stage 1 (C = 256, half-resolution grid): the <256, 4, 1> instantiation
    X1, Y1, Z1 = X // 2, Y // 2, Z // 2
    x1 = ops.to_split(torch.randn(B, X1, Y1, Z1, 256, device=dev) * 0.5)
    w21, ks1 = ops.repack_conv_weight(torch.randn(256, 256, 3, 3, 3) * 0.02)
    w21 = w21.to(dev)
    st1 = torch.zeros(B, 32, 2, dtype=torch.float64, device=dev)
    ms_1 = _time_cuda(lambda: ops.conv(x1, w21, ks1, gn_stats=st1, cpg=8), dev, flush=flush)
    fl_1 = 2.0 * 27 * 256 * 256 * B * X1 * Y1 * Z1
    ach_1 = fl_1 / (ms_1 * 1e-3) / 1e12
    conv256 = {"kernel": f"gemm_bf16x3_kernel<256, 4, 1> (conv3d 3x3x3, C=256, {X1}x{Y1}x{Z1})", "bound": "tensor", "achieved": ach_1,
               "peak": peak["tf"], "unit": "TFLOP/s", "frac": ach_1 / peak["tf"], "passes": PASSES,
               "frac_of_3pass_ceiling": PASSES * ach_1 / peak["tf"], "traffic": None, "ms_per_launch": ms_1,
               "peak_src": f"bf16 dense burst, {peak['src']}",
               "note": f"algorithmic FLOPs 2*27*256*256*V = {fl_1 / 1e9:.1f} GF per launch"}
    del x1
    # ---- 3. voxel pooling (fused lift-splat), with and without the prologue (depth softmax, NCHW->NHWC, geometry)
    gc = synth.grid_config(GRID)
    fH, fW = INPUT_SIZE[0] // DOWNSAMPLE, INPUT_SIZE[1] // DOWNSAMPLE
    dd, feat = synth.lift_inputs(B, N_CAMS, 112, fH, fW, C_TRANS, seed=0)
    dd, feat = dd.to(dev), feat.to(dev)
    cams = {k: v.to(dev) for k, v in synth.workload_cameras(WL, B).items()}
    vt = pipe.vt
    dxbx = vt._host_params()
    geom = vt.get_geometry(**cams)
    prob, feat_cl = ops.lift_prologue(dd, feat)
    BN = B * N_CAMS
    dd4, feat4 = dd.view(BN, 112, fH, fW), feat.view(BN, C_TRANS, fH, fW)
    cam_args = [cams[k] for k in ("rots", "trans", "intrins", "post_rots", "post_trans", "bda")]

    def fused(twin):  # the shipped call (occ_lift_splat_fused: memset + lift_front_kernel + vp_pool_kernel)
        return ops.lift_splat_fused(dd4, feat4, vt.frustum.data, *cam_args, B, N_CAMS, *dxbx, vt.grid_size(), with_split=twin)

    ms_f32 = _time_cuda(lambda: fused(False), dev, flush=flush)
    ms_twin = _time_cuda(lambda: fused(True), dev, flush=flush)
    ms_pool = _time_cuda(lambda: ops.lift_splat(prob, feat_cl, geom, B, N_CAMS, *dxbx, vt.grid_size(), with_split=False), dev, flush=flush)
    npts = B * N_CAMS * 112 * fH * fW
    V = B * X * Y * Z
    grid_b = V * C_TRANS * 4
    by = npts * 4 + B * N_CAMS * fH * fW * C_TRANS * 4 + grid_b          # SURVEY 8(d) fused-lift formula, geometry recomputed (0)
    by_pool = by + npts * 12                                              # the same with a materialised geometry tensor
    gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9                   # noqa: E731
    pool = {"kernel": f"occ_lift_splat_fused = memset + lift_front_kernel (depth softmax, NHWC transpose, geometry, voxel index, "
                      f"lists) + vp_pool_kernel ({N_CAMS} cams -> {X}x{Y}x{Z}), fp32 grid only", "bound": "hbm",
            "achieved": gbs(by, ms_f32), "peak": peak["hbm"], "unit": "GB/s", "frac": gbs(by, ms_f32) / peak["hbm"],
            "traffic": None, "ms_per_launch": ms_f32,
            "shipped_with_s32_twin": {"ms": ms_twin, "bytes": by + grid_b, "achieved": gbs(by + grid_b, ms_twin),
                                      "frac": gbs(by + grid_b, ms_twin) / peak["hbm"],
                                      "frac_algorithmic_bytes_only": gbs(by, ms_twin) / peak["hbm"]},
            "index_and_pool_kernels_only": {"ms": ms_pool, "bytes": by_pool, "achieved": gbs(by_pool, ms_pool),
                                            "frac": gbs(by_pool, ms_pool) / peak["hbm"]},
            "peak_src": peak["src"],
            "note": f"algorithmic bytes n_pts*4 + N*fH*fW*C*4 + (geometry recomputed in the kernel: 0) + V*C*4 = {by / 1e6:.0f} MB per "
                    f"launch, all three launches of the call timed together; the pipeline's call also writes the S32 twin of the grid "
                    f"({grid_b / 1e6:.0f} MB, operand of the encoder's first conv): 'shipped_with_s32_twin' counts those bytes as traffic; "
                    f"'index_and_pool_kernels_only' = vp_index_geom + vp_pool on a materialised geometry tensor (+ n_pts*12 bytes)"}
    return conv, {"window_attn": wattn, "swin_qkv_attn_fused": fused_attn, "conv_c256": conv256, "voxel_pool": pool}


DUMP_BYTES = 48 * 1000 * 1000


def sample_outputs(voxels, labels):
    """Host copies of one step's outputs for --dump-outputs (module docstring): voxels (B, K, X, Y, Z) float32 and
    labels (B, X, Y, Z) at every voxel, or at a fixed seeded sample of voxels when that would exceed DUMP_BYTES."""
    B, K = voxels.shape[:2]
    nvox = labels.numel()
    n = min(nvox, DUMP_BYTES // (8 + 4 * K + 4))
    if n == nvox:
        idx = torch.arange(nvox)
    else:
        idx = torch.randperm(nvox, generator=torch.Generator().manual_seed(0))[:n].sort().values
    d = idx.to(voxels.device)
    per_b = nvox // B
    vox = voxels.reshape(B, K, per_b)[d // per_b, :, d % per_b]  # (n, K)
    return {"voxel_index": idx.double().numpy(),
            "output_voxels": vox.float().cpu().numpy(),
            "output_labels": labels.reshape(-1)[d].float().cpu().numpy()}


def run_b200(args, rank, world, local_rank):
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    from occformer_b200 import dist_eval, ops
    global PASSES
    if args.precision == "bf16":
        ops.set_precision("bf16")
        PASSES = 1
    peak = peaks()
    pipe = Pipeline(dev, args.batch)
    host = host_inputs(args.batch, seed=0)
    resident = {k: v.to(dev) for k, v in host.items()}
    flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    g = torch.Generator().manual_seed(1234 + rank)
    gt = torch.randint(0, CLASSES, (args.batch, *OCC_SIZE), generator=g).to(torch.uint8).to(dev)  # synthetic ground truth
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- value: inputs resident in HBM
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # nvidia-smi needs ~1 s to deliver its first sample: start before the warm-up
    for _ in range(args.warmup):
        pipe.run(resident)
    barrier()
    # The step is a fixed sequence of kernel launches on static shapes: capture it once in a CUDA graph and replay
    # (the same kernels on the same buffers; only the CPU-side launch cost disappears).
    graph, graph_out, launches_per_step = None, None, None
    if not args.no_graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            pipe.run(resident)  # allocator warm-up on the capture stream
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        l0 = ops.LAUNCH_COUNT[0]
        graph = torch.cuda.CUDAGraph()
        # capture on the stream of the warm-up above: per-stream caches of the package (window-layout token buffers, conv
        # workspaces) are then already allocated and zero-initialised outside the graph
        with torch.cuda.graph(graph, stream=side):
            graph_out = pipe.run(resident)
        launches_per_step = ops.LAUNCH_COUNT[0] - l0
        for _ in range(2):
            graph.replay()
        barrier()

    def step_resident():
        if graph is not None:
            graph.replay()
            return graph_out
        return pipe.run(resident)
    launches0 = ops.LAUNCH_COUNT[0]
    evs = []
    for i in range(args.steps):
        flush.fill_(float(i))  # L2 flush between timed iterations (untimed)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = step_resident()
        b.record()
        evs.append((a, b))
    barrier()
    launches = (launches_per_step * args.steps) if graph is not None else ops.LAUNCH_COUNT[0] - launches0
    t_dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    clocks = sampler.stop() if rank == 0 else None
    # copied now: the e2e steps below overwrite the graph's output buffers
    dump = sample_outputs(out, pipe.labels) if args.dump_outputs and rank == 0 else None

    # ---------------------------------------------------------------- e2e: host buffers in, host result out
    # every step: H2D of the step's inputs from pinned host memory, the registered modules' forward, D2H of the per-voxel
    # class labels (uint8; what the reference's evaluation loop consumes, occupancyformer.py:238-243), the evaluation
    # counts of the step (confusion-matrix kernel) and -- with more than one rank -- the path's only collective, the
    # all-gather of the packed count vector (apis/test.py:195-212), INSIDE the timed region.
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    e2e_steps = args.steps
    totals = torch.zeros(3 + 3 * CLASSES, dtype=torch.int64, device=dev)

    def step_e2e():
        if graph is not None:  # static device buffers: H2D into the graph's inputs, replay, D2H of its output
            for k, v in host.items():
                resident[k].copy_(v, non_blocking=True)
            graph.replay()
        else:
            pipe.run({k: v.to(dev, non_blocking=True) for k, v in host.items()})
        out_host.copy_(pipe.labels, non_blocking=True)
        counts = dist_eval.ssc_counts(pipe.labels, gt, CLASSES)
        totals.add_(dist_eval.reduce_counts(counts))

    out_host = torch.empty((args.batch, *OCC_SIZE), dtype=torch.uint8).pin_memory()
    for _ in range(2):
        step_e2e()
    barrier()
    totals.zero_()
    d2h = out_host.numel() * out_host.element_size()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(e2e_steps):
        step_e2e()
    b.record()
    barrier()
    t_e2e_ms = a.elapsed_time(b)

    # max over ranks
    if world > 1:
        t = torch.tensor([t_dev_ms, t_e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_dev_ms, t_e2e_ms = float(t[0]), float(t[1])
    total_samples = args.batch * world * args.steps
    value = total_samples / (t_dev_ms * 1e-3)
    e2e_val = args.batch * world * e2e_steps / (t_e2e_ms * 1e-3)
    scores = dist_eval.ssc_scores(totals.cpu(), CLASSES)
    eval_info = {"collective": (f"all_gather of {totals.numel()} int64 per rank per step (NCCL), inside the e2e timed region"
                                if world > 1 else "none (1 rank)"),
                 "voxels_scored": int(totals[3:3 + CLASSES].sum() + totals[3 + 2 * CLASSES:].sum()),
                 "iou_ssc_mean_vs_random_gt": scores["iou_ssc_mean"]}
    if rank != 0:
        return
    roof, roof_extra = rooflines(pipe, dev, peak)
    cpu = None
    if not args.no_cpu_baseline:
        threads = cpu_threads()
        per, seg, k, warm = cpu_measure(threads, 2, 100.0)
        cpu = {"value": 1.0 / per, "unit": UNIT, "cores": threads, "kind": "port", "segments_s": seg,
               "sample": f"1 sample of {WORKLOAD} (connected: {', '.join(STAGES_ALL)}) through the CPU oracle port (torch fp32, "
                         f"{threads} threads of {os.cpu_count()} cores): 1 warm-up ({warm:.1f} s) + median of {k} timed = {per:.1f} s"}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("f32 (split-bf16 hi/lo operands, 3 tensor-core passes per contraction, f32 accumulate + storage)"
                      if PASSES == 3 else
                      "bf16 operands, single tensor-core pass, f32 accumulate + storage (--precision bf16: NOT the graded "
                      "configuration -- outside the 1e-3 tolerance, no reference twin; see tests/test_gpu_bf16_mode.py)"),
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": args.batch, "global_batch": args.batch * world,
                       "parallelism": f"dp{world}", "stages": pipe.stages(),
                       "api": "registry-built modules, forward() / simple_test() of each (connected: encoder pyramid -> neck -> head)",
                       "launch": "cuda_graph_replay" if graph is not None else "eager",
                       "l2": "192 MiB flush write between timed steps; activations (328 MB/tensor) exceed L2",
                       "input": "post-DepthNet maps (depth logits + context) + camera matrices; image backbone / DepthNet are "
                                "in front of the hot path (SURVEY 8(f)3)"},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": t_e2e_ms / e2e_steps},
            "gpu_launches": launches, "roofline": roof, "roofline_extra": roof_extra, "cpu_baseline": cpu, "eval": eval_info}
    if dump is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4,
                    help="samples per GPU per step (4 = BASELINE.json configs[3]: batch 32 over 8 GPUs)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="nusc_200", choices=["nusc_200", "nusc_ref", "kitti", "nusc_r101"],
                    help="nusc_200 = BASELINE.json configs[2] (the metric's configuration); kitti = configs[1]")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying a captured CUDA graph")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16"],
                    help="fp32 (default, graded): three bf16 passes on split operands; bf16: single pass (config 5's mode)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    set_workload(args.workload)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl b200 needs a CUDA device; there is no CPU fallback for the hot path")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()

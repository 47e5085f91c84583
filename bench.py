#!/usr/bin/env python
"""bench.py - synthesized audio samples/sec @ batch 64 + VQ-index bit-exact rate (BASELINE.json metric, config C4).

    python bench.py --gpus N --steps K --warmup W [--impl b200|reference|torch_gpu] [--config c4|c2|c3] [--dump-outputs DIR]

One "step" = one pass of the synthesis hot path over one batch of 64 synthetic utterances U
(SURVEY.md §8: 64 phones, 8-s prompt -> 500 mel frames, durations forced to 8 -> 512 mel
frames -> 64 prosody tokens -> 131,072 samples):  mel front end (STFT+mel) -> MRTE ->
ADM autoregressive decode -> length regulator -> max-pool -> PLM autoregressive decode ->
VQ decode + mel decoder -> HiFi-GAN, plus the re-vocoding of the prompt that the reference's
forward() prepends (models/megatts2.py:371-373; its samples are NOT counted in the metric).
Weights: seeded random init of the reference architecture (no checkpoints exist offline); data: synthetic,
utterance i of the global batch is a pure function of seed 1234 + i.  N > 1: one process per GPU (torchrun),
the global batch of N x 64 utterances is split with megatts2_b200.sharding.shard_bounds (weak scaling, no
data-path collective); after the timed regions the prosody ids of every shard are gathered on rank 0 over NCCL
(sharding.gather_variable) and one shard is recomputed there to check the C5 contract "per-shard identical to
single-GPU".

Arms:  --impl b200       the product (this repo's CUDA path)                      [default]
       --impl reference  the reference's CPU path (oracle port: the reference is un-installable - no setup.py,
                         un-vendored deps), batch 1 like infer.py, one utterance per worker, all host cores
       --impl torch_gpu  the same port executed by stock PyTorch on the GPU (cuBLAS/cuDNN fp32, TF32 off and on):
                         the strongest existing implementation (BASELINE.md section 3); never the reference arm
       --config c2       BASELINE config 2: STFT+mel kernel over 10k synthetic 16 kHz 3-s clips (HBM roofline)
       --config c3       BASELINE config 3: PLM autoregressive decode, 512 prosody tokens, batch 16 (reference-faithful)

Output: ONE JSON line (contract in the task statement) with `roofline`, `cpu_baseline`, `e2e`, `clocks`,
`gpu_launches` and the parity half of the metric: `vq_index_bit_exact_rate`, `duration_exact_rate`, `mel_l1`.

--dump-outputs DIR (product arm): after the timed steps, what the last timed step returned to its caller is written as
DIR/<name>.npy - c4: `wav` (batch, 1, samples) of rank 0's shard; c2: `mel` (clips, 80, frames); c3: `ids` (16, 512) -
in float32 (ids in float64, exact).  Inputs and weights are seeded, so two builds run with the same arguments can be
compared array for array.  An output larger than DUMP_BYTES is cut to a fixed, seeded sample of its rows (dim 0).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU = 64
TP, TM_FRAMES, DUR = 64, 500, 8
PROMPT_SAMPLES = (TM_FRAMES - 1) * 256 + 128          # 1 + L // 256 == 500
SAMPLES_PER_UTT = TP * DUR * 256                      # 131,072 mel-aligned samples (the vocoder also emits 10 pad frames)
METRIC = "synthesized_audio_samples_per_sec_batch64"
UNIT = "samples/s"
SEED0 = 1234
THREADS_PER_WORKER = 16                               # the CPU arm: concurrent batch-1 workers of this many torch threads
MAX_WORKERS = 4                                       # (measured on the 128-cpu GPU box, profiles/r2b_cpu_arm_sweep.log: the batch-1
#                                                       AR loops stream 0.7 GB of weights per step and are memory-bound - 4 x 16
#                                                       threads is the fastest split; 16 x 8 is 4 % slower, 1 x 64 is 2x slower)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_gpu"])
    ap.add_argument("--config", default="c4", choices=["c4", "c2", "c3"])
    ap.add_argument("--batch", type=int, default=B_PER_GPU, help="utterances per GPU (default: the C4 batch, 64)")
    ap.add_argument("--check-utts", type=int, default=16, help="utterances of the batch checked against the CPU oracle")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the bounded CPU leg (profiling runs)")
    ap.add_argument("--no-prompt-revocode", action="store_true", help="leave out the prompt re-vocoding of forward()")
    ap.add_argument("--cpu-workers", type=int, default=0, help="concurrent batch-1 CPU workers (0 = cpus / 16, at most 4)")
    ap.add_argument("--cpu-threads", type=int, default=0, help="torch threads per CPU worker (0 = 16)")
    ap.add_argument("--clips", type=int, default=10000, help="--config c2: number of 3-s clips")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the product's outputs (--impl b200)")
    return args


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


DUMP_BYTES = 64 * 10**6                               # --dump-outputs: at most this many bytes over all arrays
DUMP_SEED = 0


def dump_outputs(d, arrays):
    """arrays {name: tensor} -> d/<name>.npy: floating point as float32, integers as float64 (exact).  An array over its
    share of DUMP_BYTES keeps a sample of its rows (dim 0), in order, drawn from DUMP_SEED: the same rows on every run."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        t = t.detach().cpu()
        t = t.float() if t.is_floating_point() else t.double()
        row_bytes = t[0].numel() * t.element_size()
        if t.numel() * t.element_size() > share:
            keep = share // row_bytes
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(DUMP_SEED))[:keep].sort().values
            log(f"dump: {name} keeps a seeded sample of {keep} of its {t.shape[0]} rows")
            t = t[rows]
        np.save(os.path.join(d, name + ".npy"), t.numpy())
        log(f"dump: {os.path.join(d, name + '.npy')} {tuple(t.shape)} {t.dtype}")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thr = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        self.thr = threading.Thread(target=self._read, daemon=True)
        self.thr.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------ model + data
def build_modules():
    """Random-init (seeded) product modules of the reference architecture, built on the HOST (so that the CPU
    workers of the checker / reference arm can rebuild bit-identical weights from the same seeds)."""
    import yaml
    from megatts2_b200.models.megatts2 import HIFIGAN, MegaG
    from megatts2_b200.utils.utils import instantiate_class
    cfg = os.path.join(ROOT, "configs")
    torch.manual_seed(0)
    G = MegaG.from_hparams(os.path.join(cfg, "config_gan.yaml"))
    cb = G.vqpe.vq.vq.layers[0]._codebook
    cb.embed.normal_()
    cb.embed_avg.copy_(cb.embed)
    cb.inited.fill_(1.0)
    torch.manual_seed(1)
    plm = instantiate_class((), yaml.safe_load(open(os.path.join(cfg, "config_plm.yaml")))["model"]["plm"])
    torch.manual_seed(2)
    adm = instantiate_class((), yaml.safe_load(open(os.path.join(cfg, "config_adm.yaml")))["model"]["adm"])
    with torch.no_grad():    # keep the AR duration regression bounded on random weights
        adm.dt_linear_emb.weight.mul_(0.02)
    torch.manual_seed(3)
    hifi = HIFIGAN.from_hparams(random_init=True)
    return G, plm, adm, hifi


def build_product(device):
    from megatts2_b200.models.megatts2 import Megatts
    G, plm, adm, hifi = build_modules()
    return Megatts(generator=G, plm=plm, adm=adm, hifi_gan=hifi, device=device)


def state_dicts(G, plm, adm, hifi):
    return tuple({n: v.detach().cpu() for n, v in m.state_dict().items()} for m in (G, plm, adm, hifi.generator))


def utterance(idx):
    """utterance `idx` of the global batch: prompt audio (PROMPT_SAMPLES,) and phone ids (TP,), seed 1234 + idx"""
    g = torch.Generator().manual_seed(SEED0 + idx)
    wav = torch.rand(PROMPT_SAMPLES, generator=g) * 2 - 1
    phone = torch.randint(0, 320, (TP,), generator=g)
    return wav, phone


def make_inputs(indices, pin=True):
    ws, ps = zip(*(utterance(i) for i in indices))
    wav, phone = torch.stack(ws), torch.stack(ps)
    if pin and torch.cuda.is_available():
        wav, phone = wav.pin_memory(), phone.pin_memory()
    forced = torch.full((len(indices), TP), DUR, dtype=torch.int32)
    return wav, phone, forced


def gpu_step(tts, wav_d, phone_d, forced_d, revocode=True, intermediates=False, overlap=None):
    from megatts2_b200.modules.tokenizer import extract_mel_spec
    mel = extract_mel_spec(wav_d, frames_major=True)                  # (B, 500, 80)
    return tts.synthesize(phone_d, mel, forced_durations=forced_d, prompt_mels=mel if revocode else None,
                          return_intermediates=intermediates, overlap_prompt=overlap)


# ------------------------------------------------------------------------------------------ CPU workers (oracle port)
_W = {}


def _worker_init(threads):
    torch.set_num_threads(threads)
    from oracle import weights as W
    G, plm, adm, hifi = build_modules()
    _W["sd"] = state_dicts(G, plm, adm, hifi)
    _W["cfgs"] = (W.G_CFG, W.PLM_CFG, W.ADM_CFG, W.HIFIGAN_CFG)


def _worker_utt(job):
    """the reference's path for ONE utterance, batch 1 as infer.py runs it; returns ids / durations / mel + seconds"""
    idx, revocode = job
    from oracle import ref_megatts2 as R
    wav, phone = utterance(idx)
    forced = torch.full((1, TP), DUR, dtype=torch.int32)
    t0 = time.perf_counter()
    mel = R.mel_spectrogram(wav[None]).transpose(1, 2)
    g, p, a, h = _W["sd"]
    ref = R.synthesize(g, p, a, h, phone[None], mel, _W["cfgs"], forced_durations=forced)
    if revocode:
        R.hifigan_generator(R.SD(h), mel.transpose(1, 2), _W["cfgs"][3])      # models/megatts2.py:371-372
    dt = time.perf_counter() - t0
    chk = float(g["decoder.last_layer.weight"].double().sum() + p["predict_layer.weight"].double().sum())
    return dict(idx=idx, secs=dt, p_codes=ref["p_codes"][0].numpy(), dt=ref["dt"][0].numpy(),
                mel=ref["mel"][0].transpose(0, 1).contiguous().numpy(), weights_checksum=chk)


class CpuPool:
    def __init__(self, workers, threads=0):
        import multiprocessing as mp
        ncpu = os.cpu_count() or 1
        tpw = threads if threads > 0 else THREADS_PER_WORKER
        self.workers = workers if workers > 0 else max(1, min(MAX_WORKERS, ncpu // tpw))
        self.threads = max(1, min(tpw, ncpu // self.workers))
        self.pool = mp.get_context("spawn").Pool(self.workers, initializer=_worker_init, initargs=(self.threads,))
        self.pool.map(_noop, range(self.workers))      # every worker has imported torch and rebuilt the weights

    def run(self, indices, revocode):
        return self.pool.map(_worker_utt, [(i, revocode) for i in indices], chunksize=1)

    def close(self):
        self.pool.close()
        self.pool.join()


def _noop(i):
    time.sleep(0.2)
    return i


# ------------------------------------------------------------------------------------------ the product arm
def run_b200(args):
    from megatts2_b200 import _lib as L
    from megatts2_b200 import ops, pack, sharding
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    revocode = not args.no_prompt_revocode
    log("building product modules")
    tts = build_product(dev)
    lo, hi = sharding.shard_bounds(world * B, world)[rank]            # this rank's slice of the global batch
    wav_h, phone_h, forced = make_inputs(range(lo, hi))
    wav_d, phone_d, forced_d = wav_h.to(dev), phone_h.to(dev), forced.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    n_out = 256 * (TP * DUR + 10) + (256 * (TM_FRAMES + 10) if revocode else 0)
    out_h = torch.empty(B, 1, n_out, dtype=torch.float32).pin_memory()
    lib = L.lib()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- set-up passes (untimed, not counted as warm-up): the first builds the packed-weight plans and grows the
    # workspace, the second captures the AR drivers' CUDA graphs, and the two after a capture still show one-off host-side
    # costs of the first replays (measured: profiles/r2j2_stage_times_6_passes.log)
    from megatts2_b200 import graphs
    for _ in range(4 if graphs.enabled() else 1):
        out = gpu_step(tts, wav_d, phone_d, forced_d, revocode)
    torch.cuda.synchronize()
    # ---- the W warm-up steps of the contract
    for _ in range(max(args.warmup, 1)):
        out = gpu_step(tts, wav_d, phone_d, forced_d, revocode)
    torch.cuda.synchronize()
    log("warm-up done")

    # ---- timed region 1: device-resident inputs (`value`)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    n0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        flush.zero_()                                                   # L2 flush between timed iterations
        out = gpu_step(tts, wav_d, phone_d, forced_d, revocode)
    e1.record()
    barrier()
    timed_out = out if args.dump_outputs else None
    clocks = sampler.stop() if rank == 0 else None
    launches = ops.launch_count() - n0
    ms = e0.elapsed_time(e1)
    log(f"timed region: {ms / args.steps:.1f} ms/step")

    # ---- timed region 2: end to end through the public API with HOST buffers (`e2e`)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        flush.zero_()
        w = wav_h.to(dev, non_blocking=True)
        ph = phone_h.to(dev, non_blocking=True)
        out = gpu_step(tts, w, ph, forced_d, revocode)
        out_h.copy_(out, non_blocking=True)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    log(f"e2e region: {ms_e2e / args.steps:.1f} ms/step")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"wav": timed_out})

    if dist is not None:
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = t.tolist()
    total_samples = world * B * SAMPLES_PER_UTT * args.steps
    value = total_samples / (ms / 1e3)
    e2e_value = total_samples / (ms_e2e / 1e3)

    # ---- C5 contract: every shard's ids, gathered over NCCL, equal a single-GPU run of the same global indices
    inter = gpu_step(tts, wav_d, phone_d, forced_d, revocode, intermediates=True)
    shard_identity = None
    if dist is not None:
        ids = inter["p_codes"]                                          # (B, T8) int64 on this rank
        lens = torch.full((ids.shape[0],), ids.shape[1], dtype=torch.int64, device=dev)
        gathered = sharding.gather_variable(ids, lens)                  # [(rows_r, lens_r)] over ranks, via NCCL
        if rank == 0:
            chk = world - 1                                             # recompute the LAST rank's shard here
            clo, chi = sharding.shard_bounds(world * B, world)[chk]
            cw, cp, cf = make_inputs(range(clo, chi), pin=False)
            mine = gpu_step(tts, cw.to(dev), cp.to(dev), cf.to(dev), revocode, intermediates=True)["p_codes"]
            theirs = gathered[chk][0]
            shard_identity = {"global_batch": world * B, "gathered_rows": int(sum(g[0].shape[0] for g in gathered)), "checked_shard": chk,
                              "global_indices": [clo, chi], "ids_equal": bool(torch.equal(mine, theirs)),
                              "how": "prosody ids of every rank gathered on rank 0 with sharding.gather_variable over NCCL; "
                                     "rank 0 re-ran the checked shard's global indices itself"}
            log(f"shard identity: {shard_identity['ids_equal']}")

    result = None
    if rank == 0:
        # ---- roofline leg: per-launch CUDA events around every tap-GEMM launch of ONE step
        # (single stream for this leg: with the prompt re-vocode overlapped on its side stream the per-launch times of two
        #  concurrently running kernels would be summed)
        from megatts2_b200 import graphs
        lib.mtts_profile_begin()
        with graphs.disabled():            # the profile records events between launches: eager enqueue, no graph replay
            gpu_step(tts, wav_d, phone_d, forced_d, revocode, overlap=False)
        gms, gfl, gn = C.c_double(), C.c_double(), C.c_int64()
        L.check(lib.mtts_profile_end(C.byref(gms), C.byref(gfl), C.byref(gn)))
        log(f"roofline leg: {gn.value} tap-GEMM launches, {gms.value:.1f} ms, {gfl.value / 1e12:.2f} TFLOP")
        sp = (C.c_double * 6)()
        lib.mtts_profile_split(sp)
        pk, pk_src = peaks()
        peak = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops")))
        step_ms = ms / args.steps
        engine = pack.default_engine()
        mma_per_product = {pack.ENGINE_F16X2: 3, pack.ENGINE_BF16X3: 6}.get(engine, 0)
        scheme = {pack.ENGINE_F16X2: "f16x2 (two fp16 operand planes, residual scaled by 2^11; 3 MMAs per fp32-grade product)",
                  pack.ENGINE_BF16X3: "bf16x3 (three bf16 operand planes; 6 MMAs per fp32-grade product)"}.get(engine, "fp32 FFMA")

        def cls(ms_, fl_, n_):
            return {"ms_per_step": round(ms_, 2), "tflop_per_step": round(fl_ / 1e12, 3), "launches_per_step": int(n_),
                    "achieved_tflops": round(fl_ / (ms_ / 1e3) / 1e12, 2) if ms_ > 0 else 0.0,
                    "share_of_step": round(ms_ / step_ms, 3)}
        classes = {"fp32_ffma_tapconv_kernel": cls(sp[0], sp[1], sp[2]),
                   "tcgen05_tap_gemm_kernels (incl. their activation-split kernels)": cls(sp[3], sp[4], sp[5])}
        dom_tc = sp[3] >= sp[0]
        d_ms, d_fl = (sp[3], sp[4]) if dom_tc else (sp[0], sp[1])
        achieved = d_fl / (d_ms / 1e3) / 1e12 if d_ms > 0 else 0.0
        traffic, traffic_note = measured_traffic()
        roofline = {"bound": "tensor",
                    "kernel": (f"conv_tc_kernel (tcgen05 tap-GEMM: every Linear / Conv1d / ConvTranspose1d; operands {scheme}; "
                               "single-CTA and cta_group::2 pair variants)" if dom_tc else "tapconv_kernel (fp32 FFMA tap-GEMM)"),
                    "achieved": round(achieved, 3), "peak": peak, "unit": "TFLOP/s", "frac": round(achieved / peak, 5),
                    "traffic": traffic, "traffic_note": traffic_note,
                    "peak_source": f"{pk_src} dense bf16 (sustained). achieved = algorithmic fp32-grade FLOPs (2*M*N*K) / CUDA-event "
                                   f"time of the launches; the {scheme.split(' ')[0]} scheme issues {mma_per_product} 16-bit MMAs per such "
                                   f"FLOP pair, so its ceiling is peak/{mma_per_product}",
                    "frac_of_scheme_ceiling": round(achieved / (peak / mma_per_product), 4) if dom_tc and mma_per_product else None,
                    "classes": classes}
        parity, cpu = (None, None) if args.no_cpu_baseline else cpu_check(args, inter, lo, revocode)
        result = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C4: full synthesis MRTE+ADM+PLM+decoder+HiFi-GAN (+mel front end"
                                   + (", + re-vocoding of the 500-frame prompt as forward() does" if revocode else "") + "), "
                                   f"batch {B} synthetic utterances per GPU (64 phones, 500-frame prompt, "
                                   "512 mel frames, 64 prosody tokens, 131072 counted samples each)",
                       "global_batch": world * B, "parallelism": f"replicas x{world} (batch split, no data-path collective)",
                       "l2": "256 MiB flush write between timed iterations; working set (1.57 GB weights) >> 126 MB L2",
                       "weights": "seeded random init of the reference architecture", "ar_semantics": "reference-faithful "
                       "non-causal full recompute per step (models/megatts2.py:165-181, 257-275)",
                       "tensor_core_operands": scheme,
                       "unpinned": "HiFi-GAN (speechbrain, restated from the published architecture) and the speechbrain mel wrapper "
                                   "are parity-unpinned (SURVEY.md 8c); everything else is pinned on the reference itself"},
            "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "ms_per_step": round(ms_e2e / args.steps, 3),
                    "h2d_bytes_per_step": world * (wav_h.numel() * 4 + phone_h.numel() * 8),
                    "d2h_bytes_per_step": world * out_h.numel() * 4},
            "gpu_launches": int(launches),
            "hbm_peak_bytes": int(torch.cuda.max_memory_allocated(dev)),
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        if parity is not None:
            result.update(parity)
        if shard_identity is not None:
            result["shard_identity"] = shard_identity
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return result


def measured_traffic():
    """dram__bytes_read + dram__bytes_write per launch of the dominant kernel class, from the committed ncu capture of
    this command (tools/summarize_ncu.py -> profiles/r2_traffic.json); null until a capture exists."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(p):
        return None, "no ncu capture committed yet"
    with open(p) as f:
        d = json.load(f)
    return d.get("dominant_kernel_dram_bytes_per_launch"), d.get("note", "profiles/r2_traffic.json")


def mel_traffic(args):
    """Measured DRAM bytes of one mel_kernel launch on config C2 (ncu capture committed under profiles/); only valid for the
    default 10 000 clips."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if args.clips != 10000 or not os.path.exists(p):
        return None
    with open(p) as f:
        return json.load(f).get("mel_kernel_dram_bytes_per_launch")


def cpu_check(args, gpu, lo, revocode):
    """The oracle port (CPU restatement of the reference, batch 1 like the reference) run by concurrent workers on this
    box's host cores over `check_utts` utterances of this rank's batch: it is the CHECKER of the GPU arm's prosody ids /
    durations / mel (the parity half of the metric), and its wall time is the `cpu_baseline`."""
    n = min(args.check_utts, args.batch)
    pool = CpuPool(args.cpu_workers, args.cpu_threads)
    log(f"cpu check: {n} utterances on {pool.workers} workers x {pool.threads} threads ({os.cpu_count()} host cpus)")
    t0 = time.perf_counter()
    res = pool.run([lo + i for i in range(n)], revocode)
    wall = time.perf_counter() - t0
    pool.close()
    ids_ok = ids_n = dur_ok = dur_n = 0
    mel_l1 = 0.0
    p_codes, dt, mel = gpu["p_codes"].cpu(), gpu["dt"].cpu(), gpu["mel"].cpu()
    for r in res:
        i = r["idx"] - lo
        ids_ok += int((torch.from_numpy(r["p_codes"]) == p_codes[i]).sum()); ids_n += r["p_codes"].size
        dur_ok += int((torch.from_numpy(r["dt"]) == dt[i]).sum()); dur_n += r["dt"].size
        mel_l1 += (torch.from_numpy(r["mel"]) - mel[i]).abs().mean().item() / len(res)
    secs = [r["secs"] for r in res]
    parity = {"vq_index_bit_exact_rate": ids_ok / max(ids_n, 1), "duration_exact_rate": dur_ok / max(dur_n, 1),
              "mel_l1": mel_l1, "parity_checked_utterances": len(res),
              "parity_note": f"prosody VQ ids ({ids_n}), ADM durations ({dur_n}) and decoder mel of {len(res)} of the {args.batch} "
                             "utterances vs the CPU oracle (batch 1 each); bars: ids / durations bit-exact, mel L1 <= 1e-4"}
    cpu = {"value": round(len(res) * SAMPLES_PER_UTT / wall, 1), "unit": UNIT, "cores": pool.workers * pool.threads,
           "kind": "port",
           "sample": f"{len(res)} of the {args.batch} utterances U, batch 1 each (the reference's infer() is batch-1 only) on "
                     f"{pool.workers} concurrent workers x {pool.threads} torch threads of {os.cpu_count()} host cpus, "
                     f"{wall:.1f} s wall",
           "single_stream": {"value": round(SAMPLES_PER_UTT / statistics.median(secs), 1), "unit": UNIT,
                             "threads": pool.threads, "median_s_per_utterance": round(statistics.median(secs), 2),
                             "note": "one worker's rate while the other workers run (what one infer.py process gets)"},
           "rtf": round(wall / (len(res) * SAMPLES_PER_UTT / 16000.0), 4)}
    return parity, cpu


# ------------------------------------------------------------------------------------------ reference arm (CPU)
def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port: the reference
    cannot be pip-installed - it has no setup.py / pyproject and needs un-vendored speechbrain) on this box's
    host cores, batch 1 as infer.py does; a step = one utterance U on EVERY worker concurrently (all cores busy)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    revocode = not args.no_prompt_revocode
    pool = CpuPool(args.cpu_workers, args.cpu_threads)
    W = pool.workers
    log(f"reference arm: {W} workers x {pool.threads} torch threads of {os.cpu_count()} host cpus")
    nxt = 0
    for _ in range(min(args.warmup, 1)):       # one warm-up pass is enough on the CPU (each is ~10 s)
        pool.run(range(nxt, nxt + W), revocode); nxt += W
    t0 = time.perf_counter()
    secs = []
    for i in range(args.steps):
        secs += [r["secs"] for r in pool.run(range(nxt, nxt + W), revocode)]; nxt += W
        log(f"reference arm: step {i + 1}/{args.steps} at {time.perf_counter() - t0:.1f} s")
    dt = time.perf_counter() - t0
    pool.close()
    v = args.steps * W * SAMPLES_PER_UTT / dt
    return {"impl": "reference", "metric": METRIC, "value": round(v, 1), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"C4 utterance U through the reference's CPU path (oracle port), batch 1 per worker (the "
                                   f"reference's infer() loops are batch-1 only), {W} utterances per step on {W} concurrent workers"
                                   + (", prompt re-vocoding included" if revocode else "")},
            "cpu_baseline": {"value": round(v, 1), "unit": UNIT, "cores": W * pool.threads, "kind": "port",
                             "sample": f"{args.steps} steps x {W} utterances U (131072 samples each), {W} workers x "
                                       f"{pool.threads} torch threads of {os.cpu_count()} host cpus",
                             "single_stream": {"value": round(SAMPLES_PER_UTT / statistics.median(secs), 1), "unit": UNIT,
                                               "threads": pool.threads}},
            "e2e": {"value": round(v, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


# ------------------------------------------------------------------------------------------ stock PyTorch on the GPU
def run_torch_gpu(args):
    """--impl torch_gpu: the oracle port (the reference's own torch ops) executed by stock PyTorch on cuda:0 at batch 64 -
    cuBLAS / cuDNN fp32 with TF32 off (the parity-grade setting) and, as a stated fast mode, TF32 on - with the id-exact
    rate of each against the product's ids.  The strongest existing implementation to beat (BASELINE.md section 3)."""
    from oracle import ref_megatts2 as R
    from oracle import weights as W
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    B = args.batch
    revocode = not args.no_prompt_revocode
    G, plm, adm, hifi = build_modules()
    sds = tuple({k: v.to(dev) for k, v in sd.items()} for sd in state_dicts(G, plm, adm, hifi))
    cfgs = (W.G_CFG, W.PLM_CFG, W.ADM_CFG, W.HIFIGAN_CFG)
    wav, phone, forced = make_inputs(range(B), pin=False)
    wav, phone, forced = wav.to(dev), phone.to(dev), forced.to(dev)
    # the product's ids on the same batch (the comparison the judge asked for)
    from megatts2_b200.models.megatts2 import Megatts
    tts = Megatts(generator=G, plm=plm, adm=adm, hifi_gan=hifi, device=dev)
    ours = gpu_step(tts, wav, phone, forced, revocode, intermediates=True)
    ours_ids, ours_mel = ours["p_codes"].clone(), ours["mel"].clone()
    del tts, ours
    torch.cuda.empty_cache()

    def step():
        with torch.device(dev):
            mel = R.mel_spectrogram(wav).transpose(1, 2)
            out = R.synthesize(*sds, phone, mel, cfgs, forced_durations=forced)
            if revocode:
                R.hifigan_generator(R.SD(sds[3]), mel.transpose(1, 2), cfgs[3])
        return out
    modes = {}
    for name, tf32 in (("fp32", False), ("tf32", True)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
        for _ in range(max(1, min(args.warmup, 2))):
            out = step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            out = step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        modes[name] = {"value": round(B * SAMPLES_PER_UTT / (ms / 1e3), 1), "unit": UNIT, "ms_per_step": round(ms, 2),
                       "ids_equal_to_product_rate": float((out["p_codes"] == ours_ids).float().mean()),
                       "mel_l1_vs_product": float((out["mel"].transpose(1, 2) - ours_mel).abs().mean())}
        log(f"torch_gpu {name}: {ms:.1f} ms/step")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    m = modes["fp32"]
    return {"impl": "torch_gpu", "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"C4 batch {B}: the oracle port's torch ops on cuda (cuBLAS / cuDNN), allow_tf32 = False",
                       "note": "stock PyTorch eager; no last-row pruning, no fused kernels; same weights / inputs as the product arm"},
            "modes": modes}


# ------------------------------------------------------------------------------------------ config C2 (mel front end)
def run_c2(args):
    """BASELINE config 2: the STFT + mel-filterbank kernel over `clips` synthetic 16 kHz 3-s clips on one B200, against
    the HBM roofline (algorithmic bytes = 48000*4 in + 188*80*4 out = 252,160 B per clip, SURVEY.md 8d)."""
    from megatts2_b200 import ops
    from megatts2_b200.modules.tokenizer import extract_mel_spec
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    n, Ls = args.clips, 48000
    g = torch.Generator().manual_seed(SEED0 + 2)
    wav_h = (torch.rand(n, Ls, generator=g) * 2 - 1).pin_memory()
    wav = wav_h.to(dev)                                                 # 1.92 GB > L2
    for _ in range(max(args.warmup, 3)):
        mel = extract_mel_spec(wav)
    torch.cuda.synchronize()
    n0 = ops.launch_count()
    sampler = ClockSampler(0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        mel = extract_mel_spec(wav)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    launches = ops.launch_count() - n0
    out_h = torch.empty(mel.shape, dtype=torch.float32).pin_memory()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        m2 = extract_mel_spec(wav_h.to(dev, non_blocking=True))
        out_h.copy_(m2, non_blocking=True)
    f1.record()
    torch.cuda.synchronize()
    ms_e2e = f0.elapsed_time(f1) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"mel": mel})
    pk, pk_src = peaks()
    bytes_per_clip = Ls * 4 + 80 * (1 + Ls // 256) * 4
    gbs = n * bytes_per_clip / (ms / 1e3) / 1e9
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import ref_megatts2 as R
        torch.set_num_threads(min(32, os.cpu_count() or 1))
        k = 256
        t0 = time.perf_counter()
        ref = R.mel_spectrogram(wav_h[:k])
        dt = time.perf_counter() - t0
        l1 = (ref - mel[:k].cpu()).abs().mean().item()
        cpu = {"value": round(k / dt, 1), "unit": "clips/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"{k} of the {n} clips in one torch.stft batch", "mel_l1_vs_gpu": l1}
    return {"metric": "mel_clips_per_sec", "value": round(n / (ms / 1e3), 1), "unit": "clips/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"C2: STFT (1024/256, periodic Hann, reflect) + 80-bin slaney mel + log over {n} clips of 3 s @ 16 kHz",
                       "l2": "input 1.92 GB + output 0.60 GB per step >> 126 MB L2"},
            "e2e": {"value": round(n / (ms_e2e / 1e3), 1), "unit": "clips/s", "h2d_bytes_per_step": n * Ls * 4,
                    "d2h_bytes_per_step": int(mel.numel()) * 4},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "mel_kernel", "achieved": round(gbs, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                         "frac": round(gbs / pk["hbm_gbs"], 4), "traffic": mel_traffic(args), "peak_source": pk_src,
                         "algorithmic_bytes_per_clip": bytes_per_clip},
            "cpu_baseline": cpu}

# ------------------------------------------------------------------------------------------ config C3 (PLM decode, T = 512)
def run_c3(args):
    """BASELINE config 3: MegaPLM.infer - the reference-faithful NON-causal full-recompute greedy decode
    (models/megatts2.py:165-181) - of 512 prosody tokens at batch 16 on one B200.  A step = one whole decode.
    Parity: at sampled steps t the oracle's last-row logits for the GPU's own prefix must pick the GPU's id (a greedy decode
    is exactly the sequence for which that holds at every step)."""
    import ctypes as C
    from megatts2_b200 import _lib as L
    from megatts2_b200 import graphs, ops
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    B, T = 16, 512
    tts = build_product(dev)
    g = torch.Generator().manual_seed(SEED0 + 3)
    tc_h = torch.relu(torch.randn(B, T, 512, generator=g)).pin_memory()
    tc = tc_h.to(dev)
    for _ in range(4 if graphs.enabled() else 1):        # set-up passes: plans, graph capture, first replays
        ids = tts.plm.infer(tc)
    for _ in range(max(1, min(args.warmup, 2))):
        ids = tts.plm.infer(tc)
    torch.cuda.synchronize()
    steps = args.steps
    n0 = ops.launch_count()
    sampler = ClockSampler(0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ids = tts.plm.infer(tc)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / steps
    launches = ops.launch_count() - n0
    ids_h = torch.empty(B, T, dtype=torch.int64).pin_memory()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(steps):
        ids_h.copy_(tts.plm.infer(tc_h.to(dev, non_blocking=True)), non_blocking=True)
    f1.record()
    torch.cuda.synchronize()
    ms_e2e = f0.elapsed_time(f1) / steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"ids": ids})
    # roofline leg: algorithmic FLOPs and CUDA-event time of the tap-GEMM launches of ONE decode (eager enqueue)
    lib = L.lib()
    lib.mtts_profile_begin()
    with graphs.disabled():
        tts.plm.infer(tc)
    gms, gfl, gn = C.c_double(), C.c_double(), C.c_int64()
    L.check(lib.mtts_profile_end(C.byref(gms), C.byref(gfl), C.byref(gn)))
    pk, pk_src = peaks()
    peak = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops")))
    ach = gfl.value / 1e12 / (gms.value / 1e3)
    # causal KV-cache decode (opt-in, SURVEY 8f-1) of the same shape, for scale
    tts.plm.infer_causal(tc)
    torch.cuda.synchronize()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    tts.plm.infer_causal(tc)
    c1.record()
    torch.cuda.synchronize()
    parity, cpu = None, None
    if not args.no_cpu_baseline:
        from oracle import ref_megatts2 as R
        from oracle import weights as W
        torch.set_num_threads(min(64, os.cpu_count() or 1))
        sd = R.SD(state_dicts(*build_modules())[1])
        codes = torch.cat([torch.full((1, 1), 1024, dtype=torch.int64), ids[:1].cpu()], 1)      # BOS + the GPU's ids of sequence 0
        checked, agree, secs = [], 0, {}
        for t in (0, 1, 31, 127, 255, 383, 511):
            t0 = time.perf_counter()
            lg = R.plm_step_logits(sd, tc_h[:1, : t + 1], codes[:, : t + 1], W.PLM_CFG)
            secs[t] = time.perf_counter() - t0
            top2 = lg[0].topk(2).values
            ok = int(lg[0].argmax()) == int(codes[0, t + 1])
            checked.append({"t": t, "equal": ok, "top2_gap": float(top2[0] - top2[1])})
            agree += ok
        parity = {"sequence": 0, "steps_checked": checked, "rate": agree / len(checked)}
        # CPU time of one sequence's decode: the measured step times interpolated over t (a step's cost grows with t)
        ts = sorted(secs)
        total = 0.0
        for t in range(T):
            lo = max([u for u in ts if u <= t]); hi = min([u for u in ts if u >= t])
            total += secs[lo] if lo == hi else secs[lo] + (secs[hi] - secs[lo]) * (t - lo) / (hi - lo)
        cpu = {"value": round(T / total, 2), "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "7 decode steps of one sequence timed, the other steps interpolated over t (one sequence ~ %.0f s)" % total}
    return {"metric": "plm_prosody_tokens_per_sec", "value": round(B * T / (ms / 1e3), 1), "unit": "tokens/s", "n_gpus": 1,
            "steps": steps, "warmup": args.warmup, "ms_per_step": round(ms, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C3: MegaPLM.infer, 512 prosody tokens, batch 16: non-causal full recompute per step as the "
                                   "reference does (the final layer's out-projection / FFN for the last row only, the only "
                                   "row consumed)",
                       "l2": "weights 0.6 GB + activations per step >> 126 MB L2", "weights": "seeded random init",
                       "causal_kv_cache_decode_ms": round(c0.elapsed_time(c1), 2)},
            "e2e": {"value": round(B * T / (ms_e2e / 1e3), 1), "unit": "tokens/s", "h2d_bytes_per_step": int(tc_h.numel()) * 4,
                    "d2h_bytes_per_step": B * T * 8},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "conv_tc_kernel", "achieved": round(ach, 1), "peak": peak, "unit": "TFLOP/s",
                         "frac": round(ach / peak, 4), "frac_of_scheme_ceiling": round(3 * ach / peak, 4), "traffic": None,
                         "peak_source": pk_src, "tflop_per_decode": round(gfl.value / 1e12, 1),
                         "tap_gemm_ms_per_decode": round(gms.value, 1)},
            "vq_index_bit_exact_rate": None if parity is None else parity["rate"], "parity": parity, "cpu_baseline": cpu}


def main():
    args = parse()
    if args.impl == "reference":
        res = run_reference(args)
    else:
        if not torch.cuda.is_available():
            print(json.dumps({"error": "no CUDA device: bench.py measures the CUDA path only (no CPU fallback)"}))
            return 1
        if args.impl == "torch_gpu":
            res = run_torch_gpu(args)
        elif args.config == "c2":
            res = run_c2(args)
        elif args.config == "c3":
            res = run_c3(args)
        else:
            res = run_b200(args)
    if res is not None:
        print(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main())

"""bench.py — LLaVA-1.5 multimodal forward path on B200 (BASELINE.json metric: prefill+decode tokens/s).

  python bench.py [--gpus N --steps K --warmup W]            our sm_100a path (one process per GPU under torchrun)
  python bench.py --impl reference [...]                     the reference's CPU path (oracle port) on host cores

A "step" is one pass of the hot path over one batch of synthetic input: encode_images (CLIP ViT-L/14-336 +
mlp2x_gelu) -> splice -> LLaMA prefill over 576 image tokens + 128 text tokens -> 256 greedy decode tokens,
i.e. BASELINE.json configs[1] (LLaVA-1.5-7B bf16, 336 px, bs=1 per GPU). Random-init weights of that
architecture and synthetic inputs (no network for checkpoints/datasets).

value   : tokens/s = n_gpus * B * (S_prefill + N_decode) / (max-over-ranks device time per step), inputs resident
          in HBM, CUDA events on the launching stream.
e2e     : same metric through the public API model.generate(input_ids, images=...) with HOST (pinned) inputs:
          H2D of pixels + ids and D2H of the generated ids inside the timed region.
roofline: the decode step (one launch of the persistent decode megakernel: all layers' weight-streaming GEMV
          phases + split-KV attention + lm_head + argmax), HBM-bound: algorithmic bytes/step = W + B*(Lc+1)*kv
          (SURVEY §8d) over the measured step time, against MEASURED_PEAKS.json hbm_gbs.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "llava-plus-codebase_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
os.environ.setdefault("TRANSFORMERS_OFFLINE", "1")
os.environ.setdefault("HF_HUB_OFFLINE", "1")

import torch  # noqa: E402

MODELS = {
    "7b": dict(name="LLaVA-1.5-7B", hidden=4096, inter=11008, layers=32, heads=32),
    "13b": dict(name="LLaVA-1.5-13B", hidden=5120, inter=13824, layers=40, heads=40),
}
VOCAB, P_IMG, VIT_GF, IMAGE_TOKEN = 32000, 576, 366.03, -200


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="7b", choices=list(MODELS))
    ap.add_argument("--batch", type=int, default=1, help="samples per GPU")
    ap.add_argument("--prompt", type=int, default=128, help="text tokens (one <image> placeholder is added)")
    ap.add_argument("--new", type=int, default=256, help="greedy decode tokens")
    ap.add_argument("--fp8", action="store_true",
                    help="BASELINE configs[4]: e4m3 decoder weights/activations for decode at batch >= 7 ")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the side measurements of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (image features, last-position "
                         "prefill logits, generated token ids) as DIR/<name>.npy, at most 64 MB in all")
    return ap.parse_args()


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
        return float(pk["hbm_gbs"]), float(pk["bf16_tflops"]), "measured"
    except Exception:
        return 6650.0, 1590.0, "fallback"


def algorithmic_work(m, B, S, N, fp8=False):
    h, I, L = m["hidden"], m["inter"], m["layers"]
    layer_params = 4 * h * h + 3 * h * I
    w_bytes = 2 * (L * (layer_params + 2 * h) + h + VOCAB * h)     # decode weight stream (bf16), SURVEY §8d
    if fp8:  # 1-byte Linear weights + one fp32 scale per output channel; norms stay bf16
        w_bytes = L * (layer_params + 4 * (5 * h + 2 * I) + 2 * 2 * h) + 2 * h + VOCAB * (h + 4)
    kv_per_tok = 2 * 2 * h * L                                     # K+V bf16, all layers, per token per sample
    prefill_flops = B * (2 * S * layer_params * L + 2 * S * S * h * L + 2 * h * VOCAB)
    encode_flops = B * (VIT_GF * 1e9 + 2 * P_IMG * (1024 * h + h * h))
    # decode step j (j = 0..N-2) runs against Lc = S + j cached tokens
    steps = max(N - 1, 1)
    avg_lc = S + (steps - 1) / 2.0
    decode_bytes_per_step = w_bytes + B * (avg_lc + 1) * kv_per_tok
    return dict(w_bytes=w_bytes, kv_per_tok=kv_per_tok, prefill_flops=prefill_flops, encode_flops=encode_flops,
                decode_bytes_per_step=decode_bytes_per_step)


# ---------------------------------------------------------------------------------------------------------
# clocks (sampled DURING the timed region)
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons, pw = [], [], set(), []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------
# reference CPU path (oracle port) — bounded sample, extrapolated
# ---------------------------------------------------------------------------------------------------------
_CPU_WEIGHTS = {}


CPU_THREADS = 16  # PyTorch's CPU GEMV/GEMM get SLOWER with every hardware thread of a many-core host (measured on this pool's
                  # 128-thread hosts in round 1: 16 threads 13.1 tok/s, 64 threads 9.7, 128 threads 3.7): a fixed, stated count


_CPU_PIN = {}


def _physical_cores():
    """One logical CPU per physical core, in id order (the first hyper-thread sibling of each core), from sysfs."""
    allowed = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    seen, cores = set(), []
    for c in allowed:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
        except OSError:
            sib = str(c)
        if sib not in seen:
            seen.add(sib)
            cores.append(c)
    return cores


def cpu_threads():
    """Fixed thread count, PINNED: the intra-op pool is sized to CPU_THREADS and the process is restricted to that many distinct
    physical cores (lowest ids) for the duration of the CPU arm, so the figure does not depend on where the scheduler happens to
    put 16 threads on a 128-thread host. `cpu_unpin()` restores the previous affinity."""
    n = min(CPU_THREADS, os.cpu_count() or 1)
    torch.set_num_threads(n)
    if hasattr(os, "sched_setaffinity") and "prev" not in _CPU_PIN:
        try:
            prev = os.sched_getaffinity(0)
            cores = _physical_cores()[:n]
            if len(cores) == n:
                os.sched_setaffinity(0, cores)
                _CPU_PIN.update(prev=prev, cores=cores)
        except OSError:
            pass
    return n


def cpu_unpin():
    prev = _CPU_PIN.pop("prev", None)
    if prev is not None:
        try:
            os.sched_setaffinity(0, prev)
        except OSError:
            pass


def pick_cpu_dtype():
    """The reference runs whatever dtype the user loads; on a host without AMX-bf16, bf16 GEMMs are far slower
    than fp32 in PyTorch. Time a small matmul in both and use the faster (the kinder baseline)."""
    best, best_t = torch.float32, None
    for dt in (torch.float32, torch.bfloat16):
        a, b = torch.randn(512, 2048).to(dt), torch.randn(2048, 2048).to(dt)
        a @ b
        t0 = time.perf_counter()
        for _ in range(3):
            a @ b
        t = time.perf_counter() - t0
        if best_t is None or t < best_t:
            best, best_t = dt, t
    return best


def cpu_reference_sample(m, S, N, sample_layers=8, decode_steps=4, dtype=None):
    """Times the reference's algorithm (oracle/llava_oracle.py, HF-bf16 rounding points) on the host cores at
    the full LLaVA dims on a bounded sample: ViT+projector in full, `sample_layers` of the decoder layers for a
    full S-token prefill and `decode_steps` decode steps, lm_head measured separately; the per-layer time is
    extrapolated to all layers (layer cost is uniform). Returns tokens/s for the whole step + the breakdown."""
    from oracle import llava_oracle as O

    cpu_threads()
    if dtype is None:
        dtype = pick_cpu_dtype()
    cfg = O.make_config(hidden=m["hidden"], inter=m["inter"], layers=sample_layers, heads=m["heads"])
    g = torch.Generator().manual_seed(0)
    key = (m["name"], str(dtype))
    if _CPU_WEIGHTS.get("key") != key:  # built once per process (max sample_layers = 8 decoder layers)
        full = O.make_config(hidden=m["hidden"], inter=m["inter"], layers=8, heads=m["heads"])
        w = {}
        for k, shape, kind in O.weight_shapes(full):
            t = torch.empty(*shape, dtype=dtype).normal_(0.0, O.init_std(kind, shape), generator=g)
            w[k] = t + 1.0 if kind == "g" else t
        _CPU_WEIGHTS.update(key=key, w=w)
    w = _CPU_WEIGHTS["w"]
    images = torch.randn(1, 3, 336, 336, generator=g)
    ids = torch.randint(3, VOCAB, (1, S - P_IMG + 1), generator=g)
    ids[0, 5] = IMAGE_TOKEN
    cfg0 = dict(cfg, layers=0)
    with torch.no_grad():
        t0 = time.perf_counter()
        feats = O.encode_images(w, images, cfg, dtype=dtype)
        t_enc = time.perf_counter() - t0
        embeds, _, _, _ = O.prepare_multimodal(w, ids, None, cfg, dtype=dtype, image_features=list(feats))
        O.llama_forward(w, embeds[:, :64], cfg, dtype=dtype)  # warm-up (thread pool, allocator)
        t0 = time.perf_counter()
        _, kv = O.llama_forward(w, embeds, cfg, dtype=dtype)          # the reference runs lm_head on all S positions
        t_pre_L = time.perf_counter() - t0
        t0 = time.perf_counter()
        O.llama_forward(w, embeds, cfg0, dtype=dtype)
        t_pre_0 = time.perf_counter() - t0
        e = embeds[:, -1:]
        t_dec_L = 0.0
        for _ in range(decode_steps):
            t0 = time.perf_counter()
            _, kv = O.llama_forward(w, e, cfg, kv=kv, dtype=dtype)
            t_dec_L += time.perf_counter() - t0
        t_dec_L /= decode_steps
        t0 = time.perf_counter()
        for _ in range(decode_steps):
            O.llama_forward(w, e, cfg0, dtype=dtype)
        t_dec_0 = (time.perf_counter() - t0) / decode_steps
    L = m["layers"]
    per_layer_pre = max(t_pre_L - t_pre_0, 0.0) / sample_layers
    per_layer_dec = max(t_dec_L - t_dec_0, 0.0) / sample_layers
    t_prefill = t_pre_0 + per_layer_pre * L
    t_decode_step = t_dec_0 + per_layer_dec * L
    total = t_enc + t_prefill + (N - 1) * t_decode_step
    return dict(value=(S + N) / total, unit="tokens/s", cores=torch.get_num_threads(), kind="port",
                dtype="bf16" if dtype == torch.bfloat16 else "f32", extrapolated=True, sampled_layers=sample_layers,
                full_step_s=total,
                sample=(f"EXTRAPOLATED: oracle port ({str(dtype).replace('torch.', '')}, the faster of fp32/bf16 on this host; "
                        f"{torch.get_num_threads()} threads fixed, pinned to cores {_CPU_PIN.get('cores', 'unpinned')}, host has {os.cpu_count()}) at full {m['name']} dims: ViT+projector "
                        f"1 image in full, {sample_layers} of {L} decoder layers for an S={S} prefill (lm_head on all positions, "
                        f"as the reference does) and {decode_steps} decode steps, per-layer time extrapolated x{L}/{sample_layers}"),
                breakdown=dict(encode_s=t_enc, prefill_s=t_prefill, decode_step_s=t_decode_step,
                               prefill_tok_s=S / t_prefill, decode_tok_s=1.0 / t_decode_step),
                measured_s=t_enc + t_pre_L + t_pre_0 + decode_steps * (t_dec_L + t_dec_0))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    m = MODELS[args.model]
    S = P_IMG + args.prompt
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        # warm-up steps use a smaller sample (thread pools, allocator); timed steps the bounded sample
        last = cpu_reference_sample(m, S, args.new, sample_layers=1 if i < args.warmup else 8,
                                    decode_steps=1 if i < args.warmup else 4)
        if i >= args.warmup:
            vals.append(last)
    value = sum(v["value"] for v in vals) / len(vals)
    total_s = (S + args.new) / value
    sample_s = sum(v["measured_s"] for v in vals) / len(vals)
    out = {
        "impl": "reference", "metric": "prefill+decode tokens/s", "value": value, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        # a timed step is the bounded sample (8 of 32 layers, 4 decode steps); `value` extrapolates it to the full workload
        "ms_per_step": sample_s * 1e3, "extrapolated": True, "sampled_layers": last["sampled_layers"],
        "extrapolated_full_step_ms": total_s * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": last["dtype"], "data": "synthetic",
        "config": workload_config(args, m, S),
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": last["cores"], "kind": "port", "extrapolated": True,
                         "sampled_layers": last["sampled_layers"], "sample": last["sample"], "breakdown": last["breakdown"]},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


def workload_config(args, m, S):
    return {"workload": f"{m['name']} bf16, one 336px image/sample, bs={args.batch}/GPU: {P_IMG} image tokens + "
                        f"{args.prompt} text prefill (S={S}), {args.new}-token greedy decode (BASELINE.json configs[1])",
            "global_batch": args.batch * args.gpus, "seq_len": S, "new_tokens": args.new, "parallelism": f"dp{args.gpus} replicas",
            "l2": "working set (13.5 GB weights streamed every decode step) >> 126 MB L2; no flush needed"}


# ---------------------------------------------------------------------------------------------------------
# our path
# ---------------------------------------------------------------------------------------------------------
def build_model(m, device, max_batch, max_seq):
    from helpers import write_clip_config_dir, make_llava_config
    from llava.model import LlavaLlamaForCausalLM
    from oracle.llava_oracle import make_config, weight_shapes, init_std  # shapes/init table only (no compute)

    cfg = make_config(hidden=m["hidden"], inter=m["inter"], layers=m["layers"], heads=m["heads"])
    clip_dir = write_clip_config_dir(cfg)
    model = LlavaLlamaForCausalLM(make_llava_config(cfg, clip_dir), device=device, max_batch=max_batch,
                                  max_seq=max_seq, max_images=min(max_batch, 16))
    model.get_vision_tower().load_model(random_init=True)
    model.to(device=device, dtype=torch.bfloat16)
    gen = torch.Generator(device=device).manual_seed(0)
    sd = model.state_dict()
    kinds = {k: (shape, kind) for k, shape, kind in weight_shapes(cfg)}
    with torch.no_grad():
        for k, p in sd.items():
            shape, kind = kinds[k]
            p.normal_(0.0, init_std(kind, shape), generator=gen)
            if kind == "g":
                p.add_(1.0)
    model.invalidate_engine()
    return model.eval()


def synth_host_inputs(B, Lt, seed):
    g = torch.Generator().manual_seed(seed)
    images_host = torch.randn(B, 3, 336, 336, generator=g).pin_memory()
    ids_host = torch.randint(3, VOCAB, (B, Lt), generator=g)
    ids_host[:, 0] = 1
    ids_host[:, 5] = IMAGE_TOKEN
    return images_host, ids_host.pin_memory()


def measure_device_resident(engine, m, B, S, N, steps, warmup, seed=1, fp8=False, world=1, dev=None, sampler=None,
                            isolate_decode=False, return_outputs=False):
    """One workload through the C-ABI with every input already in HBM: encode_images -> splice -> prefill -> N-1 greedy decode
    steps, timed with CUDA events on the launching stream. Returns per-stage ms (max over ranks) and derived rates, and with
    `return_outputs` the last timed step's results as host tensors."""
    import numpy as np
    from llava import _b2
    from llava._b2 import replicas
    from llava.model.llava_arch import build_source_index

    Lt = S - P_IMG + 1
    images_host, ids_host = synth_host_inputs(B, Lt, seed)
    pixels = images_host.to(dev, torch.bfloat16)
    ids_np = ids_host.numpy().astype(np.int64)
    src, _, _, _, lens = build_source_index(ids_np, np.ones_like(ids_np, bool), np.full_like(ids_np, -100),
                                            B * P_IMG, [P_IMG] * B, None, "right")
    src_dev = torch.from_numpy(src.reshape(-1)).to(dev)
    kv = engine.new_kv(B, S + N + 8)
    out_tokens = torch.empty(max(N - 1, 1), B, dtype=torch.int32, device=dev)

    def device_step(ev=None):
        if ev: ev[0].record()
        feats = engine.encode_images(pixels)
        if ev: ev[1].record()
        embeds = engine.splice(src_dev, feats.view(-1, feats.shape[-1]), B, S)
        kv.reset()
        logits = engine.prefill(kv, embeds, lens, _b2.LOGITS_LAST)
        first = engine.argmax(logits)
        if ev: ev[2].record()
        if N > 1:
            engine.decode_greedy(kv, first, N - 1, out=out_tokens)
        if ev: ev[3].record()
        return feats, logits, first

    for _ in range(warmup):
        device_step()
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.start()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
    launches0 = _b2.launch_count()
    for i in range(steps):
        last = device_step(evs[i])
    torch.cuda.synchronize()
    launches = _b2.launch_count() - launches0
    clocks = sampler.stop() if sampler is not None else None
    outputs = None
    if return_outputs:
        feats, logits, first = last
        outputs = {"tokens": torch.cat([first[None], out_tokens[:N - 1]]).t().double().cpu(),
                   "prefill_logits": logits.float().cpu(), "image_features": feats.float().cpu()}
    t_enc = sum(e[0].elapsed_time(e[1]) for e in evs) / steps
    t_pre = sum(e[1].elapsed_time(e[2]) for e in evs) / steps
    t_dec = sum(e[2].elapsed_time(e[3]) for e in evs) / steps
    t_total = evs[0][0].elapsed_time(evs[-1][3]) / steps  # ms per step, back to back
    t_total, t_enc, t_pre, t_dec = (replicas.max_over_ranks(t, dev) for t in (t_total, t_enc, t_pre, t_dec))
    engine.check_async_error()
    dec_iso = None
    if isolate_decode and N > 1:
        # the same decode steps timed on their own: inside the step they start right behind a tensor-bound prefill of B*S
        # tokens, i.e. under the power cap's reduced SM clock (MEASURED_PEAKS.json: 1230 MHz sustained vs 1965 MHz)
        ts = []
        for _ in range(2):
            feats = engine.encode_images(pixels)
            embeds = engine.splice(src_dev, feats.view(-1, feats.shape[-1]), B, S)
            kv.reset()
            first = engine.argmax(engine.prefill(kv, embeds, lens, _b2.LOGITS_LAST))
            torch.cuda.synchronize()
            time.sleep(0.25)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            engine.decode_greedy(kv, first, N - 1, out=out_tokens)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / (N - 1))
        dec_iso = min(ts)
    kv.close()
    work = algorithmic_work(m, B, S, N, fp8=fp8)
    hbm_peak, tf_peak, _ = peaks()
    steps_dec = max(N - 1, 1)
    dec_ms = t_dec / steps_dec
    return dict(t_total=t_total, t_enc=t_enc, t_pre=t_pre, t_dec=t_dec, dec_step_ms=dec_ms, launches=launches, clocks=clocks,
                dec_step_ms_isolated=dec_iso,
                work=work, out_tokens=out_tokens, images_host=images_host, ids_host=ids_host, outputs=outputs,
                decode_gbs=work["decode_bytes_per_step"] / (dec_ms * 1e-3) / 1e9,
                decode_frac=work["decode_bytes_per_step"] / (dec_ms * 1e-3) / 1e9 / hbm_peak,
                prefill_tflops=work["prefill_flops"] / (t_pre * 1e-3) / 1e12,
                encode_tflops=work["encode_flops"] / (t_enc * 1e-3) / 1e12)


DUMP_BYTES = 64 << 20


def dump_outputs(path, outputs):
    """Writes each host tensor as <path>/<name>.npy (float64 token ids, float32 otherwise). An array that does not fit in
    what is left of DUMP_BYTES keeps a fixed, seeded sample of its rows (last dimension kept whole); the sampled row
    indices go to <name>_rows.npy."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES
    for name, t in outputs.items():
        a = t.numpy()
        if a.nbytes > left:
            rows = a.reshape(-1, a.shape[-1])
            k = max(1, left // (rows.shape[1] * a.itemsize + 8) - 1)
            idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], size=k, replace=False))
            a = rows[idx]
            np.save(os.path.join(path, f"{name}_rows.npy"), idx.astype(np.float64))
            left -= idx.size * 8 + 128
        np.save(os.path.join(path, f"{name}.npy"), a)
        left -= a.nbytes + 128  # .npy header


def config_line(name, m, B, S, N, r, fp8=False):
    hbm_peak, tf_peak, peak_kind = peaks()
    return {"workload": name, "model": m["name"], "batch": B, "seq_len": S, "new_tokens": N,
            "value": B * (S + N) / (r["t_total"] * 1e-3), "unit": "tokens/s", "ms_per_step": r["t_total"],
            "decode_tok_s": B * max(N - 1, 1) / (r["t_dec"] * 1e-3), "decode_ms_per_token_step": r["dec_step_ms"],
            "prefill_tok_s": B * S / (r["t_pre"] * 1e-3), "images_per_s": B / (r["t_enc"] * 1e-3),
            "dtype": "e4m3 decoder Linears in decode, bf16 elsewhere" if fp8 else "bf16",
            "roofline": {"bound": "hbm", "kernel": "decode step", "achieved": r["decode_gbs"], "peak": hbm_peak, "unit": "GB/s",
                         "frac": r["decode_frac"], "algorithmic_bytes_per_step": r["work"]["decode_bytes_per_step"],
                         "peak_source": peak_kind},
            "decode_isolated": None if r.get("dec_step_ms_isolated") is None else {
                "ms_per_token_step": r["dec_step_ms_isolated"],
                "frac": r["work"]["decode_bytes_per_step"] / (r["dec_step_ms_isolated"] * 1e-3) / 1e9 / hbm_peak,
                "how": "the same N-1 decode steps timed on their own after a 0.25 s pause (not right behind the B*S-token prefill)"},
            "clocks": r.get("clocks"),
            "prefill_frac_of_bf16_peak": r["prefill_tflops"] / tf_peak, "encode_frac_of_bf16_peak": r["encode_tflops"] / tf_peak}


def extra_configs(args, dev, model7b):
    """The other halves of BASELINE.json's metric ("bs=1/32", 13B, ViT bs=256, fp8) as bounded side measurements in the
    same process (N=1 only), each with its own roofline fraction from CUDA events. Short decode runs (64 steps): the
    step time is flat in this regime."""
    out = []
    hbm_peak, tf_peak, peak_kind = peaks()
    S, N, steps, warm = P_IMG + args.prompt, 64, 2, 2

    def rebuild(model, max_batch, max_images):
        model.engine_limits(max_batch=max_batch, max_seq=S + N + 8, max_images=max_images)
        model.invalidate_engine()
        return model._ensure_engine()

    # configs[2]: encode_images only, 256 images in chunks of 64
    m7 = MODELS["7b"]
    eng = rebuild(model7b, 32, 64)
    g = torch.Generator().manual_seed(7)
    px = torch.randn(256, 3, 336, 336, generator=g).to(dev, torch.bfloat16)
    for _ in range(2):
        eng.encode_images(px)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        eng.encode_images(px)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    flops = 256 * (VIT_GF * 1e9 + 2 * P_IMG * (1024 * m7["hidden"] + m7["hidden"] ** 2))
    out.append({"workload": "BASELINE configs[2]: CLIP ViT-L/14-336 + 7B projector encode_images, bs=256 (chunks of 64)",
                "value": 256 / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms,
                "roofline": {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                             "frac": flops / (ms * 1e-3) / 1e12 / tf_peak, "peak_source": peak_kind}})
    del px
    # the same 256 images starting from uint8 HWC frames on the HOST: H2D + PIL-exact resize / pad / normalise kernels
    # (llava/_b2/preprocess.py, replaces mm_utils.process_images) + encode_images, wall clock
    try:
        import numpy as np
        from llava._b2.preprocess import ClipPreprocessor
        pre = ClipPreprocessor(model7b.get_vision_tower().image_processor, device=dev, image_aspect_ratio="pad")
        rng = np.random.default_rng(0)
        frames = [rng.integers(0, 256, (480, 640, 3), dtype=np.uint8) for _ in range(32)] * 8
        eng.encode_images(pre(frames))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(2):
            eng.encode_images(pre(frames))
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 2
        out[-1]["from_uint8_host_frames"] = {"value": 256 / dt, "unit": "images/s", "ms_per_step": dt * 1e3,
                                             "input": "256 x uint8 [480,640,3] on the host, image_aspect_ratio=pad",
                                             "h2d_bytes_per_step": 256 * 480 * 640 * 3}
    except Exception as e:
        out[-1]["from_uint8_host_frames"] = {"error": repr(e)[:300]}
    # the "bs=32" half of the metric, 7B
    r = measure_device_resident(eng, m7, 32, S, N, steps, warm, dev=dev, isolate_decode=True, sampler=ClockSampler(dev.index or 0))
    out.append(config_line("LLaVA-1.5-7B bf16 bs=32: 576+%d prefill, %d-token decode" % (args.prompt, N), m7, 32, S, N, r))
    # configs[4]: fp8-weight decode, bs=64
    try:
        eng = rebuild(model7b, 64, 16)
        eng.enable_fp8_decode()
        r = measure_device_resident(eng, m7, 64, S, N, steps, warm, dev=dev, fp8=True, isolate_decode=True,
                                    sampler=ClockSampler(dev.index or 0))
        out.append(config_line("BASELINE configs[4]: LLaVA-1.5-7B fp8-weight decode bs=64", m7, 64, S, N, r, fp8=True))
    except Exception as e:  # reported, never hidden
        out.append({"workload": "BASELINE configs[4]", "error": repr(e)[:300]})
    model7b.invalidate_engine()
    return out


def extra_13b(args, dev):
    m = MODELS["13b"]
    S, N = P_IMG + args.prompt, 64
    model = build_model(m, dev, 32, S + N + 8)
    eng = model._ensure_engine()
    r = measure_device_resident(eng, m, 32, S, N, 2, 2, dev=dev, isolate_decode=True, sampler=ClockSampler(dev.index or 0))
    line = config_line("BASELINE configs[3]: LLaVA-1.5-13B bf16 bs=32 per GPU: 576+%d prefill, %d-token decode" % (args.prompt, N),
                       m, 32, S, N, r)
    model.invalidate_engine()
    del model
    torch.cuda.empty_cache()
    return line


class _QueueStreamer:
    """put()/end() into a queue drained by the caller's thread — the shape of transformers.TextIteratorStreamer without
    a tokenizer (llava/serve/model_worker.py:166 builds one per request)."""

    def __init__(self):
        import queue
        self.q = queue.Queue()

    def put(self, value):
        self.q.put(value)

    def end(self):
        self.q.put(None)


def measure_e2e_stream(model, ids_host, images_host, N, steps, warmup):
    """generate() exactly as the reference's worker calls it (llava/serve/model_worker.py:166-188): from a non-main Thread,
    with a streamer drained by this thread and a keyword-style stopping criterion that inspects the tail of the ids at
    every token. Wall clock around the whole request (thread start to join), host buffers in, host ids out."""
    import threading

    class TailCriterion:  # same per-token work as KeywordsStoppingCriteria: compare the tail against keyword ids
        def __init__(self, start_len):
            self.start_len, self.kw = start_len, torch.tensor([VOCAB + 1, VOCAB + 2])  # never matches

        def __call__(self, output_ids, scores, **kw):
            return bool((output_ids[0, -2:] == self.kw).all()) if output_ids.shape[1] - self.start_len >= 2 else False

    def one():
        st, res = _QueueStreamer(), {}
        crit = TailCriterion(ids_host.shape[1])

        def work():
            res["out"] = model.generate(inputs=ids_host, images=images_host, do_sample=False, temperature=0.0, top_p=1.0,
                                        max_new_tokens=N, streamer=st, stopping_criteria=[crit], use_cache=True, eos_token_id=[])
        th = threading.Thread(target=work)
        t0 = time.perf_counter()
        th.start()
        n, first_at = 0, None
        while True:
            v = st.q.get(timeout=120)
            if v is None:
                break
            n += 1
            if n == 2 and first_at is None:  # put #1 is the prompt, #2 the first generated token
                first_at = time.perf_counter() - t0
        th.join()
        return time.perf_counter() - t0, first_at, res["out"]

    for _ in range(warmup):
        one()
    ts, firsts = [], []
    for _ in range(steps):
        t, f, out = one()
        ts.append(t); firsts.append(f)
    return sum(ts) / len(ts), sum(firsts) / len(firsts), out


def ncu_traffic_from_profile():
    """dram__bytes_read.sum + dram__bytes_write.sum of one decode_mega_kernel launch, parsed at run time from the newest committed
    `ncu --set full` summary under profiles/ (lines `metric  value  unit`); null when no capture is committed."""
    import glob
    import re
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_prof_mega_ncu_full.txt"))):
        txt = open(path).read()
        vals = []
        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            mt = re.search(r"^" + re.escape(name) + r"\s+([\d.,]+)\s+(\w+)\s*$", txt, re.M)
            if mt and mt.group(2) in unit:
                vals.append(float(mt.group(1).replace(",", "")) * unit[mt.group(2)])
        if len(vals) == 2:
            best = (vals[0] + vals[1], os.path.basename(path))
    return best


def run_ours(args):
    import torch.distributed as dist
    from llava import _b2
    from llava._b2 import replicas

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun)"
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    m = MODELS[args.model]
    B, N = args.batch, args.new
    Lt = args.prompt + 1
    S = args.prompt + P_IMG
    model = build_model(m, dev, B, S + N + 8)
    engine = model._ensure_engine()
    if args.fp8:
        if B < 7:
            raise ValueError("--fp8 only changes decode at batch >= 7 per GPU (smaller batches keep the bf16 paths)")
        engine.enable_fp8_decode()

    stream = torch.cuda.Stream(device=dev)
    hbm_peak, tf_peak, peak_kind = peaks()
    with torch.cuda.stream(stream), torch.no_grad():
        # ---------------- device-resident arm ----------------
        r = measure_device_resident(engine, m, B, S, N, args.steps, args.warmup, seed=1 + rank, fp8=args.fp8, world=world,
                                    dev=dev, sampler=ClockSampler(local) if rank == 0 else None,
                                    return_outputs=bool(args.dump_outputs) and rank == 0)
        if r["outputs"] is not None:
            dump_outputs(args.dump_outputs, r.pop("outputs"))
        images_host, ids_host, out_tokens = r["images_host"], r["ids_host"], r["out_tokens"]
        tokens_per_step = world * B * (S + N)
        value = tokens_per_step / (r["t_total"] * 1e-3)

        # ---------------- end-to-end arm: public API, host buffers ----------------
        e2e = e2e_stream = None
        if not args.no_e2e:
            def api_step():
                # eos disabled (SURVEY §8d: every run does exactly N steps; random-init logits can hit id 2 by chance)
                return model.generate(ids_host, images=images_host, do_sample=False, max_new_tokens=N, use_cache=True,
                                      eos_token_id=[])
            for _ in range(max(1, min(args.warmup, 2))):
                api_step()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                out = api_step()
            e1.record()
            torch.cuda.synchronize()
            assert out.shape == (B, Lt + N) and out.device.type == "cpu"
            # the API path and the device-resident path must generate the same ids (same kernels, same inputs)
            ids_equal = bool(torch.equal(out[:, Lt + 1:].to(torch.int32), out_tokens.t().cpu()))
            t_e2e = replicas.max_over_ranks(e0.elapsed_time(e1) / args.steps, dev)
            e2e = {"value": tokens_per_step / (t_e2e * 1e-3), "unit": "tokens/s", "ms_per_step": t_e2e,
                   "h2d_bytes_per_step": int(images_host.numel() * 4 + ids_host.numel() * 8 + B * S * 4),
                   "d2h_bytes_per_step": int(B * N * 4), "ids_equal_device_resident_arm": ids_equal}
            if rank == 0 and B == 1:
                t_s, t_first, out_s = measure_e2e_stream(model, ids_host, images_host, N, max(2, min(args.steps, 5)), 1)
                e2e_stream = {"value": B * (S + N) / t_s, "unit": "tokens/s", "ms_per_step": t_s * 1e3,
                              "first_token_ms": t_first * 1e3, "ids_equal_plain_generate": bool(torch.equal(out_s.cpu(), out)),
                              "how": "generate(streamer=queue streamer, stopping_criteria=[tail criterion]) on a worker Thread, "
                                     "wall clock thread start -> join, host buffers (llava/serve/model_worker.py:166-188 pattern)"}
        # eval-harness gather of the generated ids over NCCL (outside the timed region; never on the hot path)
        if world > 1:
            replicas.gather_rows(out_tokens.t().contiguous(), world * B)

        configs = None
        if rank == 0 and world == 1 and not args.no_configs and args.model == "7b" and B == 1 and not args.fp8:
            configs = extra_configs(args, dev, model)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if configs is not None:
        model.invalidate_engine()
        del model, engine
        torch.cuda.empty_cache()
        with torch.cuda.stream(stream), torch.no_grad():
            try:
                configs.append(extra_13b(args, dev))
            except Exception as e:
                configs.append({"workload": "BASELINE configs[3]", "error": repr(e)[:300]})
    work = r["work"]
    steps_dec = max(N - 1, 1)
    traffic = ncu_traffic_from_profile() if (args.model == "7b" and B == 1) else None
    mega = B <= 2
    out = {
        "metric": "prefill+decode tokens/s", "value": value, "unit": "tokens/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["t_total"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "e4m3 decoder Linears in decode (per-channel / per-token scales), bf16 elsewhere" if args.fp8 else "bf16",
        "data": "synthetic",
        "config": workload_config(args, m, S),
        "breakdown": {"encode_images_ms": r["t_enc"], "prefill_ms": r["t_pre"], "decode_ms": r["t_dec"],
                      "decode_ms_per_token": r["dec_step_ms"], "images_per_s": world * B / (r["t_enc"] * 1e-3),
                      "prefill_tok_s": world * B * S / (r["t_pre"] * 1e-3),
                      "decode_tok_s": world * B * steps_dec / (r["t_dec"] * 1e-3),
                      "prefill_tflops": r["prefill_tflops"], "prefill_frac_of_bf16_peak": r["prefill_tflops"] / tf_peak,
                      "encode_tflops": r["encode_tflops"], "encode_frac_of_bf16_peak": r["encode_tflops"] / tf_peak},
        "roofline": {"bound": "hbm", "achieved": r["decode_gbs"], "peak": hbm_peak, "unit": "GB/s",
                     "frac": r["decode_frac"], "traffic": traffic[0] if traffic else None,
                     "traffic_source": traffic[1] if traffic else None, "peak_source": peak_kind,
                     "kernel": ("decode_mega_kernel: one persistent cooperative launch per generated token (all layers' GEMV phases "
                                "streamed through a TMA smem ring, attention, lm_head, argmax)") if mega else
                               "decode step (CUDA graph of the per-layer decode kernels)",
                     "algorithmic_bytes_per_launch": work["decode_bytes_per_step"],
                     "avg_launch_ms": r["dec_step_ms"]},
        "e2e": e2e, "e2e_stream": e2e_stream, "gpu_launches": int(r["launches"]), "clocks": r["clocks"],
    }
    if configs is not None:
        out["configs"] = configs
    if not args.no_cpu_baseline and world == 1:
        cpu_reference_sample(m, S, N, sample_layers=1, decode_steps=1)   # warm-up: thread pool, allocator, weights
        cbs = [cpu_reference_sample(m, S, N) for _ in range(2)]
        cpu_unpin()
        cb = dict(cbs[-1])
        cb["value"] = sum(c["value"] for c in cbs) / len(cbs)
        out["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "breakdown", "extrapolated", "sampled_layers")}
        out["cpu_baseline"]["samples_tok_s"] = [c["value"] for c in cbs]
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py (our arm) needs a B200; there is no CPU fallback. Use --impl reference for the CPU arm.")
        run_ours(args)


if __name__ == "__main__":
    main()

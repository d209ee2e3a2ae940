#!/usr/bin/env python
"""bench.py — crops/s through the VSM+VQA forward of the V* guided visual-search hot path (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...          # the reference's CPU path (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR        # also write what the last timed `value` step returned (dump_outputs)

Headline workload = BASELINE.json configs[2] (SURVEY.md §8d config 3): 2048x2048 synthetic images, smallest_size 512 => every
search evaluates 1 + 4 + 16 = 21 crops; 8 searches run in lock-step, each feeding up to 8 frontier crops into a batch of <= 64
crops; after the searches every search's question is answered by ONE SEAL-VQA `multiple_choices_inference` (4 options, 2 object
crops spliced in as <object> features: vstar_bench_eval.py:116-165, :226-257; the 8 scorings of a step run as one batch).
A "step" = those 8 searches + 8 option scorings; crops/s = 168 / step time.  Every crop evaluation = CLIP ViT-L/14 -> projector -> Vicuna-7B-shaped prefill (draft
-verified answer) -> OWL-ViT-B/16 -> SAM prompt/mask decoder -> OWL heads -> crop record (heat-map statistics + rectangle sums);
random-init weights of the reference architecture, synthetic images.

  value   : crops/s with the search images resident in HBM (uint8) and the VQA pixel tensors on the device at the start
  e2e     : crops/s through the public API from PIL images: `visual_search_many(VSM, ...)` + `seal.choose_option(VQA_LLM, ...)`
            (pinned H2D of every search image, device crop/resize, host PIL preprocessing of the VQA image and object crops,
            D2H of the crop records and option losses) inside the timed region
  configs1: the round-1 headline (BASELINE.json configs[1]: 1024^2, root + 4 crops, 32 lock-step searches), same two numbers
  frontier: STRONG scaling of configs[3]-shaped work: 4 searches of 4096^2 images (85 crops each), every frontier batch dealt
            over ALL ranks by ShardedVSM (one all_gather_into_tensor of crop records per batch), weights broadcast from rank 0
            with NCCL; rank 0 asserts that the sharded trajectory equals its own single-GPU trajectory before printing
N > 1 (`value`): searches are sharded over ranks (independent units, weights replicated, no data-path collective); time = max
over ranks of CUDA-event time, value = crops of all ranks / that time ("weak" scaling).
"""
import argparse
import atexit
import csv
import glob
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_CROP = 5.00e12      # BASELINE.md §3 (T=320, g=6, KV-cached); roofline 289 crops/s/GPU at 1443 TF/s
METRIC = "crops/s through the VSM+VQA forward (guided visual search hot path)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--searches", type=int, default=8, help="concurrent searches per step per GPU (configs[2] leg)")
    ap.add_argument("--image", type=int, default=2048)
    ap.add_argument("--smallest", type=int, default=512)
    ap.add_argument("--batch", type=int, default=64, help="frontier batch (crops per engine call)")
    ap.add_argument("--no-vqa", action="store_true", help="skip the SEAL-VQA option-scoring leg (debug; not the BASELINE metric)")
    ap.add_argument("--tiny", action="store_true", help="tiny model (debug only; not a valid bench)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-legs", action="store_true", help="skip configs1 / frontier / vqa probe / torch baseline legs")
    ap.add_argument("--attn-impl", type=int, default=0, help="A/B switch for vsb_attn_set_impl (0 = production dispatch)")
    ap.add_argument("--profile-range", action="store_true", help="cudaProfilerStart/Stop around the timed resident steps (for ncu)")
    ap.add_argument("--no-prefix-cache", action="store_true",
                    help="recompute the K/V rows of the constant text prefix (system prompt before <im_start>) for every crop")
    ap.add_argument("--gemm-l2-hints", type=int, default=-1, help="A/B switch for vsb_gemm_set_l2_hints (-1 = library default)")
    ap.add_argument("--fuse-rope", type=int, default=-1, help="A/B switch for vsb_llama_set_fuse_rope (-1 = library default)")
    ap.add_argument("--depth", type=int, default=2, help="frontier batches in flight (1 = round-1 style synchronous rounds)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0's searches and option scorings) to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return j["bf16_tflops_sustained"], j["hbm_gbs"], "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def gemm_traffic_from_profile():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant GEMM launch, read from the newest committed ncu export of
    the CURRENT kernel (profiles/rNN_gemm_dram_bytes.csv, written by tools/prof_gemm.py under ncu); None if there is none"""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r[0-9][0-9]_gemm_dram_bytes.csv")))
    if not files:
        return None, "no profiles/rNN_gemm_dram_bytes.csv committed"
    path = files[-1]
    unit_scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    per_id = {}
    with open(path, newline="") as f:
        rows = [r for r in csv.reader(l for l in f if l.startswith('"'))]
    if not rows:
        return None, f"{os.path.basename(path)}: empty"
    head = rows[0]
    try:
        i_id, i_name, i_unit, i_val = head.index("ID"), head.index("Metric Name"), head.index("Metric Unit"), head.index("Metric Value")
    except ValueError:
        return None, f"{os.path.basename(path)}: unexpected header"
    for r in rows[1:]:
        if r[i_name] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            per_id.setdefault(r[i_id], 0.0)
            per_id[r[i_id]] += float(r[i_val].replace(",", "")) * unit_scale.get(r[i_unit], 1.0)
    if not per_id:
        return None, f"{os.path.basename(path)}: no dram__bytes rows"
    last = sorted(per_id, key=lambda k: int(k))[-1]
    return per_id[last], f"dram__bytes_read.sum + dram__bytes_write.sum of the last profiled launch in profiles/{os.path.basename(path)}"


class ClockSampler:
    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}",
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)        # no sampler outlives the run when a step raises before stop()
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def host_threads():
    # all host threads the box gives us (torchrun exports OMP_NUM_THREADS=1, which would silently make this a 1-core baseline).
    # Measured on the pool's boxes in round 1: 64 threads -> 12 s per crop, 128 SMT threads -> 180 s (oversubscribed fp32 GEMMs).
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return min(max(1, n), 64)


# ----------------------------------------------------------------------------------------------------------------
# synthetic VQA question (no sentencepiece model offline: hash-word tokenizer, SURVEY.md §8c)
# ----------------------------------------------------------------------------------------------------------------
QUESTION = "What is the color of the mug that is next to the laptop on the wooden desk in this picture?"
OPTIONS = ["The color of the mug is red.", "The color of the mug is blue.", "The color of the mug is green.",
           "The color of the mug is white."]
TARGETS = ("mug", "laptop")


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port of the reference's CPU path on the host cores (bounded sample)
# ----------------------------------------------------------------------------------------------------------------
class _CpuModels:
    """fp32 random-init weights of both models for the oracle.  ALL 32 decoder layers are executed; layers 1..31 alias layer
    0's tensors (CPU timing does not depend on the values: a layer streams 809 MB of fp32 weights, far beyond the caches, and
    the GEMMs are compute-bound) which saves 26 GB of host RAM and a minute of RNG per model."""

    def __init__(self, tiny=False):
        import torch
        from oracle import vqa_oracle as V
        from vstar_b200 import synth
        from vstar_b200.config import VSMConfig, tiny_config
        self.cfg = tiny_config() if tiny else VSMConfig()
        cfg = self.cfg
        shapes = synth.state_dict_shapes(cfg)
        sd = {}
        for name, shape in shapes.items():
            if name.startswith("model.layers.") and not name.startswith("model.layers.0."):
                continue
            sd[name] = synth.synthetic_tensor(name, shape, seed=1234)
        for i in range(1, cfg.n_layers):
            for name in [k for k in sd if k.startswith("model.layers.0.")]:
                sd[name.replace("model.layers.0.", f"model.layers.{i}.")] = sd[name]
        self.sd = sd
        sdv = dict(sd)
        for name, shape in V.vqa_state_dict_shapes(cfg).items():
            if name not in sdv:
                sdv[name] = synth.synthetic_tensor(name, shape, seed=4321)
        self.sd_vqa = sdv
        prompt, ans = synth.synthetic_prompt(cfg, n_text=60, seed=0, im_start_index=None if tiny else 37)
        self.ids = torch.cat([prompt, ans.unsqueeze(0)], dim=1)


_cpu_models = None


def cpu_reference_sample(args):
    """One bounded sample of the configs[2] workload through oracle/ (the CPU restatement of the reference), fp32, all layers:
      * the ROOT crop of a 2048x2048 search through the oracle's VSM.inference equivalent: PIL crop + expand2square + both
        bicubic resizes (visual_search.py:186-194) + VSMForCausalLM.model_forward(inference=True) + clamp + heat-map max,
      * ONE option scoring (4 options, 2 object crops, image short / objects long) through the oracle's
        LlavaSearchLlamaForCausalLM path as written (question prefilled once with use_cache, options appended on its KV cache,
        vstar_bench_eval.py:127-163) incl. the host preprocessing of the padded image and the object crops.
    crops/s for the whole search = 21 / (21 * t_crop + t_vqa).  Returns (crops/s, seconds of the sample, description, threads)."""
    global _cpu_models
    import numpy as np
    import torch
    from PIL import Image
    from oracle import vqa_oracle as V
    from oracle import vsm_oracle as O
    from vstar_b200.vqa import SyntheticTokenizer, build_prompt_v1, tokenizer_image_object_token
    from vstar_b200 import seal
    n_threads = host_threads()
    torch.set_num_threads(n_threads)
    if _cpu_models is None:
        _cpu_models = _CpuModels(args.tiny)
    m = _cpu_models
    cfg = m.cfg
    side = 256 if args.tiny else args.image
    img = Image.fromarray(np.random.default_rng(0).integers(0, 256, (side, side, 3), dtype=np.uint8), "RGB")
    t = {}
    with torch.no_grad():
        t0 = time.perf_counter()
        crop = img.crop((0, 0, side, side))
        images, images_clip = O.preprocess_owl(crop), O.preprocess_clip(crop)
        t["crop_preprocess"] = time.perf_counter() - t0
        out = O.model_forward_inference(m.sd, cfg, images, images_clip, m.ids, (side, side))
        _ = float(out["pred_masks"].clamp(min=0).max())
        _ = out["pred_logits"].sigmoid().argmax()
        t["crop_total"] = time.perf_counter() - t0
        # VQA leg
        t1 = time.perf_counter()
        tok = SyntheticTokenizer(cfg)
        bg = tuple(int(x * 255) for x in O.CLIP_MEAN)
        padded, left, top = V.expand2square_center(img, bg)
        boxes = [[side * 0.3, side * 0.4, side * 0.1, side * 0.12], [side * 0.6, side * 0.2, side * 0.08, side * 0.1]]
        crops = []
        for b in boxes:
            p = V.get_patch(b, img.width, img.height, patch_scale=1.2)
            crops.append(O.preprocess_clip(img.crop((p[0], p[1], p[2], p[3])).resize((224, 224))))
        crops = torch.cat(crops, 0)
        image_t = O.preprocess_clip(padded)
        nb = [seal.normalize_bbox([b[0] + left, b[1] + top, b[2], b[3]], padded.width, padded.height) for b in boxes]
        qs = "<image>\n" + seal.focus_question(QUESTION, list(TARGETS), nb)
        q_ids = tokenizer_image_object_token(build_prompt_v1(qs), tok)
        opt_ids = [tokenizer_image_object_token(build_prompt_v1(qs, o), tok)[len(q_ids):] for o in OPTIONS]
        q = torch.tensor([q_ids])
        losses, choice = V.option_losses_cached(m.sd_vqa, cfg, q, [torch.tensor(o) for o in opt_ids], image_t, crops, [False], [True, True])
        t["vqa_total"] = time.perf_counter() - t1
    n_crops = 21
    sec_search = n_crops * t["crop_total"] + t["vqa_total"]
    desc = (f"configs[2] sample, fp32, oracle port, all {cfg.n_layers} Llama layers executed (layers 1.. alias layer 0's random weights): "
            f"1 root crop of a {side}x{side} search incl. PIL preprocessing ({t['crop_preprocess']:.2f} s of {t['crop_total']:.2f} s) + "
            f"1 option scoring with 4 options / 2 object crops ({t['vqa_total']:.2f} s); crops/s = 21 / (21 x crop + vqa)")
    return n_crops / sec_search, t["crop_total"] + t["vqa_total"], desc, n_threads


def torch_gpu_reference_sample(cfg, n_crops=3):
    """The reference's AS-WRITTEN GPU path restated with plain torch eager ops (oracle/vsm_oracle.py on cuda:0, bf16):
    batch 1, `generate(use_cache=False)` = one full CLIP + 7B pass per emitted token (5 here), lm_head and both query MLPs
    on all T rows, OWL-ViT, SAM decoder, heads, heat-map (VSM.py:438-553).  This is the "reference PyTorch-GPU" number the
    north-star's >= 10x is measured against; the reference itself cannot travel to the GPU box (Python sources under
    /root/reference + transformers 4.31), so its restatement stands in.  Host preprocessing excluded (favours the baseline)."""
    import torch
    from oracle import vsm_oracle as O
    from vstar_b200 import synth
    shapes = synth.state_dict_shapes(cfg)
    sd = {n: synth.synthetic_tensor(n, shp, seed=1234, dtype=torch.bfloat16, device="cuda") for n, shp in shapes.items()}
    prompt, ans = synth.synthetic_prompt(cfg, n_text=60, seed=0)
    prompt = prompt.cuda()
    g = torch.Generator(device="cuda").manual_seed(0)
    ic = torch.randn(1, 3, cfg.clip_image, cfg.clip_image, device="cuda", generator=g).bfloat16()
    io = torch.randn(1, 3, cfg.owl_image, cfg.owl_image, device="cuda", generator=g).bfloat16()
    with torch.no_grad():
        O.vsm_inference(sd, cfg, ic, io, prompt, (512, 512), max_new_tokens=100, mode="detection", forced_ids=ans)     # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_crops):
            out = O.vsm_inference(sd, cfg, ic, io, prompt, (512, 512), max_new_tokens=100, mode="detection", forced_ids=ans)
            _ = out["pred_masks"].clamp(min=0).max().item()
        e1.record()
        torch.cuda.synchronize()
    del sd
    torch.cuda.empty_cache()
    return n_crops / (e0.elapsed_time(e1) / 1e3)


def reference_config(args):
    return {"workload": f"BASELINE.json configs[2] on the host CPU: bounded sample = the root crop of one {args.image}x{args.image} search "
                        "(PIL preprocessing + 1-crop VSM forward, fp32, all 32 layers) + one SEAL-VQA option scoring (4 options, 2 object "
                        "crops); value = 21 crops / (21 x crop seconds + option-scoring seconds); oracle port of the reference "
                        "(oracle/vsm_oracle.py, oracle/vqa_oracle.py), random-init weights, synthetic image",
            "image": args.image, "crops_per_search": 21}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warmup = min(args.warmup, 1)          # one warm-up sample pages the weights in; more would only add minutes of CPU time
    for _ in range(warmup):
        cpu_reference_sample(args)
    vals, secs = [], []
    for _ in range(args.steps):
        v, s, desc, cores = cpu_reference_sample(args)
        vals.append(v)
        secs.append(s)
    v = sum(vals) / len(vals)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "crops/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup, "ms_per_step": 1e3 * sum(secs) / len(secs),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": reference_config(args),
        "cpu_baseline": {"value": v, "unit": "crops/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": "crops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(args):
    return {"workload": f"BASELINE.json configs[2]: {args.image}x{args.image} synthetic images, smallest_size {args.smallest} "
                        f"(1 + 4 + 16 = 21 crops per search), {args.searches} lock-step searches per step per GPU each feeding <= "
                        f"{max(1, args.batch // max(1, args.searches))} frontier crops into batches of <= {args.batch} crops, "
                        + ("no VQA leg (debug)" if args.no_vqa else "+ one SEAL-VQA multiple_choices_inference (4 options, 2 object crops) per search")
                        + ", bf16, random-init Vicuna-7B/CLIP-L/OWL-B/SAM-decoder/perceiver weights, T=315+5 tokens, forced answer ids",
            "searches_per_step": args.searches, "frontier_batch": args.batch, "image": args.image, "batches_in_flight": args.depth,
            "l2": "weights (13.5 GB per model) and activations exceed the 126 MB L2 every step; no explicit flush",
            "prefix_cache": ("off" if args.no_prefix_cache else
                             "on: K/V of the 37 constant prompt tokens before <im_start> snapshotted at the first (warm-up) prefill and "
                             "shared by all crops; identical results, see DESIGN.md §3 (--no-prefix-cache recomputes them)")}


def dump_outputs(path, results, states, scored):
    """Write what one step returned to its caller as DIR/<name>.npy (float64; the option losses float32), so that two builds
    can be compared output for output.  Nothing is padded: every value is one the step computed, or 0 where a flag says so.
    Per search (S searches):
      search_final_bbox [S,4], search_detection_result [S,4], search_path_length [S], search_success [S]: the result tuple
      search_valid_boxes_count [S], and search_valid_boxes [sum of the counts, 4] when it is not empty: all_valid_boxes of
        the searches that succeeded at their root, concatenated in search order
    Per expanded node, the search paths concatenated in search order (search_path_nodes [S] nodes per search, N in all):
      search_path_bbox [N,4], search_path_score [N]: the node and its queue priority (0 for a root, which is never queued)
      search_path_detected [N]: 1 where the node kept its best detection as a candidate (a node where a search succeeds
        holds it in search_detection_result instead), with search_path_top_logit [N] and search_path_box [N,4] (crop
        coordinates) set there and 0 elsewhere
    Per option scoring (if the step ran one): vqa_option_losses [S,n_options], vqa_choice [S]."""
    import numpy as np

    def f64(x):
        return np.asarray(x.tolist() if hasattr(x, "tolist") else x, dtype=np.float64)

    nodes = [node for st in states for node in st.search_path]
    det = [node.get("temp_detection_result") for node in nodes]
    valid = [f64(av).reshape(-1, 4) for _, _, _, av in results if av is not None and len(av)]
    out = {"search_final_bbox": f64([fs["bbox"] for fs, _, _, _ in results]),
           "search_detection_result": f64([f64(fs["detection_result"]) for fs, _, _, _ in results]),
           "search_path_length": f64([pl for _, pl, _, _ in results]),
           "search_success": f64([bool(ok) for _, _, ok, _ in results]),
           "search_valid_boxes_count": f64([0 if av is None else len(av) for _, _, _, av in results]),
           "search_path_nodes": f64([len(st.search_path) for st in states]),
           "search_path_bbox": f64([f64(node["bbox"]) for node in nodes]),
           "search_path_score": f64([0.0 if node["score"] is None else float(node["score"]) for node in nodes]),
           "search_path_detected": f64([d is not None for d in det]),
           "search_path_top_logit": f64([0.0 if d is None else float(d[0]) for d in det]),
           "search_path_box": f64([np.zeros(4) if d is None else f64(d[1]) for d in det])}
    if valid:
        out["search_valid_boxes"] = np.concatenate(valid)
    if scored is not None:
        out["vqa_option_losses"] = np.stack([f64(losses) for losses, _ in scored]).astype(np.float32)
        out["vqa_choice"] = f64([choice for _, choice in scored])
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from PIL import Image

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL prints its version banner to STDOUT when the first communicator comes up; keep stdout for the one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    from vstar_b200 import _lib, ops, seal, synth
    from vstar_b200.config import VSMConfig, tiny_config
    from vstar_b200.engine import VSMEngine, VSMWeights
    from vstar_b200.sharded import ShardedVSM, broadcast_loader
    from vstar_b200.visual_search import visual_search_many
    from vstar_b200.vqa import VQA_LLM, VQAEngine, VQAWeights, build_prompt_v1, tokenizer_image_object_token
    from vstar_b200.vsm import VSM

    if args.attn_impl:
        _lib.call("vsb_attn_set_impl", args.attn_impl)
    if args.gemm_l2_hints >= 0:
        _lib.call("vsb_gemm_set_l2_hints", args.gemm_l2_hints)
    if args.fuse_rope >= 0:
        _lib.call("vsb_llama_set_fuse_rope", args.fuse_rope)
    cfg = tiny_config() if args.tiny else VSMConfig()
    t0 = time.time()

    # ---- weights.  N > 1: only rank 0 "reads the checkpoint" (generates the tensors); every rank builds its replica through
    # broadcast_loader = one NCCL broadcast per tensor over NVLink (SURVEY.md §8e).  Timed with a device sync on both sides.
    shapes = synth.state_dict_shapes(cfg)
    vshapes = synth.vqa_state_dict_shapes(cfg)

    def gen(table, seed):
        return lambda n: synth.synthetic_tensor(n, table[n], seed=seed, device="cuda", dtype=torch.bfloat16)

    bcast = None
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        tb = time.perf_counter()
        load_vsm = broadcast_loader(gen(shapes, 1234) if rank == 0 else None, src=0, device="cuda",
                                    index={k: (tuple(v), torch.bfloat16) for k, v in shapes.items()})
        load_vqa = broadcast_loader(gen(vshapes, 4321) if rank == 0 else None, src=0, device="cuda",
                                    index={k: (tuple(v), torch.bfloat16) for k, v in vshapes.items()})
    else:
        load_vsm, load_vqa = gen(shapes, 1234), gen(vshapes, 4321)
    weights = VSMWeights(cfg, load_vsm)
    vqa_weights = None if args.no_vqa else VQAWeights(cfg, load_vqa)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        sec = time.perf_counter() - tb
        nbytes = load_vsm.stats["bytes"] + (load_vqa.stats["bytes"] if vqa_weights is not None else 0)
        bcast = {"bytes": nbytes, "seconds": sec, "GBps": nbytes / sec / 1e9, "tensors": load_vsm.stats["tensors"] + load_vqa.stats["tensors"],
                 "collective": "ncclBroadcast per tensor (torch.distributed.broadcast), rank 0 generates, includes rank 0's tensor generation"}
    engine = VSMEngine(weights, max_tokens=384)
    engine.prefix_cache = not args.no_prefix_cache
    prompt, ans = synth.synthetic_prompt(cfg, n_text=60, seed=0, im_start_index=None if args.tiny else 37)

    class BenchVSM(VSM):
        """synthetic tokenisation (no sentencepiece model offline): fixed 60-id prompt, forced 5-id answer (SURVEY.md §8d)"""

        def _ids(self, question):
            return prompt[0].tolist()

    vsm = BenchVSM(engine=engine, forced_answer_ids=ans.tolist(), frontier_batch=args.batch)
    vqa = None if args.no_vqa else VQA_LLM(engine=VQAEngine(vqa_weights))
    if vqa is not None:
        vqa.use_device_images(vsm)        # option-scoring pixels are cut / resized on the GPU from the resident search image
    load_s = time.time() - t0
    kw = dict(confidence_high=2.0, target_cue_threshold=-1e9, target_cue_threshold_minimum=-1e9)

    def images_for(n, side, base):
        return [Image.fromarray(np.random.default_rng(base + i).integers(0, 256, (side, side, 3), dtype=np.uint8), "RGB") for i in range(n)]

    def search_result_of(res):
        """two object boxes per search in image coordinates: the final detection and the root's best box (deterministic)"""
        final_step, _pl, _ok, _av = res
        out = []
        for name, step in zip(TARGETS, (final_step, None)):
            if step is None:
                b = final_step["detection_result"].clone() * 0.5
                patch = [0, 0]
            else:
                b, patch = step["detection_result"].clone(), step["bbox"]
            b[0] += patch[0]
            b[1] += patch[1]
            b[2:] = b[2:].clamp(min=8.0)
            out.append({"bbox": b.tolist(), "name": name})
        return out

    def make_leg(S, side, smallest, with_vqa, seed_base):
        images = images_for(S, side, seed_base)
        jobs = [(im, TARGETS[0], smallest) for im in images]
        state = dict(vqa_resident=None, trajectories=None)

        def vqa_public(results):
            # the call a user makes after the searches (vstar_bench_eval.py:226-257): PIL crops, host CLIP preprocessing, H2D
            return seal.choose_options(vqa, [(im, QUESTION, OPTIONS, list(TARGETS), search_result_of(r)) for im, r in zip(images, results)])

        def stage_vqa(results):
            """device-resident inputs of the same option scorings (built once from a warm-up run; searches are deterministic)"""
            staged = []
            for im, r in zip(images, results):
                sr = search_result_of(r)
                req = seal.option_request(vqa, im, QUESTION, OPTIONS, list(TARGETS), sr)
                staged.append(vqa._choice_item(*req))
            return staged

        def step(resident):
            if not resident:
                vsm.release()          # public path: every search image is uploaded (pinned H2D) inside the step
            results, states = visual_search_many(vsm, jobs, batch_size=args.batch, depth=args.depth, **kw)
            choices = scored = None
            if with_vqa:
                if resident:
                    if state["vqa_resident"] is None:
                        state["vqa_resident"] = stage_vqa(results)
                    scored = vqa.engine.option_losses_batch(state["vqa_resident"])
                    choices = [c for _, c in scored]
                else:
                    choices = vqa_public(results)
            state["last"] = (results, states, scored)       # what this step returned, for --dump-outputs
            traj = [[tuple(s["bbox"]) for s in st.search_path] for st in states]
            if state["trajectories"] is None:
                state["trajectories"] = (traj, choices)
            else:                       # in-run determinism check: every step walks the same trajectories and picks the same options
                assert state["trajectories"][0] == traj, "search trajectory changed between steps"
            return sum(st.n_evals for st in states), states

        return step, jobs, state

    def timed_steps(step, n, resident):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        crops = 0
        for _ in range(n):
            c, _ = step(resident)
            crops += c
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
            c = torch.tensor([crops], device="cuda", dtype=torch.float64)
            dist.all_reduce(c)
            crops = int(c[0])
        return ms, crops

    side = 256 if args.tiny else args.image
    smallest = 64 if args.tiny else args.smallest
    step2, jobs2, st2 = make_leg(args.searches, side, smallest, not args.no_vqa, 1000 * rank)

    # ---- e2e leg: public API from PIL images
    for _ in range(args.warmup):
        step2(False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    h2d0, d2h0 = vsm.h2d_bytes, vsm.d2h_bytes
    e2e_ms, e2e_crops = timed_steps(step2, args.steps, False)
    bytes_h2d = (vsm.h2d_bytes - h2d0) // args.steps
    bytes_d2h = (vsm.d2h_bytes - d2h0) // args.steps
    if vqa is not None:      # VQA leg: pixels come from the resident search image (no extra H2D); prompt ids up, 4 option NLL vectors down
        bytes_h2d += args.searches * 8 * 700
        bytes_d2h += args.searches * 4 * 40

    # ---- device-resident leg
    for _ in range(max(1, args.warmup)):
        step2(True)
    ops.profile_begin()
    launches0 = _lib.launches
    if args.profile_range:           # `ncu --profile-from-start off`: capture exactly the timed resident steps
        torch.cuda.profiler.start()
    dev_ms, dev_crops = timed_steps(step2, args.steps, True)
    if args.profile_range:
        torch.cuda.profiler.stop()
    launches = _lib.launches - launches0
    gemm_flops, gemm_ms, gemm_n = ops.profile_end()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *st2["last"])
    prefix_rows = engine._P

    peak_tf, peak_hbm, peak_src = peaks()
    flops_per_crop = FLOPS_PER_CROP - 2.0 * prefix_rows * 6.476e9
    if engine.tail_only and not args.tiny:      # last layer: o-proj + MLP only on the 5 consumed rows of each crop
        flops_per_crop -= 2.0 * (320 - prefix_rows - 5) * (cfg.hidden * cfg.hidden + 3 * cfg.hidden * cfg.intermediate)
    value = dev_crops / (dev_ms / 1e3)
    e2e = e2e_crops / (e2e_ms / 1e3)
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    traffic, traffic_note = gemm_traffic_from_profile()
    out = {
        "metric": METRIC, "value": value, "unit": "crops/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args),
        "e2e": {"value": e2e, "unit": "crops/s", "h2d_bytes_per_step": bytes_h2d, "d2h_bytes_per_step": bytes_d2h,
                "ms_per_step": e2e_ms / args.steps, "host_prep_s_total": vsm.timers["prep"]},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                     "traffic": traffic, "traffic_note": traffic_note, "kernel": "gemm_bf16_tcgen05_kernel", "launches": gemm_n,
                     "gemm_time_share_of_step": gemm_ms / dev_ms if dev_ms > 0 else None,
                     "how": "sum(2*M*N*K) / sum(CUDA-event duration) over every GEMM launch of the timed region (VSM and VQA); peak = " + peak_src,
                     "whole_path_frac": value / world * flops_per_crop / (peak_tf * 1e12),
                     "whole_path_note": ("crops/s/GPU x %.2f TFLOP/crop executed / peak; conservative: the VQA option scoring inside the step "
                                         "(~4 TFLOP per search) is NOT counted as useful work (BASELINE.md §3 counts 5.00 TFLOP/crop at "
                                         "T=320; %d constant prefix rows per crop are served from the shared-prefix KV snapshot, and the last "
                                         "decoder layer runs o-proj/MLP on the 5 consumed rows only)" % (flops_per_crop / 1e12, prefix_rows))},
        "crops_per_step": dev_crops // args.steps, "load_s": load_s,
        "draft_verify": engine.stats,          # (live dict: also counts the graph captures / replays of the later legs)
        "weight_broadcast": bcast,
        "parity_in_run": {"trajectories_identical_across_steps_and_legs": True,
                          "vqa_choices": st2["trajectories"][1]},
    }

    extra = not args.no_extra_legs
    # ---- configs[1] leg (round-1 headline workload) -------------------------------------------------------------------
    if extra:
        try:
            s1 = 8 if args.tiny else 32
            step1, jobs1, _ = make_leg(s1, 256 if args.tiny else 1024, 128 if args.tiny else 512, False, 5000 + 1000 * rank)
            for _ in range(2):
                step1(False)
            ms_a, c_a = timed_steps(step1, 3, False)
            step1(True)
            ms_b, c_b = timed_steps(step1, 3, True)
            out["configs1"] = {"workload": f"BASELINE.json configs[1]: 1024x1024, smallest 512 (root + 4 crops), {s1} lock-step searches, "
                                           f"frontier batch {args.batch}, no VQA leg (as in round 1)",
                               "value": c_b / (ms_b / 1e3), "e2e": c_a / (ms_a / 1e3), "unit": "crops/s", "steps": 3}
        except Exception as e:
            out["configs1"] = {"error": repr(e)}

    # ---- weak-cue leg: every root takes the context-cue branch (visual_search.py:427-443): 1 'vqa' + 1 'segmentation' model
    # call per search on top of its 5 detections, batched across the lock-step searches by the controller -----------------
    if extra and rank == 0:
        try:
            from vstar_b200 import noun_chunks
            noun_chunks.set_nlp(lambda text: [])       # synthetic answers carry no parsable nouns: "region {phrase}" prompts
            sw = 4 if args.tiny else 16
            w_images = images_for(sw, 256 if args.tiny else 1024, 7000)
            w_jobs = [(im, TARGETS[0], 128 if args.tiny else 512) for im in w_images]
            kw_weak = dict(confidence_high=2.0, target_cue_threshold=1e9, target_cue_threshold_decay=0.0, target_cue_threshold_minimum=-1e9)
            cue_sizes = []

            def wstep():
                from vstar_b200.visual_search import SearchController, SearchState
                states = [SearchState(img, name, ss, **kw_weak) for img, name, ss in w_jobs]
                ctl = SearchController(vsm, None, args.batch, depth=args.depth)
                ctl.run(states)
                cue_sizes[:] = ctl.cue_batches
                assert all("context_cue" in st.search_path[0] for st in states)
                return sum(st.n_evals for st in states)

            wstep()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n_w, det = 3, 0
            for _ in range(n_w):
                det += wstep()
            e1.record()
            torch.cuda.synchronize()
            ms_w = e0.elapsed_time(e1)
            # the same with FREE-RUNNING cue answers (no forced ids): batched exact greedy decoding of 24 tokens per weak node
            free_vsm = BenchVSM(engine=engine, frontier_batch=args.batch)
            free_vsm.vqa_max_new_tokens = 24
            free_vsm.draft_ids, free_vsm.forced_answer_ids = vsm.draft_ids, None

            class CueVSM:          # detections through the forced-answer VSM (random weights never emit [LOC]), cue calls unforced
                frontier_batch = args.batch

                def __getattr__(self, name):
                    return getattr(vsm, name)

                def inference_many(self, regions, questions, mode, **kw_):
                    return (free_vsm if mode == "vqa" else vsm).inference_many(regions, questions, mode, **kw_)

            def wstep_free():
                from vstar_b200.visual_search import SearchController, SearchState
                states = [SearchState(img, name, ss, **kw_weak) for img, name, ss in w_jobs]
                SearchController(CueVSM(), None, args.batch, depth=args.depth).run(states)
                return sum(st.n_evals for st in states)

            wstep_free()
            torch.cuda.synchronize()
            t_free = time.perf_counter()
            det_free = wstep_free()
            torch.cuda.synchronize()
            t_free = time.perf_counter() - t_free
            out["weak_cue"] = {"free_running_cue_answers": {"crops_per_s": det_free / t_free, "ms_per_step": t_free * 1e3,
                                                            "what": "cue answers decoded greedily (24 new tokens, VSMEngine.generate_many: one "
                                                                    "batched prefill + one decode step per token for all weak nodes of a round)"},
                               "workload": f"{sw} lock-step searches of 1024x1024 images (root + 4 crops) whose ROOT takes the context-cue branch: "
                                           "5 detection evaluations + 1 'vqa' + 1 'segmentation' model call per search, the cue calls batched "
                                           "across the searches (synthetic forced answer, so no free-running decode)",
                               "crops_per_s": det / (ms_w / 1e3), "model_calls_per_s": (det + 2 * sw * n_w) / (ms_w / 1e3),
                               "cue_batches": [list(c) for c in cue_sizes], "steps": n_w}
            noun_chunks.set_nlp(None)
        except Exception as e:
            out["weak_cue"] = {"error": repr(e)}

    # ---- full SEAL loop (configs[4] "full SEAL VQA+VSM loop", vstar_bench_eval.py:186-273) on one GPU: free-form answers for 8
    # images in ONE continuous-batched decode, the guided searches for the "missing objects" (2 per image), option scoring ----
    if extra and rank == 0 and vqa is not None:
        try:
            n_img = 2 if args.tiny else 8
            l_side, l_small = (256, 64) if args.tiny else (2048, 512)
            l_images = images_for(n_img, l_side, 8000)
            new_tokens = 24

            def loop_step():
                t = {}
                torch.cuda.synchronize(); t0 = time.perf_counter()
                bg = tuple(int(x * 255) for x in vqa.image_processor.image_mean)
                padded = [seal.expand2square_center(im, bg)[0] for im in l_images]
                vqa.free_form_inference_batch(padded, [QUESTION] * n_img, max_new_tokens=new_tokens, originals=l_images)   # random weights: text unused
                torch.cuda.synchronize(); t["free_form_ms"] = (time.perf_counter() - t0) * 1e3; t1 = time.perf_counter()
                # random-init weights never emit the "missing objects" sentence: take the canned one the real model gives
                missing = seal.parse_missing_objects(seal.MISSING_OBJECTS_MSG + " " + ", ".join(TARGETS) + ".")
                jobs_l = [(im, name, l_small) for im in l_images for name in missing]
                res_l, _ = visual_search_many(vsm, jobs_l, batch_size=args.batch, depth=args.depth, **kw)
                torch.cuda.synchronize(); t["search_ms"] = (time.perf_counter() - t1) * 1e3; t2 = time.perf_counter()
                samples = []
                for k, im in enumerate(l_images):
                    sr = seal.collect_search_results(missing, res_l[k * len(missing):(k + 1) * len(missing)])
                    samples.append((im, QUESTION, OPTIONS, missing, sr))
                seal.choose_options(vqa, samples)
                torch.cuda.synchronize(); t["options_ms"] = (time.perf_counter() - t2) * 1e3
                t["total_ms"] = (time.perf_counter() - t0) * 1e3
                t["crops"] = len(jobs_l) * 21
                return t

            loop_step()
            ts = [loop_step() for _ in range(2)]
            best = min(ts, key=lambda x: x["total_ms"])
            vsm.release()
            out["seal_loop"] = {"workload": f"{n_img} V*Bench-style samples of {l_side}x{l_side} images end to end from PIL images: free-form answer "
                                            f"(continuous-batched greedy decode, {new_tokens} new tokens forced by max_new_tokens), 2 guided searches per "
                                            "image (21 crops each, lock-step), option scoring with the found objects (batched)",
                                "samples_per_s": n_img / (best["total_ms"] / 1e3), "crops_per_s": best["crops"] / (best["total_ms"] / 1e3),
                                **{k: best[k] for k in ("free_form_ms", "search_ms", "options_ms", "total_ms")}}
        except Exception as e:
            out["seal_loop"] = {"error": repr(e)}

    # ---- frontier leg: ONE set of searches, every batch sharded over all ranks (strong scaling) ----------------------
    if extra:
        try:
            fs_n, f_side, f_small = (2, 256, 64) if args.tiny else (4, 4096, 512)
            f_images = images_for(fs_n, f_side, 9000)                   # the SAME images on every rank (SPMD controller)
            f_jobs = [(im, TARGETS[0], f_small) for im in f_images]
            front = ShardedVSM(vsm, device="cuda") if world > 1 else vsm
            # scheduling only (the work is the same for every N): keep >= 32 crops per rank in a full frontier batch
            f_batch = max(args.batch, 32 * world)

            def fstep():          # search images stay resident in HBM across steps (as in `value`): the leg times evaluation + gather
                return visual_search_many(front, f_jobs, batch_size=f_batch, depth=args.depth, **kw)

            # parity first: the sharded trajectories against this rank's own single-GPU run of the same searches
            vsm.release()
            _, ref_states = visual_search_many(vsm, f_jobs, batch_size=args.batch, depth=args.depth, **kw)       # single-GPU schedule
            _, sh_states = fstep()
            ref_traj = [[tuple(s["bbox"]) for s in st.search_path] for st in ref_states]
            sh_traj = [[tuple(s["bbox"]) for s in st.search_path] for st in sh_states]
            same = ref_traj == sh_traj
            scores_equal = all(a["score"] == b["score"] for sa, sb in zip(ref_states, sh_states)
                               for a, b in zip(sa.search_path[1:], sb.search_path[1:]) if tuple(a["bbox"]) == tuple(b["bbox"])) and same
            # if the orders differ, they may only differ between nodes whose priorities are closer than the bf16 score tolerance
            worst = 0.0
            same_sets = all(sorted(a) == sorted(b) for a, b in zip(ref_traj, sh_traj))
            if not same and same_sets:
                for sa, sb in zip(ref_states, sh_states):
                    pos = {tuple(n["bbox"]): i for i, n in enumerate(sb.search_path)}
                    nodes = sa.search_path
                    for i in range(1, len(nodes)):
                        for j in range(i + 1, len(nodes)):
                            if pos[tuple(nodes[i]["bbox"])] > pos[tuple(nodes[j]["bbox"])]:
                                worst = max(worst, abs(float(nodes[i]["score"]) - float(nodes[j]["score"])))
            if world > 1:
                flag = torch.tensor([1.0 if same else 0.0, 1.0 if same_sets else 0.0, -worst], device="cuda")
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                same, same_sets, worst = bool(flag[0] > 0), bool(flag[1] > 0), float(-flag[2])
            assert same_sets and worst < 3e-3, ("sharded frontier diverged from the single-GPU run beyond near-ties", worst)
            g0 = (front.gathered_bytes, front.gathers) if world > 1 else (0, 0)
            fstep()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n_f, crops_f = 3, 0
            for _ in range(n_f):
                _, sts = fstep()
                crops_f += sum(len(st.search_path) for st in sts)
            e1.record()
            torch.cuda.synchronize()
            ms_f = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms_f], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms_f = float(t[0])
            g1 = (front.gathered_bytes, front.gathers) if world > 1 else (0, 0)
            rounds = max(1, (g1[1] - g0[1]) // (n_f + 1))
            out["frontier"] = {
                "workload": f"BASELINE.json configs[3]-shaped: {fs_n} searches of {f_side}x{f_side} images (resident in HBM), smallest {f_small} "
                            f"({crops_f // n_f // fs_n} crops each), ONE controller, every frontier batch (<= {f_batch} crops) dealt "
                            f"round-robin over all {world} ranks; total work is the same for every N",
                "scaling": "strong", "value": crops_f / (ms_f / 1e3), "unit": "crops/s", "steps": n_f, "ms_per_step": ms_f / n_f,
                "collective": ("ncclAllGather (all_gather_into_tensor) of fixed-size crop records, one per frontier batch" if world > 1
                               else "none (single GPU: the strong-scaling baseline)"),
                "gather_rounds_per_step": rounds if world > 1 else 0,
                "gathered_bytes_per_round": (g1[0] - g0[0]) // max(1, g1[1] - g0[1]) if world > 1 else 0,
                "trajectory_equal_to_single_gpu": same, "queue_priorities_bit_equal": bool(scores_equal),
                "largest_priority_gap_of_an_inverted_pair": worst,
            }
        except AssertionError:
            raise
        except Exception as e:
            out["frontier"] = {"error": repr(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rank-0-only probes ---------------------------------------------------------------------------------------
    if extra and vqa is not None:
        try:
            out["vqa"] = vqa_probe(vqa, st2, peak_hbm, args)
        except Exception as e:
            out["vqa"] = {"error": repr(e)}
    if extra and world == 1:
        try:
            # latency of ONE visual_search() call on its own, public API, configs[1] (root + 4 crops) and configs[2] (21 crops)
            lat = {}
            for name, side_l, small_l in (("configs1_5crops", 1024, 512), ("configs2_21crops", 2048, 512)):
                if args.tiny:
                    side_l, small_l = side_l // 8, small_l // 8
                im = images_for(1, side_l, 77)
                for _ in range(5):        # the first calls of a shape run eagerly, later ones replay its CUDA graph
                    vsm.release()
                    torch.cuda.synchronize()
                    t1 = time.perf_counter()
                    visual_search_many(vsm, [(im[0], "mug", small_l)], batch_size=args.batch, depth=args.depth, **kw)
                    torch.cuda.synchronize()
                    lat[name] = (time.perf_counter() - t1) * 1e3
            out["search_latency_ms"] = lat["configs1_5crops"]
            out["search_latency_ms_by_config"] = lat
        except Exception as e:
            out["search_latency_ms"] = None
            out["search_latency_error"] = repr(e)
    if not args.no_cpu_baseline and world == 1:
        try:
            tg = torch_gpu_reference_sample(cfg)
            out["torch_gpu_baseline"] = {"value": tg, "unit": "crops/s", "ratio_configs1_value": (out.get("configs1", {}).get("value") or 0) / tg,
                                         "what": "reference as-written GPU path restated in plain torch eager bf16 (batch 1, uncached greedy "
                                                 "generate = 5 full CLIP+7B passes, lm_head/fcs on all rows), cuda:0, host prep excluded, no VQA leg"}
        except Exception as e:
            out["torch_gpu_baseline"] = {"value": None, "what": f"failed: {e!r}"}
        try:
            v, sec, desc, cores = cpu_reference_sample(args)
            out["cpu_baseline"] = {"value": v, "unit": "crops/s", "cores": cores, "kind": "port", "sample": desc, "sample_seconds": sec}
        except Exception as e:   # the baseline leg must never take the GPU number down
            out["cpu_baseline"] = {"value": None, "unit": "crops/s", "cores": None, "kind": "port", "sample": f"failed: {e!r}"}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def vqa_probe(vqa, st2, peak_hbm, args):
    """SEAL-VQA numbers on the bench's own inputs (device timings, CUDA events): prefill, option scoring, ms/token of the
    continuous-batched greedy decode at B = 1 / 8 / 16 with the HBM fraction (every decode step reads the 13.5 GB of weights)"""
    import torch
    eng = vqa.engine
    staged = st2["vqa_resident"]
    q_ids, opt_ids, img_d, crops_d = staged[0][:4]

    def ev_time(fn, n=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def prefill():
        x = eng.build_embeds(q_ids, img_d, crops_d, [False], [True, True])
        eng.prefill_embeds(x)
        return x.shape[0]

    T = prefill()
    res = {"prompt_tokens": T, "prefill_ms": ev_time(prefill),
           "option_scoring_ms": ev_time(lambda: eng.option_losses(q_ids, opt_ids, img_d, crops_d, [False], [True, True])),
           "option_scoring_ms_per_question_batch_of_%d" % len(staged): ev_time(lambda: eng.option_losses_batch(staged)) / len(staged),
           "how": "option scoring = CLIP + both projectors on 3 images, question prefill, ONE pass over all 4 options (segment-masked "
                  "attention on the question's KV rows); batch = questions of equal spliced length share both passes"}
    wbytes = 2.0 * (32 * (4 * 4096 * 4096 + 3 * 4096 * 11008) + 32004 * 4096) if not args.tiny else None
    for B in (1, 8, 16):
        reqs = [(q_ids, img_d, crops_d, [False], [True, True])] * B
        xs = [eng.build_embeds(*r) for r in reqs]
        logits, Tpad, lens = eng.prefill_ragged(xs, reserve=64)
        toks = [5] * B
        steps = 16

        def run():
            for s in range(steps):
                eng.decode_ragged(toks, lens, Tpad, s)

        ms = ev_time(run, n=2) / steps
        res[f"decode_ms_per_step_B{B}"] = ms
        res[f"decode_tokens_per_s_B{B}"] = B / (ms / 1e3)
        if wbytes:
            res[f"decode_hbm_frac_B{B}"] = wbytes / (ms / 1e3) / (peak_hbm * 1e9)
    return res


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)

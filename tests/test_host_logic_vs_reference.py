"""Differential tests of the host logic (integer geometry, priority queue order, prompt strings, placeholder splicing,
padding, patch geometry, noun chunks, visualisation files) against the reference's own modules (visual_search.py:54-112,
:226-283, :339-389, conversation.py, mm_utils.py, vstar_bench_eval.py:21-76), on seeded random inputs.

The reference's answers are recorded in tests/golden/host_logic.npz by oracle/make_golden.py (GOLDEN_ONLY=host_logic),
which imports the input generators below, so both sides see the same inputs.  Images and written files are recorded as
SHA-256 digests of their bytes, so those comparisons stay bit-exact."""
import hashlib
import json
import os
import queue
import tempfile

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "host_logic.npz")


# ---------------------------------------------------------------- inputs (shared with oracle/make_golden.py:case_host_logic)
def boxes(n, seed):
    rng = np.random.default_rng(seed)
    for _ in range(n):
        w, h = int(rng.integers(1, 9000)), int(rng.integers(1, 9000))
        yield [int(rng.integers(0, 5000)), int(rng.integers(0, 5000)), w, h]


def split_inputs():
    return list(boxes(3000, 1)) + [[0, 0, 100, 200], [0, 0, 200, 100], [3, 5, 7, 14], [3, 5, 14, 7], [0, 0, 1, 1], [0, 0, 2, 3]]


def refine_inputs():
    """[(W, H, b, c)]: image size, a box to refine and a second box for iou(b, c)"""
    rng = np.random.default_rng(2)
    out = []
    for _ in range(2000):
        W, H = int(rng.integers(10, 4000)), int(rng.integers(10, 4000))
        b = [float(rng.uniform(-50, W)), float(rng.uniform(-50, H)), float(rng.uniform(1, W)), float(rng.uniform(1, H))]
        c = [float(rng.uniform(0, W)), float(rng.uniform(0, H)), float(rng.uniform(1, W)), float(rng.uniform(1, H))]
        out.append((W, H, b, c))
    return out


def pop_order(prioritize, scores):
    """push Prioritize(-score, index) for every score, popping once after every third push like the search does, then
    drain: the popped indices in order"""
    q, out = queue.PriorityQueue(), []
    for i, s in enumerate(scores):
        q.put(prioritize(-s, i))
        if i % 3 == 2:
            out.append(q.get().item)
    while not q.empty():
        out.append(q.get().item)
    return out


def pop_inputs():
    rng = np.random.default_rng(3)
    return [np.round(rng.uniform(0, 1, 40), 1 if trial % 2 else 3).astype(np.float32) for trial in range(50)]     # many exact ties


PROMPT_QUESTIONS = ["Please locate the red mug in this image.", "According to the common sense knowledge and possible visual "
                    "cues, what is the most likely location of the dog in the image?", "x"]
VQA_QUESTION = "<image>\nAdditional visual information to focus on: mug <object> at location [0.1,0.2,0.3,0.4]; dog <object>.\n{}"
VQA_ANSWERS = (None, "the mug is red")
PAD_SIZES = [(300, 200), (200, 300), (256, 256), (1, 9), (513, 512)]
PAD_BG = (122, 116, 104)
PATCH_SCALES = (None, 1.2, 0.5)


def pad_image(i, w, h):
    from tests.helpers import synth_image
    return synth_image(50 + i, w, h)


def patch_inputs():
    rng = np.random.default_rng(5)
    out = []
    for _ in range(2000):
        W, H = int(rng.integers(50, 3000)), int(rng.integers(50, 3000))
        out.append((W, H, [float(rng.uniform(0, W)), float(rng.uniform(0, H)), float(rng.uniform(1, W)), float(rng.uniform(1, H))]))
    return out


def noun_chunk_inputs():
    """(phrases, chunk lists): the answers of tests.helpers.VQA_ANSWERS, random phrases over the rule parser's lexicon, and
    random (start, end) chunk lists for filter_chunk_list"""
    from tests.helpers import FakeNLP, VQA_ANSWERS as CUE_ANSWERS
    rng = np.random.default_rng(7)
    words = sorted(FakeNLP.NOUNS | FakeNLP.PRONS | FakeNLP.ADJS | FakeNLP.DETS | FakeNLP.PREPS | FakeNLP.RELS) + ["and", "somewhere", "high", "is"]
    phrases = [a.split("most likely to appear")[-1].strip().rstrip(".") for a in CUE_ANSWERS]
    for _ in range(3000):
        phrases.append(" ".join(rng.choice(words, size=int(rng.integers(1, 12)))))
    chunk_lists = [[tuple(sorted(rng.integers(0, 30, 2).tolist())) for _ in range(int(rng.integers(0, 8)))] for _ in range(2000)]
    return phrases, chunk_lists


# (image seed, w, h, smallest, stub hot mode, search kwargs) of the two searches whose visualisation files are compared
VIS_CASES = ((29, 640, 480, 224, None, dict(confidence_high=2.0, target_cue_threshold=9.5, target_cue_threshold_minimum=9.5)),
             (25, 700, 600, 224, "small", dict()))
VIS_TARGET_BBOX = [30, 40, 50, 60]


def digest(data):
    return hashlib.sha256(data).hexdigest()


def image_digest(img):
    return digest(np.ascontiguousarray(np.asarray(img)).tobytes())


def dir_digests(d):
    return {f: digest(open(os.path.join(d, f), "rb").read()) for f in sorted(os.listdir(d))}


# ---------------------------------------------------------------- checks of the product against the recorded answers
_gold = None


def golden():
    global _gold
    if _gold is None:
        with np.load(GOLD) as z:
            _gold = {k: z[k] for k in z.files}
    return _gold


def golden_json(key):
    return json.loads(str(golden()[key]))


def check_split_and_sub_patches():
    from vstar_b200 import visual_search as VS
    g = golden()
    n_14 = n_41 = 0
    for i, b in enumerate(split_inputs()):
        nw, nh = VS.split_4subpatches(b)
        assert (nw, nh) == tuple(g["split_nwnh"][i].tolist())
        n_14 += (nw, nh) == (1, 4)
        n_41 += (nw, nh) == (4, 1)
        got = VS.get_sub_patches(b, nw, nh)
        assert list(got[0]) == g["split_subs"][i].tolist() and got[1:] == tuple(g["split_strides"][i].tolist())
        # children tile the parent exactly (last row / column takes the remainder)
        assert sum(p[2] * p[3] for p in got[0]) == b[2] * b[3]
    assert n_14 > 100 and n_41 > 100


def check_refine_bbox_and_iou():
    from vstar_b200 import visual_search as VS
    g = golden()
    for i, (W, H, b, c) in enumerate(refine_inputs()):
        assert VS.refine_bbox(list(b), W, H) == g["refine_bbox"][i].tolist()
        assert VS.iou(b, c) == float(g["iou"][i])


def check_prioritize_pop_order_with_ties():
    """the expansion order IS the heap order of (Prioritize(-score, item)) incl. its tie behaviour (no tiebreak key)"""
    from vstar_b200 import visual_search as VS
    g = golden()
    for trial, scores in enumerate(pop_inputs()):
        assert pop_order(VS.Prioritize, scores) == g["pop_order"][trial].tolist()


def check_prompts_and_token_splicing():
    """prompt strings of both conversation templates and the <image>/<object> placeholder splicing (they define T and the
    255-row offset): ours vs the reference's conversation.py / mm_utils.py, with the synthetic word-hash tokenizer on both"""
    from vstar_b200 import vqa, vsm
    from vstar_b200.config import tiny_config
    want = golden_json("prompts")
    tok = vsm.SyntheticTokenizer(tiny_config())
    for q, w in zip(PROMPT_QUESTIONS, want["vsm"]):
        # VSM wrapper (visual_search.py:176-184) and the other template the CLI accepts (visual_search.py:48)
        assert vsm.build_prompt(q, "llava_v1", True) == w["llava_v1"]
        for use_se in (True, False):
            assert vsm.build_prompt(q, "llava_llama_2", use_se) == w[f"llava_llama_2_se{int(use_se)}"]
        ours = vsm.tokenizer_image_token(w["llava_v1"], tok)
        assert ours == w["ids"] and ours.count(-200) == 1
    for q, w in zip(PROMPT_QUESTIONS, want["vqa"]):
        # SEAL VQA LLM (vstar_bench_eval.py:79-85, :112-116, :136-139)
        qs = VQA_QUESTION.format(q)
        for answer, wa in zip(VQA_ANSWERS, w):
            prompt = vqa.build_prompt_v1(qs, answer)
            assert prompt == wa["prompt"]
            ours = vqa.tokenizer_image_object_token(prompt, tok)
            assert ours == wa["ids"] and ours.count(-200) == 1 and ours.count(-300) == 2


def check_padding_and_patch_geometry():
    """both expand2square variants (top-left paste for the VSM, centred for the VQA LLM) and VQA_LLM.get_patch"""
    from vstar_b200 import seal, vqa, vsm
    want = golden_json("padding")
    for i, ((w, h), wv) in enumerate(zip(PAD_SIZES, want)):
        img = pad_image(i, w, h)
        a = vsm.expand2square(img, PAD_BG)
        assert [a.width, a.height, image_digest(a)] == wv["vsm"]
        b, left, top = seal.expand2square_center(img, PAD_BG)
        assert [b.width, b.height, image_digest(b), left, top] == wv["vqa"]
    get_patch = vqa.VQA_LLM.get_patch
    g = golden()["get_patch"]
    for i, (W, H, bbox) in enumerate(patch_inputs()):
        for j, scale in enumerate(PATCH_SCALES):
            assert get_patch(None, bbox, W, H, patch_scale=scale) == g[i, j].tolist()


def check_noun_chunks():
    """extract_noun_chunks / get_noun_chunks / filter_chunk_list (visual_search.py:54-112) with the SAME deterministic parser
    on both sides (spaCy is not installed offline): random phrases from the rule parser's lexicon + hand-made trees"""
    from tests.helpers import FakeNLP
    from vstar_b200 import noun_chunks as NC
    want = golden_json("noun_chunks")
    nlp = FakeNLP()
    phrases, chunk_lists = noun_chunk_inputs()
    assert len(phrases) == len(want["chunks"]) and len(chunk_lists) == len(want["filtered"])
    n_multi = n_one = n_zero = 0
    for ph, w_chunks, w_spans in zip(phrases, want["chunks"], want["spans"]):
        got = NC.extract_noun_chunks(ph, nlp)
        assert got == w_chunks, (ph, got, w_chunks)
        n_multi += len(got) > 1
        n_one += len(got) == 1
        n_zero += len(got) == 0
        doc = nlp(ph)
        assert len(doc) == len(w_spans)
        for t, (a0, a1, b0, b1) in zip(doc, w_spans):
            assert NC.get_noun_chunks(t) == (a0, a1) and NC.subtree_span(t) == (b0, b1)
    assert n_multi > 100 and n_one > 100 and n_zero > 10
    for chunks, w in zip(chunk_lists, want["filtered"]):
        assert NC.filter_chunk_list(chunks) == [tuple(c) for c in w]


def check_visualisation_files():
    """visualize=True: the files visualize_search_path writes (visual_search.py:339-376) from the reference and from the product,
    on the same stub search: same file names, byte-identical JPEGs and context_cue.txt"""
    from tests.helpers import FakeNLP, NumpyScorer, StubVSM, synth_image
    from vstar_b200 import noun_chunks
    from vstar_b200 import visual_search as VS
    want = golden_json("visualisation")
    noun_chunks.set_nlp(FakeNLP())
    try:
        for (seed, w, h, smallest, hot, kw), wv in zip(VIS_CASES, want):
            img = synth_image(seed, w, h)
            with tempfile.TemporaryDirectory() as d:
                r = VS.visual_search(StubVSM(hot), img, "mug", VIS_TARGET_BBOX, smallest, visualize=True, save_path=d,
                                     scorer=NumpyScorer(), **kw)
                files = dir_digests(d)
            assert [r[1], r[2]] == [wv["path_length"], wv["success"]]
            fa = sorted(files)
            assert fa == sorted(wv["files"]) and "whole_image.jpg" in fa and "context_cue.txt" in fa and any(f.endswith("_heatmap.jpg") for f in fa), fa
            for f in fa:
                assert files[f] == wv["files"][f], f
    finally:
        noun_chunks.set_nlp(None)


CHECKS = ["check_visualisation_files", "check_noun_chunks", "check_split_and_sub_patches", "check_refine_bbox_and_iou",
          "check_prioritize_pop_order_with_ties", "check_prompts_and_token_splicing", "check_padding_and_patch_geometry"]


@pytest.mark.parametrize("name", CHECKS)
def test_against_live_reference(name):
    """the product against the answers the reference's modules gave on the same inputs"""
    globals()[name]()

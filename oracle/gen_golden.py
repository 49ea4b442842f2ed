"""TEST INFRASTRUCTURE. Generates tests/golden/*.npz by running the REAL reference (through
oracle/reference_shim.py) in the build container:   python -m oracle.gen_golden [--full]

The .npz files hold everything needed to replay the case without the reference: the config, the weight seed
(weights are re-drawn by visrag_b200.weights.random_state_dict), the page sizes + pixel seed (pages are
re-drawn by synth_pages), the query strings, and the reference outputs (fp32 embeddings, score top-k,
slice geometry).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import warnings

import numpy as np
from PIL import Image

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
warnings.filterwarnings("ignore")

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

from visrag_b200.synth import QUERY_PREFIX, synth_pages, synth_queries  # noqa: E402,F401


def geometry_cases():
    sizes = [(224, 224), (448, 448), (336, 336), (1344, 1344), (564, 3040), (1114, 1670), (700, 900), (1200, 500),
             (500, 1200), (640, 480), (2000, 300), (300, 2000), (449, 449), (1000, 1000), (896, 448), (447, 448)]
    rs = np.random.RandomState(11)
    for _ in range(150):
        sizes.append((int(rs.randint(100, 1500)), int(rs.randint(100, 1500))))
    return sizes


def gen_geometry():
    """Slice geometry from the reference's own slice_image (modeling_minicpmv.py:482-537)."""
    from oracle import reference_shim as RS

    RS._import_reference()
    from openmatch.modeling.modeling_minicpmv.modeling_minicpmv import slice_image

    rows = []
    for (w, h) in geometry_cases():
        src, patches, grid = slice_image(Image.new("RGB", (w, h)), 9, 448, 14)
        g = grid if grid is not None else [0, 0]
        pw, ph = (patches[0][0].size if patches else (0, 0))
        rows.append([w, h, src.size[0], src.size[1], g[0], g[1], pw, ph, sum(len(r) for r in patches)])
    np.savez(os.path.join(GOLDEN_DIR, "geometry_v1.npz"), cases=np.asarray(rows, dtype=np.int64),
             columns=np.asarray(["W", "H", "src_w", "src_h", "grid_x", "grid_y", "patch_w", "patch_h", "n_patches"]))
    print("geometry:", len(rows), "cases")


def gen_model_case(name, cfg, weight_seed, page_sizes, page_seed, n_queries, query_seed, topk):
    import torch
    from oracle import reference_shim as RS
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict

    sd = random_state_dict(cfg, weight_seed)
    model = RS.build_reference_model(cfg, sd, attn_implementation="sdpa")
    tok = StubTokenizer(cfg.vocab)
    pages = synth_pages(page_sizes, page_seed)
    queries = synth_queries(n_queries, query_seed)
    p_items = [{"id": f"d{i}", "text": "", "image": im} for i, im in enumerate(pages)]
    q_items = [{"id": f"q{i}", "text": t, "image": None} for i, t in enumerate(queries)]
    # the reference encodes in batches; padding must not matter -> encode pages in two uneven batches
    half = max(1, len(p_items) // 2)
    p = np.concatenate([RS.encode(model, tok, p_items[:half], False), RS.encode(model, tok, p_items[half:], False)])
    q = RS.encode(model, tok, q_items, True)
    # reference scoring: torch.matmul + torch.topk (dense_retriever.py:25-30)
    S = torch.matmul(torch.from_numpy(q), torch.from_numpy(p).T)
    ts, ti = torch.topk(S, min(topk, p.shape[0]), dim=1)
    np.savez(os.path.join(GOLDEN_DIR, f"{name}.npz"), config=json.dumps(cfg.to_dict()), weight_seed=weight_seed,
             page_sizes=np.asarray(page_sizes, dtype=np.int64), page_seed=page_seed, queries=np.asarray(queries),
             query_seed=query_seed, page_reps=p.astype(np.float32), query_reps=q.astype(np.float32),
             topk_scores=ts.numpy(), topk_indices=ti.numpy())
    print(name, "pages", p.shape, "queries", q.shape)


REAL_PAGES = os.path.join(GOLDEN_DIR, "real_pages.npz")


def gen_real_pages():
    """The reference's own example inputs, kept as the ENCODED bytes the reference ships (data, not code): the two
    (query, page) rows of examples/training_data/0.parquet and the demo's cat/dog photos
    (visrag_scripts/demo/retriever/test_image, README.md:315-319). Decoded with PIL at test time."""
    import pyarrow.parquet as pq
    from oracle.reference_shim import REF_ROOT

    t = pq.read_table(os.path.join(REF_ROOT, "examples", "training_data", "0.parquet"))
    out, queries = {}, []
    for i in range(t.num_rows):
        out[f"parquet{i}"] = np.frombuffer(t.column("image")[i].as_py()["bytes"], dtype=np.uint8)
        queries.append(t.column("query")[i].as_py())
    for n in ("cat.jpeg", "dog.jpg"):
        with open(os.path.join(REF_ROOT, "visrag_scripts", "demo", "retriever", "test_image", n), "rb") as f:
            out[n.split(".")[0]] = np.frombuffer(f.read(), dtype=np.uint8)
    np.savez(REAL_PAGES, queries=np.asarray(queries), **out)
    print("real pages:", {k: v.size for k, v in out.items()})


def full_v2_spec():
    """>= 32 pages (>= 8 multi-slice + the reference's 4 real example images) and >= 8 queries: a corpus on which the
    top-5 ranking is a real statement (VERDICT r01 'next' #1)."""
    single = [(448, 448), (400, 500), (300, 600), (224, 224), (336, 336), (420, 420), (500, 390), (448, 448), (360, 540),
              (640, 300), (448, 448), (280, 280), (512, 384), (384, 512), (448, 448), (330, 600), (600, 330), (448, 440),
              (224, 224), (436, 452)]
    multi = [(700, 900), (640, 480), (1000, 700), (900, 450), (1344, 336), (600, 600), (800, 1000), (448, 900)]
    spec = [{"kind": "doc", "size": list(s), "seed": 5000 + i} for i, s in enumerate(single + multi)]
    spec += [{"kind": "noise", "size": list(s), "seed": 6000 + i} for i, s in enumerate([(448, 448), (448, 448), (224, 224), (640, 480)])]
    spec += [{"kind": "real", "name": n} for n in ("parquet0", "parquet1", "cat", "dog")]
    return spec


def gen_spec_case(name, cfg, weight_seed, spec, n_queries, query_seed, topk, batch=6):
    """Like gen_model_case, for a page list described by a spec (see tests/helpers.pages_from_spec)."""
    import time

    import torch
    from oracle import reference_shim as RS
    from tests.helpers import pages_from_spec, real_queries
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict

    sd = random_state_dict(cfg, weight_seed)
    model = RS.build_reference_model(cfg, sd, attn_implementation="sdpa")
    tok = StubTokenizer(cfg.vocab)
    pages = pages_from_spec(spec)
    queries = synth_queries(n_queries, query_seed) + [QUERY_PREFIX + q for q in real_queries()]
    p_items = [{"id": f"d{i}", "text": "", "image": im} for i, im in enumerate(pages)]
    q_items = [{"id": f"q{i}", "text": t, "image": None} for i, t in enumerate(queries)]
    t0 = time.time()
    parts = []
    for s in range(0, len(p_items), batch):  # the reference's own batch loop, right-padded batches of mixed pages
        parts.append(RS.encode(model, tok, p_items[s:s + batch], False))
        print(f"  pages {s + len(parts[-1])}/{len(p_items)}  {time.time() - t0:.0f}s", flush=True)
    p = np.concatenate(parts)
    q = RS.encode(model, tok, q_items, True)
    S = torch.matmul(torch.from_numpy(q), torch.from_numpy(p).T)      # dense_retriever.py:25-30
    ts, ti = torch.topk(S, topk, dim=1)
    full = np.sort(S.numpy(), axis=1)[:, ::-1]
    gaps = full[:, :topk] - full[:, 1:topk + 1]
    np.savez(os.path.join(GOLDEN_DIR, f"{name}.npz"), config=json.dumps(cfg.to_dict()), weight_seed=weight_seed,
             page_spec=json.dumps(spec), queries=np.asarray(queries), query_seed=query_seed,
             page_reps=p.astype(np.float32), query_reps=q.astype(np.float32), topk_scores=ts.numpy(),
             topk_indices=ti.numpy(), min_gap=np.float32(gaps.min()))
    print(name, "pages", p.shape, "queries", q.shape, "min score gap inside top-(k+1):", gaps.min(), "median", np.median(gaps))


POOLINGS = ("lasttoken", "mean", "cls")
HIDDEN_ROWS = 16  # hidden-state rows kept per sequence (seeded sample, first and last valid position always in)


def hidden_row_sample(n, seed):
    rs = np.random.RandomState(seed)
    mid = np.sort(rs.choice(np.arange(1, n - 1), HIDDEN_ROWS - 2, replace=False))
    return np.concatenate([[0], mid, [n - 1]]).astype(np.int64)


def gen_reference_checks():
    """What the reference computes on the inputs of tests/test_oracle_vs_reference.py, so those comparisons run without it:
    embeddings and a seeded sample of hidden-state rows of VisRAG_Ret, the other poolings, `_retrieve_one_shard` on a
    pickle shard, and the run-file / MRR functions of utils.py."""
    import tempfile

    import torch
    from oracle import reference_shim as RS
    from oracle import restated as O
    from tests.helpers import REFERENCE_CHECKS, pooling_inputs, restatement_inputs, scoring_inputs
    from visrag_b200.retriever import save_shard
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict

    out = {}
    cfg, seed, texts, pages, queries = restatement_inputs()
    sd = random_state_dict(cfg, seed)
    model = RS.build_reference_model(cfg, sd, attn_implementation="sdpa")
    tok = StubTokenizer(cfg.vocab)
    items = [{"id": str(i), "text": t, "image": im} for i, (t, im) in enumerate(zip(texts, pages))]
    out["restate_page_reps"] = RS.encode(model, tok, items, False)
    out["restate_query_reps"] = RS.encode(model, tok, [{"id": f"q{i}", "text": t, "image": None} for i, t in enumerate(queries)], True)
    hs, mask = RS.hidden_states(model, tok, texts, pages)
    n = mask.sum(1).astype(np.int64)
    pos = np.stack([hidden_row_sample(int(n[b]), b) for b in range(len(n))])
    out.update(restate_hidden_len=n, restate_hidden_pos=pos,
               restate_hidden_rows=np.stack([hs[b, pos[b]] for b in range(len(n))]).astype(np.float32))

    cfg, seed, texts, images = pooling_inputs()
    sd = random_state_dict(cfg, seed)
    items = [{"id": str(i), "text": t, "image": im} for i, (t, im) in enumerate(zip(texts, images))]
    for pooling in POOLINGS:
        model = RS.build_reference_model(cfg, sd, attn_implementation="sdpa", pooling=pooling)
        out[f"pooling_{pooling}"] = RS.encode(model, tok, items, False)

    RS._import_reference()
    from openmatch import utils as ref_utils
    from openmatch.retriever.dense_retriever import _retrieve_one_shard as ref_retrieve

    Q, D, lookup = scoring_inputs()
    with tempfile.TemporaryDirectory() as tmp:
        shard = os.path.join(tmp, "embeddings.corpus.rank.0")
        save_shard(shard, D, lookup)  # the project's writer, the reference's reader
        s_ref, i_ref, look_ref = ref_retrieve(shard, torch.from_numpy(Q), 10, "cpu")
        assert look_ref == lookup
        s, i = s_ref.numpy(), i_ref.numpy()
        run = {f"q{q}": {lookup[j]: float(s[q, r]) for r, j in enumerate(i[q])} for q in range(len(Q))}
        qrel = {f"q{q}": {lookup[int(i[q, q % 10])]: 1} for q in range(len(Q))}
        trec = os.path.join(tmp, "run.trec")
        ref_utils.save_as_trec(run, trec)
        trec_text = open(trec).read()
        loaded = ref_utils.load_from_trec(trec)
    out.update(score_topk_scores=s, score_topk_ids=i.astype(np.int64), trec_text=np.asarray(trec_text),
               trec_loaded=np.asarray(json.dumps(loaded)),
               mrr=np.asarray(json.dumps({"10": ref_utils.eval_mrr(qrel, run, 10), "3": ref_utils.eval_mrr(qrel, run, 3)})))
    assert np.array_equal(O.score_topk(Q, D, 10)[1], i)
    np.savez_compressed(REFERENCE_CHECKS, **out)
    print("reference checks:", {k: v.shape for k, v in out.items()})


def gen_driver_run():
    """The reference's own driver (src/openmatch/driver/eval.py, unmodified) drives this project's drop-in
    DRModelForInference on a synthetic checkpoint directory: setup_model -> DRModelForInference.build, the reference's
    distributed_parallel_embedding_inference writes the pickle shards, its retrieve phase writes the run file. The
    embeddings come from the oracle on the CPU (the device math is the only thing replaced). Stores the shard names,
    their contents and the run file, which tests/test_dropin_reference_driver.py compares the project's own driver
    path against."""
    import pickle
    import tempfile
    import types

    import torch
    from oracle import reference_shim as RS
    from oracle import restated as O
    from tests.helpers import DRIVER_RUN, driver_run_args, driver_run_inputs
    from visrag_b200 import inference as I
    from visrag_b200 import modeling as M
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict, save_checkpoint

    R = RS._import_reference()
    pytrec_eval = types.ModuleType("pytrec_eval")  # absent here; only used for the metrics log, which is not stored

    class RelevanceEvaluator:
        def __init__(self, qrels, measures):
            self.qrels = qrels

        def evaluate(self, run):
            rec = I.recall_at_k(self.qrels, run, 10)
            return {qid: {"recall_10": rec[qid]} for qid in rec if qid != "all"}

    pytrec_eval.RelevanceEvaluator = RelevanceEvaluator
    pytrec_eval.compute_aggregated_measure = lambda measure, values: float(np.mean(values)) if values else 0.0
    sys.modules["pytrec_eval"] = pytrec_eval
    import openmatch.driver.eval as ev
    from openmatch.inference import distributed_parallel_embedding_inference as ref_inference

    cfg, seed, corpus, queries = driver_run_inputs()
    sd = random_state_dict(cfg, seed)
    loaded = {}

    class HostBackbone(M.VisRAGRetB200):
        def __init__(self, cfg_, state_dict, device="cuda:0"):
            self.config, self.device, self.dtype, self.training = cfg_, torch.device("cpu"), torch.bfloat16, False
            loaded["cfg"], loaded["sd"] = cfg_, {k: v.float() for k, v in state_dict.items()}

    class HostDR(M.DRModelForInference):
        def encode(self, items, model, head, is_query=False, **kwargs):
            if items is None:
                return None, None
            reps = O.encode(loaded["sd"], loaded["cfg"], kwargs["tokenizer"], items["text"], items["image"],
                            pooling=self.pooling, max_inp_length=kwargs.get("max_inp_length", 2048))
            return None, torch.from_numpy(reps)

    backbone = M.VisRAGRetB200
    M.VisRAGRetB200, ev.DRModelForInference = HostBackbone, HostDR
    try:
        with tempfile.TemporaryDirectory() as tmp:
            ckpt = os.path.join(tmp, "VisRAG-Ret-synthetic")
            save_checkpoint(ckpt, cfg, sd)
            args = driver_run_args(os.path.join(tmp, "out"), "cpu")
            model = ev.setup_model(args, R["ModelArguments"](model_name_or_path=ckpt, pooling="wmean", normalize=True))
            assert loaded["cfg"] == cfg
            tok = StubTokenizer(cfg.vocab)
            kw = {"tokenizer": tok, "max_inp_length": 2048}
            ref_inference(dataset=corpus, model=model, args=args, dataset_type="corpus", split_save=True, model_additional_args=kw)
            ref_inference(dataset=queries, model=model, args=args, dataset_type="query", split_save=False, model_additional_args=kw)
            names = sorted(f for f in os.listdir(args.output_dir) if f.startswith("embeddings."))
            shards = [pickle.load(open(os.path.join(args.output_dir, f), "rb")) for f in names]
            qrels = os.path.join(tmp, "qrels.tsv")
            with open(qrels, "w") as f:
                f.write("query-id\tcorpus-id\tscore\n" + "".join(f"{q['id']}\td0\t1\n" for q in queries))
            args.phase = "retrieve"
            ev.retrieve(types.SimpleNamespace(from_hf_repo=False, qrels_path=qrels), args)
            trec_text = open(os.path.join(args.output_dir, "test.0.trec")).read()
    finally:
        M.VisRAGRetB200 = backbone
        del sys.modules["pytrec_eval"]
    out = {"shard_names": np.asarray(names), "trec_text": np.asarray(trec_text)}
    for n, (emb, ids) in zip(names, shards):
        out[f"{n}:reps"] = np.asarray(emb, dtype=np.float32)
        out[f"{n}:ids"] = np.asarray(ids)
    np.savez_compressed(DRIVER_RUN, **out)
    print("driver run:", {k: v.shape for k, v in out.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--full", action="store_true", help="also generate the full-size (3.1 B parameter) case")
    ap.add_argument("--full-v2", action="store_true", help="only generate full_v2 (36 pages, 10 queries, top-5; ~15 min of CPU)")
    ap.add_argument("--tiny-v2", action="store_true", help="only generate tiny_v2 (same corpus as full_v2, tiny model)")
    ap.add_argument("--checks", action="store_true", help="only generate reference_checks and driver_run (~1 min of CPU)")
    a = ap.parse_args()
    from visrag_b200.config import VisRAGConfig as _C

    if a.checks:
        gen_reference_checks()
        gen_driver_run()
        return

    if a.full_v2 or a.tiny_v2:
        if not os.path.exists(REAL_PAGES):
            gen_real_pages()
        if a.tiny_v2:
            gen_spec_case("tiny_v2", _C.tiny(), 1234, full_v2_spec(), 8, 25, 5)
        if a.full_v2:
            gen_spec_case("full_v2", _C.full(), 4321, full_v2_spec(), 8, 25, 5)
        return
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    from visrag_b200.config import VisRAGConfig

    gen_geometry()
    sizes = [(224, 224), (448, 448), (224, 224), (700, 900), (760, 141), (1200, 500), (320, 240), (448, 448)]
    gen_model_case("tiny_v1", VisRAGConfig.tiny(), 1234, sizes, 7, 4, 5, 5)
    if a.full:
        gen_model_case("full_v1", VisRAGConfig.full(), 4321, [(448, 448), (224, 224), (640, 480)], 17, 3, 15, 3)


if __name__ == "__main__":
    main()

"""Shared test helpers: synthetic pages/queries (same generators the golden script used) and golden loading."""
import json
import os

import numpy as np
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
REFERENCE_CHECKS = os.path.join(GOLDEN, "reference_checks.npz")
DRIVER_RUN = os.path.join(GOLDEN, "driver_run.npz")
from visrag_b200.synth import QUERY_PREFIX, synth_doc_pages, synth_pages  # noqa: E402,F401


def load_case(name):
    from visrag_b200.config import VisRAGConfig

    z = np.load(os.path.join(GOLDEN, f"{name}.npz"), allow_pickle=False)
    cfg = VisRAGConfig(**json.loads(str(z["config"])))
    if "page_spec" in z.files:
        pages = pages_from_spec(json.loads(str(z["page_spec"])))
    else:
        pages = synth_pages(z["page_sizes"], int(z["page_seed"]))
    queries = [str(q) for q in z["queries"]]
    return cfg, int(z["weight_seed"]), pages, queries, z


def _real():
    return np.load(os.path.join(GOLDEN, "real_pages.npz"), allow_pickle=False)


def real_queries():
    """The two queries of the reference's examples/training_data/0.parquet (query i belongs to page parquet{i})."""
    return [str(q) for q in _real()["queries"]]


def pages_from_spec(spec):
    """[{kind: doc|noise, size, seed} | {kind: real, name}] -> PIL RGB pages (real ones decoded from the shipped bytes)."""
    import io

    out = []
    for e in spec:
        if e["kind"] == "doc":
            out.append(synth_doc_pages([tuple(e["size"])], e["seed"])[0])
        elif e["kind"] == "noise":
            out.append(synth_pages([tuple(e["size"])], e["seed"])[0])
        else:
            out.append(Image.open(io.BytesIO(_real()[e["name"]].tobytes())).convert("RGB"))
    return out


def cosine_rows(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


# ---- inputs of the comparisons with the reference (its outputs on them: oracle/gen_golden.py --checks)
def restatement_inputs():
    """Inputs of tests/test_oracle_vs_reference.py::test_restatement_equals_reference_on_fresh_inputs."""
    from visrag_b200.config import VisRAGConfig

    pages = synth_pages([(300, 300), (1000, 600), (448, 448)], 21)
    texts = ["", "doc text", ""]
    queries = [QUERY_PREFIX + "what is shown", QUERY_PREFIX + "x"]
    return VisRAGConfig.tiny(), 777, texts, pages, queries


def pooling_inputs():
    """Inputs of tests/test_oracle_vs_reference.py::test_other_poolings_equal_reference_on_a_ragged_batch."""
    from visrag_b200.config import VisRAGConfig

    page = synth_pages([(448, 448)], 5)[0]
    texts = [QUERY_PREFIX + "a", QUERY_PREFIX + "a much longer query about the page content", ""]
    return VisRAGConfig.tiny(), 778, texts, [None, None, page]


def scoring_inputs():
    """Inputs of tests/test_oracle_vs_reference.py::test_score_topk_and_run_files_equal_reference."""
    rs = np.random.RandomState(12)
    D = rs.randn(500, 64).astype(np.float32)
    D /= np.linalg.norm(D, axis=1, keepdims=True)
    Q = rs.randn(7, 64).astype(np.float32)
    Q /= np.linalg.norm(Q, axis=1, keepdims=True)
    return Q, D, [f"doc{i}" for i in range(len(D))]


def driver_run_inputs():
    """Checkpoint weights, corpus and queries of tests/test_dropin_reference_driver.py."""
    from visrag_b200.config import VisRAGConfig
    from visrag_b200.synth import synth_doc_pages

    pages = synth_doc_pages([(448, 448)] * 7 + [(700, 900), (640, 300), (448, 448)], 31)
    corpus = [{"id": f"d{i}", "text": "", "image": im} for i, im in enumerate(pages)]
    queries = [{"id": f"q{i}", "text": QUERY_PREFIX + t, "image": None} for i, t in enumerate(["revenue table", "climate"])]
    return VisRAGConfig.tiny(), 77, corpus, queries


def driver_run_args(output_dir, device):
    """The encode arguments of the run: batch 3 and max_inmem_docs 6, so the corpus is flushed in two shards."""
    from types import SimpleNamespace

    return SimpleNamespace(phase="encode", device=device, output_dir=output_dir, per_device_eval_batch_size=3,
                           dataloader_num_workers=0, dataloader_pin_memory=False, fp16=False, max_inmem_docs=6, world_size=1,
                           process_index=0, retrieve_depth=4, trec_save_path=None)

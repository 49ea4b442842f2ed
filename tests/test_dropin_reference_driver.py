"""The drop-in classes on the path the REAL reference driver takes, against what that driver produced.

tests/golden/driver_run.npz holds the outputs of the reference's `src/openmatch/driver/eval.py`, imported unmodified and
driving this package's `DRModelForInference` on a synthetic checkpoint directory (oracle/gen_golden.py --checks):
setup_model -> DRModelForInference.build, its distributed_parallel_embedding_inference (inference.py:53-172) writing
the pickle shards, its retrieve phase (eval.py:210-232) writing the run file. Only the device math was replaced there
(oracle embeddings on the CPU). Here the same checkpoint goes through the same calls of this package on the GPU:
`build` (what setup_model calls, eval.py:118-134), `.to` / `.eval`, `inference.distributed_parallel_embedding_inference`
and `retriever.distributed_parallel_retrieve` + `save_as_trec`; the shards and the run must be the reference driver's."""
import os

import numpy as np
import pytest

from tests.helpers import DRIVER_RUN, cosine_rows, driver_run_args, driver_run_inputs

pytestmark = pytest.mark.gpu


def test_reference_driver_drives_the_dropin_classes(tmp_path):
    from types import SimpleNamespace

    from visrag_b200 import inference as I
    from visrag_b200 import retriever as R
    from visrag_b200.modeling import DRModelForInference
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict, save_checkpoint

    ref = np.load(DRIVER_RUN, allow_pickle=False)
    cfg, seed, corpus, queries = driver_run_inputs()
    ckpt = str(tmp_path / "VisRAG-Ret-synthetic")
    save_checkpoint(ckpt, cfg, random_state_dict(cfg, seed))
    margs = SimpleNamespace(model_name_or_path=ckpt, pooling="wmean", normalize=True, cache_dir=None)
    model = DRModelForInference.build(model_args=margs, cache_dir=margs.cache_dir)
    assert model.to("cuda:0") is model and model.eval() is model
    assert model.pooling == "wmean" and model.normalize is True and model.lm_q.config == cfg

    args = driver_run_args(str(tmp_path / "out"), "cuda:0")
    kw = {"tokenizer": StubTokenizer(cfg.vocab), "max_inp_length": 2048}
    I.distributed_parallel_embedding_inference(corpus, model, args, dataset_type="corpus", split_save=True, model_additional_args=kw)
    I.distributed_parallel_embedding_inference(queries, model, args, dataset_type="query", split_save=False, model_additional_args=kw)
    names = sorted(f for f in os.listdir(args.output_dir) if f.startswith("embeddings."))
    assert names == [str(n) for n in ref["shard_names"]]  # flush rule of inference.py:112 at max_inmem_docs=6
    for n in names:
        emb, ids = R.load_shard(os.path.join(args.output_dir, n))
        assert ids == [str(i) for i in ref[f"{n}:ids"]], n
        assert cosine_rows(emb, ref[f"{n}:reps"]).min() >= 0.9999, n

    args.phase = "retrieve"
    run = R.distributed_parallel_retrieve(args, args.retrieve_depth)
    I.save_as_trec(run, os.path.join(args.output_dir, "test.0.trec"))
    ref_path = str(tmp_path / "reference.trec")
    with open(ref_path, "w") as f:
        f.write(str(ref["trec_text"]))
    ref_run = I.load_from_trec(ref_path)
    got_run = I.load_from_trec(os.path.join(args.output_dir, "test.0.trec"))
    assert set(got_run) == set(ref_run) == {q["id"] for q in queries}
    for qid, docs in ref_run.items():
        got = got_run[qid]
        assert set(got) == set(docs), qid  # union of per-shard top-4 (dense_retriever.py:88-92)
        assert max(got, key=got.get) == max(docs, key=docs.get), qid
        assert max(abs(got[d] - docs[d]) for d in docs) <= 2e-3, qid

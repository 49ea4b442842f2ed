"""Pins the oracle against the REAL reference: tests/golden/reference_checks.npz holds what the unmodified reference
computed on these inputs (oracle/gen_golden.py --checks), so the comparison runs on any machine."""
import json
import pickle

import numpy as np
import pytest

from tests import helpers as H


@pytest.fixture(scope="module")
def ref():
    return np.load(H.REFERENCE_CHECKS, allow_pickle=False)


def test_restatement_equals_reference_on_fresh_inputs(ref):
    from oracle import restated as O
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict

    cfg, seed, texts, pages, queries = H.restatement_inputs()
    sd = random_state_dict(cfg, seed)
    tok = StubTokenizer(cfg.vocab)
    p = O.encode(sd, cfg, tok, texts, pages)
    assert np.abs(p - ref["restate_page_reps"]).max() < 2e-6
    assert np.abs(O.encode(sd, cfg, tok, queries, [None, None]) - ref["restate_query_reps"]).max() < 2e-6
    # B1 boundary: hidden states of the valid positions (a seeded sample of rows of every sequence)
    _, hid = O.encode(sd, cfg, tok, texts, pages, return_hidden=True)
    for b, h in enumerate(hid):
        assert h.shape[0] == int(ref["restate_hidden_len"][b])
        assert np.abs(h[ref["restate_hidden_pos"][b]] - ref["restate_hidden_rows"][b]).max() < 5e-5


@pytest.mark.parametrize("pooling", ["lasttoken", "mean", "cls"])
def test_other_poolings_equal_reference_on_a_ragged_batch(ref, pooling):
    """SURVEY.md §8f.4: the pooling variants of `dense_retrieval_model.py:170-218` on a right-padded batch of unequal
    lengths (the oracle and the engine pool unpadded sequences; this pins that they mean the same thing)."""
    from oracle import restated as O
    from visrag_b200.tokenizer_stub import StubTokenizer
    from visrag_b200.weights import random_state_dict

    cfg, seed, texts, images = H.pooling_inputs()
    sd = random_state_dict(cfg, seed)
    got = O.encode(sd, cfg, StubTokenizer(cfg.vocab), texts, images, pooling=pooling)
    assert np.abs(got - ref[f"pooling_{pooling}"]).max() < 2e-6, pooling


def test_score_topk_and_run_files_equal_reference(ref, tmp_path):
    """The scoring side of the path against the REAL reference functions: `_retrieve_one_shard`
    (`retriever/dense_retriever.py:13-34`) on a pickle shard, `save_as_trec` / `load_from_trec` / `eval_mrr`
    (`utils.py:125-175,285-308`). Random unit vectors: no score ties, so torch.topk's unspecified tie order cannot differ."""
    from oracle import restated as O
    from visrag_b200 import inference as I
    from visrag_b200 import retriever as R

    Q, D, lookup = H.scoring_inputs()
    shard = str(tmp_path / "embeddings.corpus.rank.0")
    R.save_shard(shard, D, lookup)  # our writer; the reference's reader takes element 0 as the matrix, element 1 as the ids
    data = pickle.load(open(shard, "rb"))
    assert np.array_equal(np.asarray(data[0]), D) and data[1] == lookup
    s, i = O.score_topk(Q, D, 10)
    assert np.array_equal(i, ref["score_topk_ids"]) and np.abs(s - ref["score_topk_scores"]).max() < 1e-6
    # run files and MRR, built from the reference's scores: our writer gives the reference's file byte for byte, our
    # reader gives what the reference's reader gave, our MRR what its MRR gave
    s_ref, i_ref = ref["score_topk_scores"], ref["score_topk_ids"]
    run = {f"q{q}": {lookup[j]: float(s_ref[q, r]) for r, j in enumerate(i_ref[q])} for q in range(len(Q))}
    qrel = {f"q{q}": {lookup[int(i_ref[q, q % 10])]: 1} for q in range(len(Q))}
    ours = str(tmp_path / "ours.trec")
    I.save_as_trec(run, ours)
    assert open(ours).read() == str(ref["trec_text"])
    assert I.load_from_trec(ours) == json.loads(str(ref["trec_loaded"]))
    mrr = json.loads(str(ref["mrr"]))
    assert I.eval_mrr(qrel, run, 10) == mrr["10"]
    assert I.eval_mrr(qrel, run, 3) == mrr["3"]

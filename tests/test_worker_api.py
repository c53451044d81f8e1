"""prediction() / custom_prediction() / result-dict parity with the reference worker's behaviour
(worker.py:248-458, 564-645), exercised on CPU with a stub in place of the engine (the decode and the
input builder are host logic; the engine itself is covered by the -m gpu tests)."""
import numpy as np
import pytest
import torch

from vilbert_b200 import worker_api as W
from vilbert_b200 import _lib as L


class StubModel:
    """Returns fixed logits in the 10-tuple layout and records what it was called with."""
    _device = 0

    def __init__(self, seed=0):
        self.g = torch.Generator().manual_seed(seed)
        self.calls = []

    def __call__(self, question, features, spatials, segment_ids, input_mask, image_mask, co_mask, task_tokens,
                 output_all_attention_masks=False, select=None):
        B, V = features.shape[0], features.shape[1]
        self.calls.append(dict(B=B, q=tuple(question.shape), select=select, task=task_tokens.clone()))
        r = lambda *s: torch.randn(*s, generator=self.g)
        return (r(B, 3129), r(B, 1533), r(B, 1), r(B // 2, 2) if B % 2 == 0 else r(B, 2), r(B, 3), None, r(B, V, 1),
                None, r(B, question.shape[1] + 1, 1), [])


def _reference_decode(out, task_id, N, spatials, infos):
    """Direct restatement of worker.py:295-386 (softmax over view(-1), full sort descending, first N)."""
    pick = {"1": 0, "2": 0, "15": 1, "12": 3, "13": 4, "7": 2, "11": 6, "4": 6, "16": 6}[task_id]
    prob = torch.softmax(out[pick].view(-1), dim=0)
    val, idx = torch.sort(prob, 0, True)
    return val, idx


def _req(n_img, V=5, T=37):
    g = torch.Generator().manual_seed(1)
    return (torch.randint(0, 100, (1, T)), torch.randn(n_img, V, 2048, generator=g), torch.rand(n_img, V, 5, generator=g),
            torch.zeros(1, T, dtype=torch.long), torch.ones(1, T, dtype=torch.long), torch.ones(n_img, V, dtype=torch.uint8),
            torch.zeros(n_img, V, T), torch.tensor([[1]]))


@pytest.mark.parametrize("task_id,n_img", [("1", 1), ("15", 1), ("13", 1), ("12", 2), ("7", 4), ("11", 1), ("4", 1), ("16", 1)])
def test_prediction_matches_reference_decode(task_id, n_img):
    W.model = StubModel(seed=3)
    infos = [{"image_width": 640, "image_height": 480}] * n_img
    req = _req(n_img)
    ans = W.prediction(*req, task_id, infos)
    call = W.model.calls[-1]
    # text is replicated for pair / retrieval tasks (worker.py:266-284); only the task's head is requested
    assert call["B"] == n_img and call["q"] == (2 if task_id == "12" else n_img if task_id == "7" else 1, 37)
    assert call["select"] == W.TASK_OUTPUT[task_id]
    ref_model = StubModel(seed=3)
    q = req[0].repeat(call["q"][0], 1)
    out = ref_model(q, *req[1:7], req[7].repeat(call["q"][0], 1))
    N = n_img if task_id == "7" else 3
    val, idx = _reference_decode(out, task_id, N, req[2], infos)
    if task_id in W.GROUNDING_TASKS:
        assert isinstance(ans, list) and len(ans) == 3
        for i, a in enumerate(ans):
            box = req[2][0][idx[i]][:4].tolist()
            assert a == {"y1": int(box[1] * 480), "y2": int(box[3] * 480), "x1": int(box[0] * 640), "x2": int(box[2] * 640),
                         "confidence": pytest.approx(val[i].item() * 100, rel=1e-6)}
    else:
        n_out = {"12": 2, "13": 3, "7": n_img}.get(task_id, 3)
        assert len(ans["top3_answer"]) == n_out == len(ans["top3_confidence"])
        assert ans["top3_confidence"] == pytest.approx([val[i].item() for i in range(n_out)], rel=1e-6)
        if task_id == "7":
            assert ans["top3_answer"] == [idx[i].item() for i in range(n_out)]
        if task_id == "12":
            assert set(ans["top3_answer"]) == {"True", "False"}
        if task_id == "13":
            assert set(ans["top3_answer"]) == {"contradiction (false)", "neutral", "entailment (true)"}


def test_prediction_validation():
    """Image-count asserts and the unreachable task "2" (accepted by the decode, rejected by the validator)."""
    W.model = StubModel()
    one = [{"image_width": 1, "image_height": 1}]
    with pytest.raises(AssertionError):
        W.prediction(*_req(2), "1", one * 2)
    with pytest.raises(AssertionError):
        W.prediction(*_req(1), "12", one)
    with pytest.raises(AssertionError):
        W.prediction(*_req(1), "7", one)
    with pytest.raises(AssertionError):
        W.prediction(*_req(11), "7", one * 11)
    for bad in ("2", "3", "99", "abc"):
        with pytest.raises(ValueError, match="task not valid"):
            W.prediction(*_req(1), bad, one)


def test_label_maps():
    W.model = StubModel(seed=5)
    W.label_maps["vqa"] = [f"ans{i}" for i in range(3129)]
    ans = W.prediction(*_req(1), "1", [{"image_width": 1, "image_height": 1}])
    assert all(a.startswith("ans") for a in ans["top3_answer"])
    W.label_maps["vqa"] = None
    ans = W.prediction(*_req(1), "1", [{"image_width": 1, "image_height": 1}])
    assert all(a.startswith("<vqa:") for a in ans["top3_answer"])


VOCAB = {t: i for i, t in enumerate(["[PAD]", "[UNK]", "[CLS]", "[SEP]", "what", "is", "the", "man", "hold", "##ing",
                                     "?", "color", "of", "un", "##aff", "##able", ","])}


def test_wordpiece_tokenizer():
    tok = W.WordpieceTokenizer(VOCAB)
    assert tok.tokenize("What is the man holding?") == ["what", "is", "the", "man", "hold", "##ing", "?"]
    assert tok.tokenize("unaffable, xyz") == ["un", "##aff", "##able", ",", "[UNK]"]
    ids = tok.add_special_tokens_single_sentence(tok.encode("what is the color"))
    assert ids == [2, 4, 5, 6, 11, 3]


def test_build_inputs_matches_worker_layout():
    """worker.py:402-455: pad to 37 without truncation, global mean row first, 5-d normalised boxes with
    [0,0,1,1,1] first, ones image mask, zero co-attention mask."""
    tok = W.WordpieceTokenizer(VOCAB)
    g = torch.Generator().manual_seed(2)
    feats = [torch.rand(7, 2048, generator=g), torch.rand(7, 2048, generator=g)]
    boxes = np.array([[10, 20, 110, 220], [0, 0, 640, 480], [5, 5, 50, 40], [1, 2, 3, 4], [100, 100, 200, 300],
                      [300, 50, 600, 400], [20, 30, 40, 50]], dtype=np.float32)
    infos = [{"image_width": 640, "image_height": 480, "bbox": boxes}, {"image_width": 320, "image_height": 240, "bbox": boxes / 2}]
    text, f, s, seg, im, vm, co, task = W.build_inputs("what is the man holding?", [12], feats, infos, torch.device("cpu"), tok)
    assert text.shape == (1, 37) and text.dtype == torch.long
    assert text[0, :9].tolist() == [2, 4, 5, 6, 7, 8, 9, 10, 3] and text[0, 9:].sum() == 0
    assert im[0, :9].tolist() == [1] * 9 and im[0, 9:].sum() == 0 and seg.sum() == 0
    assert f.shape == (2, 8, 2048) and torch.allclose(f[0, 0], feats[0].mean(0), atol=1e-6) and torch.equal(f[1, 1:], feats[1])
    assert s.shape == (2, 8, 5) and s[0, 0].tolist() == [0, 0, 1, 1, 1]
    x1, y1, x2, y2 = boxes[0]
    assert s[0, 1].tolist() == pytest.approx([x1 / 640, y1 / 480, x2 / 640, y2 / 480, (y2 - y1) * (x2 - x1) / (640 * 480)])
    assert torch.allclose(s[0, 1:], s[1, 1:], atol=1e-6)            # same boxes at half resolution normalise identically
    assert vm.dtype == torch.uint8 and vm.shape == (2, 8) and vm.all()
    assert co.shape == (2, 8, 37) and co.sum() == 0 and task.tolist() == [[12]]
    # longer than 37 tokens: not truncated (worker.py:408 only pads)
    long_q = " ".join(["what"] * 50)
    text, *_ = W.build_inputs(long_q, [1], feats[:1], infos[:1], torch.device("cpu"), tok)
    assert text.shape == (1, 52)


def test_shape_result():
    a = {"top3_answer": ["yes", "no", "2"], "top3_confidence": [0.71234, 0.2, 0.05]}
    assert W.shape_result("1", a, ["x"]) == {"task_id": "1", "result": [{"answer": "yes", "confidence": 71.23},
                                                                         {"answer": "no", "confidence": 20.0},
                                                                         {"answer": "2", "confidence": 5.0}]}
    b = {"top3_answer": ["True", "False"], "top3_confidence": [0.9, 0.1]}
    assert W.shape_result("12", b, ["x", "y"])["result"] == [{"answer": "True", "confidence": 90.0}, {"answer": "False", "confidence": 10.0}]
    r = {"top3_answer": [2, 0, 1], "top3_confidence": [0.5, 0.3, 0.2]}
    paths = ["/srv/media/demo/a1.jpg", "/srv/media/demo/b2.jpg", "/srv/media/demo/c3.jpg"]
    assert W.shape_result("7", r, paths) == {"task_id": "7", "image_name_list": ["demo/c3.jpg", "demo/a1.jpg", "demo/b2.jpg"],
                                             "confidence_list": [50.0, 30.0, 20.0]}
    g = [{"x1": 1, "y1": 2, "x2": 3, "y2": 4, "confidence": 55.5555}] * 3
    assert W.shape_result("11", g, ["p"], ["n0", "n1", "n2"]) == {"task_id": "11", "image_name_list": ["n0", "n1", "n2"],
                                                                  "confidence_list": [55.56] * 3}


# ----------------------------------------------------------------------------------------------- micro-batching (SURVEY 8f-4)
class RowModel:
    """Deterministic stand-in whose outputs for a row depend on that row only (as the real forward does), except the NLVR2
    head, which consumes adjacent rows as one pair ([UPSTREAM] pooled.view(-1, 2048); worker.py:266-276)."""
    _device = 0

    def __init__(self):
        g = torch.Generator().manual_seed(11)
        self.w = {k: torch.randn(2048 + 1, n, generator=g) for k, n in (("vqa", 3129), ("gqa", 1533), ("logit", 1), ("tri", 3),
                                                                         ("bin", 2))}
        self.wv = torch.randn(2048 + 5, generator=g)
        self.calls = []

    def __call__(self, question, features, spatials, segment_ids, input_mask, image_mask, co_mask, task_tokens,
                 output_all_attention_masks=False, select=None):
        B, V = features.shape[0], features.shape[1]
        self.calls.append(dict(B=B, select=select))
        x = torch.cat([features.float().mean(1), (question * input_mask).sum(1, keepdim=True).float() * 1e-3 +
                       task_tokens.float()], dim=1)
        vl = (torch.cat([features.float(), spatials.float()], dim=2) @ self.wv).unsqueeze(-1) + x[:, -1].view(B, 1, 1)
        pair = (x.view(B // 2, 2, -1).sum(1) @ self.w["bin"]) if B % 2 == 0 else x @ self.w["bin"]
        return (x @ self.w["vqa"], x @ self.w["gqa"], x @ self.w["logit"], pair, x @ self.w["tri"], None, vl, None,
                torch.zeros(B, question.shape[1] + 1, 1), [])


def _rand_req(task_id, n_img, V, seed, T=37):
    g = torch.Generator().manual_seed(seed)
    L_ = int(torch.randint(5, 20, (1,), generator=g))
    q = torch.zeros(1, T, dtype=torch.long)
    q[0, :L_] = torch.randint(1, 1000, (L_,), generator=g)
    im = (q != 0).long()
    return (q, torch.rand(n_img, V, 2048, generator=g), torch.rand(n_img, V, 5, generator=g), torch.zeros(1, T, dtype=torch.long),
            im, torch.ones(n_img, V, dtype=torch.uint8), torch.zeros(n_img, V, T), torch.tensor([[int(task_id)]]), task_id,
            [{"image_width": 640, "image_height": 480}] * n_img)


def _same(a, b):
    if isinstance(a, list):
        assert [(x["x1"], x["y1"], x["x2"], x["y2"]) for x in a] == [(x["x1"], x["y1"], x["x2"], x["y2"]) for x in b]
        assert [x["confidence"] for x in a] == pytest.approx([x["confidence"] for x in b], rel=1e-3)
    else:                       # (the stub's CPU matmul rounds differently for different batch sizes; the engine does not)
        assert a["top3_answer"] == b["top3_answer"]
        assert a["top3_confidence"] == pytest.approx(b["top3_confidence"], rel=1e-3, abs=1e-6)


def test_prediction_batch_equals_one_request_at_a_time():
    W.label_maps.update(vqa=None, gqa=None)
    reqs = [_rand_req("1", 1, 9, 1), _rand_req("12", 2, 9, 2),      # NLVR2 would start on row 1 -> filler row in front
            _rand_req("7", 4, 9, 3), _rand_req("11", 1, 9, 4), _rand_req("13", 1, 9, 5), _rand_req("12", 2, 9, 6),
            _rand_req("15", 1, 9, 7), _rand_req("1", 1, 21, 8),      # other region count -> its own model call
            _rand_req("16", 1, 21, 9), _rand_req("12", 1, 9, 10)]    # invalid: NLVR2 with one image
    W.model = RowModel()
    single = []
    for r in reqs[:-1]:
        single.append(W.prediction(*r))
    W.model = RowModel()
    got = W.prediction_batch(reqs, bucket=1)
    assert len(W.model.calls) == 2                                    # one per (T, V) group
    assert sorted(c["B"] for c in W.model.calls) == [2, 14]          # 1 + filler + 2 + 4 + 1 + 1 + 2 + 1 = 13 -> even 14
    assert all(c["select"] == L.OUT_TASK_HEADS for c in W.model.calls)   # fixed select: one plan per shape, whatever is pending
    W.model = RowModel()
    got8 = W.prediction_batch(reqs)                                   # default: batches padded to multiples of 8
    assert sorted(c["B"] for c in W.model.calls) == [8, 16]
    for a, b in zip(got8[:-1], single):
        _same(a, b)
    for a, b in zip(got[:-1], single):
        _same(a, b)
    assert isinstance(got[-1], AssertionError) and "2 images" in str(got[-1])


def test_prediction_batch_nlvr2_pair_lands_on_even_row_after_even_sized_request(monkeypatch):
    """ADVICE r1: task 1 (1 row), task 7 (2 rows), task 12: the filler must be ONE row so the pair starts at row 4, and the
    binary logits must be those of the pair itself (compared as logits, not only as the top answer)."""
    W.label_maps.update(vqa=None, gqa=None)
    monkeypatch.setattr(W, "_decode", lambda task_id, out, spatials, infos: out)     # raw sliced outputs
    for seed in range(6):
        reqs = [_rand_req("1", 1, 9, 100 + seed), _rand_req("7", 2, 9, 200 + seed), _rand_req("12", 2, 9, 300 + seed),
                _rand_req("7", 3, 9, 400 + seed), _rand_req("12", 2, 9, 500 + seed)]
        W.model = RowModel()
        single = [W.prediction(*r) for r in reqs]
        for bucket in (1, 8):
            W.model = RowModel()
            got = W.prediction_batch(reqs, bucket=bucket)
            for i in (2, 4):
                assert got[i][3].shape == (1, 2)
                assert torch.allclose(got[i][3], single[i][3], rtol=1e-4, atol=1e-4), (seed, bucket, i)
            assert torch.allclose(got[1][2], single[1][2], rtol=1e-4, atol=1e-4)


def test_micro_batch_worker_close_cancels_queued_messages():
    import concurrent.futures as cf
    W.label_maps.update(vqa=None, gqa=None)
    W.model = RowModel()
    W.tokenizer = W.WordpieceTokenizer(VOCAB)
    worker = W.MicroBatchWorker(max_rows=4, max_wait_ms=1.0)
    worker.close()
    fut = worker.submit({"image_path": ["/m/demo/a.jpg"], "question": "what", "socket_id": "s", "task_id": "1"},
                        [torch.rand(3, 2048)], [{"image_width": 4, "image_height": 4, "bbox": np.zeros((3, 4), dtype=np.float32)}])
    with pytest.raises(cf.CancelledError):
        fut.result(timeout=5)
    # a message that slipped in behind the sentinel is cancelled by close() as well
    worker2 = W.MicroBatchWorker(max_rows=4, max_wait_ms=1.0)
    worker2._q.put(None)
    late = cf.Future()
    worker2._q.put(({"task_id": "1"}, [], [], late))
    worker2.close()
    with pytest.raises(cf.CancelledError):
        late.result(timeout=5)


def test_micro_batch_worker_round_trip(monkeypatch):
    """Messages in the sender's schema (demo/sender.py:19-24) go in, WebSocket result dicts (worker.py:564-649) come out, and
    concurrent messages share a model call.  The stub computes on the CPU, so the worker is kept on its CPU path even where a
    GPU is present (test_gpu_round2.py::test_micro_batch_worker_on_engine runs it on the engine)."""
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    W.label_maps.update(vqa=None, gqa=None)
    W.model = RowModel()
    W.tokenizer = W.WordpieceTokenizer(VOCAB)
    g = torch.Generator().manual_seed(5)
    boxes = np.array([[10, 20, 110, 220], [0, 0, 640, 480], [5, 5, 50, 40]], dtype=np.float32)

    def det(n):
        return ([torch.rand(3, 2048, generator=g) for _ in range(n)],
                [{"image_width": 640, "image_height": 480, "bbox": boxes} for _ in range(n)])
    msgs = [({"image_path": ["/m/demo/a.jpg"], "question": "what is the man holding?", "socket_id": "s1", "task_id": "1"}, *det(1)),
            ({"image_path": ["/m/demo/a.jpg", "/m/demo/b.jpg"], "question": "the man is holding", "socket_id": "s2", "task_id": "12"}, *det(2)),
            ({"image_path": ["/m/demo/a.jpg", "/m/demo/b.jpg", "/m/demo/c.jpg"], "question": "what color", "socket_id": "s3", "task_id": "7"}, *det(3)),
            ({"image_path": ["/m/demo/a.jpg"], "question": "the man", "socket_id": "s4", "task_id": "11"}, *det(1)),
            ({"image_path": ["/m/demo/a.jpg"], "question": "what", "socket_id": "s5", "task_id": "99"}, *det(1))]
    expect = []
    for body, feats, infos in msgs[:-1]:          # handle_request() with the tensors kept on the CPU (no GPU in this suite)
        tid = body["task_id"]
        args = W.build_inputs(body["question"], [int(tid)], feats, infos, torch.device("cpu"))
        expect.append(W.shape_result(tid, W.prediction(*args, tid, infos), body["image_path"]))
    W.model = RowModel()
    worker = W.MicroBatchWorker(max_rows=64, max_wait_ms=300.0)
    futs = [worker.submit(*m) for m in msgs]
    res = [f.result(timeout=60) for f in futs[:-1]]
    with pytest.raises(ValueError):
        futs[-1].result(timeout=60)
    worker.close()
    assert [r["socket_id"] for r in res] == ["s1", "s2", "s3", "s4"]
    for r, e in zip(res, expect):
        assert r["result"]["task_id"] == e["task_id"]
        if "result" in e:
            assert [x["answer"] for x in r["result"]["result"]] == [x["answer"] for x in e["result"]]
            assert [x["confidence"] for x in r["result"]["result"]] == pytest.approx([x["confidence"] for x in e["result"]], abs=0.02)
        else:
            assert r["result"]["image_name_list"] == e["image_name_list"]
            assert r["result"]["confidence_list"] == pytest.approx(e["confidence_list"], abs=0.02)
    # all five messages were pending together: ONE model call -- 1 + filler (NLVR2 onto an even row) + 2 + 3 + 1 rows = 8
    assert [c["B"] for c in W.model.calls] == [8]

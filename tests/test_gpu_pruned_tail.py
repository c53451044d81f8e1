"""Pruned tail on the GPU engine.  `-m gpu`.

When no selected output reads a stream's sequence, the stream's last layer after the last connection layer (T11 and V5 in the
12/6/6 schedule) runs everything after its QKV projection on row 0 of each sample -- the only row the poolers read.  Every kernel
computes a row from that row alone in a fixed order, so the selected outputs must keep their bits.  The reference is the same
engine with debug_taps=True: asking for the sequence outputs forces the full tail.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

NAMES = ["vil_prediction", "vil_prediction_gqa", "vil_logit", "vil_binary_prediction", "vil_tri_prediction",
         "vision_prediction", "vision_logit", "linguisic_prediction", "linguisic_logit"]


def _selects():
    from vilbert_b200 import _lib as L
    pooled = [L.OUT_VIL_PREDICTION, L.OUT_VIL_PREDICTION_GQA, L.OUT_VIL_LOGIT, L.OUT_VIL_BINARY_PREDICTION,
              L.OUT_VIL_TRI_PREDICTION]
    union = 0
    for s in pooled:
        union |= s
    return pooled + [union,
                     L.OUT_VIL_PREDICTION | L.OUT_VISION_LOGIT,          # only the text tail is pruned
                     L.OUT_VIL_PREDICTION | L.OUT_LINGUISIC_LOGIT]       # only the image tail is pruned


SELECT_IDS = ["vqa", "gqa", "vil_logit", "binary", "tri", "pooled_union", "vqa+vision_logit", "vqa+linguisic_logit"]


def _engine(oracle, **kw):
    import vilbert_b200 as vb
    cfg = vb.BertConfig.from_dict(oracle.config.to_dict())
    m = vb.VILBertForVLTasks.from_pretrained(oracle.state_dict(), config=cfg, num_labels=oracle.num_labels, **kw)
    return m.eval().cuda(0)


def _inputs(oracle, B, Tin, V, seed, pad=0):
    from oracle import vilbert_ref as R
    inp = list(R.make_inputs(B, Tin, V, seed=seed, vocab_size=oracle.config.vocab_size, pad_regions=pad))
    inp[1] = inp[1][..., :oracle.config.v_feature_size].contiguous()
    return [t.cuda() for t in inp]


def _assert_same(got, want, select, tag):
    n = 0
    for i, name in enumerate(NAMES):
        if not select & (1 << i):
            assert got[i] is None and want[i] is None
            continue
        assert torch.equal(got[i], want[i]), (tag, name, float((got[i] - want[i]).abs().max()))
        n += 1
    assert n > 0


def _check(eng, inp, select, tag):
    got = eng(*inp, select=select)
    want, _ = eng(*inp, select=select, debug_taps=True)
    torch.cuda.synchronize()
    _assert_same(got, want, select, tag)


@pytest.fixture(scope="module")
def tiny_engines(tiny_oracle):
    e = {k: _engine(tiny_oracle, compute_dtype=k) for k in ("fp16", "bf16")}
    yield e
    for m in e.values():
        m.close()


@pytest.fixture(scope="module")
def full_engines(full_oracle):
    e = {k: _engine(full_oracle, compute_dtype=k) for k in ("fp16", "bf16")}
    yield e
    for m in e.values():
        m.close()


# (B, Tin, V, pad): odd and even batches, ragged text, padded regions, and sequences beyond one 64-key block (T = 71, V = 101)
TINY_SHAPES = [(1, 12, 10, 0), (3, 30, 36, 3), (4, 22, 14, 2), (3, 70, 101, 7)]


@pytest.mark.parametrize("sel", range(8), ids=SELECT_IDS)
@pytest.mark.parametrize("B,Tin,V,pad", TINY_SHAPES)
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_tiny_pruned_equals_full_tail(tiny_oracle, tiny_engines, dt, B, Tin, V, pad, sel):
    select = _selects()[sel]
    _check(tiny_engines[dt], _inputs(tiny_oracle, B, Tin, V, 300 + B, pad), select, (dt, B, Tin, V, SELECT_IDS[sel]))


@pytest.mark.parametrize("sel", range(8), ids=SELECT_IDS)
@pytest.mark.parametrize("B", [2, 64])
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_full_pruned_equals_full_tail(full_oracle, full_engines, dt, B, sel):
    select = _selects()[sel]
    _check(full_engines[dt], _inputs(full_oracle, B, 30, 36, 500 + B, pad=2), select, (dt, B, SELECT_IDS[sel]))


def test_host_api_and_slot(tiny_oracle, tiny_engines):
    """vb200_forward_host and workspace slot 1 pick the pruned plan too, and return the full tail's bits."""
    from vilbert_b200 import _lib as L
    eng = tiny_engines["fp16"]
    inp = _inputs(tiny_oracle, 4, 20, 12, 8, pad=1)
    select = L.OUT_VIL_PREDICTION | L.OUT_VIL_LOGIT
    want, _ = eng(*inp, select=select, debug_taps=True)
    got = eng(*inp, select=select, slot=1)
    torch.cuda.synchronize()
    _assert_same(got, want, select, "slot1")
    hin = [t.cpu().pin_memory() for i, t in enumerate(inp) if i != 6]
    out = {"vil_prediction": torch.empty(4, tiny_oracle.num_labels).pin_memory(), "vil_logit": torch.empty(4, 1).pin_memory()}
    eng.forward_host(*hin, out, select=select, slot=1)
    assert torch.equal(out["vil_prediction"], want[0].cpu()) and torch.equal(out["vil_logit"], want[2].cpu())
    # a sequence output through the host entry point gets the full-tail plan
    T = 20 + (1 if eng._dims["task_specific_tokens"] else 0)
    out_seq = {"vil_prediction": torch.empty(4, tiny_oracle.num_labels).pin_memory(),
               "sequence_output_t": torch.empty(4, T, tiny_oracle.config.hidden_size).pin_memory()}
    eng.forward_host(*hin, out_seq, select=L.OUT_VIL_PREDICTION)
    _, taps = eng(*inp, select=L.OUT_VIL_PREDICTION, debug_taps=True)
    torch.cuda.synchronize()
    assert torch.equal(out_seq["sequence_output_t"], taps["sequence_output_t"].cpu())


@pytest.mark.parametrize("which", ["tiny", "full"])
def test_forward_cached_vil_logit(which, tiny_oracle, full_oracle, tiny_engines, full_engines):
    """Retrieval suffix plans prune like full plans: cached-state scores equal the plain forward and the full-tail forward."""
    from vilbert_b200 import _lib as L
    oracle, eng = (tiny_oracle, tiny_engines["fp16"]) if which == "tiny" else (full_oracle, full_engines["fp16"])
    cap, img = _inputs(oracle, 5, 22, 14, 71), _inputs(oracle, 4, 22, 14, 72, pad=2)
    q, seg, im = cap[0], cap[3], cap[4]
    f, s, vm = img[1], img[2], img[5]
    task = torch.full((5, 1), 7, dtype=torch.long).cuda()
    ts, vs = eng.encode_text(q, seg, im, task), eng.encode_image(f, s, vm)
    ci = torch.tensor([0, 0, 1, 2, 3, 4, 4, 2, 1], dtype=torch.int32)
    ii = torch.tensor([0, 3, 1, 2, 0, 3, 1, 1, 2], dtype=torch.int32)
    got = eng.forward_cached(ts, ci, vs, ii, select=L.OUT_VIL_LOGIT)
    cl, il = ci.long().cuda(), ii.long().cuda()
    args = (q[cl], f[il], s[il], seg[cl], im[cl], vm[il], None, task[cl])
    plain = eng(*args, select=L.OUT_VIL_LOGIT)
    full, _ = eng(*args, select=L.OUT_VIL_LOGIT, debug_taps=True)
    torch.cuda.synchronize()
    assert torch.equal(got[2], plain[2]) and torch.equal(got[2], full[2])


def test_plan_info_launches_and_flops(full_oracle, full_engines):
    """Same launch count; the executed FLOPs drop by exactly the B * (L - 1) rows the two tails no longer compute."""
    from vilbert_b200 import _lib as L
    eng = full_engines["bf16"]
    c = full_oracle.config
    B, Tin, V = 64, 30, 36
    T = Tin + (1 if eng._dims["task_specific_tokens"] else 0)
    n1, f1 = eng.plan_info(B, Tin, V, L.OUT_VIL_PREDICTION)
    eng.set_option("prune_tail", 0)
    try:
        n0, f0 = eng.plan_info(B, Tin, V, L.OUT_VIL_PREDICTION)
    finally:
        eng.set_option("prune_tail", 1)
    H, I, Hv, Iv = c.hidden_size, c.intermediate_size, c.v_hidden_size, c.v_intermediate_size

    def tail(rows_dropped, L_, h, inter):
        # attention-out projection, FFN-in, FFN-out (2 FLOPs per MAC) + attention (QK^T and PV over L keys per query row)
        return 2.0 * rows_dropped * (h * h + 2 * h * inter) + 4.0 * rows_dropped * L_ * h
    expect = tail(B * (T - 1), T, H, I) + tail(B * (V - 1), V, Hv, Iv)
    assert n1 == n0
    assert abs((f0 - f1) - expect) <= 1e-9 * f0, (f0, f1, expect)


def test_prune_option_bit_identical(full_oracle, full_engines):
    """set_option("prune_tail", 0 / 1) rebuilds the plans; both give the same bits."""
    from vilbert_b200 import _lib as L
    eng = full_engines["fp16"]
    inp = _inputs(full_oracle, 64, 30, 36, 1234)
    select = L.OUT_VIL_PREDICTION | L.OUT_VIL_LOGIT
    pruned = eng(*inp, select=select)
    torch.cuda.synchronize()
    eng.set_option("prune_tail", 0)
    try:
        full = eng(*inp, select=select)
        torch.cuda.synchronize()
    finally:
        eng.set_option("prune_tail", 1)
    _assert_same(pruned, full, select, "prune_tail")

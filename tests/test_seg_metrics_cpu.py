"""CPU: segmentation and classification metrics against ground truth (oracle/metrics_ref.py, metrics.py,
ug_seg_metrics_desc, PipelineRunner.plan(seg_metrics=...)).

* metrics_ref against brute-force all-pairs distances on random small masks (exact integer squared distances and the
  percentile), closed forms (single pixels, concentric squares, the full frame whose surface is the border ring) and the
  empty-set conventions;
* the device's fp64 restatement of np.percentile's linear method (index, lerp, no contraction) against np.percentile;
* classification_metrics against sklearn (confusion_matrix, precision_recall_fscore_support, roc_auc_score ovr),
  with a class missing from the labels;
* the C-ABI mirror of the descriptor: sizeof(ug_op) unchanged, the field layout of include/ugnet.h, kind 20, symbols;
* lowering (stub engine): the op last, the plan keys, the io names of plan images, the ValueError cases, default
  programs unchanged;
* a ragged source_frame=True, seg_metrics="source" pipeline program emulated whole by the descriptor interpreter.
"""
import ctypes
import math
import re

import numpy as np
import pytest
import torch

import ugnet_b200  # noqa: F401
from oracle import metrics_ref, program_ref, ragged_ref, cam_ref, source_ref
from ugnet_b200 import engine as E
from ugnet_b200 import lower, metrics
from ugnet_b200.util import ragged

from test_abi import ROOT
from test_lowering_cpu import _FakeEngine, _gnet_sd, _unet_sd
from test_plan import _parse
from test_source_frame_cpu import _normalised, _sources, _states

OP_BYTES = 280
S = 224


@pytest.fixture()
def fake_engine(monkeypatch):
    monkeypatch.setattr(E.Engine, "get", classmethod(lambda cls, device=0: _FakeEngine()))


def _brute(p, g):
    """(counts, HD, HD95) from all-pairs distances between the surfaces (4-neighbour rule written out)."""
    def surf(x):
        pad = np.pad(x, 1)
        inner = pad[:-2, 1:-1] & pad[2:, 1:-1] & pad[1:-1, :-2] & pad[1:-1, 2:]
        return x & ~inner
    p, g = p != 0, g != 0
    counts = (int((p & g).sum()), int((p & ~g).sum()), int((g & ~p).sum()))
    a, b = np.argwhere(surf(p)), np.argwhere(surf(g))
    if len(a) == 0 and len(b) == 0:
        return counts, math.nan, math.nan
    if len(a) == 0 or len(b) == 0:
        return counts, math.inf, math.inf
    sq = ((a[:, None, :] - b[None, :, :]) ** 2).sum(-1)
    d_pg, d_gp = np.sqrt(sq.min(1).astype(np.float64)), np.sqrt(sq.min(0).astype(np.float64))
    return counts, max(d_pg.max(), d_gp.max()), max(np.percentile(d_pg, 95), np.percentile(d_gp, 95))


def _same(a, b):
    return (math.isnan(a) and math.isnan(b)) or a == b


def test_reference_against_all_pairs():
    rng = np.random.default_rng(3)
    for k in range(120):
        H, W = (int(v) for v in rng.integers(1, 24, 2))
        dens = rng.uniform(0, 1, 2)
        p = (rng.random((H, W)) < dens[0]).astype(np.uint8) * (255 if k % 3 == 0 else 1)
        g = (rng.random((H, W)) < dens[1]).astype(np.uint8) * (7 if k % 2 else 1)
        got, want = metrics_ref.seg_metrics(p, g), _brute(p, g)
        assert got[0] == want[0] and _same(got[1], want[1]) and _same(got[2], want[2]), k
        sp, sg = metrics_ref.surface(p), metrics_ref.surface(g)
        if sp.any() and sg.any():
            a, b = np.argwhere(sp), np.argwhere(sg)
            assert np.array_equal(metrics_ref.directed_sq(sp, sg), ((a[:, None] - b[None]) ** 2).sum(-1).min(1))


def test_reference_closed_forms_and_empty_sets():
    z = np.zeros((20, 30), np.uint8)
    p, g = z.copy(), z.copy()
    p[2, 3], g[7, 15] = 1, 1
    c, hd, hd95 = metrics_ref.seg_metrics(p, g)
    assert c == (0, 1, 1) and hd == hd95 == math.sqrt(5 ** 2 + 12 ** 2)
    p, g = z.copy(), z.copy()                                     # concentric squares two pixels apart
    p[5:15, 5:15], g[3:17, 3:17] = 1, 1
    # d_PG is 2 everywhere; of the 52 pixels of dG, 40 are at 2, 8 at sqrt(5) and the 4 corners at sqrt(8), so
    # the 95th percentile (virtual index 48.45) lies among the corners
    c, hd, hd95 = metrics_ref.seg_metrics(p, g)
    assert c == (100, 0, 96) and hd == hd95 == math.sqrt(8)
    assert metrics_ref.seg_metrics(g, p) == ((100, 96, 0), math.sqrt(8), math.sqrt(8))
    full = np.ones((9, 13), np.uint8)                            # full frame: the surface is the border ring
    s = metrics_ref.surface(full)
    assert s.sum() == 2 * 9 + 2 * 13 - 4 and not s[1:-1, 1:-1].any()
    assert metrics_ref.seg_metrics(full, full) == ((117, 0, 0), 0.0, 0.0)
    c, hd, hd95 = metrics_ref.seg_metrics(z, z)
    assert c == (0, 0, 0) and math.isnan(hd) and math.isnan(hd95)
    assert metrics_ref.seg_metrics(p, z)[1:] == (math.inf, math.inf)
    assert metrics_ref.seg_metrics(z, g)[1:] == (math.inf, math.inf)
    dice, iou = metrics.dice_iou(torch.tensor([[3, 1, 2], [0, 5, 0], [0, 0, 0], [4, 0, 0]]))
    assert dice[0] == 6 / 9 and iou[0] == 3 / 6 and math.isnan(dice[1]) and math.isnan(iou[2])
    assert dice[3] == 1.0 and iou[3] == 1.0


def _pct95_device(keys):
    """The device's arithmetic: order statistics lo / hi of the integer keys, then the fp64 lerp."""
    k = np.sort(keys)
    n = len(k)
    v = float(n - 1) * 0.95
    lo = int(math.floor(v))
    hi = min(lo + 1, n - 1)
    g = v - lo
    a, b = math.sqrt(float(k[lo])), math.sqrt(float(k[hi]))
    diff = b - a
    return b - diff * (1.0 - g) if g >= 0.5 else a + diff * g


def test_percentile_restatement_is_bit_exact():
    rng = np.random.default_rng(5)
    for n in list(range(1, 300)) + [int(v) for v in rng.integers(300, 200_000, 40)]:
        keys = rng.integers(0, 2 * 1791 ** 2, n) if n % 2 else rng.integers(0, 30, n)
        assert _pct95_device(keys) == np.percentile(np.sqrt(keys.astype(np.float64)), 95), n


def test_classification_metrics_against_sklearn():
    from sklearn.metrics import confusion_matrix, precision_recall_fscore_support, roc_auc_score
    rng = np.random.default_rng(8)
    for missing in (None, 4):
        y = rng.integers(0, 6, 200)
        if missing is not None:
            y[y == missing] = 0
        logits = torch.from_numpy(rng.standard_normal((200, 6)) + np.eye(6)[y] * 1.5).float()
        m = metrics.classification_metrics(logits, torch.from_numpy(y))
        pred = logits.argmax(1).numpy()
        assert np.array_equal(m["confusion"], confusion_matrix(y, pred, labels=list(range(6))))
        p, r, f, _ = precision_recall_fscore_support(y, pred, labels=list(range(6)), zero_division=0)
        assert np.allclose(m["precision"], p, rtol=0, atol=1e-12) and np.allclose(m["recall"], r, rtol=0, atol=1e-12)
        assert np.allclose(m["f1"], f, rtol=0, atol=1e-12) and abs(m["macro_f1"] - f.mean()) < 1e-12
        assert m["accuracy"] == float((pred == y).mean())
        prob = torch.softmax(logits.double(), 1).numpy()
        for k in range(6):
            if k == missing:
                assert math.isnan(m["auroc"][k])
            else:
                assert abs(m["auroc"][k] - roc_auc_score(y == k, prob[:, k])) < 1e-12
        if missing is None:
            assert abs(m["macro_auroc"] - roc_auc_score(y, prob, multi_class="ovr")) < 1e-12
        else:
            assert abs(m["macro_auroc"] - np.mean([m["auroc"][k] for k in range(6) if k != missing])) < 1e-15
    with pytest.raises(ValueError):
        metrics.classification_metrics(torch.zeros(3, 5), torch.zeros(3, dtype=torch.long))


def test_descriptor_fits_the_op_union_and_mirrors_the_header():
    assert ctypes.sizeof(E.Op) == OP_BYTES
    assert ctypes.sizeof(E.SegMetricsDesc) <= ctypes.sizeof(E._OpUnion) == ctypes.sizeof(E.ConvDesc)
    assert E._DESC_KIND[E.SegMetricsDesc] == E.OP_SEG_METRICS == 20
    assert E._SINGLE_ENTRY[20] == "ug_seg_metrics"
    assert {"ug_seg_metrics", "ug_seg_metrics_workspace_bytes"} <= set(E.EXPORTED_SYMBOLS)
    src = open(f"{ROOT}/include/ugnet.h").read()
    body = re.search(r"typedef struct ug_seg_metrics_desc \{(.*?)\} ug_seg_metrics_desc;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [re.findall(r"\w+", part)[-1] for part in decl.split(",")]
    assert names == [f for f, _ in E.SegMetricsDesc._fields_]
    assert E.SegMetricsDesc.workspace_bytes.offset == 56 and E.SegMetricsDesc.B.offset == 72
    assert ctypes.sizeof(E.SegMetricsDesc) == 88
    assert re.search(r"UG_OP_SEG_METRICS\s*=\s*20", src)
    assert re.search(r"int ug_seg_metrics\(ug_handle h, const ug_seg_metrics_desc\* d, void\* stream\);", src)
    assert re.search(r"size_t ug_seg_metrics_workspace_bytes\(int B, long long capacity_px\);", src)


KW = [{"source": (300, 400)}, {"source": "ragged", "capacity": 70_000}]


def test_seg_metrics_lowering(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    for kw in [{}] + KW:
        for frame in ("input", "source"):
            if frame == "source" and not kw:
                continue
            sf = frame == "source"
            base = pipe.plan(4, source_frame=sf, **kw)["program"].descs
            ws = pipe.plan(4, source_frame=sf, seg_metrics=frame, **kw)
            descs = ws["program"].descs
            assert len(descs) == len(base) + 1 and isinstance(descs[-1], E.SegMetricsDesc)
            assert _normalised(descs[:-1]) == _normalised(base)
            d = descs[-1]
            pred = ws["mask"] if frame == "input" else ws["src_mask"]
            assert d.pred == pred.data_ptr() and d.gt == ws["gt_mask"].data_ptr() and not d.status
            assert ws["gt_mask"].shape == pred.shape and ws["gt_mask"].dtype == torch.uint8
            assert d.counts == ws["seg_counts"].data_ptr() and ws["seg_counts"].shape == (4, 3)
            assert d.hd == ws["seg_hd"].data_ptr() and ws["seg_hd"].dtype == torch.float64
            assert d.workspace == ws["seg_workspace"].data_ptr() and d.workspace_bytes == ws["seg_workspace"].numel()
            assert d.workspace_bytes >= pred.numel() * 5
            assert any(t is ws["seg_workspace"] for t in ws["program"].keepalive)
            if frame == "source" and kw["source"] == "ragged":
                assert d.index == ws["src_index"].data_ptr() and d.capacity_px == pred.numel() and d.Hs == 0
            else:
                assert not d.index and (d.Hs, d.Ws) == ((S, S) if frame == "input" else kw["source"])
            assert pipe.plan(4, source_frame=sf, seg_metrics=frame, **kw) is ws
            assert pipe.plan(4, source_frame=sf, **kw)["program"].descs is not descs
    with pytest.raises(ValueError):
        pipe.plan(2, source=(300, 400), seg_metrics="source")          # needs source_frame=True
    with pytest.raises(ValueError):
        pipe.plan(2, seg_metrics="sources")
    with pytest.raises(ValueError):
        pipe(torch.zeros((2, 3, S, S)), gt_masks=torch.zeros((2, S, S), dtype=torch.uint8), metrics_frame="source")
    with pytest.raises(ValueError):
        pipe(torch.zeros((2, 3, S, S)), gt_masks=torch.zeros((2, 100, S), dtype=torch.uint8))
    with pytest.raises(ValueError):
        pipe([np.zeros((30, 40, 3), np.uint8)], gt_masks=[np.zeros((30, 41), np.uint8)], metrics_frame="source")


@pytest.mark.parametrize("kw", [{}] + KW)
def test_default_programs_are_unchanged_by_metrics_plans(fake_engine, kw):
    a = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    b = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    want = _normalised(a.plan(2, **kw)["program"].descs)
    b.plan(2, seg_metrics="input", **kw)
    if kw:
        b.plan(2, source_frame=True, seg_metrics="source", **kw)
    assert _normalised(b.plan(2, **kw)["program"].descs) == want


def test_plan_image_lists_the_metrics_io(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=1)
    for kw, frame, n_px in [({}, "input", 2 * S * S), ({"source": (300, 400)}, "source", 2 * 300 * 400),
                            ({"source": "ragged", "capacity": 70_000}, "source", ragged.capacity(70_000))]:
        image = pipe.export_plan(2, source_frame=frame == "source", seg_metrics=frame, **kw)
        _, _, n_ops, relocs, ios, op_bytes = _parse(image)
        assert op_bytes == OP_BYTES
        sizes = {n.split(b"\0")[0].decode(): b for n, _, _, _, b in ios}
        assert sizes["gt_mask"] == n_px and sizes["seg_counts"] == 2 * 12 and sizes["seg_hd"] == 2 * 16
        fields = ["pred", "gt", "counts", "hd", "workspace"] + (["index"] if kw.get("source") == "ragged" else [])
        last = [r for r in relocs if r[0] == n_ops - 1]
        assert sorted(r[1] for r in last) == sorted(E.Op.u.offset + getattr(E.SegMetricsDesc, f).offset for f in fields)
        plain = {n.split(b"\0")[0].decode() for n, _, _, _, _ in _parse(pipe.export_plan(2, **kw))[4]}
        assert not plain & {"gt_mask", "seg_counts", "seg_hd"}


def _ellipse(H, W, cy, cx, ry, rx):
    y, x = np.mgrid[:H, :W]
    return (((y - cy) / ry) ** 2 + ((x - cx) / rx) ** 2 <= 1).astype(np.uint8) * 255


def test_ragged_metrics_program_matches_oracle(fake_engine):
    """A ragged source_frame=True, seg_metrics="source" program emulated whole in fp64 (shadow mode)."""
    shapes = [(300, 400), (224, 224), (57, 230)]
    src = _sources(shapes, 31)
    gts = [_ellipse(h, w, h / 2, w / 2, h / 3, w / 4) for h, w in shapes]
    gts[2][:] = 0                                                # empty ground truth
    pipe = lower.PipelineRunner(*_states(), "cpu", micro_batch=3)
    part = ragged.pack(src, 3, max_side=8 * S)
    ws = pipe.feed_ragged(part, source_frame=True, seg_metrics="source")
    gp = ragged.pack(gts, 1)
    ws["gt_mask"][:gp.n_px].copy_(gp.data)
    em = metrics_ref.SegMetricsProgramRef(list(ws["program"].keepalive) + [pipe.unet.w_blob, pipe.gnet.w_blob],
                                          "shadow", program_ref.weight_names(pipe.unet, pipe.gnet))
    for d in ws["program"].descs:
        em.op(d)
    kinds = {type(d) for d in ws["program"].descs}
    assert kinds <= (program_ref.COVERED_KINDS | ragged_ref.RAGGED_KINDS | cam_ref.CAM_KINDS
                     | source_ref.SOURCE_FRAME_KINDS | metrics_ref.SEG_METRICS_KINDS)
    assert isinstance(ws["program"].descs[-1], E.SegMetricsDesc)
    mask = em.mem.tensor(ws["src_mask"]).numpy().astype(np.uint8)
    counts = em.mem.tensor(ws["seg_counts"]).numpy()
    hd = em.mem.tensor(ws["seg_hd"]).numpy()
    for i, (H, W) in enumerate(shapes):
        off = int(part.table["px_offset"][i])
        c, h, h95 = metrics_ref.seg_metrics(mask[off:off + H * W].reshape(H, W), gts[i])
        assert tuple(counts[i]) == c and _same(hd[i, 0], h) and _same(hd[i, 1], h95), i
    assert counts[2][0] == counts[2][2] == 0


def test_interpreter_rejects_bad_entries():
    shapes = [(20, 30), (7, 1), (40, 40), (9, 9)]
    rng = np.random.default_rng(2)
    p = ragged.pack([(rng.random(s) < 0.5).astype(np.uint8) for s in shapes], 1)
    g = ragged.pack([(rng.random(s) < 0.5).astype(np.uint8) for s in shapes], 1)
    cap = p.n_px + 3
    table = p.table.copy()
    table[1]["px_offset"] = -1
    table[2]["W"] = 8 * S + 1
    table[3]["px_offset"] = cap - 2
    index = ragged.table_tensor(table)
    pred, gt = torch.zeros(cap, dtype=torch.uint8), torch.zeros(cap, dtype=torch.uint8)
    pred[:p.n_px], gt[:p.n_px] = p.data, g.data
    counts = torch.full((4, 3), 9, dtype=torch.int32)
    hd = torch.full((4, 2), 9.0, dtype=torch.float64)
    status = torch.full((4,), 9, dtype=torch.int32)
    work = torch.zeros(64, dtype=torch.uint8)
    d = E.SegMetricsDesc(pred.data_ptr(), gt.data_ptr(), index.data_ptr(), status.data_ptr(), counts.data_ptr(),
                         hd.data_ptr(), work.data_ptr(), 64, cap, 4, 0, 0)
    em = metrics_ref.SegMetricsProgramRef([pred, gt, index, counts, hd, status, work], "shadow")
    em.op(d)
    assert em.mem.tensor(status).tolist() == [0, 1, 1, 1]
    got_c, got_h = em.mem.tensor(counts).numpy(), em.mem.tensor(hd).numpy()
    assert (got_c[1:] == 0).all() and np.isnan(got_h[1:]).all()
    c, h, h95 = metrics_ref.seg_metrics(p.data[:600].numpy().reshape(20, 30), g.data[:600].numpy().reshape(20, 30))
    assert tuple(got_c[0]) == c and got_h[0, 0] == h and got_h[0, 1] == h95

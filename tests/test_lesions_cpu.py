"""CPU: connected components of a mask (oracle/lesions_ref.py, lesions.py, ug_lesions_desc,
PipelineRunner.plan(lesions=..., roi=...)).

* lesions_ref against a brute-force BFS flood fill on 200 random small masks for both connectivities, its numbering
  against scipy.ndimage.label, and its partition, areas, boxes and centroids against cv2.connectedComponentsWithStats
  after relabelling; central moments against cv2.moments of each component;
* lesions.derive against closed forms (axis-aligned rectangles, a rasterised ellipse) and lesions_ref.measurements;
* the C-ABI mirror: the ug_lesion layout, the descriptor's field list, sizeof(ug_op) unchanged, kind 21, symbols;
* lowering (stub engine): op order, the bbox of roi="largest" reading lesion_mask, plan keys and io, ValueError cases,
  default programs unchanged;
* uniform and ragged programs with lesions and roi="largest" emulated whole by LesionsProgramRef.
"""
import collections
import ctypes
import math
import re

import cv2
import numpy as np
import pytest
import torch
from scipy import ndimage

import ugnet_b200  # noqa: F401
from oracle import cam_ref, lesions_ref, metrics_ref, program_ref, ragged_ref, roi_ref, source_ref
from ugnet_b200 import engine as E
from ugnet_b200 import lesions as L
from ugnet_b200 import lower
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


def _bfs(mask, connectivity):
    """Labels by breadth-first flood fill in raster order of the seeds."""
    H, W = mask.shape
    lab = np.zeros((H, W), np.int32)
    nb = [(0, 1), (1, 0), (0, -1), (-1, 0)]
    if connectivity == 8:
        nb += [(1, 1), (1, -1), (-1, 1), (-1, -1)]
    n = 0
    for y in range(H):
        for x in range(W):
            if mask[y, x] and not lab[y, x]:
                n += 1
                lab[y, x] = n
                q = collections.deque([(y, x)])
                while q:
                    cy, cx = q.popleft()
                    for dy, dx in nb:
                        ny, nx = cy + dy, cx + dx
                        if 0 <= ny < H and 0 <= nx < W and mask[ny, nx] and not lab[ny, nx]:
                            lab[ny, nx] = n
                            q.append((ny, nx))
    return lab, n


def _random_masks(count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for k in range(count):
        H, W = (int(v) for v in rng.integers(1, 40, 2))
        out.append((rng.random((H, W)) < rng.uniform(0.05, 0.9)).astype(np.uint8) * (1, 255)[k % 2])
    return out


@pytest.mark.parametrize("conn", [4, 8])
def test_oracle_equals_flood_fill_and_scipy(conn):
    for m in _random_masks(200, 3 + conn):
        lab, n = lesions_ref.label(m, conn)
        want, wn = _bfs(m != 0, conn)
        assert n == wn and np.array_equal(lab, want)
        st = ndimage.generate_binary_structure(2, 1 if conn == 4 else 2)
        assert np.array_equal(lab, ndimage.label(m != 0, structure=st)[0])


@pytest.mark.parametrize("conn", [4, 8])
def test_oracle_table_against_cv2(conn):
    for m in _random_masks(200, 11 + conn):
        lab, n, rows, main = lesions_ref.table(m, conn, K=32)
        cn, clab, stats, cent = cv2.connectedComponentsWithStats((m != 0).astype(np.uint8), connectivity=conn,
                                                                 ltype=cv2.CV_32S)
        assert cn - 1 == n
        # same partition: a one-to-one map between the two labellings
        fg = lab > 0
        pairs = set(zip(lab[fg].tolist(), clab[fg].tolist()))
        assert len(pairs) == n and len({a for a, _ in pairs}) == n and len({b for _, b in pairs}) == n
        to_cv = dict(pairs)
        for r in rows[:min(n, 32)]:
            c = to_cv[int(r["label"])]
            x, y, w, h, a = stats[c]
            assert (r["area"], r["x0"], r["y0"], r["x1"], r["y1"]) == (a, x, y, x + w, y + h)
            A = int(r["area"])
            assert math.isclose(int(r["sx"]) / A, cent[c][0], rel_tol=1e-12, abs_tol=1e-12)
            assert math.isclose(int(r["sy"]) / A, cent[c][1], rel_tol=1e-12, abs_tol=1e-12)
            mo = cv2.moments((clab == c).astype(np.uint8), binaryImage=True)
            sh = L.derive(r[None])
            for ours, key in ((sh.mu20[0], "mu20"), (sh.mu02[0], "mu02"), (sh.mu11[0], "mu11")):
                assert math.isclose(ours, mo[key] / mo["m00"], rel_tol=1e-9, abs_tol=1e-9 * (1 + abs(mo["mu20"] /
                                    mo["m00"]) + abs(mo["mu02"] / mo["m00"]))), (key, ours, mo[key] / mo["m00"])
        # order: area descending, label ascending; main mask = row 0's component
        keys = [(-int(r["area"]), int(r["label"])) for r in rows[:min(n, 32)]]
        assert keys == sorted(keys) and (rows[min(n, 32):]["label"] == 0).all()
        assert np.array_equal(main, (lab == rows[0]["label"]).astype(np.uint8) if n else np.zeros_like(main))
        surf = metrics_ref.surface(m)
        for r in rows[:min(n, 32)]:
            assert r["boundary"] == int((surf & (lab == r["label"])).sum())


def test_derived_measurements_closed_forms():
    m = np.zeros((60, 80), np.uint8)
    m[10:20, 5:45] = 1                                 # 40 wide, 10 tall
    m[30:55, 60:65] = 1                                # 5 wide, 25 tall
    lab, n, rows, _ = lesions_ref.table(m, 8, K=4)
    sh = L.derive(rows)
    # a w x h rectangle of pixels: mu20 = (w^2 - 1) / 12, mu02 = (h^2 - 1) / 12, mu11 = 0
    assert sh.mu20[0] == (40 ** 2 - 1) / 12 and sh.mu02[0] == (10 ** 2 - 1) / 12 and sh.mu11[0] == 0
    assert sh.orientation[0] == 0.0 and sh.cx[0] == 24.5 and sh.cy[0] == 14.5
    assert math.isclose(sh.major_axis[0], 4 * math.sqrt((40 ** 2 - 1) / 12))
    assert math.isclose(sh.orientation[1], math.pi / 2) and math.isclose(sh.minor_axis[1], 4 * math.sqrt(2))
    assert math.isclose(sh.eccentricity[1], math.sqrt(1 - 2 / ((25 ** 2 - 1) / 12)))
    assert math.isclose(sh.equivalent_diameter[0], math.sqrt(4 * 400 / math.pi))
    assert np.isnan(sh.cx[2]) and np.isnan(sh.orientation[3])
    # a rasterised ellipse, semi-axes 60 and 25, turned by 0.5 rad: axes within a pixel, orientation within 0.01
    y, x = np.mgrid[:200, :200].astype(np.float64)
    t = 0.5
    u, v = (x - 100) * math.cos(t) + (y - 100) * math.sin(t), -(x - 100) * math.sin(t) + (y - 100) * math.cos(t)
    e = ((u / 60) ** 2 + (v / 25) ** 2 <= 1).astype(np.uint8)
    lab, n, rows, _ = lesions_ref.table(e, 8, K=1)
    sh = L.derive(rows)
    assert n == 1 and abs(sh.major_axis[0] - 120) < 1 and abs(sh.minor_axis[0] - 50) < 1
    assert abs(sh.orientation[0] - t) < 0.01 and abs(sh.eccentricity[0] - math.sqrt(1 - (25 / 60) ** 2)) < 0.01
    ref = lesions_ref.measurements(lab, 1)
    for k in L.Shape._fields:
        assert math.isclose(getattr(sh, k)[0], ref[k], rel_tol=1e-9, abs_tol=1e-9), k


def test_lesion_row_and_descriptor_mirror_the_header():
    assert ctypes.sizeof(E.Op) == OP_BYTES
    assert ctypes.sizeof(E.LesionsDesc) <= ctypes.sizeof(E._OpUnion) == ctypes.sizeof(E.ConvDesc)
    assert ctypes.sizeof(E.Lesion) == L.LESION_DTYPE.itemsize == 72
    assert [f for f, _ in E.Lesion._fields_] == list(L.LESION_DTYPE.names)
    assert all(getattr(E.Lesion, f).offset == L.LESION_DTYPE.fields[f][1] for f in L.LESION_DTYPE.names)
    assert E._DESC_KIND[E.LesionsDesc] == E.OP_LESIONS == 21 and E._SINGLE_ENTRY[21] == "ug_lesions"
    assert {"ug_lesions", "ug_lesions_workspace_bytes"} <= set(E.EXPORTED_SYMBOLS)
    src = open(f"{ROOT}/include/ugnet.h").read()
    for name, struct in (("ug_lesions_desc", E.LesionsDesc), ("ug_lesion", E.Lesion)):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), src, flags=re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        names = []
        for decl in body.split(";"):
            decl = decl.strip()
            if decl:
                names += [re.findall(r"\w+", part)[-1] for part in decl.split(",")]
        assert names == [f for f, _ in struct._fields_]
    assert ctypes.sizeof(E.LesionsDesc) == 104 and E.LesionsDesc.K.offset == 96
    assert re.search(r"UG_OP_LESIONS\s*=\s*21", src)
    assert re.search(r"int ug_lesions\(ug_handle h, const ug_lesions_desc\* d, void\* stream\);", src)
    assert re.search(r"size_t ug_lesions_workspace_bytes\(int B, long long capacity_px, int K\);", src)
    lib = E.load_library()
    assert lib.ug_lesions_workspace_bytes(4, 1000, 8) > 4000
    assert lib.ug_lesions_workspace_bytes(4, 1000, 0) == lib.ug_lesions_workspace_bytes(4, 1000, 33) == 0


KW = [{}, {"source": (300, 400)}, {"source": "ragged", "capacity": 70_000}]


def test_lesions_lowering(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    for kw in KW:
        base = pipe.plan(4, **kw)["program"].descs
        for lesions, roi in (("input", "all"), (None, "largest"), ("input", "largest")):
            ws = pipe.plan(4, lesions=lesions, roi=roi, **kw)
            descs = ws["program"].descs
            assert len(descs) == len(base) + 2                       # one op per micro-batch
            pos = [k for k, d in enumerate(descs) if isinstance(d, E.LesionsDesc)]
            bbox = [k for k, d in enumerate(descs) if isinstance(d, E.BBoxDesc)]
            assert [k + 1 for k in pos] == bbox                      # right after the UNet, right before the bbox
            for j, (k, b) in enumerate(zip(pos, bbox)):
                d = descs[k]
                sl = slice(2 * j, 2 * j + 2)
                assert d.mask == ws["mask"][sl].data_ptr() and d.main_mask == ws["lesion_mask"][sl].data_ptr()
                assert d.labels == ws["lesion_labels"][sl].data_ptr() and d.lesions == ws["lesions"][sl].data_ptr()
                assert d.count == ws["lesion_count"][sl].data_ptr() and not d.index and not d.status
                assert (d.B, d.Hs, d.Ws, d.connectivity, d.K) == (2, S, S, 8, 8)
                want = ws["lesion_mask"] if roi == "largest" else ws["mask"]
                assert descs[b].mask == want[sl].data_ptr()
            assert ws["lesions"].shape == (4, 8, 9) and ws["lesion_labels"].dtype == torch.int32
            rest = [d for d in descs if not isinstance(d, E.LesionsDesc)]
            if roi == "all":
                assert _normalised(rest) == _normalised(base)
            assert pipe.plan(4, lesions=lesions, roi=roi, **kw) is ws
        if kw:
            sf = pipe.plan(4, source_frame=True, **kw)["program"].descs
            ws = pipe.plan(4, source_frame=True, lesions="source", **kw)
            descs = ws["program"].descs
            assert len(descs) == len(sf) + 1 and isinstance(descs[-1], E.LesionsDesc)
            assert _normalised(descs[:-1]) == _normalised(sf)
            d = descs[-1]
            assert d.mask == ws["src_mask"].data_ptr() and d.labels == ws["src_lesion_labels"].data_ptr()
            assert ws["src_lesion_labels"].shape == ws["src_mask"].shape
            if kw["source"] == "ragged":
                assert d.index == ws["src_index"].data_ptr() and d.capacity_px == ws["src_mask"].numel()
            else:
                assert not d.index and (d.Hs, d.Ws) == kw["source"]
    with pytest.raises(ValueError):
        pipe.plan(2, source=(300, 400), lesions="source")            # needs source_frame=True
    with pytest.raises(ValueError):
        pipe.plan(2, lesions="both")
    with pytest.raises(ValueError):
        pipe.plan(2, roi="biggest")
    with pytest.raises(ValueError):
        pipe(torch.zeros((2, 3, S, S)), lesions="source")
    with pytest.raises(ValueError):
        L.check_args(6, 8)
    with pytest.raises(ValueError):
        L.check_args(8, 33)


@pytest.mark.parametrize("kw", KW)
def test_default_programs_are_unchanged_by_lesion_plans(fake_engine, kw):
    a = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    b = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    want = _normalised(a.plan(2, **kw)["program"].descs)
    b.plan(2, lesions="input", roi="largest", **kw)
    if kw:
        b.plan(2, source_frame=True, lesions="source", **kw)
    assert _normalised(b.plan(2, **kw)["program"].descs) == want


def test_plan_image_lists_the_lesion_io(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=1)
    image = pipe.export_plan(2, source="ragged", capacity=70_000, source_frame=True, lesions="source", roi="largest")
    _, _, n_ops, relocs, ios, op_bytes = _parse(image)
    assert op_bytes == OP_BYTES
    sizes = {n.split(b"\0")[0].decode(): b for n, _, _, _, b in ios}
    cap = ragged.capacity(70_000)
    assert sizes["lesion_labels"] == 2 * S * S * 4 and sizes["lesion_mask"] == 2 * S * S
    assert sizes["lesion_count"] == 8 and sizes["lesions"] == 2 * 8 * 72
    assert sizes["src_lesion_labels"] == cap * 4 and sizes["src_lesion_mask"] == cap
    assert sizes["src_lesion_count"] == 8 and sizes["src_lesions"] == 2 * 8 * 72
    last = [r for r in relocs if r[0] == n_ops - 1]
    fields = ["mask", "index", "labels", "main_mask", "lesions", "count", "workspace"]
    assert sorted(r[1] for r in last) == sorted(E.Op.u.offset + getattr(E.LesionsDesc, f).offset for f in fields)
    plain = {n.split(b"\0")[0].decode() for n, _, _, _, _ in _parse(pipe.export_plan(2))[4]}
    assert not any("lesion" in n for n in plain)


def _blobs(H, W, seed):
    """Three disjoint blobs of different sizes, the largest away from the image's centre."""
    m = np.zeros((H, W), np.uint8)
    m[5:25, 8:40] = 255
    m[H - 12:H - 4, W - 15:W - 6] = 255
    m[H // 2, W // 2] = 255
    return m


@pytest.mark.parametrize("kw", [{}, {"source": "ragged", "capacity": 70_000}])
def test_largest_roi_program_matches_oracle(fake_engine, kw):
    """A roi="largest" program (with lesions="source" for the ragged one) emulated whole in fp64 (shadow mode): the
    lesion table, the main mask and the bbox of the main mask of the emulated UNet mask."""
    pipe = lower.PipelineRunner(*_states(), "cpu", micro_batch=2)
    if kw:
        shapes = [(300, 400), (57, 230)]
        part = ragged.pack(_sources(shapes, 5), 3, max_side=8 * S)
        ws = pipe.feed_ragged(part, source_frame=True, lesions="source", roi="largest")
    else:
        ws = pipe.plan(2, roi="largest", lesions="input")
        ws["x_in"].copy_(torch.from_numpy(np.random.default_rng(4).random((2, 3, S, S)).astype(np.float32)))
    em = lesions_ref.LesionsProgramRef(list(ws["program"].keepalive) + [pipe.unet.w_blob, pipe.gnet.w_blob],
                                       "shadow", program_ref.weight_names(pipe.unet, pipe.gnet))
    for d in ws["program"].descs:
        em.op(d)
    kinds = {type(d) for d in ws["program"].descs}
    assert kinds <= (program_ref.COVERED_KINDS | ragged_ref.RAGGED_KINDS | cam_ref.CAM_KINDS
                     | source_ref.SOURCE_FRAME_KINDS | metrics_ref.SEG_METRICS_KINDS | lesions_ref.LESIONS_KINDS)
    mask = em.mem.tensor(ws["mask"]).numpy().astype(np.uint8)
    main = em.mem.tensor(ws["lesion_mask"]).numpy().astype(np.uint8)
    boxes = em.mem.tensor(ws["boxes"]).numpy()
    table = em.mem.tensor(ws["lesions"]).numpy().astype(np.int64)
    for i in range(2):
        lab, n, rows, want_main = lesions_ref.table(mask[i], 8, 8)
        assert np.array_equal(main[i], want_main)
        assert np.array_equal(table[i], rows.view(np.int64).reshape(8, 9))
        assert tuple(boxes[i]) == roi_ref.bbox_from_mask(want_main)
        assert int(em.mem.tensor(ws["lesion_count"])[i]) == n
    if kw:
        sm = em.mem.tensor(ws["src_mask"]).numpy().astype(np.uint8)
        cnt = em.mem.tensor(ws["src_lesion_count"]).numpy()
        for i, (H, W) in enumerate(shapes):
            off = int(part.table["px_offset"][i])
            lab, n, rows, _ = lesions_ref.table(sm[off:off + H * W].reshape(H, W), 8, 8)
            assert cnt[i] == n


def test_interpreter_rejects_bad_entries():
    shapes = [(20, 30), (7, 1), (40, 40), (9, 9)]
    rng = np.random.default_rng(2)
    p = ragged.pack([(rng.random(s) < 0.5).astype(np.uint8) for s in shapes], 1)
    cap = p.n_px + 3
    table = p.table.copy()
    table[1]["px_offset"] = -1
    table[2]["W"] = 8 * S + 1
    table[3]["px_offset"] = cap - 2
    index = ragged.table_tensor(table)
    mask = torch.zeros(cap, dtype=torch.uint8)
    mask[:p.n_px] = p.data
    labels = torch.full((cap,), -7, dtype=torch.int32)
    main = torch.full((cap,), 7, dtype=torch.uint8)
    rows = torch.full((4, 8, 9), 9, dtype=torch.int64)
    count = torch.full((4,), 9, dtype=torch.int32)
    status = torch.full((4,), 9, dtype=torch.int32)
    work = torch.zeros(64, dtype=torch.uint8)
    d = E.LesionsDesc(mask.data_ptr(), index.data_ptr(), status.data_ptr(), labels.data_ptr(), main.data_ptr(),
                      rows.data_ptr(), count.data_ptr(), work.data_ptr(), 64, cap, 4, 0, 0, 4, 8)
    em = lesions_ref.LesionsProgramRef([mask, index, labels, main, rows, count, status, work], "shadow")
    em.op(d)
    assert em.mem.tensor(status).tolist() == [0, 1, 1, 1]
    assert em.mem.tensor(count).tolist()[1:] == [0, 0, 0]
    assert (em.mem.tensor(rows)[1:] == 0).all()
    lab, n, r, m = lesions_ref.table(p.data[:600].numpy().reshape(20, 30), 4, 8)
    assert np.array_equal(em.mem.tensor(labels)[:600].numpy().reshape(20, 30), lab)
    assert (em.mem.tensor(labels)[600:] == -7).all()                # nothing written through rejected entries

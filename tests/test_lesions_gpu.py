"""GPU: connected components of a mask (ug_lesions, programs built with lesions=... / roi="largest",
PipelineRunner / TwoStagePipeline(..., lesions=..., roi=...), lesions.label, infer.grade_images(..., lesions=...)).

* ug_lesions alone on ragged batches of edge cases (empty, full frame, 1x1, 1x1792, 1792x1, 1792x1792, checkerboards,
  diagonals, a spiral, a serpentine, concentric rings, blobs straddling every tile border, noise at densities 0.1, 0.5
  and 0.6, more components than rows and ties in area), packed with gaps under poisoned guard bands, for connectivity
  4 and 8 and K = 1, 8 and 32: labels, count, rows and main mask equal oracle/lesions_ref exactly; bad table entries
  rejected without a read or write; gaps and guards untouched; two runs bit-identical;
* a uniform batch through lesions.label; descriptors with a bad connectivity or K rejected, nothing written;
* the pipeline: 70 mixed-size images with lesions="source" against the oracle on the call's own src_mask; a 256-image
  batch with lesions="input" bit-identical to the default; roi="largest" boxes and crops against roi_ref on the
  oracle's main mask of the engine's own mask, and bit-identical to the default where a mask has at most one
  component;
* an op-by-op replay of a roi="largest" program, its plan image through the C ABI against the Python call, and
  grade_images' lesions.csv.
"""
import csv

import numpy as np
import pytest
import torch

from guard import guarded

pytestmark = pytest.mark.gpu
S = 224


@pytest.fixture(scope="module")
def trained():
    from oracle import fixtures
    return fixtures.trained_unet_state(device="cuda"), fixtures.trained_googlenet_state(device="cuda")


def _spiral(n, pitch=4):
    """Archimedean spiral bands of width pitch / 2: long winding components."""
    y, x = np.mgrid[:n, :n] - (n - 1) / 2
    t = (np.hypot(y, x) - pitch * np.arctan2(y, x) / (2 * np.pi)) % pitch
    return (t < pitch / 2).astype(np.uint8)


def _cases(rng):
    """Edge-case masks (0/1 or 0/255)."""
    yy, xx = np.mgrid[:300, :300]
    out = [np.zeros((40, 50), np.uint8), np.ones((64, 70), np.uint8) * 255, np.ones((1, 1), np.uint8),
           np.zeros((1, 1), np.uint8), (rng.random((1, 1792)) < 0.5).astype(np.uint8),
           (rng.random((1792, 1)) < 0.5).astype(np.uint8), ((yy + xx) % 2).astype(np.uint8),
           (((yy - xx) % 5) == 0).astype(np.uint8), (((yy + xx) % 7) == 0).astype(np.uint8) * 255, _spiral(257)]
    ser = np.zeros((250, 250), np.uint8)                               # a serpentine: rows joined at alternate ends
    ser[::2] = 1
    ser[1::4, -1] = 1
    ser[3::4, 0] = 1
    out.append(ser)
    r = np.hypot(yy - 150.0, xx - 140.0)
    out.append(((r.astype(int) % 6) < 2).astype(np.uint8))          # concentric rings
    tiles = np.zeros((130, 200), np.uint8)                           # blobs across every tile border and corner
    for ty in range(31, 130, 32):
        for tx in range(31, 200, 32):
            tiles[ty - 1:ty + 2, tx - 1:tx + 2] = 1
            tiles[ty + 2, tx + 2] = 1                                  # a diagonal link (8-connected only)
    out.append(tiles)
    for p in (0.1, 0.5, 0.6):
        out.append((rng.random((480, 333)) < p).astype(np.uint8))
    ties = np.zeros((60, 90), np.uint8)                              # 12 components of area 4, then 3 of area 9
    for k in range(12):
        ties[2 + 4 * (k // 6):4 + 4 * (k // 6), 3 + 10 * (k % 6):5 + 10 * (k % 6)] = 1
    for k in range(3):
        ties[30:33, 5 + 20 * k:8 + 20 * k] = 1
    out.append(ties)
    out.append((rng.random((1792, 1792)) < 0.55).astype(np.uint8))
    out += [(rng.random(tuple(int(v) for v in rng.integers(1, 400, 2))) < rng.uniform(0.05, 0.7)).astype(np.uint8)
            for _ in range(8)]
    return out


def _run(engine, masks, conn, K, rng, rejected=()):
    from oracle import lesions_ref
    from ugnet_b200 import engine as E
    from ugnet_b200.util import ragged
    B = len(masks)
    table = np.zeros(B, ragged.ENTRY)
    off = 0
    for i, m in enumerate(masks):                                   # packed with gaps of 0..6 pixels
        off += int(rng.integers(0, 7))
        table[i] = (off, m.shape[0], m.shape[1])
        off += m.size
    cap = off + 5
    host = np.full(cap, 3, np.uint8)                                # gaps hold foreground values
    for (o, H, W), m in zip(table, masks):
        host[o:o + H * W] = m.reshape(-1)
    bad = table.copy()
    for i, how in zip(rejected, ("neg", "side", "cap")):
        if how == "neg":
            bad[i]["px_offset"] = -3
        elif how == "side":
            bad[i]["W"] = 8 * S + 1
        else:
            bad[i]["px_offset"] = cap - 2
    index = ragged.table_tensor(bad, "cuda")
    mask, m_ok = guarded((cap,), 5, torch.uint8)
    mask.copy_(torch.from_numpy(host))
    labels, l_ok = guarded((cap,), -9, torch.int32)
    main, mm_ok = guarded((cap,), 7, torch.uint8)
    rows, r_ok = guarded((B, K, 9), -9, torch.int64)
    count, c_ok = guarded((B,), -9, torch.int32)
    status, s_ok = guarded((B,), 9, torch.int32)
    nbytes = E.load_library().ug_lesions_workspace_bytes(B, cap, K)
    work, w_ok = guarded((nbytes,), 0xA5, torch.uint8)
    d = E.LesionsDesc(mask.data_ptr(), index.data_ptr(), status.data_ptr(), labels.data_ptr(), main.data_ptr(),
                      rows.data_ptr(), count.data_ptr(), work.data_ptr(), nbytes, cap, B, 0, 0, conn, K)
    ref = lesions_ref.LesionsProgramRef([mask, index, labels, main, rows, count, status, work], "real")
    outs = ref.op(d)
    engine.run_op(d)
    torch.cuda.synchronize()
    for o in outs:
        assert o.ratio(ref.mem.read(o.region, o.idx)) <= 1.0, (o.name, conn, K)
    for ok in (m_ok, l_ok, mm_ok, r_ok, c_ok, s_ok, w_ok):
        ok()
    assert status.tolist() == [1 if i in rejected else 0 for i in range(B)]
    assert torch.equal(mask.cpu(), torch.from_numpy(host))
    # untouched gaps between images and nothing written through rejected entries
    written = np.zeros(cap, bool)
    for i, (o, H, W) in enumerate(table):
        if i not in rejected:
            written[o:o + H * W] = True
    lab_h = labels.cpu().numpy()
    assert (lab_h[~written] == -9).all() and (main.cpu().numpy()[~written] == 7).all()
    assert not count[list(rejected)].any() and not rows[list(rejected)].any()
    first = (labels.clone(), main.clone(), rows.clone(), count.clone())
    engine.run_op(d)
    torch.cuda.synchronize()
    for a, b in zip(first, (labels, main, rows, count)):
        assert torch.equal(a, b)
    return d


@pytest.mark.parametrize("conn,K", [(8, 8), (4, 8), (8, 1), (4, 32)])
def test_lesions_op_edge_cases_under_guards(engine, conn, K):
    rng = np.random.default_rng(31 + conn + K)
    masks = _cases(rng)
    d = _run(engine, masks, conn, K, rng, rejected=(3, 7, 12))
    if conn == 8 and K == 8:
        from ugnet_b200 import engine as E
        for field, val in (("connectivity", 6), ("connectivity", 0), ("K", 0), ("K", 33)):
            bad = E.LesionsDesc.from_buffer_copy(d)
            setattr(bad, field, val)
            with pytest.raises(RuntimeError):
                engine.run_op(bad)
        small = E.LesionsDesc.from_buffer_copy(d)
        small.workspace_bytes = d.workspace_bytes - 1
        with pytest.raises(RuntimeError):
            engine.run_op(small)


def test_bad_descriptor_writes_nothing(engine):
    from ugnet_b200 import lesions as L
    m = torch.ones((2, 30, 40), dtype=torch.uint8, device="cuda")
    labels, main, count, rows = L.outputs(2, m, 8, "cuda")
    for t in (labels, main, count, rows):
        t.fill_(3)
    ws = L.workspace(2, m.numel(), 8, "cuda")
    for conn, K in ((6, 8), (8, 0), (8, 33)):
        d = L.lesions_desc(m, labels, main, rows, count, ws, 2, conn, K, Hs=30, Ws=40)
        with pytest.raises(RuntimeError):
            engine.run_op(d)
        torch.cuda.synchronize()
        for t in (labels, main, count, rows):
            assert bool((t == 3).all())


def test_label_uniform_and_list(engine):
    from oracle import lesions_ref
    from ugnet_b200 import lesions as L
    rng = np.random.default_rng(5)
    m = (rng.random((6, 224, 224)) < 0.5).astype(np.uint8) * 255
    res = L.label(torch.from_numpy(m).cuda(), connectivity=4, top_k=5)
    for i in range(6):
        lab, n, rows, main = lesions_ref.table(m[i], 4, 5)
        assert int(res.count[i]) == n and np.array_equal(res.labels[i].cpu().numpy(), lab)
        assert np.array_equal(res.main_masks[i].cpu().numpy(), main) and np.array_equal(res.table[i], rows)
    sh = L.derive(res.table)
    assert np.array_equal(np.nan_to_num(sh.major_axis), np.nan_to_num(res.derived.major_axis))
    lst = [m[0][:100, :37], m[1][:1, :1], m[2]]
    res = L.label(lst)
    for i, x in enumerate(lst):
        lab, n, rows, main = lesions_ref.table(x, 8, 8)
        assert int(res.count[i]) == n and np.array_equal(res.labels[i].cpu().numpy(), lab)
        assert np.array_equal(res.table[i], rows)


def _procedural():
    from oracle import fixtures
    return (fixtures.procedural_state(fixtures.unet_template(), seed=7),
            fixtures.procedural_state(fixtures.googlenet_template(), seed=11))


def test_pipeline_source_lesions_mixed_sizes(engine):
    from oracle import lesions_ref
    from ugnet_b200.pipeline import TwoStagePipeline
    from test_ragged_gpu import _rgb_sources
    pipe = TwoStagePipeline(*_procedural(), micro_batch=32, cls_batch=64)
    imgs = _rgb_sources(70, seed=43, lo=2, hi=1200)
    out = pipe(imgs, return_source=True, lesions="source")
    base = pipe(imgs, return_source=True)
    for got, want in zip(out[:3], base[:3]):
        assert torch.equal(got, want)
    les = out[4]
    multi = 0
    for i, sm in enumerate(out[3].masks):
        lab, n, rows, main = lesions_ref.table(sm.cpu().numpy(), 8, 8)
        assert int(les.count[i]) == n and np.array_equal(les.labels[i].cpu().numpy(), lab), i
        assert np.array_equal(les.main_masks[i].cpu().numpy(), main) and np.array_equal(les.table[i], rows), i
        multi += n > 1
    print(f"\n  70 mixed sizes: {multi} source masks with more than one component")
    assert multi > 0


def test_pipeline_input_lesions_and_largest_roi(engine):
    from oracle import lesions_ref, roi_ref
    from ugnet_b200.lower import PipelineRunner
    rng = np.random.default_rng(8)
    x = torch.from_numpy(rng.random((256, 3, S, S)).astype(np.float32)).cuda()
    pipe = PipelineRunner(*_procedural(), "cuda:0", micro_batch=64, cls_batch=256)
    m, b, c, lg = pipe(x, return_logits=True)
    u8 = pipe.plan(256)["u8"].clone()
    m2, b2, c2, lg2, les = pipe(x, return_logits=True, lesions="input")
    assert torch.equal(m, m2) and torch.equal(b, b2) and torch.equal(c, c2) and torch.equal(lg, lg2)
    assert torch.equal(pipe.plan(256, lesions="input")["u8"], u8)
    m3, b3, c3, lg3, les3 = pipe(x, return_logits=True, lesions="input", roi="largest")
    assert torch.equal(m, m3) and torch.equal(lg, lg3)
    assert torch.equal(les.labels, les3.labels) and np.array_equal(les.table, les3.table)
    u8l = pipe.plan(256, lesions="input", roi="largest")["u8"].cpu().numpy()
    mh, xh = m.cpu().numpy(), x.cpu().numpy()
    single, n_multi = [], 0
    for i in range(256):
        lab, n, rows, main = lesions_ref.table(mh[i], 8, 8)
        assert np.array_equal(les.labels[i].cpu().numpy(), lab) and np.array_equal(les.table[i], rows)
        box = roi_ref.bbox_from_mask(main)
        assert tuple(b3[i].tolist()) == box, i
        crop = roi_ref.roi_crop_resize_u8(xh[i], box)
        assert np.array_equal(u8l[i], crop), i
        if n <= 1:
            single.append(i)
        n_multi += n > 1
    print(f"\n  256 noise inputs: {n_multi} masks with more than one component")
    assert n_multi > 0 and single
    s = torch.tensor(single, device="cuda")
    assert torch.equal(b3[s], b[s]) and torch.equal(c3[s], c[s])


def test_replay_plan_image_and_grade_images(engine, monkeypatch, tmp_path):
    import test_program_replay_gpu as replay
    from oracle import lesions_ref
    from ugnet_b200 import engine as E
    from ugnet_b200 import lesions as L
    from ugnet_b200.infer import grade_images
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged
    from test_ragged_gpu import _gray_images, _rgb_sources
    monkeypatch.setattr(replay, "_interpreter", lesions_ref.interpreter)
    monkeypatch.setitem(replay._INT, torch.int64, torch.int64)
    pipe = PipelineRunner(*_procedural(), "cuda:0", micro_batch=4, cls_batch=8)
    imgs = _rgb_sources(8, seed=47, lo=30, hi=900)
    part = ragged.pack(imgs, 3, max_side=8 * S)
    ws = pipe.feed_ragged(part, source_frame=True, lesions="source", roi="largest")
    assert isinstance(ws["program"].descs[-1], E.LesionsDesc)
    replay._replay(engine, ws["program"], [pipe.unet, pipe.gnet])
    ws["program"].run()
    torch.cuda.synchronize()
    want = {k: ws[k].clone() for k in ("boxes", "cls_logits", "lesions", "lesion_count", "src_lesions",
                                       "src_lesion_count", "src_boxes")}
    plan = E.Plan(engine, pipe.export_plan(8, source="ragged", capacity=part.n_px, source_frame=True,
                                           lesions="source", roi="largest"))
    assert {"lesions", "lesion_mask", "src_lesions", "src_lesion_labels"} <= set(plan.names)
    cap = ragged.capacity(part.n_px)
    src_u8 = torch.zeros(3 * cap, dtype=torch.uint8)
    src_u8[:part.data.numel()] = part.data.cpu()
    plan.copy_in("src_u8", src_u8)
    plan.copy_in("src_index", ragged.table_tensor(part.table))
    plan.run()
    for k, v in want.items():
        got = plan.copy_out(k, torch.empty(v.shape, dtype=v.dtype))
        assert torch.equal(got, v.cpu()), k
    plan.close()
    out = pipe(imgs, lesions="source", roi="largest")               # the Python call
    assert torch.equal(out[1], want["boxes"]) and np.array_equal(out[-1].table, L.rows(want["src_lesions"]))
    # grade_images: lesions.csv against lesions.label of the source-frame masks; result.txt unchanged with roi="all"
    sizes = [(300, 400), (224, 224), (181, 97), (57, 230), (512, 512), (2, 9), (640, 480)]
    grays = _gray_images(sizes, 5)
    names = [f"{n}.png" for n in (10, 2, 33, 4, 5, 61, 7)]
    grade_images(pipe, grays, names, save_dir=str(tmp_path / "a"))
    grade_images(pipe, grays, names, save_dir=str(tmp_path / "b"), roi="all", lesions="source")
    assert (tmp_path / "a" / "result.txt").read_bytes() == (tmp_path / "b" / "result.txt").read_bytes()
    from ugnet_b200.util.wavelet import wavelet_enhance_batch
    rgb = [wavelet_enhance_batch(torch.from_numpy(g).cuda()[None])[0] for g in grays]
    masks = pipe(rgb, return_source=True)[-1].masks
    ref = L.label(masks)
    with open(tmp_path / "b" / "lesions.csv") as f:
        got = list(csv.DictReader(f))
    want_rows = []
    for i, n in enumerate(names):
        for k in range(8):
            t = ref.table[i, k]
            if t["label"]:
                want_rows.append((int(n[:-4]), k, int(ref.count[i]), int(t["label"]), int(t["area"]),
                                  float(ref.derived.orientation[i, k])))
    want_rows.sort()
    assert [(int(r["name"]), int(r["rank"]), int(r["count"]), int(r["label"]), int(r["area"]),
             float(r["orientation"])) for r in got] == want_rows
    grade_images(pipe, grays, names, save_dir=str(tmp_path / "c"), roi="largest")
    assert (tmp_path / "c" / "result.txt").exists()

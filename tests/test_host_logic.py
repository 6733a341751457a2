"""CPU: the Python boundary mirrors the reference's surface (names, hparams, state_dict keys,
padding rules, error behaviour) and the sharding helpers work under gloo with world_size 2."""
import json
import os
from argparse import Namespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import GOLDEN
from oracle import raft_oracle as O


def test_registry_and_get_model():
    import ptlflow_b200 as pb

    assert {"raft", "raft_small"} <= set(pb.get_model_names())
    assert pb.get_model_reference("raft").__name__ == "raft"
    with pytest.raises(ValueError):
        pb.get_model_reference("not_a_model")
    m = pb.get_model("raft", args=Namespace(model=Namespace(iters=12, corr_radius=3, alternate_corr=True)))
    assert (m.iters, m.corr_radius, m.alternate_corr, m.output_stride) == (12, 3, True, 8)
    assert m.hparams.iters == 12 and m.hparams.corr_radius == 3 and not hasattr(m.hparams, "loss_fn")
    assert m.update_block.encoder.convc1.weight.shape == (256, 4 * 49, 1, 1)
    m2 = pb.get_model("raft_small", args={"model": {"init_args": {"iters": 4}}})
    assert m2.iters == 4 and m2.hidden_dim == 96


@pytest.mark.parametrize("variant", ["raft", "raft_small", "gma"])
def test_state_dict_keys_equal_reference(variant):
    import ptlflow_b200 as pb

    with open(os.path.join(GOLDEN, f"state_shapes_{variant}.json")) as f:
        ref = {k: tuple(v) for k, v in json.load(f).items()}
    mine = {k: tuple(v.shape) for k, v in pb.get_model(variant).state_dict().items()}
    assert mine == ref


def test_checkpoint_roundtrip(tmp_path):
    import ptlflow_b200 as pb

    m = pb.get_model("raft_small")
    path = tmp_path / "m.ckpt"
    torch.save({"state_dict": m.state_dict(), "hyper_parameters": {"train_size": [368, 496], "extra_params": {"a": 1}}}, path)
    m2 = pb.get_model("raft_small", ckpt_path=str(path))
    assert m2.train_size == [368, 496] and m2.extra_params == {"a": 1}
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)
    with pytest.raises(ValueError):
        pb.get_model("raft_small", ckpt_path="not_a_checkpoint_name")


@pytest.mark.parametrize("h,w", [(436, 1024), (128, 256), (132, 164), (1080, 1920), (37, 41)])
def test_padding_rule(h, w):
    from ptlflow_b200.utils.utils import InputPadder

    x = torch.arange(2 * 2 * 3 * h * w, dtype=torch.float32).reshape(2, 2, 3, h, w)
    p = InputPadder(x.shape, stride=8)
    l, r, t, b = O.pad_amounts(h, w)
    assert p._pad == [l, r, t, b] and p.pad_top_left == (t, l)
    y = p.fill(x)
    assert y.shape[-2] % 8 == 0 and y.shape[-1] % 8 == 0
    ref, _ = O.preprocess(x / x.max())
    assert y.shape == ref.shape
    assert torch.equal(p.unfill(y), x)
    if (l, r, t, b) != (0, 0, 0, 0):
        assert p.unfill(x) is x  # already un-padded tensors pass through (utils.py:87-90)


def test_preprocess_matches_oracle_and_keeps_input():
    import ptlflow_b200 as pb

    m = pb.get_model("raft")
    img = torch.rand(1, 2, 3, 37, 50)
    keep = img.clone()
    x, resizer = m.preprocess_images(img, bgr_add=-0.5, bgr_mult=2.0, bgr_to_rgb=True, resize_mode="pad", pad_mode="replicate", pad_two_side=True)
    ref, pads = O.preprocess(img)
    assert torch.equal(img, keep)
    assert torch.allclose(x, ref, atol=0, rtol=0)


def test_no_cpu_fallback():
    import ptlflow_b200 as pb
    from ptlflow_b200 import ops

    m = pb.get_model("raft_small").eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m({"images": torch.rand(1, 2, 3, 64, 64)})
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.corr_volume_build(torch.zeros(1, 8, 8, 16), torch.zeros(1, 8, 8, 16), 1)
    with pytest.raises(RuntimeError):
        m.update_block(None, None, None, None)  # parameter container, not a PyTorch implementation


def test_shard_range_tiles_exactly():
    from ptlflow_b200.sharding import shard_range

    for n in (0, 1, 7, 8, 9, 32, 1041):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(4, 2, 2)


def _gloo_worker(rank, world, port, out):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    from ptlflow_b200 import sharding

    assert sharding.init_process_group("gloo")
    lo, hi = sharding.shard_range(9, rank, world)
    sharding.barrier()
    slowest = sharding.max_over_ranks(10.0 + rank)
    total = sharding.sum_over_ranks(hi - lo)
    out.put((rank, lo, hi, slowest, total))
    dist.destroy_process_group()


def test_gloo_world_size_2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 300
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert [(r[1], r[2]) for r in res] == [(0, 5), (5, 9)]
    assert all(r[3] == 11.0 and r[4] == 9.0 for r in res)


def test_first_conv_pack_layout_matches_header():
    """ops.pack_first_conv == the layout include/ptlflow_b200.h documents for pfb_first_conv7x7s2 (built element by element here)."""
    from ptlflow_b200 import ops

    w = torch.arange(64 * 3 * 7 * 7, dtype=torch.float32).reshape(64, 3, 7, 7) / 1000.0
    pk = ops.pack_first_conv(w, torch.float32)  # [9][16 row groups][4 K groups][8 rows][8 elements]
    assert pk.shape == (9, 16, 4, 8, 8) and pk.is_contiguous()
    for j, p, co, t, c in [(0, 0, 5, 1, 0), (2, 1, 63, 7, 2), (8, 1, 0, 4, 1), (6, 0, 17, 3, 2), (3, 1, 9, 1, 0)]:
        row, col = p * 64 + co, 4 * t + c
        ky, kx = j - 2 * p, t - 1
        assert pk[j, row // 8, col // 8, row % 8, col % 8].item() == pytest.approx(w[co, c, ky, kx].item())
    # zero where the filter row / column falls outside 0..6, for the dummy window pixel t = 0 and the pad channel c = 3
    dense = pk.permute(0, 1, 3, 2, 4).reshape(9, 128, 32)
    assert not dense[0, 64:].any() and not dense[1, 64:].any()  # phase 1 sees input-row offsets 2..8 only
    assert not dense[7, :64].any() and not dense[8, :64].any()  # phase 0 sees 0..6 only
    assert not dense[:, :, 0:4].any() and not dense[:, :, 3::4].any()


def test_flow_conv_pack_layout_matches_header():
    from ptlflow_b200 import ops

    w = torch.arange(128 * 2 * 7 * 7, dtype=torch.float32).reshape(128, 2, 7, 7) / 1000.0
    pk = ops.pack_flow_conv(w, torch.float32)  # [7][16][8][8][8]
    assert pk.shape == (7, 16, 8, 8, 8)
    dense = pk.permute(0, 1, 3, 2, 4).reshape(7, 128, 64)
    for ky, co, t, c in [(0, 0, 1, 0), (6, 127, 7, 3), (3, 64, 4, 2), (2, 9, 2, 1)]:
        assert dense[ky, co, 8 * t + c].item() == pytest.approx(w[co, c & 1, ky, t - 1].item())  # hi and lo halves share the weight
    assert not dense[:, :, 0:8].any()  # window pixel t = 0 lies left of the 7 taps
    assert not dense.reshape(7, 128, 8, 8)[..., 4:].any()  # channels 4..7 of the 16-byte pixel are padding


def test_pipeline_rejects_cpu_models_and_bad_depth():
    import ptlflow_b200 as pb
    from ptlflow_b200.pipeline import FramePipeline

    m = pb.get_model("raft_small").eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        FramePipeline(m, depth=2)
    with pytest.raises(ValueError):
        FramePipeline(m, depth=0)


def test_cudnn_flags_first_in_last_out():
    """Nested / concurrent forwards must not switch cuDNN's benchmark mode off under each other (models/raft/raft.py)."""
    from ptlflow_b200.models.raft.raft import _cudnn_flags

    cd = torch.backends.cudnn
    before = (cd.enabled, cd.benchmark, cd.allow_tf32)
    with _cudnn_flags(True, False):
        assert cd.benchmark is True and cd.allow_tf32 is False
        with _cudnn_flags(False, True):  # a second forward in flight: the first one's settings stay
            assert cd.benchmark is True and cd.allow_tf32 is False
        assert cd.benchmark is True  # ... also after the inner one has left
    assert (cd.enabled, cd.benchmark, cd.allow_tf32) == before


def test_flow_io_round_trips_and_conventions(tmp_path):
    from ptlflow_b200.utils.flow_utils import AsyncFlowWriter, flow_read, flow_write

    rng = np.random.default_rng(3)
    flow = (rng.standard_normal((17, 23, 2)) * 20).astype(np.float32)
    flow[2, 3] = np.nan  # invalid pixel
    # .flo: exact, NaN <-> Middlebury sentinel
    p = tmp_path / "a.flo"
    flow_write(p, flow)
    raw = p.read_bytes()
    assert raw[:4] == b"PIEH" and np.frombuffer(raw[4:12], dtype="<u4").tolist() == [23, 17] and len(raw) == 12 + 17 * 23 * 8
    back = flow_read(p)
    assert np.array_equal(np.isnan(back), np.isnan(flow)) and np.array_equal(back[~np.isnan(back)], flow[~np.isnan(flow)])
    assert np.frombuffer(raw[12:], dtype="<f4").reshape(17, 23, 2)[2, 3, 0] == np.float32(1666666800.0)
    # KITTI png: 1/64 px quantisation, validity channel
    q = tmp_path / "a.png"
    flow_write(q, flow)
    back = flow_read(q)
    assert np.isnan(back[2, 3]).all() and np.nanmax(np.abs(back - flow)) <= 1.0 / 64 + 1e-6
    flow_write(tmp_path / "a.npy", flow)
    assert np.array_equal(np.isnan(flow_read(tmp_path / "a.npy")), np.isnan(flow))
    with pytest.raises(ValueError):
        flow_write(tmp_path / "a.xyz", flow)
    # writer pool: [2,H,W] tensors, any order of completion
    with AsyncFlowWriter(workers=2) as w:
        for k in range(5):
            w.submit(tmp_path / f"w{k}.flo", torch.full((2, 6, 7), float(k)))
    for k in range(5):
        assert (flow_read(tmp_path / f"w{k}.flo") == k).all()


def test_flow_io_agrees_with_reference_reader(tmp_path):
    """Files written here are byte for byte what the reference's own flow_write writes, its flow_read read them back
    identically, and the reference's file reads back identically here (io_flo.npz, oracle/make_golden.py make_flow_io)."""
    from helpers import load_golden
    from ptlflow_b200.utils.flow_utils import flow_read, flow_write

    recipe, g = load_golden("io_flo")
    flow = (np.random.default_rng(recipe["seed"]).standard_normal((recipe["h"], recipe["w"], 2)) * recipe["scale"]).astype(np.float32)
    flow[1, 1] = np.nan
    p = tmp_path / "x.flo"
    flow_write(p, flow)
    assert p.read_bytes() == g["ref_written"].tobytes()
    ref = g["ref_read"]
    assert np.array_equal(np.isnan(ref), np.isnan(flow)) and np.array_equal(ref[~np.isnan(ref)], flow[~np.isnan(flow)])
    (tmp_path / "y.flo").write_bytes(g["ref_written"].tobytes())
    mine = flow_read(tmp_path / "y.flo")
    assert np.array_equal(np.isnan(mine), np.isnan(flow)) and np.array_equal(mine[~np.isnan(mine)], flow[~np.isnan(flow)])


def test_frame_feeder_batches_and_splits_on_size(tmp_path):
    import cv2

    from ptlflow_b200.pipeline import FrameFeeder

    rng = np.random.default_rng(5)
    paths = []
    for k in range(5):
        h, w = (24, 32) if k < 3 else (16, 40)
        pair = []
        for f in range(2):
            img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
            path = tmp_path / f"f{k}_{f}.png"
            cv2.imwrite(str(path), img)
            pair.append((path, img))
        paths.append(pair)
    feeder = FrameFeeder([(a[0], b[0]) for a, b in paths], batch=4, dtype=torch.float32, workers=2, pin=False)
    got = list(feeder)
    assert [g[0] for g in got] == [[0, 1, 2], [3], [4]]  # batch of 4 split where the size changes, then the rest
    idx, images = got[0]
    assert images.shape == (3, 2, 3, 24, 32)
    want = torch.from_numpy(paths[1][1][1]).permute(2, 0, 1).float() / 255.0  # pair 1, second frame, BGR as cv2 reads it
    assert torch.equal(images[1, 1], want)


def test_overlapping_window_gemm_is_the_convolution():
    """CPU emulation of csrc/first_conv.cu: the packed weight tiles times the overlapping 8-pixel windows of the raw
    input rows (what the non-swizzled UMMA descriptor with LBO = 16 B, SBO = 128 B reads) equals the convolution.
    Pins the operand contract written in include/ptlflow_b200.h without a GPU."""
    import torch.nn.functional as F

    from ptlflow_b200 import ops

    g = torch.Generator().manual_seed(7)
    # ---- first encoder convolution: 7x7, stride 2, 3 -> 64, 4-channel pixels, two output rows per accumulator
    H, W = 12, 20
    x = torch.randn(1, H, W, 4, generator=g)
    x[..., 3] = 0
    wt = torch.randn(64, 3, 7, 7, generator=g)
    ref = F.conv2d(x[..., :3].permute(0, 3, 1, 2), wt, stride=2, padding=3)[0]  # [64, H/2, W/2]
    tiles = ops.pack_first_conv(wt, torch.float32).permute(0, 1, 3, 2, 4).reshape(9, 128, 32)  # [j][p*64+co][4t+c]
    Wo = W // 2
    for y in range(0, H // 2, 2):
        acc = torch.zeros(128, Wo)
        for j in range(9):
            r = 2 * y - 3 + j
            if not 0 <= r < H:
                continue  # rows outside the image contribute zero: the kernel skips their MMAs
            row = torch.zeros((2 * Wo + 8) * 4)  # buffer pixel i <-> image pixel i - 4, zero halo
            row[4 * 4 : 4 * 4 + W * 4] = x[0, r].reshape(-1)
            windows = row.as_strided((Wo, 32), (8, 1))  # output pixel n reads 8 pixels x 4 channels starting 2 pixels further
            acc += tiles[j] @ windows.T
        assert torch.allclose(acc[:64], ref[:, y], atol=1e-4)
        if y + 1 < H // 2:
            assert torch.allclose(acc[64:], ref[:, y + 1], atol=1e-4)
    # ---- convf1: 7x7, stride 1, 2 -> 128 on the hi/lo-split flow, 16-byte (8-channel) pixels
    Hf, Wf = 6, 11
    flow = torch.randn(1, Hf, Wf, 2, generator=g) * 5
    wf = torch.randn(128, 2, 7, 7, generator=g)
    reff = F.conv2d(flow.permute(0, 3, 1, 2), wf, padding=3)[0]
    tf = ops.pack_flow_conv(wf, torch.float32).permute(0, 1, 3, 2, 4).reshape(7, 128, 64)
    hi = flow.half().float()
    lo = flow - hi
    px = torch.zeros(1, Hf, Wf, 8)
    px[..., 0:2], px[..., 2:4] = hi, lo
    for y in range(Hf):
        acc = torch.zeros(128, Wf)
        for j in range(7):
            r = y + j - 3
            if not 0 <= r < Hf:
                continue
            row = torch.zeros((Wf + 8) * 8)
            row[4 * 8 : 4 * 8 + Wf * 8] = px[0, r].reshape(-1)
            acc += tf[j] @ row.as_strided((Wf, 64), (8, 1)).T
        assert torch.allclose(acc, reff[:, y], atol=1e-3)


def test_tiled_layout_index_formula():
    """The tiled-pyramid element offset of include/ptlflow_b200.h (what the CUDA kernels compute) against ops.untile_level."""
    import numpy as np
    import torch

    from ptlflow_b200 import ops

    for h, w in ((55, 128), (27, 45), (6, 16), (1, 1), (13, 33)):
        ty, tx = (h + 3) // 4, (w + 7) // 8
        dense = np.arange(3 * h * w, dtype=np.float32).reshape(3, h, w)
        tiled = np.full((3, ty * tx * 32), -1.0, dtype=np.float32)
        for y in range(h):
            for x in range(w):
                tiled[:, ((y >> 2) * tx + (x >> 3)) * 32 + (y & 3) * 8 + (x & 7)] = dense[:, y, x]
        back = ops.untile_level(torch.from_numpy(tiled), h, w).numpy()
        assert np.array_equal(back, dense)


def test_capture_gate_readers_share_writer_alone():
    """``raft._CaptureGate`` (forwards vs CUDA-graph captures): forwards overlap each other, a capture overlaps nothing, and a
    waiting capture is not starved by new forwards."""
    import threading
    import time

    from ptlflow_b200.models.raft.raft import _CaptureGate

    gate = _CaptureGate()
    lock = threading.Lock()
    state = {"readers": 0, "writers": 0, "max_readers": 0, "violations": 0}
    order = []

    def forward(tag, hold):
        with gate.forward():
            with lock:
                state["readers"] += 1
                state["max_readers"] = max(state["max_readers"], state["readers"])
                state["violations"] += state["writers"] != 0
                order.append(("f", tag))
            time.sleep(hold)
            with lock:
                state["readers"] -= 1

    def capture(tag, hold):
        with gate.capture():
            with lock:
                state["writers"] += 1
                state["violations"] += state["readers"] != 0 or state["writers"] != 1
                order.append(("c", tag))
            time.sleep(hold)
            with lock:
                state["writers"] -= 1

    ts = [threading.Thread(target=forward, args=(i, 0.15)) for i in range(3)]
    for t in ts:
        t.start()
    time.sleep(0.03)
    tc = threading.Thread(target=capture, args=("c0", 0.05))
    tc.start()  # waits for the three forwards
    time.sleep(0.03)
    late = threading.Thread(target=forward, args=("late", 0.0))
    late.start()  # arrives while the capture is waiting: must queue behind it
    for t in ts + [tc, late]:
        t.join(5)
        assert not t.is_alive()
    assert state["violations"] == 0
    assert state["max_readers"] == 3
    assert order.index(("c", "c0")) < order.index(("f", "late"))


def test_onthefly_region_gemm_is_the_lookup():
    """CPU emulation of csrc/corr_onthefly_umma.cu's algorithm (no GPU): per (8 x 16 query tile, level) ONE region of the level's
    feature map -- anchored at the smallest window origin, 32 targets wide, bands of 8 rows at stride 7 -- multiplied with the
    tile's query vectors, and every query's 9 x 9 window blended out of its own row of that product.  Pins, against the oracle's
    a4 (oracle/raft_oracle.py::alt_corr_lookup), the geometry the kernel relies on: every (window row, tap pair) lies in exactly
    one band, windows that fit the region need no other data, zero fill outside the map is the sampler's zero padding, the
    x-major channel order, and which queries are outliers (recomputed by the SIMT kernel on the GPU)."""
    R, D, K, RW = 4, 10, 9, 32
    b, c, h, w, levels = 1, 32, 19, 37, 3
    g = torch.Generator().manual_seed(5)
    f1 = torch.randn(b, c, h, w, generator=g)
    f2 = torch.randn(b, c, h, w, generator=g)
    coords = O.coords_grid(b, h, w) + torch.tensor([2.3, -1.6]).view(1, 2, 1, 1) + 1.2 * torch.randn(b, 2, h, w, generator=g)
    coords[0, :, 3, 5] = torch.tensor([-40.0, 7.0])      # window entirely outside: zeros, not an outlier
    coords[0, :, 10, 20] = torch.tensor([-3.0, 9.0])     # far left of its tile's other windows: it becomes the anchor, the
                                                         # windows more than 22 columns to its right do not fit the region
    ref = O.alt_corr_lookup(f1, f2, coords, R, levels)   # [b, levels*81, h, w]
    scale = 1.0 / np.sqrt(c)

    pyr, f = [], f2
    for lvl in range(levels):
        if lvl:
            f = torch.nn.functional.avg_pool2d(f, 2, stride=2)
        pyr.append(f[0].permute(1, 2, 0).numpy())       # [Hl, Wl, C]
    q1 = f1[0].permute(1, 2, 0).numpy()
    cx, cy = coords[0, 0].numpy(), coords[0, 1].numpy()
    out = np.zeros((h, w, levels * K * K), np.float32)
    served = np.zeros((h, w, levels), bool)
    outliers = 0
    for ty in range(0, h, 8):
        for tx in range(0, w, 16):
            ys, xs = np.meshgrid(np.arange(ty, min(ty + 8, h)), np.arange(tx, min(tx + 16, w)), indexing="ij")
            ys, xs = ys.ravel(), xs.ravel()
            for lvl in range(levels):
                Hl, Wl, _ = pyr[lvl].shape
                x, y = cx[ys, xs] / 2**lvl, cy[ys, xs] / 2**lvl
                xf, yf = np.floor(x), np.floor(y)
                fx, fy = (x - xf).astype(np.float32), (y - yf).astype(np.float32)
                x0, y0 = xf.astype(int) - R, yf.astype(int) - R
                live = (x0 + D - 1 >= 0) & (x0 < Wl) & (y0 + D - 1 >= 0) & (y0 < Hl)
                served[ys[~live], xs[~live], lvl] = True  # all-zero windows
                if not live.any():
                    continue
                bx0, by0, By = x0[live].min(), y0[live].min(), y0[live].max()
                nb = min(max((By + D - 1 - by0 + 6) // 7, 1), 8)
                # the region, zero outside the map (what the TMA unit fills in)
                reg = np.zeros((7 * nb + 1, RW, c), np.float32)
                for ry in range(reg.shape[0]):
                    for rx in range(RW):
                        yy, xx = by0 + ry, bx0 + rx
                        if 0 <= yy < Hl and 0 <= xx < Wl:
                            reg[ry, rx] = pyr[lvl][yy, xx]
                for qi in np.nonzero(live)[0]:
                    cxo, ryo = x0[qi] - bx0, y0[qi] - by0
                    if cxo + D > RW or ryo + D - 1 > 7 * nb:
                        outliers += 1
                        continue
                    qv = q1[ys[qi], xs[qi]]
                    w00, w10 = (1 - fx[qi]) * (1 - fy[qi]) * scale, fx[qi] * (1 - fy[qi]) * scale
                    w01, w11 = (1 - fx[qi]) * fy[qi] * scale, fx[qi] * fy[qi] * scale
                    hits = np.zeros(K, int)
                    for kb in range(nb):
                        band = reg[7 * kb: 7 * kb + 8].reshape(-1, c) @ qv   # this query's accumulator row of the band GEMM
                        for j in range(K):
                            rr = ryo + j - 7 * kb
                            if rr < 0 or rr > 6:
                                continue
                            hits[j] += 1
                            up, dn = band[rr * RW + cxo: rr * RW + cxo + D], band[(rr + 1) * RW + cxo: (rr + 1) * RW + cxo + D]
                            for i in range(K):
                                out[ys[qi], xs[qi], lvl * K * K + i * K + j] = w00 * up[i] + w10 * up[i + 1] + w01 * dn[i] + w11 * dn[i + 1]
                    assert (hits == 1).all(), "every window row is served by exactly one band"
                    served[ys[qi], xs[qi], lvl] = True
    assert outliers >= 1 and served[10, 20].all() and not served[8:16, 16:32].all()
    refp = ref[0].permute(1, 2, 0).numpy().reshape(h, w, levels, K * K)
    got = out.reshape(h, w, levels, K * K)
    assert served.mean() > 0.7
    err = np.abs(got - refp)[served].max()
    assert err < 2e-4, err
    assert np.abs(got[3, 5]).max() == 0 and np.abs(refp[3, 5]).max() == 0


@pytest.mark.parametrize("radius", [3, 4])
def test_tiled_lookup_blend_lane_map_covers_the_window(radius):
    """The lane -> window position map of corr_lookup_tiled_kernel's blend phase (csrc/corr_tiled.cu: rounds of 8 rows x 4 columns,
    plus one mixed round for the ninth row / column of a 9 x 9 window): every position exactly once, and within a round the
    staged rows a warp reads are 12 words apart with at most 3 words per row -- no two lanes on one bank unless on one word."""
    K = 2 * radius + 1
    npos = 3 if K == 9 else (K + 3) // 4
    seen = {}
    for k in range(npos):
        banks = {}
        for lane in range(32):
            if K == 9 and k == 2:
                i, j, act = (8, lane, lane < 17) if lane < 8 else (lane - 8, 8, lane < 17)
            else:
                i, j = (lane >> 3) + 4 * k, lane & 7
                act = j < K and i < K
            if not act:
                continue
            assert (i, j) not in seen
            seen[(i, j)] = (k, lane)
            for off in (0, 7):  # window origin inside its 8-column tile: the two extremes
                word = (j * 24 + i + off) // 2
                banks.setdefault((off, word % 32), set()).add(word)
        if not (K == 9 and k == 2):
            assert all(len(v) == 1 for v in banks.values()), f"round {k}: two different words on one bank"
    assert len(seen) == K * K

"""Generate tests/golden/*.npz by running the REAL reference (build container only).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Usage, from the repo root:

    python -m oracle.make_golden                          # everything the reference computes on the CPU
    python -m oracle.make_golden --ref-plugin [--out DIR]  # op_ref_alt_cuda_corr.npz: needs a CUDA device + oracle/_ref

Each fixture stores only the *outputs* of the reference plus a JSON recipe; inputs and
weights are rebuilt from the recipe with oracle.synth (numpy Philox, platform-stable), so
the fixtures stay small.  The reference's own tests hold no golden vectors for this path
(SURVEY.md section 4) -- these files are what pins the oracle and the CUDA path.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import tempfile
import types

import numpy as np
import torch

from . import ref_shim, synth
from . import raft_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# (fixture name, variant, model kwargs, batch, H, W, image kind, weight seed, image seed)
E2E_CASES = [
    ("e2e_raft_small_cfg1", "raft_small", dict(iters=4), 1, 128, 256, "noise", 1, 11),  # BASELINE.json configs[0] shape
    ("e2e_raft_small_b2", "raft_small", dict(iters=4), 2, 132, 164, "smooth", 2, 12),  # ragged: pads 132->136, 164->168
    ("e2e_raft_noise", "raft", dict(iters=6), 1, 132, 164, "noise", 3, 13),
    ("e2e_raft_smooth_b2", "raft", dict(iters=12), 2, 128, 192, "smooth", 4, 14),
    ("e2e_raft_altcorr", "raft", dict(iters=4, alternate_corr=True), 1, 128, 160, "noise", 5, 15),
    ("e2e_raft_r3_l3", "raft", dict(iters=3, corr_radius=3, corr_levels=3), 1, 128, 136, "smooth", 6, 16),
    ("e2e_gma", "gma", dict(iters=6), 2, 128, 192, "smooth", 7, 17),  # BASELINE.json configs[2] family
]


def _recipe(**kw) -> np.ndarray:
    return np.frombuffer(json.dumps(kw, sort_keys=True).encode(), dtype=np.uint8)


def _sampled(key: str, t: torch.Tensor, k: int) -> dict:
    """An output too large to store whole: its shape, the values at synth.sample_index(numel, k), and the sum, absolute
    sum and largest magnitude over all of it (read back by tests/helpers.check_sample)."""
    flat = t.detach().double().cpu().reshape(-1).numpy()
    return {key: flat[synth.sample_index(flat.size, k)].astype(np.float32), key + "_shape": np.array(t.shape),
            key + "_sums": np.array([flat.sum(), np.abs(flat).sum(), np.abs(flat).max()])}


def make_e2e() -> None:
    for name, variant, kwargs, b, h, w, kind, wseed, iseed in E2E_CASES:
        model = ref_shim.build_reference_model(variant, seed=wseed, **kwargs)
        img = torch.from_numpy(synth.synth_images(b, h, w, seed=iseed, kind=kind))
        with torch.no_grad():
            out = model({"images": img})
        np.savez_compressed(
            os.path.join(GOLDEN_DIR, name + ".npz"),
            recipe=_recipe(variant=variant, kwargs=kwargs, batch=b, height=h, width=w, kind=kind, wseed=wseed, iseed=iseed),
            flows=out["flows"].numpy().astype(np.float32),
            flow_small=out["flow_small"].numpy().astype(np.float32),
        )
        print(name, tuple(out["flows"].shape), "max|flow|", float(out["flows"].abs().max()))


def make_gma_ops() -> None:
    """GMA's Attention / Aggregate (gma_utils.py:32-113) as the reference's own modules compute them (heads = 1)."""
    ref_shim.load_gma()
    import ptlflow.models.gma.gma_utils as gu

    b, c, h, w = 2, 128, 6, 9
    att = gu.Attention(dim=c, heads=1, max_pos_size=160, dim_head=c, position_only=False, position_and_content=False).eval()
    agg = gu.Aggregate(dim=c, dim_head=c, heads=1).eval()
    sd = {"att.to_qk.weight": torch.from_numpy(synth.synth_tensor("att.to_qk.weight", tuple(att.to_qk.weight.shape), 71)),
          "update_block.aggregator.to_v.weight": torch.from_numpy(synth.synth_tensor("update_block.aggregator.to_v.weight", tuple(agg.to_v.weight.shape), 71)),
          "update_block.aggregator.gamma": torch.from_numpy(synth.synth_tensor("update_block.aggregator.gamma", (1,), 71))}
    att.to_qk.weight.data.copy_(sd["att.to_qk.weight"])
    agg.to_v.weight.data.copy_(sd["update_block.aggregator.to_v.weight"])
    agg.gamma.data.copy_(sd["update_block.aggregator.gamma"])
    inp = torch.relu(torch.from_numpy(synth.synth_normal("gma/inp", (b, c, h, w), 71)))
    motion = torch.from_numpy(synth.synth_normal("gma/motion", (b, c, h, w), 71))
    with torch.no_grad():
        a = att(inp)  # [b, heads, N, N]
        g = agg(a, motion)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "op_gma.npz"), recipe=_recipe(b=b, c=c, h=h, w=w, seed=71),
                        attention=a.numpy().astype(np.float32), aggregate=g.numpy().astype(np.float32))
    print("op_gma", tuple(a.shape), tuple(g.shape))


def make_warm_start() -> None:
    """Warm start: the reference's forward_interpolate_batch (scipy) and a second forward started from it."""
    ref_shim.load_raft()
    import ptlflow.utils.utils as ref_utils

    flow = torch.from_numpy(synth.synth_normal("ws/flow", (2, 2, 16, 24), 51, scale=4.0))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "op_forward_interpolate.npz"), recipe=_recipe(b=2, h=16, w=24, seed=51, scale=4.0),
                        out=ref_utils.forward_interpolate_batch(flow).numpy().astype(np.float32))
    model = ref_shim.build_reference_model("raft_small", seed=8, iters=3)
    img = torch.from_numpy(synth.synth_images(1, 128, 160, seed=18, kind="smooth"))
    with torch.no_grad():
        first = model({"images": img})
        second = model({"images": img, "prev_preds": {"flow_small": first["flow_small"]}})
    np.savez_compressed(os.path.join(GOLDEN_DIR, "e2e_raft_small_warm.npz"),
                        recipe=_recipe(variant="raft_small", kwargs=dict(iters=3), batch=1, height=128, width=160, kind="smooth", wseed=8, iseed=18),
                        first_flow_small=first["flow_small"].numpy().astype(np.float32),
                        flows=second["flows"].numpy().astype(np.float32), flow_small=second["flow_small"].numpy().astype(np.float32))
    print("warm start", tuple(second["flows"].shape), "max|flow|", float(second["flows"].abs().max()))


def make_ops() -> None:
    """Operator-level vectors straight from the reference classes (CorrBlock, BasicUpdateBlock, ...)."""
    ref_corr = ref_shim.load_raft_corr()
    ref_raft = ref_shim.load_raft()
    import ptlflow.models.raft.update as ref_update  # reference module (via shim)
    import ptlflow.models.raft.utils as ref_utils

    # --- a1-a3: volume, pyramid, lookup, incl. far out-of-bounds queries -----------------
    b, c, h, w, r, L = 2, 64, 17, 24, 4, 4  # odd H exercises the floor in pooling: 17->8->4->2
    f1 = torch.from_numpy(synth.synth_normal("ops/fmap1", (b, c, h, w), 21))
    f2 = torch.from_numpy(synth.synth_normal("ops/fmap2", (b, c, h, w), 21))
    coords = O.coords_grid(b, h, w) + torch.from_numpy(synth.synth_normal("ops/coords", (b, 2, h, w), 21, scale=6.0))
    coords[0, :, 0, 0] = torch.tensor([-40.0, 3.0])  # far outside
    coords[0, :, 0, 1] = torch.tensor([5.25, 100.0])
    coords[1, :, 1, 1] = torch.tensor([float(w - 1), float(h - 1)])  # exactly on the last pixel
    blk = ref_corr.CorrBlock(f1, f2, num_levels=L, radius=r)
    look = blk(coords)
    np.savez_compressed(
        os.path.join(GOLDEN_DIR, "op_corr_lookup.npz"),
        recipe=_recipe(b=b, c=c, h=h, w=w, radius=r, levels=L, seed=21),
        coords=coords.numpy(),
        lookup=look.numpy(),
        level_sums=np.array([float(p.double().sum()) for p in blk.corr_pyramid]),
        level_shapes=np.array([list(p.shape[-2:]) for p in blk.corr_pyramid]),
        level3=blk.corr_pyramid[3].numpy(),
    )
    print("op_corr_lookup", tuple(look.shape))

    # --- a4/a5: the reference's on-the-fly block (IterativeCorrBlock: alt_cuda_corr not built here)
    alt = ref_corr.get_corr_block(f1, f2, num_levels=L, radius=r, alternate_corr=True)
    np.savez_compressed(
        os.path.join(GOLDEN_DIR, "op_alt_corr.npz"),
        recipe=_recipe(b=b, c=c, h=h, w=w, radius=r, levels=L, seed=21, impl=type(alt).__name__),
        coords=coords.numpy(),
        lookup=alt(coords).numpy(),
    )

    # --- a6-a9: BasicUpdateBlock and SmallUpdateBlock on random tensors ----------------
    for variant, cls, hd, cd, rr in (("raft", ref_update.BasicUpdateBlock, 128, 128, 4), ("raft_small", ref_update.SmallUpdateBlock, 96, 64, 3)):
        ub = cls(4, rr, hidden_dim=hd).eval()
        sd = {"update_block." + k: torch.from_numpy(synth.synth_tensor("update_block." + k, tuple(v.shape), 31)) for k, v in ub.state_dict().items()}
        ub.load_state_dict({k[len("update_block."):]: v for k, v in sd.items()})
        bb, hh, ww = 2, 9, 13
        planes = 4 * (2 * rr + 1) ** 2
        net = torch.tanh(torch.from_numpy(synth.synth_normal("ub/net", (bb, hd, hh, ww), 31)))
        inp = torch.relu(torch.from_numpy(synth.synth_normal("ub/inp", (bb, cd, hh, ww), 31)))
        corr = torch.from_numpy(synth.synth_normal("ub/corr", (bb, planes, hh, ww), 31))
        flow = torch.from_numpy(synth.synth_normal("ub/flow", (bb, 2, hh, ww), 31, scale=3.0))
        with torch.no_grad():
            n2, mask, delta = ub(net, inp, corr, flow)
        extra = {} if mask is None else {"mask": mask.numpy()}
        np.savez_compressed(
            os.path.join(GOLDEN_DIR, f"op_update_{variant}.npz"),
            recipe=_recipe(variant=variant, b=bb, h=hh, w=ww, hidden=hd, context=cd, radius=rr, seed=31),
            net=n2.numpy(), delta=delta.numpy(), **extra,
        )
        print("op_update", variant, tuple(n2.shape))

    # --- a10: convex upsample and raft_small's bilinear upflow8 -------------------------
    m = ref_raft.raft().eval()
    flow = torch.from_numpy(synth.synth_normal("up/flow", (2, 2, 7, 10), 41, scale=3.0))
    mask = torch.from_numpy(synth.synth_normal("up/mask", (2, 576, 7, 10), 41, scale=2.0))
    np.savez_compressed(
        os.path.join(GOLDEN_DIR, "op_upsample.npz"),
        recipe=_recipe(b=2, h=7, w=10, seed=41),
        convex=m.upsample_flow(flow, mask).numpy(),
        upflow8=ref_utils.upflow8(flow).numpy(),
    )

    # --- state_dict names/shapes (restore_model's strict load contract) ------------------
    for variant in ("raft", "raft_small", "gma"):
        mm = getattr(ref_shim.load_gma() if variant == "gma" else ref_raft, variant)()
        shapes = {k: list(v.shape) for k, v in mm.state_dict().items() if k.split(".")[0] in ("fnet", "cnet", "update_block", "att")}
        with open(os.path.join(GOLDEN_DIR, f"state_shapes_{variant}.json"), "w") as f:
            json.dump(shapes, f, indent=0)
        print("state_shapes", variant, len(shapes), sum(int(np.prod(s)) for k, s in shapes.items() if "running" not in k and "num_batches" not in k))


SIBLING_SAME_AS_RAFT = ["gma", "gmflownet", "rapidflow", "rpknet", "skflow", "ms_raft_plus"]
SIBLING_PER_LEVEL_GEMM = ["sea_raft", "memfof", "flow_anything", "flowseek", "recover"]


def make_sibling_corr() -> None:
    """SURVEY.md section 8(f) rank 3 / appendix E: the CorrBlock of each sibling model's own corr.py, RAFT style
    (volume + avg-pool pyramid) at two (levels, radius) and SEA-RAFT style (one volume per level) at (3, 3)."""
    ref_shim.load_raft()
    b, c, h, w, seed = 2, 32, 17, 24, 61  # 17x24 -> 8x12 -> 4x6 -> 2x3: no 1-pixel level (the reference's sampler divides by W - 1)
    f1 = torch.from_numpy(synth.synth_normal("sib/f1", (b, c, h, w), seed))
    f2 = torch.from_numpy(synth.synth_normal("sib/f2", (b, c, h, w), seed))
    coords = O.coords_grid(b, h, w) + torch.from_numpy(synth.synth_normal("sib/c", (b, 2, h, w), seed, scale=3.0))
    out = {}
    for family in SIBLING_SAME_AS_RAFT + SIBLING_PER_LEVEL_GEMM:
        mod = importlib.import_module(f"ptlflow.models.{family}.corr")
        with torch.no_grad():
            if family in SIBLING_SAME_AS_RAFT:
                for levels, radius in ((4, 4), (2, 3)):
                    out.update(_sampled(f"{family}_l{levels}_r{radius}", mod.CorrBlock(f1, f2, num_levels=levels, radius=radius)(coords), 1024))
            else:
                out.update(_sampled(f"{family}_l3_r3", mod.CorrBlock(f1, f2, 3, 3)(coords), 1024))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "op_sibling_corr.npz"), recipe=_recipe(b=b, c=c, h=h, w=w, seed=seed), **out)
    print("op_sibling_corr", len(out) // 3, "outputs")


def make_flow_io() -> None:
    """The reference's .flo writer on a flow holding a NaN, and what its reader returns for the file this project writes."""
    from ptlflow_b200.utils.flow_utils import flow_write

    ref_shim.load_raft()
    for absent in ("png", "h5py"):  # pypng / h5py are not in this image; only the .flo branch is exercised
        sys.modules.setdefault(absent, types.ModuleType(absent))
    import ptlflow.utils.flow_utils as ref_io

    flow = (np.random.default_rng(4).standard_normal((9, 11, 2)) * 7).astype(np.float32)
    flow[1, 1] = np.nan
    with tempfile.TemporaryDirectory() as d:
        ref_io.flow_write(os.path.join(d, "ref.flo"), flow)
        flow_write(os.path.join(d, "ours.flo"), flow)
        written = np.fromfile(os.path.join(d, "ref.flo"), dtype=np.uint8)
        read = np.asarray(ref_io.flow_read(os.path.join(d, "ours.flo")), dtype=np.float32)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "io_flo.npz"), recipe=_recipe(h=9, w=11, seed=4, scale=7.0), ref_written=written, ref_read=read)
    print("io_flo", written.size, "bytes")


REF_PLUGIN_CASES = [(1, 256, 16, 24, 16, 24, 4), (2, 128, 17, 29, 8, 14, 4), (1, 64, 9, 12, 9, 12, 3), (1, 256, 55, 128, 27, 64, 4)]


def make_ref_plugin(out_dir: str) -> None:
    """The reference's own native kernel, ``alt_cuda_corr.forward(fmap1, fmap2, coords, radius)`` (oracle/_ref, built by
    oracle/build_ref.py), on a CUDA device, for the cases of tests/test_gpu_ref_plugin.py."""
    from . import build_ref

    mod = build_ref.load()
    if mod is None:
        raise RuntimeError("oracle/_ref/alt_cuda_corr.so is not built: run oracle/build_ref.py where the reference checkout is")
    dev = "cuda:0"
    out = {}
    for case in REF_PLUGIN_CASES:
        b, c, h1, w1, h2, w2, r = case
        f1 = torch.from_numpy(synth.synth_normal("rp/f1", (b, h1, w1, c), 21)).to(dev)
        f2 = torch.from_numpy(synth.synth_normal("rp/f2", (b, h2, w2, c), 21)).to(dev)
        grid = torch.stack(torch.meshgrid(torch.arange(w1, dtype=torch.float32), torch.arange(h1, dtype=torch.float32), indexing="xy"), dim=-1)
        coords = (grid[None, None] * (w2 / w1) + torch.from_numpy(synth.synth_normal("rp/c", (b, 1, h1, w1, 2), 21, scale=3.0))).contiguous().to(dev)
        (ref,) = mod.forward(f1, f2, coords, r)
        assert ref.dtype == torch.float32
        out.update(_sampled("case_" + "_".join(map(str, case)), ref, 4096))
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, "op_ref_alt_cuda_corr.npz"), recipe=_recipe(seed=21, cases=REF_PLUGIN_CASES), **out)
    print("op_ref_alt_cuda_corr", len(REF_PLUGIN_CASES), "cases on", torch.cuda.get_device_name(0))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-plugin", action="store_true", help="only op_ref_alt_cuda_corr.npz (needs a CUDA device and oracle/_ref)")
    ap.add_argument("--out", default=GOLDEN_DIR, help="where --ref-plugin writes its fixture")
    args = ap.parse_args()
    if args.ref_plugin:
        make_ref_plugin(args.out)
        return
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    make_ops()
    make_e2e()
    make_warm_start()
    make_gma_ops()
    make_sibling_corr()
    make_flow_io()
    total = sum(os.path.getsize(os.path.join(GOLDEN_DIR, f)) for f in os.listdir(GOLDEN_DIR))
    print("golden bytes:", total)


if __name__ == "__main__":
    main()

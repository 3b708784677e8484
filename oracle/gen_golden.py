"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/* by executing the UNMODIFIED reference.

Run in the build container (needs /root/reference):   python oracle/gen_golden.py
The outputs are committed; nothing under tests/ or bench.py reads /root/reference at run time.

Fixtures (all produced by reference code, not by the oracle or the product):
  slice_math.json     get_slice_intersection / get_destination_view / assemble_tensor /
                      torch's _compute_local_shape_and_global_offset on seeded random cases plus
                      the tables of the reference's own tests (tests/test_utils.py:34-119)
  direct_plan.json    DirectWeightSyncDest._build_plan op lists and pull() results for the cases
                      of tests/test_direct_weight_sync.py:103-174, for real DTensor destinations
                      built on a fake process group, and plan statistics for the Llama-3-8B
                      FSDP(N)->TP(N) layouts (meta tensors)
  store_reshard.json  LocalClient + Controller + InMemoryStore + SharedMemoryTransportBuffer:
                      put shards / reshard-get for the mesh pairs of tests/test_resharding_basic.py,
                      tests/test_resharding_ext.py and tests/test_tensor_slice.py (sha256 of results)
  reference_dropin.json  DirectWeightSyncDest._build_plan op lists for handles that carry our
                      NvlinkBuffer, plus the field names of RDMAWeightHandle / TensorSlice and the
                      methods the reference calls on a handle's rdma_buffer
  cast_vectors.npz    torch CPU .to() bit patterns for the dtype pairs the cast kernel implements

``python oracle/gen_golden.py NAME ...`` regenerates only the named fixtures.
"""

from __future__ import annotations

import asyncio
import hashlib
import itertools
import json
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_harness  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def sha(t: torch.Tensor) -> str:
    return hashlib.sha256(t.contiguous().view(torch.uint8).numpy().tobytes()).hexdigest()


def slice_to_json(s):
    if s is None:
        return None
    return {
        "offsets": list(s.offsets),
        "coordinates": None if s.coordinates is None else list(s.coordinates),
        "global_shape": list(s.global_shape),
        "local_shape": list(s.local_shape),
        "mesh_shape": None if s.mesh_shape is None else list(s.mesh_shape),
    }


def placements_to_json(pl):
    from torch.distributed.tensor.placement_types import Shard

    return [["S", p.dim] if isinstance(p, Shard) else ["R"] for p in pl]


# ------------------------------------------------------------------------------------------------
def gen_slice_math():
    from torch.distributed.tensor._utils import _compute_local_shape_and_global_offset
    from torch.distributed.tensor.placement_types import Replicate, Shard
    from torchstore.transport.types import TensorSlice
    from torchstore.utils import assemble_tensor, get_destination_view, get_local_tensor, get_slice_intersection

    rng = random.Random(1234)
    out = {"layouts": [], "intersections": [], "dest_views": [], "assemble": [], "get_local_tensor": []}

    # layouts
    for _ in range(150):
        nd = rng.randint(1, 3)
        shape = tuple(rng.randint(1, 17) for _ in range(nd))
        md = rng.randint(1, 3)
        mesh = tuple(rng.randint(1, 4) for _ in range(md))
        pl = tuple(rng.choice([Replicate()] + [Shard(d) for d in range(nd)]) for _ in range(md))
        for coord in itertools.product(*(range(m) for m in mesh)):
            shp, off = _compute_local_shape_and_global_offset(shape, mesh, list(coord), pl)
            out["layouts"].append({"global_shape": list(shape), "mesh_shape": list(mesh), "coordinate": list(coord),
                                   "placements": placements_to_json(pl), "local_shape": list(shp), "offsets": list(off)})

    def rand_slice(gshape):
        offs, shp = [], []
        for g in gshape:
            a = rng.randint(0, g - 1)
            b = rng.randint(a + 1, g)
            offs.append(a)
            shp.append(b - a)
        return TensorSlice(tuple(offs), (rng.randint(0, 3),), tuple(gshape), tuple(shp), (4,))

    for _ in range(400):
        nd = rng.randint(1, 4)
        g = tuple(rng.randint(1, 12) for _ in range(nd))
        a, b = rand_slice(g), rand_slice(g)
        if rng.random() < 0.05:
            b = TensorSlice(b.offsets, b.coordinates, tuple(x + 1 for x in g), b.local_shape, b.mesh_shape)
        r = get_slice_intersection(a, b)
        out["intersections"].append({"stored": slice_to_json(a), "wanted": slice_to_json(b), "result": slice_to_json(r)})

    for _ in range(400):
        nd = rng.randint(1, 4)
        g = tuple(rng.randint(1, 10) for _ in range(nd))
        dest_slice = rand_slice(g) if rng.random() < 0.8 else None
        dshape = dest_slice.local_shape if dest_slice is not None else g
        dest = torch.zeros(dshape)
        contiguous = True
        if rng.random() < 0.1 and len(dshape) >= 2:
            dest = torch.zeros(tuple(reversed(dshape))).permute(*reversed(range(len(dshape))))
            contiguous = dest.is_contiguous()
        fetch = rand_slice(g)
        if rng.random() < 0.6 and dest_slice is not None:
            inter = get_slice_intersection(fetch, dest_slice)
            if inter is not None:
                fetch = inter
        view = get_destination_view(dest, dest_slice, fetch)
        res = None
        if view is not None:
            # recover the index from the view's storage offset and shape
            esz = dest.element_size()
            off = (view.data_ptr() - dest.data_ptr()) // esz
            idx = []
            rem = off
            for st, e in zip(dest.stride(), view.shape):
                q = rem // st if st else 0
                rem -= q * st
                idx.append([int(q), int(q + e)])
            res = idx
        out["dest_views"].append({"dest_shape": list(dshape), "dest_contiguous": bool(contiguous),
                                  "dest_slice": slice_to_json(dest_slice), "fetch": slice_to_json(fetch), "result": res})

    # assemble: the reference's own tables (tests/test_utils.py:69-119) + random tilings
    def add_assemble(parts, offsets):
        res = assemble_tensor([torch.tensor(p) for p in parts], offsets)
        out["assemble"].append({"parts": parts, "offsets": [list(o) for o in offsets], "result": res.tolist(), "shape": list(res.shape)})

    add_assemble([[0], [1], [2], [3]], [(0,), (1,), (2,), (3,)])
    add_assemble([[1], [2]], [(1,), (2,)])
    add_assemble([[[0, 1], [10, 11]], [[2], [12]], [[3], [13]], [[4], [14]]], [(0, 0), (0, 2), (0, 3), (0, 4)])
    add_assemble([[[0, 1], [10, 11]], [[2], [12]], [[20, 21, 22]]], [(1, 1), (1, 3), (3, 1)])
    for _ in range(40):
        rows, cols = rng.randint(2, 6), rng.randint(2, 6)
        full = torch.arange(rows * cols).reshape(rows, cols) + 100
        rcut = sorted(rng.sample(range(1, rows), rng.randint(0, min(2, rows - 1))))
        ccut = sorted(rng.sample(range(1, cols), rng.randint(0, min(2, cols - 1))))
        rb = [0] + rcut + [rows]
        cb = [0] + ccut + [cols]
        parts, offs = [], []
        for i in range(len(rb) - 1):
            for j in range(len(cb) - 1):
                parts.append(full[rb[i]:rb[i + 1], cb[j]:cb[j + 1]].tolist())
                offs.append((rb[i] + 3, cb[j] + 5))
        order = list(range(len(parts)))
        rng.shuffle(order)
        add_assemble([parts[k] for k in order], [offs[k] for k in order])

    g1 = torch.tensor([0, 1, 2, 3, 4])
    for shape, off in [((1,), (0,)), ((1,), (1,)), ((1,), (2,)), ((1,), (3,))]:
        out["get_local_tensor"].append({"global": g1.tolist(), "shape": list(shape), "offset": list(off),
                                        "result": get_local_tensor(g1, shape, off).tolist()})
    g2 = torch.tensor([[0, 1, 2, 3, 4], [10, 11, 12, 13, 14]])
    for shape, off in [((2, 2), (0, 0)), ((2, 1), (0, 2)), ((2, 1), (0, 3)), ((2, 1), (0, 4))]:
        out["get_local_tensor"].append({"global": g2.tolist(), "shape": list(shape), "offset": list(off),
                                        "result": get_local_tensor(g2, shape, off).tolist()})
    return out


# ------------------------------------------------------------------------------------------------
class MockRDMABuffer:
    """tests/test_direct_weight_sync.py:27-37 semantics."""

    def __init__(self, source_bytes):
        self._source = source_bytes

    async def read_into(self, dest_byte_view):
        dest_byte_view.copy_(self._source)

    async def drop(self):
        pass


def ops_to_json(plan, handle_lists, dest_sd):
    """Describe reference _TransferOps positionally (which handle, exact?, slices)."""
    by_buf = {}
    for name, hl in handle_lists.items():
        for i, h in enumerate(hl):
            by_buf[id(h.rdma_buffer)] = (name, i, h.source_rank)
    ops = []
    for op in plan:
        name, idx, rank = by_buf[id(op.rdma_buffer)]
        ops.append({
            "name": name,
            "source_index": idx,
            "source_rank": rank,
            "exact": op.dest_tensor is None,
            "src_index": None if op.src_slices is None else [[s.start, s.stop] for s in op.src_slices],
            "dest_index": None if op.dest_slices is None else [[s.start, s.stop] for s in op.dest_slices],
        })
    return ops


LLAMA3_8B = dict(dim=4096, n_layers=32, n_heads=32, n_kv_heads=8, vocab=128256, ffn=14336)


def llama_shapes(cfg=LLAMA3_8B):
    """name -> (shape, tp placement) with the torchtitan TP plan (SURVEY.md section 8 header)."""
    d, kv = cfg["dim"], cfg["dim"] // cfg["n_heads"] * cfg["n_kv_heads"]
    out = {"tok_embeddings.weight": ((cfg["vocab"], d), ("S", 0))}
    for i in range(cfg["n_layers"]):
        p = f"layers.{i}."
        out[p + "attention.wq.weight"] = ((d, d), ("S", 0))
        out[p + "attention.wk.weight"] = ((kv, d), ("S", 0))
        out[p + "attention.wv.weight"] = ((kv, d), ("S", 0))
        out[p + "attention.wo.weight"] = ((d, d), ("S", 1))
        out[p + "feed_forward.w1.weight"] = ((cfg["ffn"], d), ("S", 0))
        out[p + "feed_forward.w2.weight"] = ((d, cfg["ffn"]), ("S", 1))
        out[p + "feed_forward.w3.weight"] = ((cfg["ffn"], d), ("S", 0))
        out[p + "attention_norm.weight"] = ((d,), ("R",))
        out[p + "ffn_norm.weight"] = ((d,), ("R",))
    out["norm.weight"] = ((d,), ("R",))
    out["output.weight"] = ((cfg["vocab"], d), ("S", 0))
    return out


def gen_direct_plan():
    import torch.distributed as dist
    from torch.distributed.device_mesh import DeviceMesh
    from torch.distributed.tensor import DTensor, Replicate, Shard
    from torch.distributed.tensor._utils import _compute_local_shape_and_global_offset
    from torch.testing._internal.distributed.fake_pg import FakeStore
    from torchstore.direct_weight_sync import DirectWeightSyncDest, RDMAWeightHandle
    from torchstore.transport.types import TensorSlice
    from torchstore.utils import to_byte_view

    def P(p):
        return Shard(p[1]) if p[0] == "S" else Replicate()

    def source_handles(full, mesh_shape, placements, device="cpu"):
        handles = []
        for rank, coord in enumerate(itertools.product(*(range(m) for m in mesh_shape))):
            shp, off = _compute_local_shape_and_global_offset(full.shape, mesh_shape, list(coord), tuple(P(p) for p in placements))
            if device == "meta":
                local = torch.empty(shp, dtype=full.dtype, device="meta")
            else:
                local = full[tuple(slice(o, o + s) for o, s in zip(off, shp))].contiguous()
            ts = TensorSlice(tuple(off), tuple(coord), tuple(full.shape), tuple(shp), tuple(mesh_shape))
            handles.append(RDMAWeightHandle(MockRDMABuffer(to_byte_view(local)), ts, rank))
        return handles

    cases = []

    # (1) the reference's own test cases: plain full-tensor destinations
    def plain_case(label, fulls, layouts):
        handle_lists = {n: source_handles(fulls[n], *layouts[n]) for n in fulls}
        dest_sd = {n: torch.zeros_like(fulls[n]) for n in fulls}
        sync = DirectWeightSyncDest()
        asyncio.run(sync.pull(handle_lists, dest_sd))
        for n in fulls:
            assert torch.equal(dest_sd[n], fulls[n])
        cases.append({
            "label": label,
            "params": {n: {"global_shape": list(fulls[n].shape), "dtype": str(fulls[n].dtype).replace("torch.", ""),
                           "fill": "arange",
                           "arange_start": int(fulls[n].flatten()[0].item()),
                           "src_mesh": list(layouts[n][0]), "src_placements": [list(p) for p in layouts[n][1]],
                           "dst_mesh": None, "dst_placements": None, "dst_rank": None} for n in fulls},
            "ops": ops_to_json(sync._plan, handle_lists, dest_sd),
            "dest_sha256": {n: sha(dest_sd[n]) for n in fulls},
        })

    big = torch.arange(512 * 512, dtype=torch.float32).reshape(512, 512)
    plain_case("exact_match", {"weight": big}, {"weight": ((1,), [("S", 0)])})
    plain_case("reshard_2_dim0", {"weight": big}, {"weight": ((2,), [("S", 0)])})
    plain_case("reshard_4_dim0", {"weight": big}, {"weight": ((4,), [("S", 0)])})
    plain_case("reshard_2_dim1", {"weight": big}, {"weight": ((2,), [("S", 1)])})
    plain_case("replicated_dedup", {"weight": big}, {"weight": ((2,), [("R",)])})
    w1 = torch.arange(100, dtype=torch.float32).reshape(10, 10)
    w2 = torch.arange(100, 200, dtype=torch.float32).reshape(10, 10)
    plain_case("multiple_params", {"layer.weight": w1, "layer.bias": w2},
               {"layer.weight": ((2,), [("S", 0)]), "layer.bias": ((1,), [("S", 0)])})

    # (2) real DTensor destinations on a fake process group: src layout -> dst layout, every dst rank
    pairs = [
        ((48, 40), (2,), [("S", 0)], (4,), [("S", 1)]),
        ((48, 40), (4,), [("S", 1)], (2,), [("S", 0)]),
        ((48, 40), (2, 2), [("S", 0), ("S", 1)], (4,), [("S", 0)]),
        ((48, 40), (2, 2), [("R",), ("S", 0)], (2, 2), [("S", 1), ("S", 0)]),
        ((48, 40), (8,), [("S", 0)], (8,), [("S", 1)]),
        ((50, 7), (4,), [("S", 0)], (3,), [("S", 0)]),       # uneven
        ((9, 5, 6), (2, 2), [("S", 0), ("S", 2)], (3,), [("S", 1)]),  # 3-D
        ((48, 40), (4,), [("S", 0)], (2, 2), [("R",), ("S", 1)]),
    ]
    for gshape, smesh, spl, dmesh, dpl in pairs:
        full = torch.arange(int(np.prod(gshape)), dtype=torch.float32).reshape(gshape)
        world = int(np.prod(dmesh))
        for drank in range(world):
            dist.init_process_group("fake", store=FakeStore(), rank=drank, world_size=world)
            try:
                mesh = DeviceMesh("cpu", torch.arange(world).reshape(dmesh))
                coord = mesh.get_coordinate()
                shp, off = _compute_local_shape_and_global_offset(full.shape, dmesh, coord, tuple(P(p) for p in dpl))
                local = torch.zeros(shp, dtype=full.dtype)
                dt = DTensor.from_local(local, mesh, tuple(P(p) for p in dpl), run_check=False, shape=full.shape, stride=full.stride())
                handle_lists = {"w": source_handles(full, smesh, spl)}
                sync = DirectWeightSyncDest()
                asyncio.run(sync.pull(handle_lists, {"w": dt}))
                expect = full[tuple(slice(o, o + s) for o, s in zip(off, shp))]
                assert torch.equal(dt._local_tensor, expect), (gshape, smesh, spl, dmesh, dpl, drank)
                cases.append({
                    "label": f"dtensor_{list(gshape)}_{list(smesh)}{spl}_to_{list(dmesh)}{dpl}_r{drank}",
                    "params": {"w": {"global_shape": list(gshape), "dtype": "float32", "fill": "arange", "arange_start": 0,
                                     "src_mesh": list(smesh), "src_placements": [list(p) for p in spl],
                                     "dst_mesh": list(dmesh), "dst_placements": [list(p) for p in dpl], "dst_rank": drank}},
                    "ops": ops_to_json(sync._plan, handle_lists, {"w": dt}),
                    "dest_sha256": {"w": sha(dt._local_tensor)},
                })
            finally:
                dist.destroy_process_group()

    # (3) Llama-3-8B plan statistics on meta tensors (metadata only)
    stats = []
    shapes = llama_shapes()
    for n in (1, 2, 4, 8):
        per_rank = []
        for drank in range(n):
            dist.init_process_group("fake", store=FakeStore(), rank=drank, world_size=n)
            try:
                mesh = DeviceMesh("cpu", torch.arange(n))
                handle_lists, dest_sd = {}, {}
                for name, (shape, tp) in shapes.items():
                    full = torch.empty(shape, dtype=torch.bfloat16, device="meta")
                    handle_lists[name] = source_handles(full, (n,), [("S", 0)], device="meta")
                    shp, off = _compute_local_shape_and_global_offset(shape, (n,), [drank], (P(tp),))
                    local = torch.empty(shp, dtype=torch.bfloat16, device="meta")
                    if n == 1:
                        dest_sd[name] = local
                    else:
                        dest_sd[name] = DTensor.from_local(local, mesh, (P(tp),), run_check=False, shape=torch.Size(shape),
                                                           stride=torch.empty(shape, device="meta").stride())
                sync = DirectWeightSyncDest()
                plan = sync._build_plan(handle_lists, dest_sd)
                n_exact = sum(1 for op in plan if op.dest_tensor is None)
                algo = 0
                ref_read = 0
                for op in plan:
                    ref_read += op.dest_byte_view.numel()
                    if op.dest_tensor is None:
                        algo += op.dest_byte_view.numel()
                    else:
                        algo += int(np.prod([s.stop - s.start for s in op.dest_slices])) * 2
                per_rank.append({"ops": len(plan), "exact_ops": n_exact, "algorithmic_bytes": algo, "reference_read_bytes": ref_read})
            finally:
                dist.destroy_process_group()
        stats.append({"n": n, "per_dest_rank": per_rank})
    return {"cases": cases, "llama3_8b_fsdp_to_tp": stats}


# ------------------------------------------------------------------------------------------------
def gen_store_reshard():
    from torch.distributed.tensor._utils import _compute_local_shape_and_global_offset
    from torch.distributed.tensor.placement_types import Replicate, Shard
    from torchstore.transport import create_transport_buffer
    from torchstore.transport.types import Request, TensorSlice

    def P(p):
        return Shard(p[1]) if p[0] == "S" else Replicate()

    async def put_shard(store, rank, key, local, ts):
        c = store.client(rank)
        req = Request(key=key, tensor_val=local, tensor_slice=ts)
        ref = c.strategy.select_storage_volume()
        tb = create_transport_buffer(ref)
        await tb.put_to_storage_volume([req])
        await c._controller.notify_put_batch.call([req.meta_only()], ref.volume_id)

    # mesh pairs of tests/test_resharding_basic.py:24-154 and tests/test_resharding_ext.py:29-133
    pairs = [
        ((2,), [("S", 0)], (4,), [("S", 0)]),
        ((4,), [("S", 0)], (2,), [("S", 0)]),
        ((2,), [("S", 0)], (2,), [("S", 1)]),
        ((2,), [("S", 1)], (4,), [("S", 0)]),
        ((4,), [("S", 1)], (2,), [("S", 1)]),
        ((2, 2), [("S", 0), ("S", 1)], (4,), [("S", 0)]),
        ((2, 2), [("S", 1), ("S", 0)], (2, 2), [("S", 0), ("S", 1)]),
        ((2, 2), [("R",), ("S", 0)], (4,), [("S", 1)]),
        ((4,), [("S", 0)], (2, 2), [("R",), ("S", 1)]),
        ((2,), [("S", 0)], (2,), [("R",)]),
    ]
    out = {"cases": []}
    full = torch.arange(512 * 512, dtype=torch.float32).reshape(512, 512)  # test_resharding_basic.py:199-205

    async def run():
        for smesh, spl, dmesh, dpl in pairs:
            nput = int(np.prod(smesh))
            nget = int(np.prod(dmesh))
            store = ref_harness.RefStore(max(nput, nget))
            key = "test_key"
            for rank, coord in enumerate(itertools.product(*(range(m) for m in smesh))):
                shp, off = _compute_local_shape_and_global_offset(full.shape, smesh, list(coord), tuple(P(p) for p in spl))
                local = full[tuple(slice(o, o + s) for o, s in zip(off, shp))].contiguous()
                ts = TensorSlice(tuple(off), tuple(coord), tuple(full.shape), tuple(shp), tuple(smesh))
                all_rep = all(p[0] == "R" for p in spl)
                if all_rep:
                    await store.client(rank).put(key, local)  # fully-replicated DTensor == plain tensor
                else:
                    await put_shard(store, rank, key, local, ts)
            results = []
            for rank, coord in enumerate(itertools.product(*(range(m) for m in dmesh))):
                shp, off = _compute_local_shape_and_global_offset(full.shape, dmesh, list(coord), tuple(P(p) for p in dpl))
                dest = torch.zeros(shp, dtype=full.dtype)
                ts = TensorSlice(tuple(off), tuple(coord), tuple(full.shape), tuple(shp), tuple(dmesh))
                got = await store.client(rank).get(key, dest, ts)
                assert got is dest
                assert torch.equal(dest, full[tuple(slice(o, o + s) for o, s in zip(off, shp))])
                results.append({"rank": rank, "local_shape": list(shp), "offsets": list(off), "sha256": sha(dest)})
            whole = await store.client(0).get(key)
            assert torch.equal(whole, full)
            out["cases"].append({"src_mesh": list(smesh), "src_placements": [list(p) for p in spl],
                                 "dst_mesh": list(dmesh), "dst_placements": [list(p) for p in dpl],
                                 "global_shape": list(full.shape), "dtype": "float32", "fill": "arange",
                                 "per_rank": results, "full_get_sha256": sha(whole)})
            store.close()

        # explicit TensorSlice gets (tests/test_tensor_slice.py:66-146)
        store = ref_harness.RefStore(1)
        t = torch.arange(100 * 100, dtype=torch.float32).reshape(100, 100)
        await store.client(0).put("t", t)
        spec = TensorSlice((10, 20), (), (100, 100), (5, 10), ())
        got = await store.client(0).get("t", tensor_slice_spec=spec)
        buf = torch.zeros(5, 10)
        got2 = await store.client(0).get("t", buf, spec)
        assert got2 is buf and torch.equal(got, t[10:15, 20:30]) and torch.equal(buf, got)
        out["tensor_slice_get"] = {"global_shape": [100, 100], "offsets": [10, 20], "local_shape": [5, 10], "sha256": sha(got)}
        # partial commit error text (tests/test_tensor_slice.py:331-396)
        store2 = ref_harness.RefStore(2)
        small = torch.arange(8 * 6, dtype=torch.float32).reshape(8, 6)
        ts0 = TensorSlice((0, 0), (0,), (8, 6), (4, 6), (2,))
        await put_shard(store2, 0, "p", small[:4].contiguous(), ts0)
        try:
            await store2.client(0).get("p")
            msg = None
        except KeyError as e:
            msg = str(e)
        assert msg and "partially committed" in msg
        out["partial_commit_error_contains"] = "partially committed"
        out["partial_commit_exists"] = await store2.client(0).exists("p")
        store.close()
        store2.close()

    asyncio.run(run())
    return out


# ------------------------------------------------------------------------------------------------
def gen_reference_dropin():
    """The reference's _build_plan fed handles that carry our NvlinkBuffer (descriptor only, as a
    destination process sees them after unpickling); tests/test_reference_dropin.py builds our plan
    from the same handles and compares it op for op."""
    import dataclasses
    import inspect
    import re

    import torchstore.direct_weight_sync as ref
    from torchstore.transport.types import TensorSlice

    import workloads
    from torchstore_b200 import direct_weight_sync as ours
    from torchstore_b200.planner import HbmDescriptor

    def fake_buffer(shape, device):
        stride = [int(np.prod(shape[i + 1:])) for i in range(len(shape))]
        desc = HbmDescriptor(region=bytes(120), shape=tuple(shape), stride=tuple(stride), dtype=torch.float32, device=device)
        return ours.NvlinkBuffer(descriptor=desc)

    def make_slice(shape, n, r, placement):
        off, shp = workloads.shard_box(shape, n, r, placement) if placement[0] == "S" else ((0,) * len(shape), tuple(shape))
        return TensorSlice(offsets=tuple(off), coordinates=(r,), global_shape=tuple(shape), local_shape=tuple(shp), mesh_shape=(n,))

    # (global shape, n source ranks, source placement, n dest ranks, dest placement)
    cases = [
        ((512, 512), 2, ("S", 0), 2, ("S", 0)),   # exact
        ((512, 512), 4, ("S", 0), 2, ("S", 1)),   # reshard
        ((96, 40), 4, ("S", 0), 3, ("S", 1)),     # uneven
        ((64,), 4, ("R",), 2, ("R",)),            # replicated dedup
        ((128, 64), 8, ("S", 0), 1, ("R",)),      # replicated reader (config 3)
    ]
    out = {"cases": []}
    for shape, n_src, sp, n_dst, dp in cases:
        per_dest = {}
        for drank in range(n_dst):
            ds = make_slice(shape, n_dst, drank, dp)
            if 0 in ds.local_shape:
                continue
            handles, rank_of = [], {}
            for r in range(n_src):
                ss = make_slice(shape, n_src, r, sp)
                if 0 in ss.local_shape:
                    continue
                buf = fake_buffer(ss.local_shape, r)
                rank_of[id(buf)] = r
                handles.append(ref.RDMAWeightHandle(rdma_buffer=buf, tensor_slice=ss, source_rank=r))
            dest = torch.zeros(ds.local_shape, dtype=torch.float32)
            # a plain destination tensor stands for "the whole tensor"; hand the reference the shard's
            # slice the way Request.from_dtensor would
            saved = ref._request_to_slice
            ref._request_to_slice = lambda req, param, _s=ds: _s
            try:
                plan = ref.DirectWeightSyncDest()._build_plan({"w": handles}, {"w": dest})
            finally:
                ref._request_to_slice = saved
            ops = []
            for op in plan:
                exact = op.dest_tensor is None
                ops.append({
                    "source_rank": rank_of[id(op.rdma_buffer)],
                    "exact": exact,
                    "src_index": None if exact else [[s.start, s.stop] for s in op.src_slices],
                    "dest_index": None if exact else [[s.start, s.stop] for s in op.dest_slices],
                    "recv_shape": None if exact else list(op.recv_buffer.shape),
                    # exact: the read lands in the caller's tensor; partial: the overlap is copied into it
                    "writes_into_dest": (op.dest_byte_view.data_ptr() == dest.data_ptr()) if exact else (op.dest_tensor is dest),
                })
            per_dest[str(drank)] = ops
        out["cases"].append({"global_shape": list(shape), "n_src": n_src, "src_placement": list(sp), "n_dst": n_dst,
                             "dst_placement": list(dp), "ops_by_dest_rank": per_dest})
    out["handle_fields"] = [f.name for f in dataclasses.fields(ref.RDMAWeightHandle)]
    out["tensor_slice_fields"] = [f.name for f in dataclasses.fields(TensorSlice)]
    out["buffer_calls"] = sorted(set(re.findall(r"\.rdma_buffer\.(\w+)\(", inspect.getsource(ref))))
    return out


# ------------------------------------------------------------------------------------------------
def gen_cast_vectors():
    rng = np.random.default_rng(7)
    edge32 = np.array([
        0x00000000, 0x80000000, 0x3F800000, 0xBF800000, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00000, 0x7F800001,
        0x7FFFFFFF, 0x00000001, 0x007FFFFF, 0x00800000, 0x3F808000, 0x3F818000, 0x3F807FFF, 0x3F808001, 0x7F7FFFFF,
        0x7F7F8000, 0x477FE000, 0x477FF000, 0x38800000, 0x387FC000, 0x33800000, 0x33000000, 0x33000001, 0x32FFFFFF,
        0x3F801000, 0x3F803000, 0x3F800FFF, 0x3F801001, 0x47800000, 0xC7800000, 0x0000FFFF, 0x00010000,
    ], dtype=np.uint32)
    rnd32 = rng.integers(0, 2**32, size=4096, dtype=np.uint64).astype(np.uint32)
    near = (np.float32(1.0) + rng.standard_normal(2048).astype(np.float32) * np.float32(0.02)).view(np.uint32)
    f32 = np.concatenate([edge32, rnd32, near])
    t32 = torch.from_numpy(f32.view(np.float32).copy())
    bf16 = t32.to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    f16 = t32.to(torch.float16).view(torch.int16).numpy().view(np.uint16)

    all16 = np.arange(0, 65536, dtype=np.uint32).astype(np.uint16)
    t_bf = torch.from_numpy(all16.view(np.int16).copy()).view(torch.bfloat16)
    t_h = torch.from_numpy(all16.view(np.int16).copy()).view(torch.float16)
    bf16_to_f32 = t_bf.to(torch.float32).view(torch.int32).numpy().view(np.uint32)
    f16_to_f32 = t_h.to(torch.float32).view(torch.int32).numpy().view(np.uint32)
    bf16_to_f16 = t_bf.to(torch.float16).view(torch.int16).numpy().view(np.uint16)
    f16_to_bf16 = t_h.to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)

    f64 = np.concatenate([
        np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, 1e-50, 1e50, 3.4028235677973366e38, 1.0000000596046448, 1.0000001788139343]),
        rng.standard_normal(1024) * 10.0 ** rng.integers(-40, 40, size=1024),
    ]).astype(np.float64)
    f64_to_f32 = torch.from_numpy(f64.copy()).to(torch.float32).view(torch.int32).numpy().view(np.uint32)
    f32_to_f64 = t32.to(torch.float64).view(torch.int64).numpy().view(np.uint64)
    return dict(f32=f32, f32_to_bf16=bf16, f32_to_f16=f16, all16=all16, bf16_to_f32=bf16_to_f32, f16_to_f32=f16_to_f32,
                bf16_to_f16=bf16_to_f16, f16_to_bf16=f16_to_bf16, f64=f64.view(np.uint64), f64_to_f32=f64_to_f32,
                f32_to_f64=f32_to_f64)


def main():
    ref_harness.import_reference()
    os.makedirs(GOLDEN, exist_ok=True)
    meta = {"reference_commit": "ed2ddb67", "torch": torch.__version__, "generator": "oracle/gen_golden.py"}
    fixtures = {"slice_math": gen_slice_math, "direct_plan": gen_direct_plan, "store_reshard": gen_store_reshard,
                "reference_dropin": gen_reference_dropin}
    wanted = sys.argv[1:] or [*fixtures, "cast_vectors"]
    unknown = set(wanted) - set(fixtures) - {"cast_vectors"}
    if unknown:
        raise SystemExit(f"unknown fixtures {sorted(unknown)}; choose from {[*fixtures, 'cast_vectors']}")
    for name, fn in fixtures.items():
        if name not in wanted:
            continue
        data = fn()
        data["_meta"] = meta
        with open(os.path.join(GOLDEN, name + ".json"), "w") as f:
            json.dump(data, f, separators=(",", ":"))
        print(name, os.path.getsize(os.path.join(GOLDEN, name + ".json")), "bytes")
    if "cast_vectors" in wanted:
        np.savez_compressed(os.path.join(GOLDEN, "cast_vectors.npz"), **gen_cast_vectors())
        print("cast_vectors", os.path.getsize(os.path.join(GOLDEN, "cast_vectors.npz")), "bytes")


if __name__ == "__main__":
    main()

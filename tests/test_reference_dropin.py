"""Drop-in proof: our ``NvlinkBuffer`` handles go through the reference's UNMODIFIED
``DirectWeightSyncDest._build_plan`` (metadata only -- torchstore/direct_weight_sync.py:221-317) and
the op list it builds must equal the one our own ``_build_plan`` builds from the same handles: same
length, same order, same exact/partial classification, same source/destination slices, same buffer
per op.  The reference's op lists were recorded by oracle/gen_golden.py into
tests/golden/reference_dropin.json.

Also checks the other half of the duck-type contract (direct_weight_sync.py:46-58): a handle with the
reference's fields carrying an ``NvlinkBuffer`` survives the pickle round trip every store put
performs, and the buffer exposes the coroutine methods the reference calls (read_into / write_from / drop).
"""

import dataclasses
import inspect
import json
import os
import pickle

import pytest
import torch

import workloads
from torchstore_b200 import direct_weight_sync as ours
from torchstore_b200.planner import HbmDescriptor
from torchstore_b200.transport.types import TensorSlice as OurSlice

with open(os.path.join(os.path.dirname(__file__), "golden", "reference_dropin.json")) as _f:
    GOLDEN = json.load(_f)


def _fake_buffer(shape, dtype, device):
    """An NvlinkBuffer as a destination process sees it after unpickling: descriptor only."""
    stride = []
    s = 1
    for e in reversed(shape):
        stride.append(s)
        s *= e
    desc = HbmDescriptor(region=bytes(120), shape=tuple(shape), stride=tuple(reversed(stride)), dtype=dtype, device=device)
    return ours.NvlinkBuffer(descriptor=desc)


def _cases():
    # (global shape, n source ranks, source placement, n dest ranks, dest placement, recorded reference ops)
    for c in GOLDEN["cases"]:
        yield (tuple(c["global_shape"]), c["n_src"], tuple(c["src_placement"]), c["n_dst"], tuple(c["dst_placement"]),
               c["ops_by_dest_rank"])


def _slice(cls, shape, n, r, placement):
    off, shp = workloads.shard_box(shape, n, r, placement) if placement[0] == "S" else ((0,) * len(shape), tuple(shape))
    return cls(offsets=tuple(off), coordinates=(r,), global_shape=tuple(shape), local_shape=tuple(shp), mesh_shape=(n,))


def _slices(index):
    return tuple(slice(a, b) for a, b in index)


@pytest.mark.parametrize("case", list(_cases()), ids=lambda c: f"{c[0]}-{c[1]}{c[2]}->{c[3]}{c[4]}")
def test_reference_build_plan_accepts_nvlink_buffers_and_matches_ours(case):
    shape, n_src, sp, n_dst, dp, ref_ops_by_rank = case

    for drank in range(n_dst):
        buf_of_rank, our_handles = {}, []
        for r in range(n_src):
            rs = _slice(OurSlice, shape, n_src, r, sp)
            if 0 in rs.local_shape:
                continue
            buf = _fake_buffer(rs.local_shape, torch.float32, r)
            buf_of_rank[r] = buf
            our_handles.append(ours.RDMAWeightHandle(rdma_buffer=buf, tensor_slice=rs, source_rank=r))
        ds_our = _slice(OurSlice, shape, n_dst, drank, dp)
        if 0 in ds_our.local_shape:
            continue
        ref_ops = ref_ops_by_rank[str(drank)]
        dest = torch.zeros(ds_our.local_shape, dtype=torch.float32)
        our_ops = ours.DirectWeightSyncDest()._build_plan({"w": our_handles}, {"w": dest}, {"w": ds_our})
        assert len(ref_ops) == len(our_ops) > 0
        for a, b in zip(ref_ops, our_ops):
            assert buf_of_rank[a["source_rank"]] is b.rdma_buffer  # same source, same order
            ref_exact = a["exact"]
            assert ref_exact == (b.dest_tensor is None)
            assert a["writes_into_dest"]  # the reference fills the caller's tensor, not a copy of it
            if not ref_exact:
                assert _slices(a["src_index"]) == tuple(b.src_slices)
                assert _slices(a["dest_index"]) == tuple(b.dest_slices)
                assert b.dest_tensor is dest
                # the reference stages the WHOLE source shard; we describe just the overlap rectangle
                assert tuple(a["recv_shape"]) == tuple(buf_of_rank[a["source_rank"]].shape)
            else:
                assert b.dest_byte_view.data_ptr() == dest.data_ptr()


def test_handle_pickles_and_duck_types_like_an_rdma_buffer():
    # our handle and slice carry exactly the reference's fields, so either side can build the other's
    assert [f.name for f in dataclasses.fields(ours.RDMAWeightHandle)] == GOLDEN["handle_fields"]
    assert [f.name for f in dataclasses.fields(OurSlice)] == GOLDEN["tensor_slice_fields"]

    buf = _fake_buffer((16, 8), torch.bfloat16, 3)
    h = ours.RDMAWeightHandle(**dict(zip(GOLDEN["handle_fields"], (buf, _slice(OurSlice, (32, 8), 2, 1, ("S", 0)), 1))))
    h2 = pickle.loads(pickle.dumps(h))
    assert h2.rdma_buffer.descriptor == buf.descriptor and h2.tensor_slice == h.tensor_slice and h2.source_rank == 1
    assert h2.rdma_buffer.nbytes == 16 * 8 * 2 and h2.rdma_buffer.dtype == torch.bfloat16
    methods = ("read_into", "write_from", "drop")  # call sites direct_weight_sync.py:143,174,339
    assert set(GOLDEN["buffer_calls"]) <= set(methods)
    for name in methods:
        assert inspect.iscoroutinefunction(getattr(h2.rdma_buffer, name))
    # CPU tensors are refused loudly (no host data plane behind this handle)
    import asyncio

    with pytest.raises(RuntimeError):
        asyncio.run(h2.rdma_buffer.read_into(torch.zeros(16 * 8 * 2, dtype=torch.uint8)))

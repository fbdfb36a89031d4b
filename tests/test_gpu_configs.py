"""BASELINE.json configs 3, 4 and 5 at full size as parity cases (config 2 is in test_gpu_parity.py,
config 1 in test_gpu_client.py).  Blobs are generated in HBM; the CPU oracle re-hashes the same bytes."""
import hashlib
import struct

import numpy as np
import pytest

import modelx_b200

pytestmark = pytest.mark.gpu
SEED = 0x6D6F64656C78


def _torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def test_config3_32_safetensors_shards_whole_file_digests(engine, oracle):
    """32 x 0.5 GB safetensors-shaped shards (8-byte LE header length + JSON header + fp16 payload):
    one reference-identical whole-file digest per shard, all 32 hashed as one lock-step batch."""
    torch = _torch()
    nshard, size = 32, 500_000_000
    buf = torch.empty(nshard * size, dtype=torch.uint8, device="cuda")
    engine.dev_gen_fill(0, buf.data_ptr(), 0, nshard * size, SEED + 3)
    # give every shard a real safetensors prefix so the bytes are shaped like the Llama-3-8B fp16 layout
    for i in range(nshard):
        hdr = ('{"model.layers.%d.mlp.down_proj.weight":{"dtype":"F16","shape":[4096,14336],"data_offsets":[0,117440512]},'
               '"model.layers.%d.mlp.up_proj.weight":{"dtype":"F16","shape":[14336,4096],"data_offsets":[117440512,234881024]}}' % (i, i)).encode()
        hdr += b" " * (-len(hdr) % 8)
        prefix = struct.pack("<Q", len(hdr)) + hdr
        buf[i * size:i * size + len(prefix)] = torch.frombuffer(bytearray(prefix), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    spans = [(buf.data_ptr() + i * size, size) for i in range(nshard)]
    got = engine.sha256_batch_ptrs(spans)
    host = buf.cpu().numpy()
    want = oracle.sha256_batch_ptrs([(host.ctypes.data + i * size, size) for i in range(nshard)], threads=32)
    assert got == want
    assert len(set(got)) == nshard
    # chunked form of the same shards: per-shard tree roots
    d_root = torch.empty(32, dtype=torch.uint8, device="cuda")
    for i in (0, 31):
        engine.dev_tree_digest(0, buf.data_ptr() + i * size, size, (8 << 20, 16 << 10, 8), 0, d_root.data_ptr())
        torch.cuda.synchronize()
        _, _, root = oracle.tree_digest_ptr(host.ctypes.data + i * size, size, 8 << 20, 16 << 10, 8, threads=32)
        assert d_root.cpu().numpy().tobytes() == root


def test_config4_140GB_blob_8MiB_chunks(engine, oracle):
    """One 140 GB blob (70B-fp16 sized) in 8 MiB chunks: 16,690 chunk digests (last chunk 2,521,088 B) and the
    root, HBM-resident, against the threaded CPU oracle on the same bytes; plus the sharded form."""
    torch = _torch()
    size = 140_000_000_000
    tp = (8 << 20, 16 << 10, 8)
    nch = -(-size // tp[0])
    assert nch == 16690 and size - (nch - 1) * tp[0] == 2_521_088
    data = torch.empty(size, dtype=torch.uint8, device="cuda")
    d_chunks = torch.empty(nch * 32, dtype=torch.uint8, device="cuda")
    d_root = torch.empty(32, dtype=torch.uint8, device="cuda")
    engine.dev_gen_fill(0, data.data_ptr(), 0, size, SEED + 4)
    engine.dev_tree_digest(0, data.data_ptr(), size, tp, d_chunks.data_ptr(), d_root.data_ptr())
    torch.cuda.synchronize()
    chunks_gpu = d_chunks.cpu().numpy().tobytes()
    root_gpu = d_root.cpu().numpy().tobytes()
    # sharded across 8 "ranks": chunk ranges hashed independently, then finished from the gathered list
    from modelx_b200 import shard
    gathered = b""
    d_part = torch.empty(shard.chunks_per_rank(nch, 8) * 32, dtype=torch.uint8, device="cuda")
    for r in range(8):
        b0, b1 = shard.byte_range(r, 8, size, tp[0])
        c0, c1 = shard.chunk_range(r, 8, nch)
        engine.dev_tree_chunks(0, data.data_ptr() + b0, b1 - b0, tp, d_part.data_ptr())
        torch.cuda.synchronize()
        gathered += d_part.cpu().numpy().tobytes()[:32 * (c1 - c0)]
    assert gathered == chunks_gpu
    assert engine.tree_finish(gathered, size, *tp) == root_gpu
    # CPU oracle over the same 140 GB, copied to the host one chunk-aligned 8 GiB slab at a time so that host memory
    # stays far below the blob size: a piece that starts on a chunk boundary hashes to exactly the chunk digests of its
    # range (docs/TREE_FORMAT.md), and the levels above the chunk list are rebuilt from those digests by hand
    slab = 1024 * tp[0]
    want_chunks = []
    for s0 in range(0, size, slab):
        host = data[s0:min(s0 + slab, size)].cpu().numpy()
        want_chunks += oracle.tree_digest_ptr(host.ctypes.data, host.size, *tp, threads=32)[0]
        del host
    del data
    level = list(want_chunks)
    while len(level) > 1:
        level = [hashlib.sha256(b"".join(level[i:i + tp[2]])).digest() for i in range(0, len(level), tp[2])]
    want_root = hashlib.sha256(b"modelx.tree.v1\0\0" + struct.pack("<QQII", size, tp[1], tp[2], 0) + level[0]).digest()
    assert len(want_chunks) == nch
    assert chunks_gpu == b"".join(want_chunks) and root_gpu == want_root


def test_config5_pull_side_verify_1000_blobs(engine, oracle):
    """1000 x 128 MB blobs with precomputed expected digests: the pull-side check (pull.go:115-123) as one
    GPU batch + compare kernel; a few expectations are corrupted on purpose."""
    torch = _torch()
    n, size = 1000, 128_000_000
    buf = torch.empty(n * size, dtype=torch.uint8, device="cuda")
    engine.dev_gen_fill(0, buf.data_ptr(), 0, n * size, SEED + 5)
    torch.cuda.synchronize()
    # expected digests from the CPU oracle (what a manifest would carry), computed on a host copy in slabs
    want = []
    slab = 100
    for s in range(0, n, slab):
        host = buf[s * size:(s + slab) * size].cpu().numpy()
        want += oracle.sha256_batch_ptrs([(host.ctypes.data + i * size, size) for i in range(slab)], threads=32)
        del host
    spans = np.zeros((n, 2), dtype=np.uint64)
    spans[:, 0] = buf.data_ptr() + np.arange(n, dtype=np.uint64) * np.uint64(size)
    spans[:, 1] = size
    d_spans = torch.from_numpy(spans.view(np.uint8).reshape(-1)).cuda()
    d_got = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    engine.dev_sha256_batch(0, d_spans.data_ptr(), n, d_got.data_ptr())
    torch.cuda.synchronize()
    assert d_got.cpu().numpy().tobytes() == b"".join(want)
    bad = {7, 500, 999}
    exp = bytearray(b"".join(want))
    for i in bad:
        exp[32 * i + 5] ^= 0x40
    d_want = torch.frombuffer(exp, dtype=torch.uint8).cuda()
    d_ok = torch.empty(n, dtype=torch.uint8, device="cuda")
    engine.dev_compare(0, d_got.data_ptr(), d_want.data_ptr(), n, d_ok.data_ptr())
    torch.cuda.synchronize()
    assert d_ok.cpu().tolist() == [int(i not in bad) for i in range(n)]

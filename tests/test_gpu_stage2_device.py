"""Stage 2 on the device (LZ4 blocks per chunk, cldn_lz4.cu): device pointers in, device pointers out. LZ4 compressors are
not canonical, so the bytes are not compared with liblz4's; what must hold is interoperability both ways with the stock
reference (which calls LZ4_compress_default / LZ4_decompress_safe per chunk, codec_common.cpp:220-299)."""
import numpy as np
import pytest

import cloudini_b200 as cb
from cloudini_b200 import synth
from test_gpu_parity import _Dev

pytestmark = pytest.mark.gpu
LZ4 = cb.CompressionOption.LZ4


def _device_encode(info, clouds):
    enc = cb.PointcloudEncoder(info)
    n_bytes = [c.size for c in clouds]
    caps = [cb.MaxCompressedSize(info, b // info.point_step, True) for b in n_bytes]
    d_in = [_Dev(src=c) if c.size else _Dev(size=16) for c in clouds]
    d_out = [_Dev(size=max(c, 16)) for c in caps]
    sizes = enc.encode_batch_device(enc.make_device_batch([t.ptr for t in d_in], n_bytes, [t.ptr for t in d_out], caps), write_header=True, want_sizes=True)
    return [bytes(o.numpy()[:s]) for o, s in zip(d_out, sizes)]


def _device_decode(info, blobs, n_bytes, fill=0):
    dec = cb.PointcloudDecoder()
    hdrs = [cb.DecodeHeader(b)[1] for b in blobs]
    d_blob = [_Dev(src=np.frombuffer(b, dtype=np.uint8)) for b in blobs]
    d_out = [_Dev(src=np.full(n_bytes, fill, dtype=np.uint8)) for _ in blobs]
    batch = dec.make_device_batch([t.ptr + h for t, h in zip(d_blob, hdrs)], [len(b) - h for b, h in zip(blobs, hdrs)], [t.ptr for t in d_out], [n_bytes] * len(blobs))
    dec.decode_batch_device(info, batch, sync=True)
    return [o.numpy() for o in d_out]


def _ref_decode(ref, blob, n_bytes, fill=0):
    out = np.full(n_bytes, fill, dtype=np.uint8)
    ref.decode(blob, out)
    return out


def _cases():
    n = 70_000
    info, cloud = synth.cloud_c2(n, seed=31)
    yield "xyzi", info, [cloud, synth.cloud_c2(n, seed=32)[1], synth.cloud_c2(n, seed=33)[1]]
    flat = np.tile(np.array([1.5, -2.25, 0.125, 7.0], dtype=np.float32), n).view(np.uint8)        # long, overlapping matches
    rnd = np.random.default_rng(5).normal(0, 50.0, (n, 4)).astype(np.float32).view(np.uint8).reshape(-1)  # nearly incompressible
    yield "flat+random", synth.info_xyzi(n), [np.array(flat), rnd]
    info, cloud = synth.cloud_c3(40_001, seed=8)                                                    # V5 sections behind the floats
    yield "c3", info, [cloud]
    info, cloud = synth.cloud_c4_mixed_frame(3)                                                      # Velodyne XYZIRT, step 22
    yield "xyzirt", info, [cloud, synth.cloud_c4_mixed_frame(4)[1]]
    yield "tiny", synth.info_xyzi(3), [synth.cloud_c2(3, seed=1)[1]]                                 # blocks below the 13-byte minimum
    # a sweep that repeats every 977 points: the stage-1 bytes repeat at a distance of a few KB, so matches span many of the
    # compressor's 128-position steps and run into the end of every chunk (last-match / last-literals rules of the block format);
    # the second cloud stops 5 points into its third chunk (a block of a few bytes behind two full ones)
    rng = np.random.default_rng(77)
    base = np.cumsum(rng.normal(0, 0.02, (977, 4)), axis=0).astype(np.float32)
    per = np.tile(base, (n // 977 + 1, 1))[:n]
    yield "periodic", synth.info_xyzi(n), [np.ascontiguousarray(per).view(np.uint8).reshape(-1)]
    m = 2 * 32768 + 5
    yield "periodic-ragged", synth.info_xyzi(m), [np.ascontiguousarray(np.tile(base, (m // 977 + 1, 1))[:m]).view(np.uint8).reshape(-1)]


@pytest.mark.parametrize("case", list(_cases()), ids=lambda c: c[0])
def test_device_lz4_interoperates_with_the_reference(ref, case):
    name, info, clouds = case
    info.compression_opt = LZ4
    n_bytes = clouds[0].size
    ours = _device_encode(info, clouds)
    for blob, cloud in zip(ours, clouds):
        theirs = ref.encode(info, cloud)
        dinfo, _ = cb.DecodeHeader(blob)
        assert dinfo.compression_opt == LZ4
        want = _ref_decode(ref, theirs, n_bytes, 0x2E)
        # the stock decoder reads our blocks: the host-pointer API hands every block to liblz4's LZ4_decompress_safe, the
        # call the reference makes per chunk (our blocks are not canonical, so the reference's answer on them is not stored)
        mine = np.full(n_bytes, 0x2E, dtype=np.uint8)
        cb.PointcloudDecoder().decode(dinfo, blob[cb.DecodeHeader(blob)[1]:], mine)
        assert np.array_equal(mine, want), name
        got = _device_decode(dinfo, [blob, theirs], n_bytes, 0x2E)                   # and we read both
        assert np.array_equal(got[0], want) and np.array_equal(got[1], want), name
    # the host-pointer API (liblz4 behind it) and the device path are interchangeable
    host_blob = cb.PointcloudEncoder(info).encode(clouds[0])
    assert np.array_equal(_device_decode(cb.DecodeHeader(host_blob)[0], [host_blob], n_bytes)[0], _ref_decode(ref, host_blob, n_bytes))


def test_device_lz4_rejects_damaged_blocks(ref):
    n = 40_000
    info, cloud = synth.cloud_c2(n, seed=3)
    info.compression_opt = LZ4
    blob = bytearray(ref.encode(info, cloud))   # liblz4's blocks: the damaged blobs are the same on every run
    dinfo, hdr = cb.DecodeHeader(bytes(blob))
    rng = np.random.default_rng(1)
    failures = 0
    for trial in range(12):
        bad = bytearray(blob)
        if trial % 3 == 0:
            bad = bad[:hdr + int(rng.integers(6, len(blob) - hdr - 1))]           # truncated
        elif trial % 3 == 1:
            bad[hdr:hdr + 4] = int(rng.integers(len(blob), 2**31)).to_bytes(4, "little")  # forged chunk size
        else:
            for _ in range(6):
                bad[hdr + 4 + int(rng.integers(0, 2000))] = int(rng.integers(0, 256))     # damaged sequences
        try:
            out = _device_decode(dinfo, [bytes(bad)], n * 16)[0]
            ok_ref = True
            try:
                want = _ref_decode(ref, bytes(bad), n * 16)
            except RuntimeError:
                ok_ref = False
            if ok_ref:
                assert np.array_equal(out, want), trial   # the damage happened to leave a valid blob: same points
        except RuntimeError:
            failures += 1
    assert failures >= 6

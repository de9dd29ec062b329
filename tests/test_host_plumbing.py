"""BASELINE config 1 — "groupByKey on 1M Int pairs, local[2], rootDir=file:///tmp/spark-s3-shuffle, LZ4 (CPU plumbing,
no GPU)" — and the host mirror's reference-compatible behaviour.  Runs without a GPU: the writer is used in
pass-through mode, i.e. exactly the reference's own situation where Spark's writers hand it bytes that are already
compressed and checksummed (shuffle/S3ShuffleMapOutputWriter.scala:91,113-115); here the ORACLE plays that upstream.
Shape follows test/S3ShuffleManagerTest.scala:56-73 (runWithSparkConf_noMapSideCombine) + :207-220 (conf).
"""
import os
import shutil
import uuid

import numpy as np
import pytest

import spark_s3_shuffle_b200 as pkg
from shuffle_model import decode_pairs, encode_pairs, oracle_read_partition
from without_gpu import rerun_without_gpu

host = pkg.host


def new_conf(tmp_path, **extra):
    conf = {
        "spark.app.id": "app-" + uuid.uuid4().hex[:12],
        "spark.shuffle.s3.rootDir": "file://" + str(tmp_path) + "/spark-s3-shuffle",  # test/…:215
        "spark.shuffle.checksum.enabled": True,
        "spark.shuffle.checksum.algorithm": "ADLER32",
        "spark.io.compression.codec": "lz4",
        "spark.shuffle.s3.gpu.enabled": False,  # pass-through: the reference's own mode
    }
    conf.update(extra)
    return conf


def test_header_symbols_are_exported():
    import ctypes, re
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                             "b200shuffle_host.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    syms = sorted(set(re.findall(r"\b(b2sh_[a-z0-9_]+)\s*\(", text)))
    assert syms == sorted(host.SYMBOLS)
    lib = ctypes.CDLL(pkg._build.build_host())
    for s in syms:
        assert hasattr(lib, s)


def test_config1_groupbykey_1m_int_pairs(tmp_path, oracle):
    conf = new_conf(tmp_path)
    d = host.S3ShuffleDispatcher(conf)
    n, n_maps, n_red = 1_000_000, 2, 2
    i = np.arange(n, dtype=np.int64)
    keys, vals = i % 1000, i
    alg = host.S3ShuffleHelper.createChecksumAlgorithm("ADLER32")
    expect = {r: [] for r in range(n_red)}
    for m in range(n_maps):
        sel = slice(m * n // n_maps, (m + 1) * n // n_maps)
        k, v = keys[sel], vals[sel]
        w = host.S3ShuffleMapOutputWriter(d, 0, m, n_red)
        cks, lens = [], []
        for r in range(n_red):
            mask = (k % n_red) == r
            raw = encode_pairs(k[mask], v[mask])
            expect[r].append((k[mask], v[mask]))
            comp = oracle.lz4block_compress(raw, 32768)  # upstream compress (Spark's wrapStream)
            cks.append(oracle.checksum(alg, comp))       # upstream MutableCheckedOutputStream
            lens.append(len(comp))
            with w.getPartitionWriter(r) as s:
                for c in range(0, len(comp), 8 << 20):    # BufferedOutputStream(8 MiB) sized writes
                    s.write(comp[c:c + (8 << 20)])
        out_lens = w.commitAllPartitions(cks)
        assert list(out_lens) == lens
        # on-disk layout (SURVEY appendix A): path scheme, BE int64 cumulative index, BE int64 checksums
        root = str(tmp_path) + "/spark-s3-shuffle/"
        base = "%s%d/%s/0/shuffle_0_%d_0" % (root, m % 10, conf["spark.app.id"], m)
        assert d.getPath("data", 0, m) == base + ".data"
        assert open(base + ".index", "rb").read() == oracle.index_bytes(lens)
        assert open(base + ".checksum", "rb").read() == oracle.be64_bytes(cks)
        assert os.path.getsize(base + ".data") == sum(lens)
        assert list(host.S3ShuffleHelper.getPartitionLengths(d, 0, m)) == [0, lens[0], lens[0] + lens[1]]
        assert list(host.S3ShuffleHelper.getChecksums(d, 0, m)) == cks
        w.close()
    # reduce side: the oracle reads what the writer laid out; compare as multisets per reducer
    for r in range(n_red):
        got = oracle_read_partition(oracle, d, 0, range(n_maps), r, "ADLER32")
        gk = np.concatenate([decode_pairs(b)[0] for _, b in got])
        gv = np.concatenate([decode_pairs(b)[1] for _, b in got])
        ek = np.concatenate([e[0] for e in expect[r]])
        ev = np.concatenate([e[1] for e in expect[r]])
        assert gk.size == ek.size == n // n_red
        assert np.array_equal(np.sort(gv), np.sort(ev))
        assert np.array_equal(np.sort(gk * (1 << 32) + gv), np.sort(ek * (1 << 32) + ev))
        # groupByKey: 1000 keys over 2 reducers, every key has n/1000 values
        uk, cnt = np.unique(gk, return_counts=True)
        assert uk.size == 500 and (cnt == n // 1000).all()
    d.removeShuffle(0)
    assert not os.path.exists(os.path.dirname(d.getPath("data", 0, 0)))
    d.close()


def test_writer_preconditions_match_the_reference(tmp_path):
    d = host.S3ShuffleDispatcher(new_conf(tmp_path))
    w = host.S3ShuffleMapOutputWriter(d, 1, 3, 4)
    s = w.getPartitionWriter(1)
    s.write(b"abc")
    s.close()
    with pytest.raises(host.RuntimeException, match="monotonically increasing reducePartitionId"):
        w.getPartitionWriter(1)  # shuffle/S3ShuffleMapOutputWriter.scala:68-70
    with pytest.raises(host.RuntimeException, match="Invalid partition id"):
        w.getPartitionWriter(4)  # :71-73
    with pytest.raises(host.IOException, match="already closed"):
        s.write(b"x")            # :175-177
    lens = w.commitAllPartitions([0, 7, 0, 0])
    assert list(lens) == [0, 3, 0, 0]
    assert list(host.S3ShuffleHelper.getPartitionLengths(d, 1, 3)) == [0, 0, 3, 3, 3]
    w.close()
    d.close()


def test_empty_map_output_writes_no_index_unless_forced(tmp_path):
    d = host.S3ShuffleDispatcher(new_conf(tmp_path))
    w = host.S3ShuffleMapOutputWriter(d, 2, 0, 3)
    w.commitAllPartitions([1, 1, 1])
    assert not os.path.exists(d.getPath("index", 2, 0))  # shuffle/S3ShuffleMapOutputWriter.scala:111
    w.close()
    d2 = host.S3ShuffleDispatcher(new_conf(tmp_path, **{"spark.shuffle.s3.alwaysCreateIndex": True}))
    w = host.S3ShuffleMapOutputWriter(d2, 2, 1, 3)
    w.commitAllPartitions([1, 1, 1])
    assert os.path.getsize(d2.getPath("index", 2, 1)) == 4 * 8
    assert os.path.getsize(d2.getPath("checksum", 2, 1)) == 3 * 8
    w.close()
    d.close()
    d2.close()


def test_checksum_algorithm_factory(tmp_path):
    H = host.S3ShuffleHelper
    assert H.createChecksumAlgorithm("ADLER32") == 1 and H.createChecksumAlgorithm("CRC32") == 2
    assert H.createChecksumAlgorithm("CRC32C") == 3  # the case the shim adds (north-star)
    with pytest.raises(host.UnsupportedOperationException, match="Unsupported shuffle checksum algorithm"):
        H.createChecksumAlgorithm("MD5")  # helper/S3ShuffleHelper.scala:100-101


def test_bad_index_length_is_a_spark_exception(tmp_path):
    d = host.S3ShuffleDispatcher(new_conf(tmp_path, **{"spark.shuffle.s3.cachePartitionLengths": False}))
    p = d.getPath("index", 5, 0)
    os.makedirs(os.path.dirname(p))
    open(p, "wb").write(b"\0" * 13)
    with pytest.raises(host.SparkException, match="Unexpected file length"):
        host.S3ShuffleHelper.getPartitionLengths(d, 5, 0)  # helper/S3ShuffleHelper.scala:112-114
    d.close()


def test_folder_prefix_and_root_normalisation(tmp_path):
    d = host.S3ShuffleDispatcher(new_conf(tmp_path, **{"spark.shuffle.s3.folderPrefixes": 3,
                                                       "spark.app.id": "app-x"}))
    assert d.getPath("checksum", 7, 11).endswith("/spark-s3-shuffle/2/app-x/7/shuffle_7_11_0.checksum")
    d.close()


def test_gpu_mode_fails_loudly_without_a_device(tmp_path):
    """No CPU fallback above the C ABI either: with spark.shuffle.s3.gpu.enabled (default) a GPU-less commit raises."""
    try:
        import torch
        if torch.cuda.is_available():
            rerun_without_gpu(__file__, "test_gpu_mode_fails_loudly_without_a_device")
            return
    except ImportError:
        pass
    d = host.S3ShuffleDispatcher(new_conf(tmp_path, **{"spark.shuffle.s3.gpu.enabled": True}))
    w = host.S3ShuffleMapOutputWriter(d, 0, 0, 1)
    with w.getPartitionWriter(0) as s:
        s.write(b"hello world" * 100)
    with pytest.raises(host.CodecException):
        w.commitAllPartitions()
    w.close()
    d.close()


def test_group_commit_queue_fails_loudly_without_a_device(tmp_path):
    """the queue is plumbing over the C ABI: no GPU, no result (never a CPU path)"""
    import torch
    if torch.cuda.is_available():
        rerun_without_gpu(__file__, "test_group_commit_queue_fails_loudly_without_a_device")
        return
    d = host.S3ShuffleDispatcher(new_conf(tmp_path))
    with pytest.raises(host.CodecException):
        d.queueCompress(1, [b"abc" * 100], bound=lambda n: n + 64)
    assert d.queueStatistics()["batches"] == 0
    d.close()


def test_single_spill_transfer_moves_file_and_writes_metadata(tmp_path, oracle):
    """shuffle/S3SingleSpillShuffleMapOutputWriter.scala:24-64 — the spill file (already compressed + checksummed by
    Spark's UnsafeShuffleWriter, played by the oracle) becomes the .data object; .checksum and .index follow."""
    d = host.S3ShuffleDispatcher(new_conf(tmp_path, **{"spark.shuffle.checksum.algorithm": "CRC32"}))
    parts = [oracle.lz4block_compress(bytes([65 + r]) * (1000 * (r + 1)), 32768) for r in range(3)] + [b""]
    spill = tmp_path / "spill.bin"
    spill.write_bytes(b"".join(parts))
    lens = [len(p) for p in parts]
    cks = [oracle.crc32(p) for p in parts]
    host.S3SingleSpillShuffleMapOutputWriter(d, 4, 9).transferMapSpillFile(spill, lens, cks)
    assert not spill.exists()
    assert open(d.getPath("data", 4, 9), "rb").read() == b"".join(parts)
    assert open(d.getPath("index", 4, 9), "rb").read() == oracle.index_bytes(lens)
    assert open(d.getPath("checksum", 4, 9), "rb").read() == oracle.be64_bytes(cks)
    got = oracle_read_partition(oracle, d, 4, [9], 1, "CRC32")
    assert got[0][1] == b"B" * 2000
    d.close()

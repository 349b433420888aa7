"""Packed contact records (include/bbk.h, BbkRecHeader) written by libbbkio's bbkio_pack_records, decoded back by a numpy
restatement of the format, and validated by bbkio_check_records.  Host code only - these tests need no GPU."""
import numpy as np
import pytest

I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
CHUNK = 4096
HEADER = np.dtype([("magic", "<u4"), ("version", "<u4"), ("rows", "<i8"), ("bytes", "<u8"), ("reserved", "<u8")])
CHUNK_REC = np.dtype([("base", "<i8", 3), ("step", "<u8", 3), ("offset", "<u8"), ("bits", "u1", 3), ("reserved", "u1", 5)])


@pytest.fixture(scope="module")
def io():
    from blueberry_b200 import build, _io
    build.build_io()
    _io.load()
    return _io


def _layout(sizes):
    starts, off = [], 0
    for n in sizes:
        starts.append(off)
        off += (int(n) + 3) & ~3
    return starts, off


def _col_bytes(n, bits):
    return (n * bits + 127) // 128 * 16


def decode(buf, rows):
    """The format as bbk.h states it, in numpy: (mid1, mid2, count) int32 columns of `rows` rows."""
    buf = np.asarray(buf, dtype=np.uint8)
    h = np.frombuffer(buf[:HEADER.itemsize].tobytes(), dtype=HEADER)[0]
    assert h["magic"] == 0x31434552 and h["version"] == 1 and h["rows"] == rows
    nc = -(-rows // CHUNK)
    table = np.frombuffer(buf[32:32 + nc * 64].tobytes(), dtype=CHUNK_REC)
    out = [np.zeros(rows, dtype=np.int64) for _ in range(3)]
    for c in range(nc):
        t = table[c]
        r0 = c * CHUNK
        n = min(CHUNK, rows - r0)
        at = int(t["offset"])
        assert at % 16 == 0
        for j in range(3):
            b = int(t["bits"][j])
            nbytes = _col_bytes(n, b)
            words = np.frombuffer(buf[at:at + nbytes].tobytes(), dtype="<u8")
            at += nbytes
            u = np.zeros(n, dtype=object)
            if b:
                big = 0
                for k, w in enumerate(words.tolist()):
                    big |= int(w) << (64 * k)
                mask = (1 << b) - 1
                u = np.array([(big >> (i * b)) & mask for i in range(n)], dtype=object)
            v = int(t["base"][j]) + int(t["step"][j]) * u
            out[j][r0:r0 + n] = np.asarray(v, dtype=np.int64)
    mid1, e, count = out
    mid2 = mid1 + e
    for x in (mid1, mid2, count):
        assert x.min(initial=0) >= I32_MIN and x.max(initial=0) <= I32_MAX
    return mid1.astype(np.int32), mid2.astype(np.int32), count.astype(np.int32)


def pack(io, shards, threads=0, capacity=None):
    rows = _layout([len(s[0]) for s in shards])[1]
    bound = io.pack_records_bound(rows)
    out = np.full(bound if capacity is None else capacity, 0xAB, dtype=np.uint8)
    n = io.pack_records(shards, out.ctypes.data, out.size, threads)
    assert n <= bound
    return out[:n].copy(), rows


def expected(shards):
    starts, rows = _layout([len(s[0]) for s in shards])
    cols = [np.zeros(rows, dtype=np.int32) for _ in range(3)]
    for a, sh in zip(starts, shards):
        for j in range(3):
            cols[j][a:a + len(sh[j])] = sh[j]
    return cols


def roundtrip(io, shards):
    buf, rows = pack(io, shards)
    io.check_records(buf.ctypes.data, buf.size, rows)
    got = decode(buf, rows)
    for g, w in zip(got, expected(shards)):
        np.testing.assert_array_equal(g, w)
    return buf, rows


def _row_major(n, R=5000, K=2000, seed=0):
    rng = np.random.default_rng(seed)
    i = np.arange(n, dtype=np.int64)
    mid1 = (i // (K + 1)) * R + R // 2
    mid2 = mid1 + (i % (K + 1)) * R
    return mid1.astype(np.int32), mid2.astype(np.int32), rng.poisson(3.0, n).astype(np.int32)


@pytest.mark.parametrize("n", [0, 1, 3, 4095, 4096, 4097, 3 * 4096 + 5])
def test_roundtrip_row_major_sizes(io, n):
    roundtrip(io, [_row_major(n, seed=n)])


def test_roundtrip_several_shards_with_padding_and_an_empty_shard(io):
    shards = [_row_major(n, seed=k) for k, n in enumerate([5, 0, 4093, 1, 6000, 3])]
    buf, rows = roundtrip(io, shards)
    assert rows == _layout([5, 0, 4093, 1, 6000, 3])[1]


def test_roundtrip_extreme_values(io):
    n = 5000
    z = np.zeros(n, dtype=np.int32)
    cases = [
        (z, z, z),                                                              # constant: 0 bits everywhere
        (np.full(n, 7, np.int32), np.full(n, -3, np.int32), np.full(n, I32_MAX, np.int32)),
        (np.full(n, I32_MIN, np.int32), np.full(n, I32_MAX, np.int32), np.full(n, I32_MIN, np.int32)),   # e = 2^32 - 1
        (np.full(n, I32_MAX, np.int32), np.full(n, I32_MIN, np.int32), np.full(n, I32_MAX, np.int32)),   # e = -(2^32 - 1)
    ]
    m1 = np.resize(np.array([I32_MIN, I32_MAX, 0, 0], np.int32), n)
    m2 = np.resize(np.array([I32_MAX, I32_MIN, 0, 1], np.int32), n)
    cases.append((m1, m2, m1))                              # e in {2^32 - 1, -(2^32 - 1), 0, 1}: span 2^33 - 2, step 1, 33 bits
    rng = np.random.default_rng(1)
    full = lambda: rng.integers(I32_MIN, I32_MAX, n, endpoint=True, dtype=np.int64).astype(np.int32)
    cases.append((full(), full(), full()))                                      # random full range, mid2 < mid1 often
    cases.append((full(), full() // 7 * 7, np.abs(full()) // 1000))
    for sh in cases:
        buf, rows = roundtrip(io, [sh])
        table = np.frombuffer(buf[32:32 + 64].tobytes(), dtype=CHUNK_REC)
        assert table["bits"].max() <= 33
    # the alternating case needs the 33-bit e
    buf, _ = pack(io, [cases[4]])
    assert np.frombuffer(buf[32:96].tobytes(), dtype=CHUNK_REC)[0]["bits"][1] == 33


def test_bytes_do_not_depend_on_the_thread_count(io):
    rng = np.random.default_rng(5)
    shards = [_row_major(70_000, seed=1), _row_major(3, seed=2), _row_major(50_001, seed=3)]
    shards.append(tuple(rng.integers(I32_MIN, I32_MAX, 9000, endpoint=True, dtype=np.int64).astype(np.int32) for _ in range(3)))
    one, _ = pack(io, shards, threads=1)
    for t in (0, 3, 64):
        other, _ = pack(io, shards, threads=t)
        assert one.tobytes() == other.tobytes()


def test_never_exceeds_the_bound_and_a_short_capacity_fails(io):
    rng = np.random.default_rng(9)
    for n in (1, 4096, 10_001):
        sh = tuple(rng.integers(I32_MIN, I32_MAX, n, endpoint=True, dtype=np.int64).astype(np.int32) for _ in range(3))
        buf, rows = pack(io, [sh])
        assert buf.size <= io.pack_records_bound(rows)
        with pytest.raises(ValueError):
            pack(io, [sh], capacity=buf.size - 16)


def test_check_rejects_malformed_buffers(io):
    buf, rows = roundtrip(io, [_row_major(3 * 4096 + 5)])

    def check(b, nbytes=None, r=rows):
        io.check_records(b.ctypes.data, b.size if nbytes is None else nbytes, r)

    check(buf)
    with pytest.raises(ValueError):                     # truncated
        check(buf, buf.size - 1)
    with pytest.raises(ValueError):                     # shorter than the header
        check(buf, 16)
    with pytest.raises(ValueError):                     # other row count
        check(buf, r=rows + 4)
    bad = buf.copy()
    bad[0] ^= 0xFF                                      # bad magic
    with pytest.raises(ValueError):
        check(bad)
    bad = buf.copy()
    tab = bad[32:32 + 4 * 64].view(CHUNK_REC)
    tab[3]["offset"] = buf.size + 4096                  # offset past the end
    with pytest.raises(ValueError):
        check(bad)
    bad = buf.copy()
    tab = bad[32:32 + 4 * 64].view(CHUNK_REC)
    tab[1]["offset"] = tab[0]["offset"]                 # offsets not increasing
    with pytest.raises(ValueError):
        check(bad)
    bad = buf.copy()
    tab = bad[32:32 + 4 * 64].view(CHUNK_REC)
    tab[2]["bits"][1] = 34                              # bits > 33
    with pytest.raises(ValueError):
        check(bad)
    bad = buf.copy()
    tab = bad[32:32 + 4 * 64].view(CHUNK_REC)
    tab[2]["bits"][0] = 33                              # 33 bits only for e
    with pytest.raises(ValueError):
        check(bad)


def test_cfg3_like_records_pack_to_at_most_3_2_bytes_per_row(io):
    """BASELINE config 3's count model (5 kb, 10 Mb cap, depth 450) on chr21, zeros kept: the compression the format is for."""
    from blueberry_b200 import synth
    nb = synth.n_bins_of(synth.HG19_LENGTHS[20], 5000)
    b = synth.make_bias([nb], 3)
    c = synth.make_contacts([nb], 5000, 10_000_000, 450.0, 7, b, keep_zeros=True)
    sh = (c["mid1"], c["mid2"], c["count"])
    buf, rows = pack(io, [sh])
    io.check_records(buf.ctypes.data, buf.size, rows)
    assert buf.size / c["mid1"].size <= 3.2
    # the decoder restatement on a few chunks of it (the whole table would take minutes in Python ints)
    part = tuple(x[:3 * 4096 + 17] for x in sh)
    roundtrip(io, [part])

"""CPU: `bench.py --dump-outputs` -- the sample of the last timed solve's fields is float32, the same seeded nodes for
every source and every run, and stays under 64 MB at config 3's size."""
import numpy as np

import bench


class _FakeContext:
    def __init__(self, fields):
        self.fields = fields

    def get_tt(self, s, out):
        out[...] = self.fields[s]
        return out


def test_dump_is_a_fixed_float32_node_sample_of_every_source(tmp_path):
    dims = (9, 7, 5)
    rng = np.random.default_rng(3)
    fields = rng.random((3,) + dims, dtype=np.float32)
    bench.dump_outputs(_FakeContext(fields), 3, dims, tmp_path / "a", "tt")
    bench.dump_outputs(_FakeContext(fields), 3, dims, tmp_path / "b", "tt")
    a = np.load(tmp_path / "a" / "tt.npy")
    assert a.dtype == np.float32 and a.shape == (3, 9 * 7 * 5)   # a box smaller than the sample is dumped whole
    assert np.array_equal(a, np.load(tmp_path / "b" / "tt.npy"))
    assert np.array_equal(a, fields.reshape(3, -1))


def test_dump_of_config3_samples_the_seeded_nodes_and_fits_in_64_mb(tmp_path):
    dims = bench.DIMS
    n = int(np.prod(dims))                                   # < 2**24: every flat index is exact in float32
    node = np.arange(n, dtype=np.float32).reshape(dims)
    bench.dump_outputs(_FakeContext(np.stack([node, -node])), 2, dims, tmp_path, "tt")
    got = np.load(tmp_path / "tt.npy")
    want = np.sort(np.random.default_rng(0).choice(n, size=bench.DUMP_NODES, replace=False))
    assert got.shape == (2, bench.DUMP_NODES) and got.dtype == np.float32
    assert np.array_equal(got[0], want.astype(np.float32))   # distinct, sorted, seeded node indices ...
    assert np.array_equal(got[1], -got[0])                   # ... and the same ones for every source
    assert 111 * got[0].nbytes <= 64 << 20

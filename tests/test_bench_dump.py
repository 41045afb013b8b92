"""bench.py --dump-outputs: the sample it writes is the timed encode's parity rows and digests of the named blocks, as float32
.npy files that stay under 64 MB for any --blocks; the same arguments select the same blocks."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_sample(tmp_path):
    nblocks = 40
    pitch = (bench.S + 15) // 16 * 16
    g = torch.Generator().manual_seed(3)
    par = torch.randint(0, 256, (nblocks * bench.M, pitch), dtype=torch.uint8, generator=g)
    dig = torch.randint(0, 256, (nblocks, bench.K + bench.M, 32), dtype=torch.uint8, generator=g)
    bench.dump_outputs(str(tmp_path / "a"), par, dig, nblocks)
    bench.dump_outputs(str(tmp_path / "b"), par, dig, nblocks)
    load = lambda run, name: np.load(os.path.join(tmp_path, run, name + ".npy"))
    names = ("parity", "digests", "parity_blocks", "digest_blocks")
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in names)
    for name in names:
        assert load("a", name).dtype in (np.float32, np.float64)
        assert np.array_equal(load("a", name), load("b", name))
    pb, db = load("a", "parity_blocks").astype(np.int64), load("a", "digest_blocks").astype(np.int64)
    assert len(pb) == bench.DUMP_PARITY_BLOCKS and len(set(pb)) == len(pb) and np.array_equal(db, np.arange(nblocks))
    want = par.view(nblocks, bench.M, pitch)[torch.from_numpy(pb)][:, :, :bench.S]
    assert np.array_equal(load("a", "parity"), want.float().numpy())
    assert np.array_equal(load("a", "digests"), dig.float().numpy())
    largest = 4 * (bench.DUMP_PARITY_BLOCKS * bench.M * bench.S + bench.DUMP_DIGEST_BLOCKS * (bench.K + bench.M) * 32)
    assert largest + 8 * (bench.DUMP_PARITY_BLOCKS + bench.DUMP_DIGEST_BLOCKS) < 64 * 10 ** 6

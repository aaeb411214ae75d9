"""python -m mapper_b200 on several devices, without a device: the --device list, and the batch dispatcher (map_batches) driven with
stand-in handles that finish out of order or fail."""
import random
import threading
import time

import numpy as np
import pytest

from mapper_b200 import __main__ as cli


@pytest.mark.parametrize("text,want", [("0", [0]), ("3", [3]), ("0,1", [0, 1]), ("2,0,1,7", [2, 0, 1, 7])])
def test_device_list(text, want):
    assert cli.parse_args(["--reference", "r.fa", "--queries", "q.fq", "--device", text]).device == want


def test_device_default():
    assert cli.parse_args(["--reference", "r.fa", "--queries", "q.fq"]).device == [0]


@pytest.mark.parametrize("text", ["0,0", "1,2,1", "-1", "0,-2", "x", "0,", ",1", "1.5", "0;1", ""])
def test_device_list_rejected(text, capsys):
    with pytest.raises(SystemExit) as e:
        cli.parse_args(["--reference", "r.fa", "--queries", "q.fq", "--device", text])
    assert e.value.code == 2
    assert "--device" in capsys.readouterr().err


class FakeHandle:
    """Records what the dispatcher asks of it; align_batch_sam sleeps a random while, so that devices finish out of order."""

    def __init__(self, rank, fail_at=None, seed=0):
        self.rank, self.fail_at, self.rng = rank, fail_at, random.Random(seed)
        self.infos, self.batches, self.collectives = [], [], []

    def counts_batch_info(self, first, keys):
        self.infos.append((first, np.asarray(keys).copy()))

    def align_batch_sam(self, batch, names, contig_names, strict=False):
        time.sleep(self.rng.random() * 0.01)
        tag = bytes(names[0][:names[1][1]]).decode()
        if tag == self.fail_at:
            q_status = np.zeros(len(batch["n_seqs"]), np.int32)
            q_status[0] = 3
            return dict(q_status=q_status, stats=np.zeros(32, np.int64)), ""
        self.batches.append(tag)
        stats = np.zeros(32, np.int64)
        stats[0] = 1000
        return dict(q_status=np.zeros(len(batch["n_seqs"]), np.int32), stats=stats), "sam of %s\n" % tag

    def comm_unique_id(self):
        self.collectives.append("uid")
        return bytes(128)

    def comm_init(self, n, rank, uid):
        self.collectives.append("comm_init")

    def counts_reduce(self):
        self.collectives.append("counts_reduce")


def fake_batches(sizes, per_query=1):
    """Array dicts as query_batches yields them: batch k has sizes[k] sequences named b<k>s<i>."""
    for k, n in enumerate(sizes):
        names = [b"b%ds%d" % (k, i) for i in range(n)]
        off = np.zeros(n + 1, np.int64)
        off[1:] = np.cumsum([len(x) for x in names])
        yield dict(packed=np.zeros(n, np.uint16), seq_word_off=np.arange(n + 1, dtype=np.int64), seq_len=np.full(n, 4, np.int32),
                   names=b"".join(names), name_off=off), per_query


def run(n_dev, sizes, ranks, fail=None, reduce=True, per_query=1):
    hs = [FakeHandle(d, fail_at=fail, seed=d) for d in range(n_dev)]
    out = []
    res = cli.map_batches(hs, fake_batches(sizes, per_query), ranks, (0.0, 1.0), (b"c", np.array([0, 1], np.int64)), out.append, reduce=reduce)
    return hs, out, res


@pytest.mark.parametrize("n_dev", [2, 3, 4])
def test_dispatch_order_and_ids(n_dev):
    sizes = [5, 3, 8, 1, 6, 4, 7, 2, 9, 3, 5, 4]
    ranks = np.random.default_rng(1).permutation(sum(sizes)).astype(np.int64)
    one, out1, res1 = run(1, sizes, ranks)
    hs, out, res = run(n_dev, sizes, ranks)
    assert out == out1 == ["sam of b%ds0\n" % k for k in range(len(sizes))]
    assert res[:2] == res1[:2] == (sum(sizes), len(sizes))
    assert res[2] == [1000 * len(h.batches) for h in hs]
    for d, h in enumerate(hs):
        assert h.batches == ["b%ds0" % k for k in range(d, len(sizes), n_dev)]
        want = one[0].infos[d::n_dev]
        assert [f for f, _ in h.infos] == [f for f, _ in want]
        for (_, a), (_, b) in zip(h.infos, want):
            assert np.array_equal(a, b)
        assert h.collectives == (["uid"] if d == 0 else []) + ["comm_init", "counts_reduce"]
    firsts = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    assert [f for f, _ in one[0].infos] == list(firsts)
    assert all(np.array_equal(k, ranks[f:f + n]) for (f, k), n in zip(one[0].infos, sizes))


def test_dispatch_without_counts():
    hs, out, _ = run(2, [3, 4, 5], None, reduce=False)
    assert len(out) == 3 and all(h.infos == [] and h.collectives == [] for h in hs)


@pytest.mark.parametrize("n_dev,fail", [(1, 0), (2, 0), (2, 5), (3, 7), (4, 11)])
def test_worker_failure(n_dev, fail):
    before = threading.active_count()
    sizes = [4] * 12
    hs = [FakeHandle(d, fail_at="b%ds0" % fail, seed=d) for d in range(n_dev)]
    out = []
    with pytest.raises(SystemExit) as e:
        cli.map_batches(hs, fake_batches(sizes), np.arange(48, dtype=np.int64), (0.0, 1.0), (b"c", np.array([0, 1], np.int64)), out.append, reduce=True)
    assert "query 'b%ds0' could not be aligned on the device (status 3)" % fail in str(e.value)
    assert out == ["sam of b%ds0\n" % k for k in range(len(out))] and len(out) <= fail
    assert all(h.collectives == [] for h in hs)
    assert threading.active_count() == before


def test_producer_failure_stops_dispatch():
    before = threading.active_count()

    def batches():
        yield from fake_batches([3, 3, 3])
        raise SystemExit("r2.fq has fewer records than r1.fq")
    hs = [FakeHandle(d) for d in range(2)]
    with pytest.raises(SystemExit, match="fewer records"):
        cli.map_batches(hs, cli.prefetch(batches()), None, (0.0, 1.0), (b"c", np.array([0, 1], np.int64)), lambda t: None, reduce=True)
    assert all(h.collectives == [] for h in hs)
    assert threading.active_count() == before


def test_prefetch_closed_early_joins_its_thread():
    before = threading.active_count()
    gen = cli.prefetch(iter(range(100)))
    assert next(gen) == 0
    gen.close()
    assert threading.active_count() == before

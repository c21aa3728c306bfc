"""Host logic of data-parallel ``train_mm.py`` (torchrun): how an epoch's batches are dealt to the ranks (accelerate's
BatchSamplerShard, split_batches=False, even_batches=True), how the test pass is split and put back into the one-GPU order,
and that without WORLD_SIZE nothing distributed is set up."""
import pytest


def test_deal_batches_world_one_is_the_batch_list():
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import deal_batches
    assert deal_batches(5, 1) == [[0], [1], [2], [3], [4]]
    assert deal_batches(0, 1) == []


def test_deal_batches_world_divides_the_count():
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import deal_batches
    assert deal_batches(6, 2) == [[0, 1], [2, 3], [4, 5]]
    assert deal_batches(8, 4) == [[0, 1, 2, 3], [4, 5, 6, 7]]
    for n, w in ((12, 3), (16, 8), (30, 5)):
        dealt = deal_batches(n, w)
        assert len(dealt) == n // w and sorted(b for step in dealt for b in step) == list(range(n))
        assert all(step[r] == s * w + r for s, step in enumerate(dealt) for r in range(w))


def test_deal_batches_fills_the_last_round_from_the_start():
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import deal_batches
    assert deal_batches(5, 2) == [[0, 1], [2, 3], [4, 0]]
    assert deal_batches(7, 4) == [[0, 1, 2, 3], [4, 5, 6, 0]]
    assert deal_batches(3, 8) == [[0, 1, 2, 0, 1, 2, 0, 1]]      # fewer batches than ranks: the list is cycled
    for n, w in ((9, 4), (31, 8), (4, 3)):
        dealt = deal_batches(n, w)
        flat = [b for step in dealt for b in step]
        assert len(dealt) == -(-n // w) and flat[:n] == list(range(n)) and flat[n:] == [i % n for i in range(len(flat) - n)]


@pytest.mark.parametrize("n,world", [(1, 2), (5, 2), (6, 2), (7, 3), (2, 4), (13, 4), (31, 8), (0, 2)])
def test_test_shards_gather_back_into_the_one_gpu_order(n, world):
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import restore_order, shard_test_batches
    shards = [shard_test_batches(n, r, world) for r in range(world)]
    assert sorted(i for s in shards for i in s) == list(range(n))
    assert all(s == list(range(r, n, world)) for r, s in enumerate(shards))
    per_rank = [[("batch", i) for i in s] for s in shards]        # what each rank computes, in its own order
    assert restore_order(per_rank) == [("batch", i) for i in range(n)]
    assert shard_test_batches(n, 0, 1) == list(range(n)) and restore_order([list(range(n))]) == list(range(n))


def test_without_world_size_nothing_distributed_is_set_up(monkeypatch):
    import torch.distributed as dist
    import erc_b200  # noqa: F401
    from erc_b200 import train_mm
    args = train_mm.parse_args(["--module=dgcn", "--device=3", "--train.batch_size=8"])

    def refuse(*a, **k):
        raise AssertionError("init_process_group called without WORLD_SIZE > 1")
    monkeypatch.setattr(dist, "init_process_group", refuse)
    for env in (None, "1"):
        if env is None:
            monkeypatch.delenv("WORLD_SIZE", raising=False)
        else:
            monkeypatch.setenv("WORLD_SIZE", env)
        p = train_mm.resolve_params(args)
        want = dict(p)
        lines = []
        assert train_mm.init_distributed(p, log=lines.append) == (0, 1)
        assert p == want and p["device"] == 3 and p["batch_size"] == 8 and not lines


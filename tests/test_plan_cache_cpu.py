"""The host-side shape policy (PlanCache) and grow-only workspaces (WorkspacePool) shared by the encoder engine, the
fused head and training, driven with fake plans and CPU buffers."""
from collections import Counter

import torch

from auto_avsr_b200._cache import PlanCache, WorkspacePool


class Fakes:
    def __init__(self):
        self.built, self.destroyed = [], Counter()

    def builder(self, key):
        def build():
            rec = ("plan", key, len(self.built))
            self.built.append(rec)
            return rec
        return build

    def destroy(self, rec):
        self.destroyed[rec] += 1


def test_no_build_before_the_graph_after_th_sighting():
    f = Fakes()
    cache = PlanCache(f.destroy, graph_after=3, max_plans=4)
    assert cache.get("a", f.builder("a")) is None
    assert cache.get("a", f.builder("a")) is None
    assert f.built == [] and len(cache) == 0
    rec = cache.get("a", f.builder("a"))
    assert f.built == [rec] and len(cache) == 1
    assert cache.get("a", f.builder("a")) is rec and len(f.built) == 1
    cache.graph_after = 1                                 # assignable: later keys capture at first sight
    assert cache.get("b", f.builder("b")) is not None and len(f.built) == 2

    f = Fakes()
    cache = PlanCache(f.destroy, graph_after=1, max_plans=4)
    rec = cache.get("a", f.builder("a"))
    assert f.built == [rec] and cache.get("a", f.builder("a")) is rec


def test_hits_refresh_recency_and_eviction_is_lru_with_one_destroy_each():
    f = Fakes()
    cache = PlanCache(f.destroy, graph_after=1, max_plans=2)
    a = cache.get("a", f.builder("a"))
    b = cache.get("b", f.builder("b"))
    assert cache.get("a", f.builder("a")) is a            # hit: "a" becomes the most recently used
    c = cache.get("c", f.builder("c"))
    assert f.destroyed == Counter({b: 1}) and len(cache) == 2
    assert cache.get("a", f.builder("a")) is a and cache.get("c", f.builder("c")) is c
    d = cache.get("d", f.builder("d"))                    # "a" is now the least recently used
    assert f.destroyed == Counter({b: 1, a: 1})
    cache.clear()
    assert len(cache) == 0 and f.destroyed == Counter({a: 1, b: 1, c: 1, d: 1})
    cache.clear()
    assert sum(f.destroyed.values()) == 4
    b2 = cache.get("b", f.builder("b"))                   # an evicted key that comes back is built again
    assert b2 is not b and len(f.built) == 5


def test_sighting_table_stays_bounded_under_distinct_keys():
    f = Fakes()
    cache = PlanCache(f.destroy, graph_after=3, max_plans=4)
    for T in range(10_000):                               # B = 1, a new T per utterance
        assert cache.get((1, T), f.builder((1, T))) is None
        assert len(cache._seen) <= 64 * 4
    assert len(cache._seen) == 64 * 4 and f.built == []
    for _ in range(2):                                    # a recent key keeps its sightings
        cache.get((1, 9_999), f.builder((1, 9_999)))
    assert len(f.built) == 1


def test_workspace_pool_one_grow_only_buffer_per_tag_device_stream():
    pool = WorkspacePool()
    cpu = torch.device("cpu")
    ws = pool.get("direct", 1000, cpu, 7)
    assert ws.dtype == torch.uint8 and ws.numel() >= 1000 and len(pool) == 1
    for n in (1000, 10, 1, ws.numel()):                   # smaller or equal requests reuse the buffer
        assert pool.get("direct", n, cpu, 7) is ws
    assert len(pool) == 1
    other = [pool.get("direct", 1000, cpu, 8), pool.get("proj", 1000, cpu, 7)]
    assert len(pool) == 3 and all(o is not ws for o in other)
    big = pool.get("direct", ws.numel() + 1, cpu, 7)
    assert big is not ws and big.numel() >= ws.numel() + 1 and len(pool) == 3
    assert pool.get("direct", 1000, cpu, 7) is big
    for n in (0, 1, 255, 4097, 10**6):
        assert pool.get("sizes", n, cpu, 0).numel() >= n

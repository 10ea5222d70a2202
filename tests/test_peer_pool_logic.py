"""CPU tests of the peer-mapped background pool's host logic: the segments of one gather (pool.peer_segments) and the
refusals PeerPool.open decides from the gathered metadata (pool.check_peer_meta)."""
import numpy as np
import pytest


def _index(rng, counts):
    owner = np.concatenate([np.full(c, r, np.int64) for r, c in enumerate(counts)])
    slot = np.concatenate([np.arange(c, dtype=np.int64) for c in counts])
    h, w = rng.integers(1, 40, owner.size), rng.integers(1, 40, owner.size)
    nbytes = 3 * h * w
    # every owner's buffer laid out as RaggedPool.append does: 16-byte aligned, images back to back
    offsets = []
    for r, c in enumerate(counts):
        sizes = nbytes[owner == r]
        offsets.append(np.concatenate([[0], np.cumsum((sizes + 15) & ~15)[:-1]]).astype(np.int64) if c else np.zeros(0, np.int64))
    src_offset = np.array([offsets[o][s] for o, s in zip(owner, slot)], dtype=np.int64)
    return owner, slot, h, w, nbytes, offsets, src_offset


@pytest.mark.parametrize("counts", [[5, 3], [4, 0, 7], [1, 1, 1, 9], [6]])
def test_peer_segments_read_each_owner_in_request_order(counts):
    """Every image lands at a 16-byte aligned offset, in request order, back to back; each segment reads 3*h*w bytes from the
    owner's base at the owner's slot offset."""
    from bgdebias_b200.pool import ShardedPool, peer_segments
    rng = np.random.default_rng(sum(counts) * 31 + len(counts))
    owner, slot, h, w, nbytes, offsets, src_offset = _index(rng, counts)
    P = owner.size
    idx = rng.integers(0, P, 24)
    app = (rng.random(24) < 0.6).astype(np.uint8)
    requests = ShardedPool.requests_of(idx, app)
    assert requests == list(dict.fromkeys(int(g) for g, a in zip(idx, app) if a))
    seg, dst, total = peer_segments(requests, owner, src_offset, nbytes)
    assert seg.dtype == np.int64 and seg.shape == (len(requests), 4)
    at = 0
    for k, g in enumerate(requests):
        r, so, do, b = seg[k].tolist()
        assert r == owner[g] and so == offsets[r][slot[g]] and b == 3 * h[g] * w[g]
        assert do == dst[k] == at and do % 16 == 0 and so % 16 == 0
        at += (b + 15) & ~15
    assert total == at
    # a batch that mixes nothing: no segment, an empty buffer
    seg0, dst0, total0 = peer_segments([], owner, src_offset, nbytes)
    assert seg0.shape == (0, 4) and dst0.size == 0 and total0 == 0


def _meta(host="node0/boot", handle=b"\x01" * 64, offset=0, error=None):
    return dict(host=host, uuid="GPU-x", handle=handle, offset=offset, bytes=4096 if handle else 0, error=error,
                offsets=np.zeros(0, np.int64))


def test_open_refuses_mismatched_hosts_and_unexportable_buffers():
    from bgdebias_b200.pool import check_peer_meta
    check_peer_meta([_meta(), _meta(handle=None), _meta(offset=512)])             # one node, an empty shard: accepted
    with pytest.raises(ValueError, match="different hosts.*attach_sharded_pool"):
        check_peer_meta([_meta(), _meta(), _meta(host="node1/boot")])
    with pytest.raises(ValueError, match="rank 1 cannot export.*expandable_segments.*attach_sharded_pool"):
        check_peer_meta([_meta(), _meta(handle=None, error="the allocation cannot be exported (expandable_segments)")])
    with pytest.raises(ValueError, match="unaligned"):
        check_peer_meta([_meta(), _meta(offset=8)])

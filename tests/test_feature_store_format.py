"""The compact feature-store format (include/graphpope_b200.h, gp_fstore_*) restated in numpy, and checked against
the C oracle: a store is uint64 [N, P, W], W = ceil(K/64); plane 0 is the reached mask, plane 1 + q bit q of the hop
count; column j is word j >> 6, bit j & 63; P = 1 + bit_length(max hop); padding and unreached hop bits are zero.
Decoding must give exactly the float32 values of the dense path (cbfs.normalise)."""
import numpy as np
import pytest

from conftest import DEEP_HUB_NAMES, micro_names

UNREACHED = 0xFFFF


def num_planes(hops: np.ndarray) -> int:
    reached = hops[hops != UNREACHED]
    return 1 + (int(reached.max()) if reached.size else 0).bit_length()


def _bits(store: np.ndarray) -> np.ndarray:
    """bool [N, P, 64 W]: bit j of every plane (little-endian words, so byte j >> 3, bit j & 7)."""
    n, p, w = store.shape
    raw = np.ascontiguousarray(store, dtype="<u8").view(np.uint8).reshape(n, p, w * 8)
    return np.unpackbits(raw, axis=-1, bitorder="little").astype(bool)


def encode(hops: np.ndarray) -> np.ndarray:
    """uint16 [N, K] hop matrix (0xFFFF = unreachable) -> uint64 [N, P, W] store."""
    n, k = hops.shape
    p, w = num_planes(hops), -(-k // 64)
    reached = hops != UNREACHED
    d = np.where(reached, hops, 0).astype(np.uint32)
    bits = np.zeros((n, p, 64 * w), dtype=bool)
    bits[:, 0, :k] = reached
    for q in range(p - 1):
        bits[:, 1 + q, :k] = (d >> q) & 1
    return np.ascontiguousarray(np.packbits(bits, axis=-1, bitorder="little")).view("<u8").reshape(n, p, w)


def decode(store: np.ndarray, k: int) -> np.ndarray:
    """uint64 [N, P, W] store -> float32 [N, K]: 1/(d+1) in IEEE fp32 where reached, else 0."""
    bits = _bits(store)[:, :, :k]
    d = np.zeros(bits.shape[::2], dtype=np.uint32)
    for q in range(store.shape[1] - 1):
        d |= bits[:, 1 + q].astype(np.uint32) << q
    inv = np.float32(1.0) / (d + 1).astype(np.float32)
    return np.where(bits[:, 0], inv, np.float32(0.0)).astype(np.float32)


def assert_round_trip(hops: np.ndarray):
    from oracle import cbfs

    n, k = hops.shape
    store = encode(hops)
    assert store.dtype == np.uint64 and store.shape == (n, num_planes(hops), -(-k // 64))
    bits = _bits(store)
    assert not bits[:, :, k:].any(), "padding past K must be zero"
    assert not bits[:, 1:, :k][np.broadcast_to((hops == UNREACHED)[:, None, :], bits[:, 1:, :k].shape)].any(), \
        "hop bits of unreached lanes must be zero"
    want = cbfs.normalise(hops)
    assert np.array_equal(decode(store, k).view(np.uint32), want.view(np.uint32))
    return store


def _oracle_hops(ei, n, anchors):
    from oracle import cbfs

    return cbfs.bfs_hops(cbfs.InCsr(ei, n), anchors)


def test_micro_graphs_round_trip(golden_small):
    for name in micro_names(golden_small):
        g = lambda key: golden_small[f"micro/{name}/{key}"]  # noqa: E731
        hops = _oracle_hops(g("edges"), int(g("n")), g("anchors"))
        assert_round_trip(hops)
        want = g("rows_f64").astype(np.float32)  # what the unmodified reference returned
        assert np.array_equal(decode(encode(hops), hops.shape[1]), want), name


@pytest.mark.parametrize("name", DEEP_HUB_NAMES)
def test_deep_and_hub_graphs_round_trip(golden_deep_hub, name):
    g = golden_deep_hub
    hops = _oracle_hops(g[f"{name}/edge_index"], int(g[f"{name}/n"]), g[f"{name}/anchors"])
    store = assert_round_trip(hops)
    assert np.array_equal(decode(store, hops.shape[1]).view(np.uint32), g[f"{name}/embedding"].view(np.uint32))
    if name == "deep_chain":
        assert int(hops[hops != UNREACHED].max()) == 4999 and store.shape[1] == 14


@pytest.mark.parametrize("k", [0, 1, 2, 8, 63, 64, 65, 257])
@pytest.mark.parametrize("max_hop", [0, 1, 15, 16, 300, 65534])
def test_every_width_and_depth(k, max_hop):
    rng = np.random.default_rng(k * 7 + max_hop)
    hops = rng.integers(0, max_hop + 1, size=(37, k)).astype(np.uint16)
    hops[rng.random((37, k)) < 0.3] = UNREACHED
    if k:
        hops[0, 0] = max_hop
    store = assert_round_trip(hops)
    assert store.shape[1] == 1 + (max_hop.bit_length() if k else 0)

#!/usr/bin/env python3
"""Mint tests/golden/ref_parity.npz and tests/golden/ref_etcd_listing.bin from the reference itself:
oracle/_ref/libxllm_ref.so (oracle/build_ref.sh compiles the reference's hash / index / routing files unmodified)
replays the seeded histories of tests/test_ref_parity.py and its answers are stored, so that test compares the
oracle with the reference without the reference's sources.

ref_parity.npz:
  xxh3_random          uint8 [n, 16]   hash_util.cpp's xxh3_128bits_hash for each test_ref_parity.xxh3_random_cases()
  hist<s>_n, hist<s>_sha256            per history of random_histories(seed s): how many answers GlobalKVCacheMgr +
                                       CacheAwareRouting gave, and the SHA-256 of those answers as little-endian int64
  replica_sizes        [round, 2]      master / replica map sizes after each upload of replica_history()
  replica_gets         [round, key, 2, 4]  master / replica (found, hbm, dram, ssd masks) of every key
  replica_final        [3, 4]          the replica's answers after a PUT + DELETE in one response, an unparsable
                                       value and a value with an extra member
ref_etcd_listing.bin (little endian; "bytes" = u32 length + data):
  u32 n_names, bytes name[n_names], u32 n_namespaces, then per namespace:
  bytes namespace, u32 n_pairs, then per pair: bytes etcd key, bytes etcd value, u64 hbm, dram, ssd masks over names

Run:  bash oracle/build_ref.sh && python tests/golden/make_ref_goldens.py   (needs the reference's sources)
"""
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

from oracle import oracle, ref  # noqa: E402
import test_ref_parity as t  # noqa: E402

WIRE_NAMES = ["10.0.0.1:8000", 'instance-"quoted"', "back\\slash", "tab\there", "nl\nname", "café",
              "日本", "sp ace", "/slash"] + ["instance-%d" % i for i in range(9, 40)]


def _bytes(b):
    return struct.pack("<I", len(b)) + b


def histories():
    out = {}
    for seed in range(t.N_SEEDS):
        answers, _, _ = t.random_histories(oracle, lambda names, bs: ref.RefIndex(names, bs, 1024), seed)
        out["hist%d_n" % seed] = np.array([a.size for a in answers], np.int64)
        out["hist%d_sha256" % seed] = np.array([np.frombuffer(t.digest(a), np.uint8) for a in answers])
    return out


def replica():
    keys, rounds = t.replica_history()
    M = ref.RefIndex(t.REPLICA_NAMES)
    Rp = ref.RefIndex(t.REPLICA_NAMES, master=False, share=M)
    sizes, gets = [], []
    for events in rounds:
        for ev in events:
            M.record(*ev)
        assert M.upload()
        sizes.append([M.size(), Rp.size()])
        gets.append([[[int(f)] + m for f, m in (M.get(k), Rp.get(k))] for k in keys])
    final = []
    Rp.batch(True)
    Rp.delete(keys[0])
    Rp.put(keys[0], hbm=["n1"])
    Rp.batch(False)
    final.append(Rp.get(keys[0]))
    Rp.put_raw(b"XLLM:CACHE:" + bytes(keys[1]), b"{not json")
    final.append(Rp.get(keys[1]))
    Rp.put_raw(b"XLLM:CACHE:" + bytes(keys[1]),
               b'{"ssd_instance_set":["n3"],"x":1,"hbm_instance_set":[],"dram_instance_set":["n2","n2"]}')
    final.append(Rp.get(keys[1]))
    return {"replica_sizes": np.array(sizes, np.int64), "replica_gets": np.array(gets, np.int64),
            "replica_final": np.array([[int(f)] + m for f, m in final], np.int64)}


def etcd_listing():
    """A random event history over 160 keys (embedded NULs included) and 40 names (escapes, UTF-8) on a reference
    master, four uploads, then the master's etcd store under the cache prefix, for the empty and a set namespace."""
    rng = np.random.default_rng(11)
    out = [struct.pack("<I", len(WIRE_NAMES))] + [_bytes(n.encode()) for n in WIRE_NAMES]
    namespaces = ["", "prod/cluster-a"]
    out.append(struct.pack("<I", len(namespaces)))
    for ns in namespaces:
        nsp = "/%s/" % ns if ns else ""    # utils.cpp:105-124
        R = ref.RefIndex(WIRE_NAMES, namespace=ns)
        keys = rng.integers(0, 256, (160, 16), dtype=np.uint8)
        keys[0, 3] = keys[1, 0] = keys[2, 15] = 0
        for _ in range(4):
            for _ in range(200):
                k = keys[int(rng.integers(0, 160))][None]
                n = WIRE_NAMES[int(rng.integers(0, len(WIRE_NAMES)))]
                what = int(rng.integers(0, 10))
                R.record(n, *((k, (), ()) if what < 6 else ((), k, ()) if what < 9 else ((), (), k)))
            assert R.upload()
        pairs = R.etcd_pairs((nsp + "XLLM:CACHE:").encode())
        assert len(pairs) == R.size() > 100
        out += [_bytes(ns.encode()), struct.pack("<I", len(pairs))]
        for k, v in pairs:
            found, m = R.get(k[-16:])
            assert found
            out += [_bytes(k), _bytes(v), struct.pack("<3Q", *m)]
    return b"".join(out)


def main():
    oracle.build()
    if not ref.available():
        sys.exit("oracle/_ref/libxllm_ref.so is not built: run oracle/build_ref.sh with the reference's sources")
    g = {"xxh3_random": np.array([np.frombuffer(ref.xxh3_128bits_hash(p, tk, s), np.uint8)
                                  for p, tk, s in t.xxh3_random_cases()])}
    g.update(histories())
    g.update(replica())
    np.savez_compressed(os.path.join(HERE, "ref_parity.npz"), **g)
    with open(os.path.join(HERE, "ref_etcd_listing.bin"), "wb") as f:
        f.write(etcd_listing())


if __name__ == "__main__":
    main()

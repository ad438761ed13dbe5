"""Rows a5-a8 / f1 / f3 pinned to the REFERENCE ITSELF.  tests/golden/ref_parity.npz and
tests/golden/ref_etcd_listing.bin hold what the reference's own hash_util.cpp, types.h, global_kvcache_mgr.cpp,
etcd_client.cpp, cache_aware_routing.cpp and InstanceMgr::get_load_metrics — compiled unmodified into
oracle/_ref/libxllm_ref.so by oracle/build_ref.sh, over an in-memory etcd — answered for the seeded histories below
(tests/golden/make_ref_goldens.py replays them on the reference and writes those files).  The restatement
(oracle/prefix_oracle.cc, oracle/xxh3_oracle.c) — which every GPU parity test compares the device against — must give
the same answers on the XXH3 known answers, on random block hashes, and on random event / upload / match / route
histories."""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(__file__)
GOLDEN = os.path.join(HERE, "golden", "ref_parity.npz")
LISTING = os.path.join(HERE, "golden", "ref_etcd_listing.bin")
N_SEEDS = 8


@pytest.fixture(scope="module")
def golden():
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def xxh3_random_cases():
    """(prev, tokens, seed) for every length the reference accepts (4n + 16 < 1024, hash_util.cpp:33), chained and
    unchained, three seeds."""
    rng = np.random.default_rng(5)
    for n in list(range(0, 252)) + [128] * 50:
        for seed in (1024, 0, 0xFFFFFFFF):
            t = rng.integers(-2**31, 2**31, size=n, dtype=np.int64).astype(np.int32)
            prev = bytes(rng.integers(0, 256, 16, dtype=np.uint8)) if rng.random() < 0.7 else None
            yield prev, t, seed


def test_xxh3_known_answers_and_random_blocks(oracle, golden):
    # SURVEY.md §8c KAT (libxxhash 0.8.2): tokens 0..255, block 128, seed 1024
    k = oracle.block_hash_chain(np.arange(256, dtype=np.int32), 128, 1024)
    assert bytes(k[0]).hex() == "a6c0e2fc92c32b1c1ccff29b710ca0d2"
    assert bytes(k[1]).hex() == "f981264b143b2d5f81fd86ed5d58d2a1"
    assert oracle.xxh3_128bits_hash(None, np.arange(16, dtype=np.int32), 1024).hex() == "1247ae96b541bccd1d2bea48ea0a97e4"
    # the chained golden vectors minted from libxxhash
    kat = json.load(open(os.path.join(HERE, "golden", "xxh3_kat.json")))
    for c in kat.get("chains", []):
        toks = np.array(c["tokens"], dtype=np.int32) if "tokens" in c else None
        if toks is None or 4 * c["block_size"] + 16 >= 1024:
            continue
        got = oracle.block_hash_chain(toks, c["block_size"], c["seed"])
        assert [bytes(x).hex() for x in got] == c["keys"]
    want = golden["xxh3_random"]
    n = 0
    for i, (prev, t, seed) in enumerate(xxh3_random_cases()):
        assert oracle.xxh3_128bits_hash(prev, t, seed) == bytes(want[i]), (t.size, seed)
        n += 1
    assert n == want.shape[0]


def _reference_survives(oracle, X, toks, bs):
    """GlobalKVCacheMgr::match dereferences hbm_instance_set.begin() inside its DRAM and SSD branches
    (global_kvcache_mgr.cpp:113-114,123-124): a matched block held only in DRAM / SSD is undefined behaviour there
    (a null-node read: the compiled reference segfaults).  Such requests can only be checked on the restatement."""
    for k in oracle.block_hash_chain(toks, bs, 1024):
        found, m = X.get(k)
        if not found or not any(m):
            return True
        if m[0] == 0:
            return False
    return True


def random_histories(oracle, make_index, seed):
    """Per seed: 150 independent histories x ~70 steps (~10 K operations): random KvCacheEvents
    (stored / offload / removed, several keys each) from random instances, uploads at random points, load-metric and
    schedulability changes, then match + route of prompts built to share prefixes with the indexed blocks.
    make_index(names, block_size) gives a fresh oracle.PrefixOracle or oracle.ref.RefIndex.  Returns one int64 array
    per history holding, in order, every answer the index gave: after each upload its size and the whole key
    universe's (found, hbm, dram, ssd masks); for each match every field; for each route ok and, when routed, the
    prefill and decode ids.  Also returns (operations, requests skipped as undefined behaviour in the reference)."""
    rng = np.random.default_rng(1000 + seed)
    n_ops = n_ub = 0
    answers = []
    for hist in range(150):
        obs = []
        n_inst = int(rng.integers(1, 13))
        names = ["inst-%d-%d" % (hist, i) for i in range(n_inst)]
        types = [int(rng.integers(0, 4)) for _ in names]
        bs = int(rng.choice([128, 16, 64, 251, 1]))
        X = make_index(names, bs)
        for n, t in zip(names, types):
            X.set_instance(n, t)
        # a few prompts; the key universe = their block keys + some foreign keys
        prompts = []
        for _ in range(4):
            nb = int(rng.integers(0, 9))
            tail = int(rng.integers(0, bs))
            prompts.append(rng.integers(0, 32000, nb * bs + tail).astype(np.int32))
        prompts.append(np.concatenate([prompts[0][:2 * bs], rng.integers(0, 32000, 3 * bs).astype(np.int32)]))
        universe = [oracle.block_hash_chain(p, bs, 1024) for p in prompts]
        universe = np.concatenate(universe + [rng.integers(0, 256, (4, 16), dtype=np.uint8)])
        for n in names:
            if rng.random() < 0.85:
                w, u = int(rng.integers(0, 6)), float(np.float32(rng.choice([0.0, 0.25, 0.5, 0.99, 1.0, rng.random()])))
                X.set_load(n, w, u)
        for step in range(int(rng.integers(40, 100))):
            op = rng.random()
            n_ops += 1
            if op < 0.45 and len(universe):
                name = names[int(rng.integers(0, n_inst))]
                pick = lambda: universe[rng.integers(0, len(universe), int(rng.integers(0, 5)))]
                kind = rng.random()
                s = pick() if kind < 0.6 else ()
                o = pick() if 0.4 < kind < 0.9 else ()
                r = pick() if kind > 0.8 else ()
                X.record(name, s, o, r)
            elif op < 0.6:
                assert X.upload() is not False
                obs.append(X.size())
                for k in universe:
                    found, m = X.get(k)
                    obs += [int(found)] + m
            elif op < 0.7:
                n = names[int(rng.integers(0, n_inst))]
                if rng.random() < 0.3:
                    X.clear_load(n)
                elif rng.random() < 0.3:
                    t, sch = int(rng.integers(0, 4)), bool(rng.random() < 0.7)
                    X.set_instance(n, t, sch)
                else:
                    w, u = int(rng.integers(0, 6)), float(np.float32(rng.random()))
                    X.set_load(n, w, u)
            else:
                toks = prompts[int(rng.integers(0, len(prompts)))]
                if rng.random() < 0.2:
                    toks = toks[:int(rng.integers(0, toks.size + 1))]
                if not _reference_survives(oracle, X, toks, bs):
                    n_ub += 1
                    continue
                m = X.match(toks)
                for f in ("hbm", "dram", "ssd"):
                    obs += [int(v) for v in m[f]]
                obs += [int(m[f]) for f in ("instances", "max_block_num", "max_matched_block_num")]
                a = X.route(toks)
                obs.append(int(a["ok"]))
                if a["ok"]:
                    obs += [a["prefill_id"], a["decode_id"]]
                    # the oracle's literal choice (same containers, same insertion history => same iteration order)
                    # must lie in its own arg-max set; -1: every candidate scored <= MIN_SCORE, the name stays empty
                    # (cache_aware_routing.cpp:65,80)
                    if "prefill_argmax" in a and a["prefill_id"] >= 0:
                        assert (a["prefill_argmax"] >> a["prefill_id"]) & 1
                    if "decode_argmax" in a and a["decode_id"] >= 0:
                        assert (a["decode_argmax"] >> a["decode_id"]) & 1
        answers.append(np.array(obs, dtype=np.int64))
    return answers, n_ops, n_ub


def digest(answers):
    """SHA-256 of one history's answers: the golden keeps this instead of the ~100 K answers of a seed."""
    return hashlib.sha256(np.ascontiguousarray(answers, dtype="<i8").tobytes()).digest()


@pytest.mark.parametrize("seed", range(N_SEEDS))
def test_random_histories_oracle_equals_reference(oracle, golden, seed):
    """After every upload the whole key universe must hold what the reference's held; every match must equal the
    reference's field by field; every routing decision must be the reference's literal choice."""
    got, n_ops, n_ub = random_histories(oracle, lambda names, bs: oracle.PrefixOracle(names, bs, 1024), seed)
    n, sha = golden["hist%d_n" % seed], golden["hist%d_sha256" % seed]
    assert len(got) == n.size
    for h, g in enumerate(got):
        assert g.size == n[h] and digest(g) == bytes(sha[h]), "history %d differs from the reference" % h
    assert n_ops > 9000 and n_ub < n_ops // 10


REPLICA_NAMES = ["n%d" % i for i in range(10)]


def replica_history():
    """update_kvcache (global_kvcache_mgr.cpp:133-175): twelve rounds of 150 random KvCacheEvents on a master, one
    upload per round.  -> (the 200 keys, [[(name, stored, offload, removed)] per round])"""
    rng = np.random.default_rng(3)
    keys = rng.integers(0, 256, (200, 16), dtype=np.uint8)
    rounds = []
    for rnd in range(12):
        events = []
        for _ in range(150):
            n = REPLICA_NAMES[int(rng.integers(0, 10))]
            k = keys[rng.integers(0, 200, int(rng.integers(1, 4)))]
            kind = rng.random()
            events.append((n,) + ((k, (), ()) if kind < 0.5 else ((), k, ()) if kind < 0.8 else ((), (), k)))
        rounds.append(events)
    return keys, rounds


def test_replica_watch_path_oracle_equals_reference(oracle, golden):
    """A reference replica follows a reference master through etcd PUT / DELETE events — one watch response per
    upload, PUTs before DELETEs, last value wins — and ends with the master's map after every round (golden
    replica_gets[round, key] = (found, hbm, dram, ssd) of master and replica); the oracle given the same events holds
    the same map."""
    P = oracle.PrefixOracle(REPLICA_NAMES)
    sizes, gets = golden["replica_sizes"], golden["replica_gets"]
    keys, rounds = replica_history()
    assert sizes.shape[0] == len(rounds)
    for rnd, events in enumerate(rounds):
        for ev in events:
            P.record(*ev)
        P.upload()
        assert (sizes[rnd] == P.size()).all()
        for i, k in enumerate(keys):
            found, m = P.get(k)
            assert (gets[rnd, i] == [int(found)] + m).all(), (rnd, i)
    # one response carrying a PUT and a DELETE of the same key: the reference applies the DELETE last (:163-172)
    final = golden["replica_final"]
    P.put(keys[0], hbm=["n1"])
    P.delete(keys[0])
    found, m = P.get(keys[0])
    assert final[0].tolist() == [int(found)] + m and not found
    # an unparsable value is skipped by the reference (:149-152): the key keeps what the master holds
    found, m = P.get(keys[1])
    assert final[1].tolist() == [int(found)] + m
    # a parsable one with extra keys is taken: {"ssd_instance_set":["n3"],"x":1,"hbm_instance_set":[],
    # "dram_instance_set":["n2","n2"]}
    P.put(keys[1], hbm=[], dram=["n2", "n2"], ssd=["n3"])
    found, m = P.get(keys[1])
    assert final[2].tolist() == [int(found)] + m == [1, 0, 4, 8]


def test_index_wire_form_against_the_reference(tmp_path):
    """host/index_wire.h reads what a reference master wrote to etcd in upload_kvcache (etcd_client.cpp:122-137) into
    the sets the reference held, and writes the same keys and — up to the order of names inside an array — the same
    JSON (tests/cpp/index_wire_ref_main.cc over tests/golden/ref_etcd_listing.bin)."""
    exe = tmp_path / "index_wire_ref_main"
    subprocess.check_call(["g++", "-std=c++17", "-O1", os.path.join(HERE, "cpp", "index_wire_ref_main.cc"), "-o",
                           str(exe)])
    p = subprocess.run([str(exe), LISTING], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and p.stdout.strip().endswith("OK"), p.stdout[-2000:]

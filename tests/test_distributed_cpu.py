"""Host-side logic of the N > 1 paths on CPU: world_size-2 gloo processes exercise the byte-range
sharding rule (bpe.cpp:864-873), the variable-length all-gather and the merge of per-rank word
exports (additivity in the word frequency), the sentence sharding of encode, and the host
alphabet / model writer of train_distributed against the oracle."""
import collections
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import _cases
from _bind import read_model, tmp_model_path
from youtokentome_b200 import distributed as D
from youtokentome_b200 import synth


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _words_export(shard):
    """A stand-in for yttm_train_export_words on the CPU: unique words of a shard as packed arrays
    (token = byte value + 5, first token 4 = the role of '▁')."""
    cnt = collections.Counter(shard.split())
    toks, offs, freq = [], [0], []
    for w, c in sorted(cnt.items()):
        toks += [4] + [b + 5 for b in w]
        offs.append(len(toks))
        freq.append(c)
    return np.asarray(toks, np.uint32), np.asarray(offs, np.uint32), np.asarray(freq, np.uint64)


def _worker(rank, world, port, text, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        pos = D.split_byte_ranges(text, world)
        shard = text[pos[rank]:pos[rank + 1]]
        t, o, f = _words_export(shard)
        toks, offs, frqs = D.all_gather_arrays(t), D.all_gather_arrays(o), D.all_gather_arrays(f)
        mt, mo, mf = D.merge_word_exports(list(zip(toks, offs, frqs)))
        total = collections.Counter()
        for i in range(len(mf)):
            total[bytes(int(x) - 5 for x in mt[mo[i] + 1:mo[i + 1]])] += int(mf[i])
        assert total == collections.Counter(text.split()), "merged exports lose or invent words"
        # encode sharding: every sentence exactly once, contiguous
        offsets = np.concatenate([[0], np.cumsum([len(s) for s in text.split(b"\n")])]).astype(np.uint64)
        lo, hi = D.shard_sentences(offsets, rank, world)
        los = [torch.zeros(2, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(los, torch.tensor([lo, hi]))
        rngs = [tuple(x.tolist()) for x in los]
        assert rngs[0][0] == 0 and rngs[-1][1] == len(offsets) - 1
        assert all(rngs[i][1] == rngs[i + 1][0] for i in range(world - 1))
        np.save(os.path.join(out_dir, "ok_%d.npy" % rank), np.asarray([1]))
    finally:
        dist.destroy_process_group()


def test_gloo_world2_sharding_and_merge(tmp_path):
    text = synth.readme_corpus(n_lines=400) + _cases.zipf().text(60_000)
    port = _free_port()
    mp.spawn(_worker, args=(2, port, text, str(tmp_path)), nprocs=2, join=True)
    assert all(os.path.exists(tmp_path / ("ok_%d.npy" % r)) for r in range(2))


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_split_byte_ranges_rule(world):
    text = _cases.zipf().text(50_000)
    pos = D.split_byte_ranges(text, world)
    assert pos[0] == 0 and pos[-1] == len(text) and all(a <= b for a, b in zip(pos, pos[1:]))
    for p in pos[1:-1]:
        assert text[p] in b" \t\n\r\x0b\x0c"           # cut only on an ASCII space (never inside UTF-8)
    # no word is split: the word multiset of the shards equals that of the text
    parts = collections.Counter()
    for a, b in zip(pos, pos[1:]):
        parts.update(text[a:b].split())
    assert parts == collections.Counter(text.split())


def test_shard_sentences_balanced():
    rng = np.random.default_rng(0)
    lens = rng.integers(1, 4000, size=5000)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    world = 8
    got = [D.shard_sentences(offsets, r, world) for r in range(world)]
    assert got[0][0] == 0 and got[-1][1] == 5000 and all(got[i][1] == got[i + 1][0] for i in range(world - 1))
    sizes = [int(offsets[hi] - offsets[lo]) for lo, hi in got]
    assert max(sizes) - min(sizes) < 2 * 4000
    assert D.shard_sentences(np.zeros(1, np.uint64), 0, 2) == (0, 0)


@pytest.mark.parametrize("cov", [1.0, 0.95])
def test_host_alphabet_and_model_writer_match_oracle(oracle, cov):
    text = _cases.zipf().text(80_000)
    m = tmp_model_path("orc")
    oracle.train(text, m, 1200, cov)
    want_c2i, want_rules, want_special = read_model(m)
    chars = [c for c in text.decode() if not c.isspace()]
    cnt = collections.Counter(chars)
    cps = np.asarray(sorted(ord(c) for c in cnt), dtype=np.uint32)
    counts = np.asarray([cnt[chr(c)] for c in cps], dtype=np.uint64)
    char2id, n_special = D.choose_alphabet(cps, counts, len(text.decode()), cov, (0, 1, 2, 3))
    out = tmp_model_path("host")
    D.write_model(out, char2id, np.zeros((0, 3), np.uint32), (0, 1, 2, 3), 1200)
    got_c2i, _, got_special = read_model(out)
    assert got_c2i == want_c2i and got_special == want_special


@pytest.mark.parametrize("special", [(0, 1, 2, 3), (-1, 0, -1, 5)])
def test_model_writer_is_byte_identical_to_the_reference(special):
    """write_model (rank 0 of train_distributed) writes the very bytes the reference's BPEState::dump does,
    char2id lines in flat_hash_map order included (the reference's file recorded by its SHA-256, see _refgolden):
    feed it the trained model un-renamed."""
    import _bind
    import _refgolden as R
    pad, unk, bos, eos = special
    text = _cases.zipf().text(60_000)
    m = tmp_model_path("orcw")
    _bind.Oracle().train(text, m, 900, 1.0, pad=pad, unk=unk, bos=bos, eos=eos)
    c2i, rules, _ = read_model(m)
    # undo rename_tokens: final ids -> internal ids (specials first, then the rest ascending)
    taken = {s for s in special if s != -1}
    free = [i for i in range(900) if i not in taken]
    back = {final: len(taken) + k for k, final in enumerate(free)}
    char2id = {cp: back[i] for cp, i in c2i.items()}
    internal = np.asarray([[back[x], back[y], back[z]] for x, y, z in rules], dtype=np.uint32).reshape(-1, 3)
    out = tmp_model_path("oursw")
    D.write_model(out, char2id, internal, special, 900)
    assert R.file_sha256(out) == R.want("distributed/model_writer/%d_%d_%d_%d" % special, lambda: R.file_sha256(
        R.train(text, 900, 1.0, pad=pad, unk=unk, bos=bos, eos=eos)))

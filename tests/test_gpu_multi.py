"""Matcher::match_list_parallel through the C ABI (include/frz_cuda.h: frz_comm_*, frz_match_list_parallel*).

Mirrors the reference's parallel == sequential tests (src/matcher/parallel.rs:104-173, tests/api_properties.rs:99-111,
626-668).  The 1-GPU tests run everywhere (a communicator over one GPU, with and without the forced all-gather + merge
leg); the 2-GPU tests need two GPUs on the box and are skipped otherwise (`gpurun --gpus 2`; their recorded output is
committed under profiles/)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpus():
    import torch
    return torch.cuda.device_count()


def _haystacks_4101():
    """The reference's own parallel test list (src/matcher/parallel.rs:104-130): matches at chunk seams, ties broken by index."""
    hs = ["nomatch"] * 4101
    for i in (0, 2047, 2048, 2049, 4095, 4096, 4100):
        hs[i] = "foo"
    for i in (5, 1000, 3000):
        hs[i] = "f_o_o"
    hs[2050] = "xfoo"
    return hs


@pytest.mark.parametrize("force_nccl", [0, 1])
def test_parallel_world1_equals_match_list(force_nccl, monkeypatch):
    """A communicator over ONE GPU: match_list_parallel == match_list (parallel.rs:29-31, threads == 1).  With
    FRZ_PARALLEL_FORCE_NCCL=1 the run still goes through the gather + k-way merge leg (one run)."""
    import frizbee_b200 as F
    from frizbee_b200 import parallel, synth
    from frizbee_b200.types import Config, SortStrategy
    monkeypatch.setenv("FRZ_PARALLEL_FORCE_NCCL", str(force_nccl))
    comm = parallel.Comm.local(1)
    data, off = synth.generate("deadbeef", 120_001, 48, 64, seed=21)
    shards = comm.shard_arrow(data, off)
    whole = F.Corpus.from_arrow(data, off)
    for sort in SortStrategy:
        for k in (0, 1, None):
            m = F.Matcher("deadbeef", Config(max_typos=k, sort=sort))
            got = comm.match_list_parallel(m, shards)
            want = m.match_list_array(whole)
            assert len(got) == len(want) and np.array_equal(got, want), (sort, k)
            m.close()
    hs = _haystacks_4101()
    d2, o2 = F.pack_host(hs)
    s2 = comm.shard_arrow(d2, o2)
    m = F.Matcher("foo", Config())
    assert [x for x in comm.match_list_parallel(m, s2)["index"]] == [x.index for x in m.match_list(hs)]
    for s in shards + s2:
        s.close()
    whole.close()
    comm.close()


def test_parallel_rank_api_world1_nccl_comm():
    """The multi-process form with a world of one rank: ncclCommInitRank, the shared host segment, the device-only result."""
    import frizbee_b200 as F
    from frizbee_b200 import parallel, synth
    from frizbee_b200.types import Config
    comm = parallel.Comm.from_rank(parallel.Comm.unique_id(), 1, 0, 0)
    data, off = synth.generate("deadbeef", 60_000, 48, 64, seed=5)
    shard = F.Corpus.from_arrow(data, off)
    m = F.Matcher("deadbeef", Config(max_typos=1))
    out = comm.host_alloc_matches(60_000)
    total, d_ptr = comm.match_list_parallel_rank(m, shard, 1000, out)
    want = m.match_list_array(shard)
    want = want.copy(); want["index"] += 1000
    assert total == len(want) and np.array_equal(np.array(out[:total]), want)
    total2, d_ptr2 = comm.match_list_parallel_rank(m, shard, 1000, None)
    assert total2 == total and d_ptr2 != 0
    # end to end on the rank: host Arrow buffers in
    total3 = comm.match_list_parallel_rank_host(m, data, off, 1000, out)
    assert total3 == total and np.array_equal(np.array(out[:total]), want)
    t = comm.last_timings(0)
    assert t["total_ms"] > 0 and t["launches"] > 0
    # capacity error reports the needed count
    small = comm.host_alloc_matches(8)
    with pytest.raises(F.FrizbeeError) as e:
        comm.match_list_parallel_rank(m, shard, 0, small)
    assert e.value.status_name == "FRZ_ERR_CAPACITY"
    comm.host_free(small)
    comm.host_free(out)
    shard.close(); m.close(); comm.close()


def test_streamed_end_to_end_call_equals_resident_corpus():
    """frz_match_list_parallel_rank_host matches the list WHILE it streams in (host.cu: frz_match_shard_streamed — the
    pipeline runs over consecutive tile ranges as their H2D chunks land, the tile scan carries the running count, only
    the sort waits for the last chunk).  2 M haystacks = 12 chunks = 3 ranges; the result must equal match_list on the
    resident corpus for the two sort strategies the streamed form serves, and for the ones that fall back (reversed)."""
    import frizbee_b200 as F
    from frizbee_b200 import parallel, synth
    from frizbee_b200.types import Config, SortStrategy
    comm = parallel.Comm.from_rank(parallel.Comm.unique_id(), 1, 0, 0)
    n = 2_000_000
    data, off = synth.generate("deadbeef", n, 48, 64, seed=17)
    off32 = off.astype(np.int32)
    whole = F.Corpus.from_arrow(data, off)
    out = comm.host_alloc_matches(n)
    for sort in (SortStrategy.ScoreThenIndexAsc, SortStrategy.IndexAsc, SortStrategy.ScoreThenIndexDesc):
        for k in (1, 0):
            m = F.Matcher("deadbeef", Config(max_typos=k, sort=sort))
            want = m.match_list_array(whole)
            for offsets in (off32, off):
                total = comm.match_list_parallel_rank_host(m, data, offsets, 7, out)
                w = want.copy(); w["index"] += 7
                assert total == len(w) and np.array_equal(np.array(out[:total]), w), (sort, k, offsets.dtype)
            m.close()
    comm.host_free(out)
    whole.close(); comm.close()


def test_sort_scratch_regrows_for_a_larger_corpus():
    """ADVICE r1 (high): a matcher whose score bound needs the two-pass sort sized its scratch by the FIRST corpus; a later,
    larger corpus must regrow it (was a device out-of-bounds write)."""
    import frizbee_b200 as F
    from frizbee_b200 import synth
    from frizbee_b200.types import Config
    from oracle import pyoracle as O
    needle = "abcdefghijklmnopqrstuvwxyzabcdefghijklmnopqrstuvwxyzabcdefgh"   # 60 bytes: score bound >= 1024
    cfg = Config(max_typos=None)
    m = F.Matcher(needle, cfg)
    assert m.score_bound() >= 1024
    lanes = m.backend_info()["prefilter_lanes"]
    small_d, small_o = synth.generate(needle, 300, 80, 128, seed=1, p_full=0.5)
    big_d, big_o = synth.generate(needle, 20_000, 80, 128, seed=2, p_full=0.5)
    for d, o in ((small_d, small_o), (big_d, big_o), (small_d, small_o)):
        got = m.match_list_host_array(d, o)
        want = O.match_list_packed([needle], cfg.with_(emulate_lanes=lanes), d, o)
        assert len(got) == len(want) and all(np.array_equal(got[f], want[f]) for f in ("index", "score", "exact"))
    m.close()


def test_c_client_on_the_gpu(tmp_path):
    """examples/ffi_demo.c — plain C against include/frz_cuda.h — on the device: match_list, match_indices, and
    match_list_parallel over min(2, #GPUs) GPUs == match_list (the Rust shim's call sequence, INTEGRATION.md)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_host_logic import _build_ffi_demo
    exe = _build_ffi_demo(tmp_path)
    n = min(2, _gpus())
    r = subprocess.run([exe, str(n)], capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout[-2000:]); sys.stderr.write(r.stderr[-2000:])
    assert r.returncode == 0, (r.stdout, r.stderr)
    assert "Match { score: 53, index: 0, exact: false }" in r.stdout
    assert f"match_list_parallel over {n} GPU(s)" in r.stdout and "parallel == sequential: yes" in r.stdout


@pytest.mark.parametrize("exchange", ["p2p", "allgather"])
def test_local_form_two_gpus(exchange, monkeypatch):
    """Single process, two GPUs (frz_comm_create_local: ncclCommInitAll + one worker thread per GPU), with both forms of
    the exchange step: P2P placement (k_place: every GPU stores its matches at their merged positions in the peers' slice
    buffers over NVLink) and the all-gather of whole runs."""
    if _gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    import frizbee_b200 as F
    from frizbee_b200 import parallel, synth
    from frizbee_b200.types import Config, SortStrategy
    monkeypatch.setenv("FRZ_PARALLEL_EXCHANGE", exchange)
    comm = parallel.Comm.local(2)
    data, off = synth.generate("deadbeef", 300_001, 48, 64, seed=33)
    shards = comm.shard_arrow(data, off)
    whole = F.Corpus.from_arrow(data, off)
    out = comm.host_alloc_matches(300_001)
    for sort in SortStrategy:
        for k in (0, 1, None):
            m = F.Matcher("deadbeef", Config(max_typos=k, sort=sort))
            got = comm.match_list_parallel(m, shards, out)
            want = m.match_list_array(whole)
            assert len(got) == len(want) and np.array_equal(np.array(got), want), (sort, k)
            m.close()
    hs = _haystacks_4101()
    d2, o2 = F.pack_host(hs)
    s2 = comm.shard_arrow(d2, o2)
    m = F.Matcher("foo", Config())
    assert [int(x) for x in comm.match_list_parallel(m, s2)["index"]] == [x.index for x in m.match_list(hs)]
    comm.host_free(out)
    for s in shards + s2:
        s.close()
    whole.close(); comm.close()


@pytest.mark.parametrize("exchange", ["p2p", "allgather"])
def test_match_list_parallel_two_gpus_torchrun(exchange):
    """One rank per GPU under torchrun (the bench's launch mode): tests/_multi_gpu_worker.py, with both forms of the
    exchange step for the host-out calls (device-only calls always all-gather; p2p maps the peers' slice buffers with cudaIpc)."""
    if _gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    world = 2
    env = dict(os.environ, FRZ_PARALLEL_TIMEOUT_S="60", FRZ_PARALLEL_EXCHANGE=exchange)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tests", "_multi_gpu_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    sys.stdout.write(r.stdout[-4000:])
    sys.stderr.write(r.stderr[-4000:])
    assert r.returncode == 0
    assert "False" not in r.stdout and "differs" not in r.stdout

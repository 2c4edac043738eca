"""Search-window input (bdx_submit_windows): the reads' window bytes -- as bytes or 4-bit codes, staged or pinned --
give the results, per-pass details and DemuxStats of bdx_submit on the full reads, which are the oracle's."""
import ctypes as C

import numpy as np
import pytest

import bdx_b200 as bdx
import hostref
import synth
import windows_cases as wc
from bdx_b200 import capi
from gpu_common import compare

pytestmark = pytest.mark.gpu
R = bdx.parse_dynamic_range
MODES = ("win", "win4", "win_pinned", "win4_pinned")


class Pinned:
    """Page-locked copies of numpy arrays (bdx_host_alloc), freed on exit."""

    def __init__(self):
        self.lib, self.ptrs = capi.load_library(), []

    def __call__(self, a):
        p = self.lib.bdx_host_alloc(max(a.nbytes, 16))
        assert p
        self.ptrs.append(p)
        out = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), (max(a.nbytes, 16),))[:a.nbytes].view(a.dtype)
        out[:] = a
        return out

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        for p in self.ptrs:
            self.lib.bdx_host_free(p)


def submit(st, config, blob, off32, mode, pin, tag=0):
    if mode == "bytes":
        st.submit(blob if blob.size else np.zeros(1, np.uint8), off32, tag=tag)
        return
    if mode == "packed":
        st.submit_packed4(config.pack4(blob), off32, tag=tag)
        return
    win, win_off = config.window_reads(blob, off32)
    packed = mode.startswith("win4")
    if packed:
        win = config.pack4(win)
    if mode.endswith("pinned"):
        win, win_off, off32 = pin(win), pin(win_off), pin(off32)
    st.submit_windows(win, win_off, off32, packed4=packed, pinned=mode.endswith("pinned"), tag=tag)


def run_modes(cfg, reads, want_stats, modes=("bytes",) + MODES):
    """{mode: (results, details, stats counters, stats overflow)} of one batch per mode on one stream."""
    blob, off = bdx.pack_reads(reads)
    off32 = off.astype(np.int32)
    out = {}
    with capi.Engine(cfg, max_reads=max(len(reads), 1), max_bytes=max(int(off[-1]), 16), want_stats=want_stats) as eng, \
            Pinned() as pin:
        st = eng.stream
        st.enable_details(True)
        for mode in modes:
            st.stats_reset()
            submit(st, eng.config, blob, off32, mode, pin)
            _, res, det = st.fetch(want_details=True)
            out[mode] = (res, det, st.stats() if want_stats else None, st.stats_overflow() if want_stats else None)
    return out


def assert_same(out, label):
    res, det, stats, ovf = out["bytes"]
    for mode, (r, d, s, o) in out.items():
        assert (r == res).all(), (label, mode, np.nonzero(r != res)[0][:5])
        assert (d == det).all(), (label, mode)
        if stats is not None:
            assert (s == stats).all(), (label, mode)
            assert (np.sort(o) == np.sort(ovf)).all(), (label, mode)


@pytest.mark.parametrize("name", sorted(wc.CASES))
def test_windows_equal_full_reads_and_oracle(name):
    rng = np.random.default_rng(sum(map(ord, name)) + 2)
    cfg, b1, b2 = wc.make_case(name, rng)
    reads = wc.make_reads(rng, b1, b2, 3000)
    want_stats = bool(cfg.summary)
    compare(cfg, reads, want_stats=want_stats, label=name)
    assert_same(run_modes(cfg, reads, want_stats), name)


def test_config3_geometry():
    import bench_configs
    cfg = bench_configs.configs()["3"][0]
    rng = np.random.default_rng(3)
    reads = synth.random_reads(rng, 4000, cfg.bc_seqs, barcodes2=cfg.bc_seqs2, min_len=150, start_hi=5)
    compare(cfg, reads, label="config3")
    assert_same(run_modes(cfg, reads, False), "config3")


@pytest.mark.parametrize("algo", ["semiglobal", "hamming"])
@pytest.mark.parametrize("rng_expr,at_end", [("1:120", False), ("end-119:end", True), ("30:180", False)])
def test_long_reads_short_search_ranges_windowed(algo, rng_expr, at_end):
    rng = np.random.default_rng(len(rng_expr) * 31 + len(algo))
    bcs = synth.random_barcodes(rng, 96, 24)
    reads = []
    for r in synth.random_reads(rng, 1200, bcs, min_len=100, max_len=118, start_hi=60):
        pad = bytes(synth.BASES[rng.integers(0, 4, int(rng.integers(500, 4000)))])
        reads.append(pad + r if at_end else r + pad)
    reads += [b"", b"ACGT" * 10]
    for kw in (dict(), dict(trim_side=3 if at_end else 5, summary=True), dict(min_delta=0.09)):
        cfg = wc.bdx.DemuxConfig(bc_seqs=bcs, bc_lengths_no_N=[24] * 96, ids=[f"a{i}" for i in range(96)],
                                 matching_algorithm=algo, ref_search_range=R(rng_expr), **kw)
        out = run_modes(cfg, reads, bool(kw.get("summary")))
        assert_same(out, f"{algo} {rng_expr} {kw}")
        if kw.get("summary") and at_end:
            assert len(out["bytes"][3]) > 0      # matches beyond the position histogram: the overflow list is used


def test_zero_read_batch_and_interleaving():
    """A zero-read windowed batch, and four windowed batches in flight interleaved with byte and packed batches."""
    rng = np.random.default_rng(12)
    cfg, b1, b2 = wc.make_case("sg_dual", rng)
    batches = [wc.make_reads(rng, b1, b2, 300 + 50 * k) for k in range(8)]
    packed = [bdx.pack_reads(b) for b in batches]
    modes = ["win", "bytes", "win4_pinned", "packed", "win_pinned", "win4", "win", "bytes"]
    with capi.Engine(cfg, max_reads=1000, max_bytes=400 * 1000) as eng, Pinned() as pin:
        want = [eng.classify_packed(blob, off) for blob, off in packed]
        st = eng.stream
        submit(st, eng.config, np.zeros(0, np.uint8), np.zeros(1, np.int32), "win", pin, tag=99)
        assert st.fetch()[0] == 99
        got, q = {}, 0
        for k, (blob, off) in enumerate(packed):
            submit(st, eng.config, blob, off.astype(np.int32), modes[k], pin, tag=k)
            q += 1
            if q == 4:
                tag, res = st.fetch()
                got[tag] = res
                q -= 1
        while q:
            tag, res = st.fetch()
            got[tag] = res
            q -= 1
    for k in range(len(packed)):
        assert (got[k] == want[k]).all(), (k, modes[k])


@pytest.mark.parametrize("mode", ["win", "win4"])
def test_graph_replay_of_windowed_chunks(mode):
    """Full-size 512-read chunks replay a captured graph from a slot's second use on; k_expand_windows runs in front
    of it, outside the graph.  24 chunks must equal one big uncaptured batch."""
    rng = np.random.default_rng(78)
    bcs = synth.random_barcodes(rng, 96, 24)
    cfg = wc.bdx.DemuxConfig(bc_seqs=bcs, bc_lengths_no_N=[24] * 96, ids=[f"a{i}" for i in range(96)],
                             ref_search_range=R("1:40"), trim_side=5, summary=True)
    B, nb = 512, 24
    reads = synth.random_reads(rng, B * nb, bcs, min_len=150, start_hi=10)
    blob, off = bdx.pack_reads(reads)
    with capi.Engine(cfg, max_reads=B * nb + 1, max_bytes=int(off[-1]) + 16) as big:
        want = big.classify_packed(blob, off)
        want_stats = big.stream.stats()
    sub_off = np.ascontiguousarray(off[:B + 1]).astype(np.int32)
    with capi.Engine(cfg, max_reads=B, max_bytes=B * 150) as eng, Pinned() as pin:
        st, got, q = eng.stream, [], 0
        for k in range(nb):
            submit(st, eng.config, blob[k * B * 150:(k + 1) * B * 150], sub_off, mode, pin, tag=k)
            q += 1
            if q == 4:
                got.append(st.fetch()[1])
                q -= 1
        while q:
            got.append(st.fetch()[1])
            q -= 1
        assert (np.concatenate(got) == want).all()
        assert (st.stats() == want_stats).all()


@pytest.mark.parametrize("idx", [0, 1, 2])
def test_golden_files_through_windows(refdata, tmp_path, idx):
    case = hostref.demo_cases(refdata)[idx]
    engines = []

    def make(cfg):
        for e in engines:
            e.close()
        engines.clear()
        engines.append(capi.Engine(cfg, max_reads=4000, windows=True))
        return engines[0].classify_reads

    assert hostref.run_case(case, str(tmp_path / "out"), make) == {0: 24, 1: 24, 2: 76}[idx]
    for e in engines:
        e.close()


def test_refusals_leave_nothing_in_flight():
    rng = np.random.default_rng(4)
    cfg, b1, b2 = wc.make_case("sg_start", rng)
    reads = wc.make_reads(rng, b1, b2, 100)
    blob, off = bdx.pack_reads(reads)
    off32 = off.astype(np.int32)
    with capi.Engine(cfg, max_reads=len(reads), max_bytes=int(off[-1])) as eng:
        st, config = eng.stream, eng.config
        win, win_off = config.window_reads(blob, off32)
        long_read = np.nonzero(np.diff(win_off) > 0)[0][0]
        bad = win_off.copy()
        bad[long_read + 1:] -= 1                       # one read's window a byte short
        first = win_off + 1                            # win_offsets[0] != 0
        big_off = np.concatenate([off32, off32[-1:] + 5])
        for w, wo, o, code in ((win, bad, off32, capi.BDX_ERR_INVALID), (win, first, off32, capi.BDX_ERR_INVALID),
                               (win, np.zeros(len(big_off), np.int32), big_off, capi.BDX_ERR_TOO_LARGE)):
            with pytest.raises(capi.BdxError) as ei:
                st.submit_windows(w, wo, o)
            assert ei.value.code == code
        with pytest.raises(capi.BdxError) as ei:
            st.submit_windows(win, win_off, off32 * 0 + np.arange(len(off32), dtype=np.int32) * 10 ** 6)
        assert ei.value.code == capi.BDX_ERR_TOO_LARGE
        with pytest.raises(capi.BdxError) as ei:                 # nothing was left in flight
            st.fetch()
        assert ei.value.code == capi.BDX_ERR_STATE
        st.submit_windows(win, win_off, off32)                    # and the stream still works
        assert len(st.fetch()[1]) == len(reads)
    wide = ["ABCDEFGHIJKLMNOP", "QRSTUVWXABCDEFGH"]
    cfg = bdx.DemuxConfig(bc_seqs=wide, bc_lengths_no_N=[16, 16], ids=["x", "y"])
    with capi.Engine(cfg, max_reads=10, max_bytes=1000) as eng:
        off32 = np.array([0, 16], np.int32)
        win, win_off = eng.config.window_reads(np.frombuffer(b"ABCDEFGHIJKLMNOP", np.uint8), off32)
        with pytest.raises(capi.BdxError) as ei:
            eng.stream.submit_windows(np.zeros(8, np.uint8), win_off, off32, packed4=True)
        assert ei.value.code == capi.BDX_ERR_INVALID
        with pytest.raises(capi.BdxError) as ei:
            eng.stream.fetch()
        assert ei.value.code == capi.BDX_ERR_STATE

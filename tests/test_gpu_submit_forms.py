"""Every way into a bdx_stream -- bdx_submit, bdx_submit_pinned, bdx_submit_packed4[_pinned], bdx_submit_windows
[_pinned] with byte and packed windows, bdx_acquire + bdx_commit -- refuses each bad batch with the same code and
text and leaves the stream able to take the next one, and gives the results and details of bdx_submit on the same
reads, also with all of them mixed on one ring of slots next to graph replay."""
import ctypes as C

import numpy as np
import pytest

import bdx_b200 as bdx
import orc
import windows_cases as wc
from bdx_b200 import capi
from test_gpu_windows import Pinned

pytestmark = pytest.mark.gpu
FORMS = ("bytes", "bytes_pinned", "packed4", "packed4_pinned", "win", "win_pinned", "win4", "win4_pinned", "acquire")
PACKED = ("packed4", "packed4_pinned", "win4", "win4_pinned")
WINDOWS = ("win", "win_pinned", "win4", "win4_pinned")
MAX_IN_FLIGHT = 4
INV, STATE, BIG = capi.BDX_ERR_INVALID, capi.BDX_ERR_STATE, capi.BDX_ERR_TOO_LARGE


def ptr(a):
    return None if a is None else a.ctypes.data


def form_input(config, blob, off, form):
    """(data, offsets, window offsets) of the batch blob / off as `form` takes it."""
    data, win_off = blob, None
    if form in WINDOWS:
        data, win_off = config.window_reads(blob, off)
    if form in PACKED:
        data = config.pack4(data)
    return data, off, win_off


def pinned(form, pin, arrays):
    """The arrays in page-locked memory for the *_pinned forms, as they are for the others."""
    if not form.endswith("pinned"):
        return arrays
    return tuple(None if a is None else pin(a) for a in arrays)


def acquire(st):
    seq_p, off_p = C.c_void_p(), C.c_void_p()
    rc = st.lib.bdx_acquire(st.handle, C.byref(seq_p), C.byref(off_p))
    return rc, (seq_p, off_p)


def stage(st, staging, data, off):
    """Copy a batch into the staging bdx_acquire handed out (as much of it as fits)."""
    seq_p, off_p = staging
    if off is not None:
        C.memmove(off_p.value, off.ctypes.data, min(off.nbytes, (st.max_reads + 1) * 4))
    if data is not None and data.size:
        C.memmove(seq_p.value, data.ctypes.data, min(data.nbytes, st.max_bytes))


def call(st, form, data, off, win_off, n, tag=0, staging=None):
    """The form's C entry points on raw pointers; their status.  staging: that of a bdx_acquire still open."""
    L, h, pin = st.lib, st.handle, form.endswith("pinned")
    if form.startswith("bytes"):
        return (L.bdx_submit_pinned if pin else L.bdx_submit)(h, ptr(data), ptr(off), n, tag)
    if form.startswith("packed4"):
        return (L.bdx_submit_packed4_pinned if pin else L.bdx_submit_packed4)(h, ptr(data), ptr(off), n, tag)
    if form in WINDOWS:
        fn = L.bdx_submit_windows_pinned if pin else L.bdx_submit_windows
        return fn(h, ptr(data), ptr(win_off), ptr(off), n, int(form in PACKED), tag)
    if staging is None:
        rc, staging = acquire(st)
        if rc:
            return rc
    stage(st, staging, data, off)
    return L.bdx_commit(h, n, tag)


def submit(st, config, pin, blob, off, form, tag, staging=None):
    d, o, w = pinned(form, pin, form_input(config, blob, off, form))
    return call(st, form, d, o, w, len(off) - 1, tag, staging)


def fetch(st, view):
    """(tag, results, details) of the oldest batch, through bdx_fetch_view or bdx_fetch."""
    if view:
        return st.fetch(want_details=True)
    tag, n = C.c_uint64(), C.c_int32()
    res = np.zeros(st.max_reads, capi.RESULT_DTYPE)
    det = np.zeros(2 * st.max_reads, capi.DETAIL_DTYPE)
    capi._check(st.lib.bdx_fetch(st.handle, C.byref(tag), C.byref(n), res.ctypes.data, det.ctypes.data))
    return tag.value, res[:n.value], det[:2 * n.value].reshape(2, n.value)


def last_error(st):
    return st.lib.bdx_last_error().decode()


def make_config(seed):
    rng = np.random.default_rng(seed)
    cfg, b1, b2 = wc.make_case("sg_dual", rng)        # two sets, search ranges, DemuxStats on
    return cfg, b1, b2


def make_batch(seed, b1, b2, n):
    blob, off = bdx.pack_reads(wc.make_reads(np.random.default_rng(seed), b1, b2, n))
    return blob, off.astype(np.int32)


def reference(st, blob, off):
    """bdx_submit's results and details on blob / off, after checking the results against the oracle."""
    capi._check(st.lib.bdx_submit(st.handle, blob.ctypes.data, off.ctypes.data, len(off) - 1, 0))
    _, res, det = st.fetch(want_details=True)
    want = orc.Oracle(st.config.cfg).classify(blob, off)
    for f in ("status", "bc1", "bc2", "keep_start", "keep_end"):
        assert (res[f] == want[f]).all(), f
    return res, det


def argument_refusals(config, blob, off, max_bytes):
    """name -> (forms, mutate(data, off, win_off, n) -> the same, code, text): the refusals a batch's own arguments
    decide, in the order the submit path checks them."""
    _, win_off = config.window_reads(blob, off)
    long_read = int(np.nonzero(np.diff(win_off) > 0)[0][0])
    first = int(np.nonzero(np.diff(off) > 0)[0][0])

    def edit(a, fn):
        a = a.copy()
        fn(a)
        return a

    def shift(a):
        a += 1

    def too_big(o):
        o[-1] = max_bytes + 1

    def decreasing(o):                                  # read first + 1 ends one byte before it starts
        o[first + 1] = o[first + 2] + 1

    def short(w):                                       # one read's window a byte short
        w[long_read + 1:] -= 1

    return {
        "null_data": (("bytes", "bytes_pinned", "packed4", "packed4_pinned"),
                      lambda d, o, w, n: (None, o, w, n), INV, "null argument"),
        "null_offsets": (FORMS[:-1], lambda d, o, w, n: (d, None, w, n), INV, "null argument"),
        "null_win_offsets": (WINDOWS, lambda d, o, w, n: (d, o, None, n), INV, "null argument"),
        "negative_n": (FORMS, lambda d, o, w, n: (d, o, w, -1), INV, "negative n_reads"),
        "n_over_max_reads": (FORMS, lambda d, o, w, n: (d, o, w, n + 1), BIG, "batch exceeds max_reads"),
        "offsets0": (FORMS, lambda d, o, w, n: (d, edit(o, shift), w, n), INV, "offsets[0] must be 0"),
        "over_max_bytes": (FORMS, lambda d, o, w, n: (d, edit(o, too_big), w, n), BIG, "batch exceeds max_bytes"),
        "decreasing": (FORMS, lambda d, o, w, n: (d, edit(o, decreasing), w, n), INV, "must be non-decreasing"),
        "win_offsets0": (WINDOWS, lambda d, o, w, n: (d, o, edit(w, shift), n), INV, "win_offsets[0] must be 0"),
        "window_short": (WINDOWS, lambda d, o, w, n: (d, o, edit(w, short), n), INV,
                         f"win_offsets do not match the search windows of the read lengths (first bad read: {long_read})"),
        "null_win": (WINDOWS, lambda d, o, w, n: (None, o, w, n), INV, "null argument"),
    }


def test_refusals_leave_the_stream_as_it_was():
    cfg, b1, b2 = make_config(11)
    blob, off = make_batch(12, b1, b2, 300)
    n = len(off) - 1
    max_bytes = int(off[-1]) + 64
    with capi.Engine(cfg, max_reads=n, max_bytes=max_bytes) as eng, Pinned() as pin:
        st, config = eng.stream, eng.config
        st.enable_details(True)
        want_res, want_det = reference(st, blob, off)

        def accepts(form, label, staging=None):
            assert submit(st, config, pin, blob, off, form, 5, staging) == 0, (label, last_error(st))
            tag, res, det = st.fetch(want_details=True)
            assert tag == 5 and (res == want_res).all() and (det == want_det).all(), label

        def refused(s, rc, launches, code, text, label):
            """rc is the refusal (code, text); no kernel ran and nothing is in flight."""
            assert rc == code, (label, rc, last_error(s))
            assert text in last_error(s), (label, last_error(s))
            assert s.launch_count == launches, label
            with pytest.raises(capi.BdxError) as ei:
                s.fetch()
            assert ei.value.code == STATE and "nothing in flight" in str(ei.value), label

        for name, (forms, mutate, code, text) in argument_refusals(config, blob, off, max_bytes).items():
            for form in forms:
                label = f"{name}/{form}"
                d, o, w, k = mutate(*form_input(config, blob, off, form), n)
                d, o, w = pinned(form, pin, (d, o, w))
                staging = None
                if form == "acquire":                   # refused by bdx_commit, which keeps the staging acquired
                    rc, staging = acquire(st)
                    assert rc == 0, label
                launches = st.launch_count
                rc = call(st, form, d, o, w, k, staging=staging)
                refused(st, rc, launches, code, text, label)
                accepts(form, label, staging)

        launches = st.launch_count
        refused(st, st.lib.bdx_acquire(st.handle, None, None), launches, INV, "null argument", "acquire/null")
        accepts("acquire", "acquire/null")
        launches = st.launch_count
        refused(st, st.lib.bdx_commit(st.handle, n, 0), launches, STATE, "bdx_commit without bdx_acquire",
                "commit_without_acquire")
        accepts("acquire", "commit_without_acquire")

        # an acquire pending: every form is refused, bdx_acquire itself as "already acquired"
        for form in FORMS:
            label = f"acquire_pending/{form}"
            rc, staging = acquire(st)
            assert rc == 0, label
            d, o, w = pinned(form, pin, form_input(config, blob, off, form))
            launches = st.launch_count
            rc = acquire(st)[0] if form == "acquire" else call(st, form, d, o, w, n)
            text = "already acquired" if form == "acquire" else "bdx_acquire pending; call bdx_commit"
            refused(st, rc, launches, STATE, text, label)
            accepts("acquire", label, staging)           # the pending batch still goes through
            accepts(form, label)

        # BDX_MAX_IN_FLIGHT batches in flight
        for form in FORMS:
            label = f"in_flight_full/{form}"
            for t in range(MAX_IN_FLIGHT):
                capi._check(st.lib.bdx_submit(st.handle, blob.ctypes.data, off.ctypes.data, n, 100 + t))
            d, o, w = pinned(form, pin, form_input(config, blob, off, form))
            launches = st.launch_count
            rc = acquire(st)[0] if form == "acquire" else call(st, form, d, o, w, n)
            for t in range(MAX_IN_FLIGHT):
                tag, res, det = st.fetch(want_details=True)
                assert tag == 100 + t and (res == want_res).all() and (det == want_det).all(), label
            refused(st, rc, launches, STATE, "BDX_MAX_IN_FLIGHT batches already in flight; call bdx_fetch", label)
            accepts(form, label)

        # a stream without staging
        empty = capi.Stream(config, max_reads=0, max_bytes=max_bytes)
        try:
            for form in FORMS:
                label = f"max_reads_0/{form}"
                d, o, w = pinned(form, pin, form_input(config, blob, off, form))
                launches = empty.launch_count
                rc = acquire(empty)[0] if form == "acquire" else call(empty, form, d, o, w, n)
                refused(empty, rc, launches, STATE, "stream has no staging (max_reads = 0)", label)
                accepts(form, label)
        finally:
            empty.close()

    # packed input on a config with more than 15 distinct barcode bytes
    wide = ["ABCDEFGHIJKLMNOP", "QRSTUVWXABCDEFGH"]
    wcfg = bdx.DemuxConfig(bc_seqs=wide, bc_lengths_no_N=[16, 16], ids=["x", "y"])
    wblob = np.frombuffer(b"ABCDEFGHIJKLMNOPQRSTUVWXABCDEFGH" * 2, np.uint8).copy()
    woff = np.array([0, 32, 64], np.int32)
    with capi.Engine(wcfg, max_reads=4, max_bytes=1000) as eng, Pinned() as pin:
        st = eng.stream
        _, wwin_off = eng.config.window_reads(wblob, woff)
        want = st.classify(wblob, woff)
        for form in PACKED:
            label = f"wide/{form}"
            d, o, w = pinned(form, pin, (np.zeros(32, np.uint8), woff, wwin_off))
            launches = st.launch_count
            rc = call(st, form, d, o, w, 2)
            refused(st, rc, launches, INV, "more than 15 distinct barcode bytes: no 4-bit packed input", label)
            st.submit(wblob, woff)                       # the stream still takes byte input
            assert (st.fetch()[1] == want).all(), label


def test_mixed_forms_on_one_ring():
    """Every form in turn, BDX_MAX_IN_FLIGHT batches in flight, twice around the forms: full-size batches, so that
    each slot captures a CUDA graph on its second use and replays it from then on."""
    cfg, b1, b2 = make_config(20)
    batches = [make_batch(30 + k, b1, b2, 400) for k in range(3)]
    n = len(batches[0][1]) - 1
    assert all(len(o) - 1 == n for _, o in batches)
    max_bytes = max(int(o[-1]) for _, o in batches)
    with capi.Engine(cfg, max_reads=n, max_bytes=max_bytes) as eng, Pinned() as pin:
        st, config = eng.stream, eng.config
        st.enable_details(True)
        want = [reference(st, blob, off) for blob, off in batches]
        order = [(FORMS[i % len(FORMS)], i % len(batches)) for i in range(2 * len(FORMS))]
        launches, pending = [], []

        def check_oldest():
            i = pending.pop(0)
            tag, res, det = fetch(st, view=i % 2 == 0)
            form, b = order[i]
            assert tag == i and (res == want[b][0]).all() and (det == want[b][1]).all(), (i, form)

        for i, (form, b) in enumerate(order):
            if len(pending) == MAX_IN_FLIGHT:
                check_oldest()
            l0 = st.launch_count
            assert submit(st, config, pin, *batches[b], form, i) == 0, (form, last_error(st))
            launches.append(st.launch_count - l0)
            pending.append(i)
        while pending:
            check_oldest()
    # each batch launches the classification kernels, plus one expansion kernel for packed or windowed input
    base = launches[0]
    for (form, _), k in zip(order, launches):
        assert k == base + (form in PACKED or form in WINDOWS), (form, k, base)

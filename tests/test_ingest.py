"""rtl_tcp ingest (SURVEY.md §8(f) row 1): wire protocol of set_*_tcp.m, byte-exact lock-step captures, and
(gpu) ingest -> gsmcal_calibrate_batch == the same bytes handed over directly."""
import struct
import time

import numpy as np
import pytest

from gsmcal import ingest
from gsmcal.rtl_tcp_replay import GREETING, ReplayDongle


def _servers(n, n_bytes, seed=0, **kw):
    rng = np.random.default_rng(seed)
    return [ReplayDongle(rng.integers(0, 256, n_bytes, dtype=np.uint8), **kw) for _ in range(n)]


def _wait_cmds(srv, n, t=2.0):
    t0 = time.time()
    while len(srv.commands) < n and time.time() - t0 < t:
        time.sleep(0.01)
    return list(srv.commands)


def _read_until_gone(ing, seconds=15.0):
    """read_capture until it raises.  After a server goes away the client still reads what the kernel had buffered (both socket
    buffers: megabytes where the host allows 4 MB buffers, hundreds of short captures), so the bound is time, not a count of reads."""
    t_end = time.time() + seconds
    while time.time() < t_end:
        ing.read_capture(ing.buffers[0])


def test_commands_match_reference_wire_format():
    srv = _servers(1, 4096)[0]
    try:
        import socket
        s = socket.create_connection((srv.host, srv.port))
        ingest.set_gain_tcp(s, 0)                # set_gain_tcp.m:13-15
        ingest.set_gain_tcp(s, 496)              # :8-11
        ingest.set_rate_tcp(s, (1625 / 6) * 1e3 * 8)   # 2166666.67 -> uint32 rounds to 2166667
        ingest.set_freq_tcp(s, 957.4e6)
        cmds = _wait_cmds(srv, 5)
        assert cmds == [(3, 0), (3, 1), (4, 496), (2, 2166667), (1, 957400000)]
        # big-endian on the wire, as MATLAB tcpip writes uint32 and rtl_tcp reads with ntohl
        assert struct.pack(">BI", 1, 957400000) == b"\x01" + (957400000).to_bytes(4, "big")
        assert s.recv(12, __import__("socket").MSG_WAITALL) == GREETING
        s.close()
    finally:
        srv.close()


def test_lockstep_captures_are_byte_exact_and_greeting_is_flushed():
    D, N = 5, 30000                               # 2N bytes per capture; stored capture is shorter -> wraps
    srvs = _servers(D, 2 * N - 1000, seed=3)
    try:
        with ingest.DongleIngest([(s.host, s.port) for s in srvs], N, 957.4e6, 2166666.67, n_threads=2) as ing:
            got = [c.copy() for c in ing.captures(3)]
            for s in srvs:
                assert _wait_cmds(s, 3) == [(3, 0), (2, 2166667), (1, 957400000)]     # gsm_sync_demod.m:72-84 order
        for k, cap in enumerate(got):
            assert cap.shape == (D, 2 * N) and cap.dtype == np.uint8
            for d, s in enumerate(srvs):
                # flush read = greeting (12 B) + first 2N-12 stream bytes; capture k starts right after it
                np.testing.assert_array_equal(cap[d], s.expected(2 * N - 12 + k * 2 * N, 2 * N))
    finally:
        for s in srvs:
            s.close()


def test_negative_gain_saturates_like_uint32():
    """MATLAB's uint32(gain) saturates at 0 (set_gain_tcp.m:10); a two's-complement wrap would ask the tuner for 4e9 tenths of a dB"""
    srv = _servers(1, 4096)[0]
    try:
        import socket
        s = socket.create_connection((srv.host, srv.port))
        ingest.set_gain_tcp(s, -7)
        assert _wait_cmds(srv, 2) == [(3, 1), (4, 0)]
        s.close()
    finally:
        srv.close()


def test_one_failing_dongle_stops_all_readers_and_leaves_sockets_usable():
    """a dongle that stalls must not leave the other reader threads writing into the buffer until their own timeout, and the
    sockets of the healthy dongles must come back blocking (a retry starts clean)"""
    D, N = 4, 20000
    srvs = _servers(D, 2 * N, seed=5)
    try:
        ing = ingest.DongleIngest([(s.host, s.port) for s in srvs], N, 957.4e6, 2166666.67, n_threads=4, timeout=1.0)
        ing.flush()
        srvs[2].close()                           # dongle 2 goes away
        time.sleep(0.2)
        t0 = time.time()
        with pytest.raises((ConnectionError, TimeoutError, OSError)):
            _read_until_gone(ing)
        assert time.time() - t0 < 20
        for d in (0, 1, 3):
            assert ing.socks[d].gettimeout() == 1.0      # handed back in blocking-with-timeout mode
        ing.close()
    finally:
        for s in srvs:
            s.close()


def test_short_stream_raises():
    srv = _servers(1, 1000)[0]
    try:
        ing = ingest.DongleIngest([(srv.host, srv.port)], 4000, 1e9, 2e6, timeout=1.0)
        ing.flush()
        srv.close()                               # server goes away mid-stream
        time.sleep(0.3)
        with pytest.raises((ConnectionError, TimeoutError, OSError)):
            _read_until_gone(ing)
        ing.close()
    finally:
        srv.close()


@pytest.mark.gpu
def test_ingest_calibrate_equals_direct(gpu):
    import torch
    from gsmcal import synth
    N = 1_020_000                                 # gsm_sync_demod.m:23-29
    specs = [synth.random_spec(seed, 2 * N + 8) for seed in (1, 2, 3)]
    raw = synth.generate_batch(specs, device="cuda").cpu().numpy()
    srvs = [ReplayDongle(raw[d]) for d in range(len(specs))]
    try:
        res = ingest.calibrate_from_dongles([(s.host, s.port) for s in srvs], N, 957.4e6, n_captures=1)[0]
    finally:
        for s in srvs:
            s.close()
    direct_in = np.stack([s.expected(2 * N - 12, 2 * N) for s in srvs])
    fs = (1625 / 6) * 1e3 * 8
    direct = gpu.calibrate_batch(direct_in, 957.4e6, gpu.gsm_SCH_training_sequence_gen(8), gpu.fir1(46, 200e3 / fs))
    assert len(res) == len(direct) == 3
    locked = 0
    for a, b in zip(res, direct):
        np.testing.assert_array_equal(a["pos_info"], b["pos_info"])
        np.testing.assert_array_equal(a["fcch_pos"], b["fcch_pos"])
        assert a["flags"] == b["flags"]
        assert a["total_sampling_ppm"] == b["total_sampling_ppm"] and a["total_carrier_ppm"] == b["total_carrier_ppm"]
        locked += int(np.isfinite(a["total_sampling_ppm"]))
    assert locked >= 2
    torch.cuda.synchronize()

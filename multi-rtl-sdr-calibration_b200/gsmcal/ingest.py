"""Streaming ingest from rtl_tcp servers into pinned double buffers (SURVEY.md §8(f) row 1).

Mirrors the capture side of the reference drivers, one TCP connection per dongle:
  * `set_gain_tcp` / `set_rate_tcp` / `set_freq_tcp`: the 5-byte rtl_tcp commands (1 command byte + uint32, network
    byte order - what MATLAB's `fwrite(tcp_obj, uint32(x), 'uint32')` puts on the wire with tcpip's default ByteOrder)
    — set_gain_tcp.m:8-16, set_rate_tcp.m:6-7, set_freq_tcp.m:6-7;
  * open -> gain -> rate -> freq -> one flush read of 2*num_sample bytes -> capture reads of 2*num_sample bytes per
    dongle (`gsm_sync_demod.m:57-98`).  Like the reference, the 12-byte "RTL0" greeting of rtl_tcp is not parsed: it
    is swallowed by the flush read (12 is even, so I/Q alignment survives).

`DongleIngest.captures()` fills one pinned [D, 2N] uint8 buffer (row d == the column `fread` returns for dongle d)
while the previous one is being calibrated: `gsmcal_calibrate_batch(raw_mem=HOST)` overlaps its own H2D copies with
its kernels, and the socket reads of the next capture overlap both (reader threads release the GIL in recv_into and
the ctypes call releases it for the whole library call).
"""
from __future__ import annotations

import selectors
import socket
import struct
import threading

import numpy as np

CMD_SET_FREQ, CMD_SET_RATE, CMD_SET_GAIN_MODE, CMD_SET_GAIN = 1, 2, 3, 4


def _send_cmd(sock: socket.socket, cmd: int, param: int) -> None:
    param = min(max(int(param), 0), 0xFFFFFFFF)                  # MATLAB's uint32() saturates (a negative gain becomes 0, not 4e9)
    sock.sendall(struct.pack(">BI", cmd, param))


def set_freq_tcp(sock: socket.socket, freq: float) -> socket.socket:
    """set_freq_tcp.m:5-7 (uint32() rounds to nearest)."""
    _send_cmd(sock, CMD_SET_FREQ, int(np.floor(freq + 0.5)))
    return sock


def set_rate_tcp(sock: socket.socket, rate: float) -> socket.socket:
    """set_rate_tcp.m:5-7."""
    _send_cmd(sock, CMD_SET_RATE, int(np.floor(rate + 0.5)))
    return sock


def set_gain_tcp(sock: socket.socket, gain: float) -> socket.socket:
    """set_gain_tcp.m:6-16: gain 0 -> automatic gain (mode 0); otherwise manual mode + gain in tenths of a dB."""
    if gain:
        _send_cmd(sock, CMD_SET_GAIN_MODE, 1)
        _send_cmd(sock, CMD_SET_GAIN, int(np.floor(gain + 0.5)))
    else:
        _send_cmd(sock, CMD_SET_GAIN_MODE, 0)
    return sock


def pinned_bytes(shape) -> np.ndarray:
    """Page-locked uint8 host buffer when a CUDA device is present (H2D at PCIe rate), pageable otherwise."""
    import torch
    if torch.cuda.is_available():
        t = torch.empty(shape, dtype=torch.uint8, pin_memory=True)
        a = t.numpy()
        _KEEP[a.ctypes.data] = t
        return a
    return np.empty(shape, dtype=np.uint8)


_KEEP: dict = {}


class DongleIngest:
    """D rtl_tcp connections read in lock-step captures of `num_sample` IQ samples each (2*num_sample bytes)."""

    def __init__(self, endpoints, num_sample: int, freq: float, rate: float, gain: float = 0, n_threads: int = 8,
                 timeout: float = 10.0, n_buffers: int = 2):
        self.endpoints = [(h, int(p)) for h, p in endpoints]
        self.num_sample = int(num_sample)
        self.timeout = float(timeout)
        self.n_threads = max(1, min(int(n_threads), len(self.endpoints)))
        self.socks = []
        for ep in self.endpoints:                                   # gsm_sync_demod.m:57-69
            s = socket.create_connection(ep, timeout=self.timeout)
            s.setsockopt(socket.IPPROTO_TCP, socket.TCP_NODELAY, 1)
            s.setsockopt(socket.SOL_SOCKET, socket.SO_RCVBUF, 4 << 20)
            self.socks.append(s)
        for s in self.socks:
            set_gain_tcp(s, gain)                                   # :72-74
        for s in self.socks:
            set_rate_tcp(s, rate)                                   # :77-79
        for s in self.socks:
            set_freq_tcp(s, freq)                                   # :82-84
        D = len(self.socks)
        self.buffers = [pinned_bytes((D, 2 * self.num_sample)) for _ in range(max(2, n_buffers))]
        self._flushed = False
        self.bytes_read = 0

    # ------------------------------------------------------------------------------------------------------------
    def _read_rows(self, buf: np.ndarray, rows: list[int], errors: list, stop: threading.Event) -> None:
        """One worker: multiplex its sockets, recv_into straight into the pinned rows.  A failure in ANY worker sets `stop`, so the
        others leave within one poll interval instead of writing into the buffer until their own timeout; the selector is always
        closed and the sockets are handed back blocking, so a retry of read_capture starts from a clean state."""
        sel = selectors.DefaultSelector()
        try:
            need = 2 * self.num_sample
            views = {d: memoryview(buf[d]) for d in rows}
            got = {d: 0 for d in rows}
            for d in rows:
                self.socks[d].setblocking(False)
                sel.register(self.socks[d], selectors.EVENT_READ, d)
            left = len(rows)
            waited = 0.0
            poll = min(0.2, self.timeout)
            while left and not stop.is_set():
                ev = sel.select(poll)
                if not ev:
                    waited += poll
                    if waited >= self.timeout:
                        raise TimeoutError(f"rtl_tcp read timed out; short rows: "
                                           f"{[(d, got[d]) for d in rows if got[d] < need][:4]}")
                    continue
                waited = 0.0
                for key, _ in ev:
                    d = key.data
                    n = key.fileobj.recv_into(views[d][got[d]:need])
                    if n == 0:
                        raise ConnectionError(f"dongle {d}: connection closed after {got[d]} of {need} bytes")
                    got[d] += n
                    if got[d] == need:
                        sel.unregister(key.fileobj)
                        left -= 1
        except Exception as e:                                      # surfaced by read_capture on the calling thread
            errors.append(e)
            stop.set()
        finally:
            sel.close()
            for d in rows:
                try:
                    self.socks[d].settimeout(self.timeout)
                except OSError:
                    pass

    def read_capture(self, buf: np.ndarray) -> np.ndarray:
        """The `fread(tcp_obj{i}, 2*num_sample, 'uint8')` loop of gsm_sync_demod.m:95-98 for all dongles at once."""
        D = len(self.socks)
        errors: list = []
        stop = threading.Event()
        parts = [list(range(t, D, self.n_threads)) for t in range(self.n_threads)]
        threads = [threading.Thread(target=self._read_rows, args=(buf, rows, errors, stop), daemon=True) for rows in parts[1:]]
        for t in threads:
            t.start()
        self._read_rows(buf, parts[0], errors, stop)
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        self.bytes_read += buf.size
        return buf

    def flush(self) -> None:
        """gsm_sync_demod.m:87-89: discard one capture's worth of bytes (this also eats the 12-byte RTL0 greeting)."""
        self.read_capture(self.buffers[0])
        self._flushed = True

    def captures(self, n: int):
        """Yield n captures; capture k+1 is read on a background thread while the consumer works on capture k.

        The yielded array is only valid until the consumer asks for the capture after the next one (ring of buffers)."""
        if not self._flushed:
            self.flush()
        nb = len(self.buffers)
        box: dict = {}

        def fill(i):
            try:
                box[i] = self.read_capture(self.buffers[i % nb])
            except Exception as e:
                box[i] = e
        th = threading.Thread(target=fill, args=(0,), daemon=True)
        th.start()
        for k in range(n):
            th.join()
            cur = box.pop(k)
            if isinstance(cur, Exception):
                raise cur
            if k + 1 < n:
                th = threading.Thread(target=fill, args=(k + 1,), daemon=True)
                th.start()
            yield cur

    def close(self) -> None:
        for s in self.socks:
            try:
                s.close()
            except OSError:
                pass
        for b in self.buffers:
            _KEEP.pop(b.ctypes.data, None)
        self.socks, self.buffers = [], []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def calibrate_from_dongles(endpoints, num_sample: int, freq: float, n_captures: int = 1, osr: int = 8,
                           coarse_dr: int = 8, gain: float = 0, details: bool = True, demod: bool = False,
                           sch_timing: bool = False, **kw):
    """gsm_sync_demod.m:57-124 with every dongle of `endpoints` in one batched library call per capture.

    Returns a list (one entry per capture) of the per-dongle result lists of `calibrate_batch`.  With demod=True the call is
    `calibrate_demod_batch` with the normal training sequences of gsm_sync_demod.m:39, so the whole per-dongle loop (:57-147: SCH_demod,
    FCCH_demod and BCCH_demod on every r_correct) runs, and each per-dongle dict carries its sch / fcch / bcch entries (details is
    ignored then).  With sch_timing=True (and demod False) the call is `calibrate_batch(..., sch_timing=True)`: each per-dongle dict
    carries its timing entry, every SCH burst timed to a fraction of a sample and the least-squares clock fit of the dongle."""
    from . import api
    fs = (1625.0 / 6.0) * 1e3 * osr
    coef = api.fir1(46, 200e3 / fs)                                 # gsm_sync_demod.m:34
    tpl = api.gsm_SCH_training_sequence_gen(osr)                    # :37
    nts = api.gsm_normal_training_sequence_gen(osr) if demod else None      # :39
    out = []
    with DongleIngest(endpoints, num_sample, freq, fs, gain, **kw) as ing:
        for buf in ing.captures(n_captures):
            if demod:
                out.append(api.calibrate_demod_batch(buf, freq, tpl, coef, osr, coarse_dr, normal_training_sequence=nts))
            else:
                out.append(api.calibrate_batch(buf, freq, tpl, coef, osr, coarse_dr, details=details, sch_timing=sch_timing))
    return out

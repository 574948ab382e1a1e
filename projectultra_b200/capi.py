"""ctypes binding of libpu_b200.so (include/pu/pu_capi.h).

This module is the thin Python view of the C ABI used by tests/ and bench.py.  numpy arrays are passed as HOST
buffers (PU_MEM_HOST), torch CUDA tensors as DEVICE buffers (PU_MEM_DEVICE) on torch's current stream.
There is no fallback of any kind: if the shared library is missing or no sm_100 GPU is usable the calls raise.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpu_b200.so")

PU_MEM_HOST, PU_MEM_DEVICE = 0, 1
DBPSK, BPSK, DQPSK, QPSK, D8PSK, QAM8, QAM16, QAM32, QAM64, QAM256 = 0, 1, 2, 3, 4, 5, 6, 7, 8, 10
R1_4, R1_3, R1_2, R2_3, R3_4, R5_6, R7_8 = range(7)
LDPC_N = 648


class PuError(RuntimeError):
    pass


class ModemConfig(C.Structure):
    """pu_modem_config: POD mirror of ultra::ModemConfig (include/ultra/types.hpp:139-234)."""
    _fields_ = [("sample_rate", C.c_uint32), ("center_freq", C.c_uint32), ("fft_size", C.c_uint32),
                ("num_carriers", C.c_uint32), ("cp_mode", C.c_uint32), ("symbol_guard", C.c_uint32),
                ("pilot_spacing", C.c_uint32), ("use_pilots", C.c_uint32), ("modulation", C.c_uint32),
                ("code_rate", C.c_uint32), ("output_scale", C.c_float), ("tx_cfo_hz", C.c_float)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PuError(f"{LIB_PATH} is missing: run `python -m projectultra_b200.build` "
                          "(the CUDA library is the product; there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.pu_status_string.restype = C.c_char_p
        L.pu_last_error.restype = C.c_char_p
        L.pu_kernel_launches.restype = C.c_uint64
        _lib = L
    return _lib


def check(status):
    if status != 0:
        L = lib()
        raise PuError(f"{L.pu_status_string(status).decode()}: {L.pu_last_error().decode()}")


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _ptr(x, ctype=None):
    if x is None:
        return None
    if _is_torch(x):
        return C.c_void_p(x.data_ptr())
    return C.c_void_p(x.ctypes.data)


def _space(*xs):
    dev = [_is_torch(x) and x.is_cuda for x in xs if x is not None]
    if any(dev) and not all(dev):
        raise PuError("mixing host and device buffers in one call")
    return PU_MEM_DEVICE if dev and dev[0] else PU_MEM_HOST


def _stream(space):
    if space == PU_MEM_DEVICE:
        import torch
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)
    return None


class Context:
    """pu_ctx: one per GPU (per process rank)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        check(lib().pu_init(int(device), C.byref(self._h)))
        self.device = device

    def close(self):
        if self._h:
            lib().pu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def sm_count(self):
        return lib().pu_device_sm_count(self._h)

    @property
    def kernel_launches(self):
        return int(lib().pu_kernel_launches(self._h))

    @property
    def transfer_bytes(self):
        """(host->device, device->host) bytes moved so far by pu_receive_decode_batch(PU_MEM_HOST) through this context."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        lib().pu_transfer_bytes(self._h, C.byref(a), C.byref(b))
        return int(a.value), int(b.value)

    def synchronize(self):
        check(lib().pu_synchronize(self._h, None))


class LdpcDecoder:
    """pu_ldpc: batched drop-in for ultra::LDPCDecoder (include/ultra/fec.hpp:48-77)."""

    def __init__(self, ctx, rate, max_iter=50):
        self.ctx = ctx
        self._h = C.c_void_p()
        check(lib().pu_ldpc_create(ctx._h, int(rate), int(max_iter), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().pu_ldpc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def k(self):
        return lib().pu_ldpc_info_bits(self._h)

    @property
    def info_bytes(self):
        return (self.k + 7) // 8

    @property
    def rate(self):
        return lib().pu_ldpc_rate(self._h)

    @property
    def num_edges(self):
        return lib().pu_ldpc_num_edges(self._h)

    def set_rate(self, rate):
        check(lib().pu_ldpc_set_rate(self._h, int(rate)))

    def set_max_iterations(self, n):
        check(lib().pu_ldpc_set_max_iterations(self._h, int(n)))

    def rows(self):
        out = []
        buf = (C.c_int32 * 16)()
        for i in range(648 - self.k):
            d = lib().pu_ldpc_row(self._h, i, buf, 16)
            out.append([buf[e] for e in range(d)])
        return out

    def frame_decode_batch(self, llr, num_codewords, frame_cap=None):
        """pu_frame_decode_batch: RxPipeline::decodeFrame for every row of llr [B, num_codewords * 648] at this decoder's rate ->
        (frames [B, frame_cap] uint8, frame_len [B], info [B, 5] = {success, frame_type, codewords ok, codewords failed, expected})."""
        tor = _is_torch(llr)
        if tor:
            import torch
            assert llr.dtype == torch.float32 and llr.dim() == 2 and llr.is_contiguous()
        else:
            llr = np.ascontiguousarray(llr, dtype=np.float32)
            if llr.ndim == 1:
                llr = llr.reshape(1, -1)
        B = llr.shape[0]
        assert llr.shape[1] == num_codewords * 648
        if frame_cap is None:
            frame_cap = num_codewords * ((lib().pu_ldpc_info_bits(self._h) + 7) // 8)
        frames = _like(llr, (B, frame_cap), np.uint8, "uint8")
        flen = _like(llr, (B,), np.int32, "int32")
        info = _like(llr, (B, 5), np.int32, "int32")
        sp = _space(llr, frames, flen, info)
        check(lib().pu_frame_decode_batch(self.ctx._h, self._h, _ptr(llr), C.c_size_t(B), C.c_size_t(num_codewords), _ptr(frames),
                                          C.c_size_t(frame_cap), _ptr(flen), _ptr(info), sp, _stream(sp)))
        return frames, flen, info

    def encode_batch(self, payload, out=None):
        """pu_ldpc_encode_batch: LDPCEncoder::encode of every row of payload [B, payload_bytes <= k / 8] uint8 (numpy => host, torch.cuda =>
        device) at this decoder's rate -> coded [B, 81] uint8.  `out` may have rows wider than 81 bytes (their padding is left as it is)."""
        B, nbytes = payload.shape
        payload, stride = _byte_rows(payload)
        out = _like(payload, (B, 81), np.uint8, "uint8") if out is None else out
        out, ostride = _byte_rows(out)
        assert out.shape[0] == B and out.shape[1] >= 81
        sp = _space(payload, out)
        check(lib().pu_ldpc_encode_batch(self._h, _ptr(payload), C.c_size_t(stride), C.c_size_t(nbytes), C.c_size_t(B), _ptr(out),
                                         C.c_size_t(ostride), sp, _stream(sp)))
        return out

    def frame_codewords(self, frame_bytes):
        """Codewords of a frame of frame_bytes bytes at this decoder's rate (pu_frame_encode_batch's query)."""
        n = C.c_size_t(0)
        check(lib().pu_frame_encode_batch(self._h, None, C.c_size_t(frame_bytes), C.c_size_t(frame_bytes), C.c_size_t(0), None, C.c_size_t(0),
                                          C.byref(n), 0, None))
        return int(n.value)

    def frame_encode_batch(self, frames, out=None):
        """pu_frame_encode_batch: v2::encodeFrameWithLDPC of every row of frames [B, frame_bytes] uint8 (numpy => host, torch.cuda => device)
        at this decoder's rate -> coded [B, n_codewords * 81] uint8.  `out` may have wider rows (their padding is left as it is).
        Returns (out, n_codewords)."""
        B, nbytes = frames.shape
        ncw = self.frame_codewords(nbytes)
        frames, stride = _byte_rows(frames)
        out = _like(frames, (B, ncw * 81), np.uint8, "uint8") if out is None else out
        out, ostride = _byte_rows(out)
        assert out.shape[0] == B and out.shape[1] >= ncw * 81
        n = C.c_size_t(0)
        sp = _space(frames, out)
        check(lib().pu_frame_encode_batch(self._h, _ptr(frames), C.c_size_t(stride), C.c_size_t(nbytes), C.c_size_t(B), _ptr(out),
                                          C.c_size_t(ostride), C.byref(n), sp, _stream(sp)))
        return out, int(n.value)

    def decode_batch(self, llr, info=None, ok=None, iters=None):
        """llr: [B, >=648] float32 (numpy => host, torch.cuda => device).  Returns (info_bytes, ok, iters)."""
        if _is_torch(llr):
            import torch
            assert llr.dtype == torch.float32 and llr.dim() == 2 and llr.stride(1) == 1
            B, stride = llr.shape[0], llr.stride(0)
            if info is None:
                info = torch.empty((B, self.info_bytes), dtype=torch.uint8, device=llr.device)
            if ok is None:
                ok = torch.empty(B, dtype=torch.uint8, device=llr.device)
            if iters is None:
                iters = torch.empty(B, dtype=torch.int32, device=llr.device)
            istride = info.stride(0)
        else:
            llr = np.ascontiguousarray(llr, dtype=np.float32)
            if llr.ndim == 1:
                llr = llr.reshape(1, -1)
            B, stride = llr.shape[0], llr.shape[1]
            if info is None:
                info = np.zeros((B, self.info_bytes), np.uint8)
            if ok is None:
                ok = np.zeros(B, np.uint8)
            if iters is None:
                iters = np.zeros(B, np.int32)
            istride = info.shape[1]
        sp = _space(llr, info, ok, iters)
        check(lib().pu_ldpc_decode_batch(self._h, _ptr(llr), C.c_size_t(stride), C.c_size_t(B), _ptr(info),
                                         C.c_size_t(istride), _ptr(ok), _ptr(iters), sp, _stream(sp)))
        return info, ok, iters

    def decode_soft(self, llr):
        """LDPCDecoder::decodeSoft on host memory -> (bytes, lastDecodeSuccess, lastIterations)."""
        x = np.ascontiguousarray(llr, dtype=np.float32)
        out = np.zeros(128 * (len(x) // 648 + 2), np.uint8)
        n, ok, it = C.c_size_t(0), C.c_int(0), C.c_int(0)
        check(lib().pu_ldpc_decode_soft(self._h, _ptr(x), C.c_size_t(len(x)), _ptr(out), C.c_size_t(len(out)),
                                        C.byref(n), C.byref(ok), C.byref(it)))
        return out[:n.value].copy(), bool(ok.value), it.value

    def decode_hard(self, coded):
        d = np.ascontiguousarray(np.frombuffer(bytes(coded), np.uint8) if isinstance(coded, (bytes, bytearray))
                                 else coded, dtype=np.uint8)
        out = np.zeros(128 * (len(d) // 81 + 2), np.uint8)
        n, ok, it = C.c_size_t(0), C.c_int(0), C.c_int(0)
        check(lib().pu_ldpc_decode_hard(self._h, _ptr(d), C.c_size_t(len(d)), _ptr(out), C.c_size_t(len(out)),
                                        C.byref(n), C.byref(ok), C.byref(it)))
        return out[:n.value].copy(), bool(ok.value), it.value


def chirp_search_stats():
    """(searches, coarse verification rounds, fine runs) of the two-tier chirp search on the current device since the last call."""
    a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    check(lib().pu_chirp_search_stats(C.byref(a), C.byref(b), C.byref(c)))
    return int(a.value), int(b.value), int(c.value)


def tools_apply_cfo(samples, cfo_hz, sample_rate=48000.0):
    """pu_tools_apply_cfo: the reference tools' FFT-Hilbert CFO injector (tools/test_iwaveform.cpp:67-118) on a copy of `samples`."""
    x = np.ascontiguousarray(samples, np.float32).copy()
    check(lib().pu_tools_apply_cfo(_ptr(x), C.c_size_t(len(x)), C.c_float(cfo_hz), C.c_float(sample_rate)))
    return x


class ToolsCfo:
    """pu_tools_cfo: the same injector on the GPU for every row of a batch, bit-identical to tools_apply_cfo row by row."""

    def __init__(self, ctx, n, cfo_hz, sample_rate=48000.0):
        self.ctx, self.n = ctx, int(n)
        self._h = C.c_void_p()
        check(lib().pu_tools_cfo_create(ctx._h, C.c_size_t(self.n), C.c_float(cfo_hz), C.c_float(sample_rate), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().pu_tools_cfo_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def apply_batch(self, x):
        """In place on the first n samples of every row of x [B, stride] (float32, rows contiguous; numpy => host, torch.cuda => device
        on torch's current stream).  Returns x."""
        if _is_torch(x):
            import torch
            assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
            B, stride = x.shape[0], x.stride(0)
        else:
            assert x.dtype == np.float32 and x.ndim == 2 and x.strides[1] == 4 and x.strides[0] % 4 == 0
            B, stride = x.shape[0], x.strides[0] // 4
        sp = _space(x)
        check(lib().pu_tools_cfo_apply_batch(self._h, _ptr(x), C.c_size_t(B), C.c_size_t(stride), sp, _stream(sp)))
        return x


def chirp_phase_cycles():
    """Cycles per phase of the two-tier chirp search since the last call (pu_chirp_phase_cycles)."""
    out = (C.c_uint64 * 8)()
    check(lib().pu_chirp_phase_cycles(out))
    return [int(v) for v in out]


def chirp_generate(sample_rate=48000.0, tx_cfo_hz=0.0):
    """ChirpSync::generate (host): [up chirp][gap][down chirp][gap]."""
    n = C.c_size_t(0)
    check(lib().pu_chirp_generate(C.c_float(sample_rate), C.c_float(tx_cfo_hz), None, C.c_size_t(0), C.byref(n)))
    out = np.zeros(n.value, np.float32)
    check(lib().pu_chirp_generate(C.c_float(sample_rate), C.c_float(tx_cfo_hz), _ptr(out), C.c_size_t(len(out)), C.byref(n)))
    return out


def ldpc_encode(rate, data):
    """LDPCEncoder::encode (host)."""
    d = np.ascontiguousarray(np.frombuffer(bytes(data), np.uint8) if isinstance(data, (bytes, bytearray)) else data,
                             dtype=np.uint8)
    out = np.zeros(81 * (len(d) * 8 // 162 + 2), np.uint8)
    n = C.c_size_t(0)
    check(lib().pu_ldpc_encode(int(rate), _ptr(d), C.c_size_t(len(d)), _ptr(out), C.c_size_t(len(out)), C.byref(n)))
    return out[:n.value].copy()


def frame_encode(rate, frame):
    """pu_frame_encode: v2::encodeFrameWithLDPC(frame, rate) (host) -> uint8 [n_codewords, 81]."""
    f = np.ascontiguousarray(np.frombuffer(bytes(frame), np.uint8) if isinstance(frame, (bytes, bytearray)) else frame, dtype=np.uint8)
    n = C.c_size_t(0)
    check(lib().pu_frame_encode(int(rate), _ptr(f), C.c_size_t(len(f)), None, C.c_size_t(0), C.byref(n)))
    out = np.zeros((n.value, 81), np.uint8)
    check(lib().pu_frame_encode(int(rate), _ptr(f), C.c_size_t(len(f)), _ptr(out), C.c_size_t(out.size), C.byref(n)))
    return out


def _byte_rows(x):
    """(x, row stride in bytes) of a 2-D uint8 array whose rows are contiguous (numpy arrays are made so)."""
    if _is_torch(x):
        import torch
        assert x.dtype == torch.uint8 and x.dim() == 2 and x.stride(1) == 1
        return x, x.stride(0)
    if not (x.dtype == np.uint8 and x.ndim == 2 and x.strides[1] == 1):
        x = np.ascontiguousarray(x, dtype=np.uint8)
    return x, x.strides[0]


def count_raw_errors(ctx, llr, coded, counters, n_bits=None, n_valid=None, coded_index=None, bins=None, strong=10.0):
    """pu_count_raw_errors on device tensors, torch's current stream: soft bits llr [B, >= n_bits] float32 (decoder order) against the
    coded bytes sent, row coded_index[b] of coded [P, >= n_bits / 8] uint8 (None = row b); positions >= n_valid[b] (int32 [B], None = all)
    and soft bits equal to +-0 are erasures.  counters: torch.int64 [n_bins, 4] (RAW_COUNTER_NAMES of linksim) accumulated in place at
    row bins[b] (None = row 0).  n_bits defaults to the width of llr."""
    import torch
    assert llr.dtype == torch.float32 and llr.dim() == 2 and llr.stride(1) == 1 and coded.dtype == torch.uint8 and coded.stride(-1) == 1
    assert counters.dtype == torch.int64 and counters.is_contiguous() and counters.shape[-1] == 4
    B = llr.shape[0]
    n = llr.shape[1] if n_bits is None else int(n_bits)
    check(lib().pu_count_raw_errors(ctx._h, _ptr(llr), C.c_size_t(llr.stride(0)), C.c_size_t(n), _ptr(n_valid), _ptr(coded),
                                    C.c_size_t(coded.stride(0)), _ptr(coded_index), _ptr(bins), C.c_size_t(B), C.c_float(strong),
                                    _ptr(counters), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return counters


def channel_interleaver_perm(bps, total=648):
    perm = np.zeros(total, np.uint32)
    inv = np.zeros(total, np.uint32)
    step = C.c_size_t(0)
    check(lib().pu_channel_interleaver_perm(C.c_size_t(bps), C.c_size_t(total), _ptr(perm), _ptr(inv), C.byref(step)))
    return perm, inv, step.value


def llr_deinterleave_batch(ctx, llr, n_blocks, bps):
    """pu_llr_deinterleave_batch: ChannelInterleaver(bps, 648)::deinterleave IN PLACE on the first n_blocks * 648 soft bits of every row
    of llr [B, stride] (float32, rows contiguous; numpy => host, torch.cuda => device on torch's current stream), each 648-bit block on
    its own.  Returns llr."""
    if _is_torch(llr):
        import torch
        assert llr.dtype == torch.float32 and llr.dim() == 2 and llr.stride(1) == 1
        B, stride = llr.shape[0], llr.stride(0)
    else:
        assert llr.dtype == np.float32 and llr.ndim == 2 and llr.strides[1] == 4 and llr.strides[0] % 4 == 0
        B, stride = llr.shape[0], llr.strides[0] // 4
    sp = _space(llr)
    check(lib().pu_llr_deinterleave_batch(ctx._h, _ptr(llr), C.c_size_t(B), C.c_size_t(stride), C.c_size_t(n_blocks), C.c_size_t(bps),
                                          sp, _stream(sp)))
    return llr


def block_interleaver_perm(rows, cols):
    perm = np.zeros(rows * cols, np.uint32)
    check(lib().pu_block_interleaver_perm(C.c_size_t(rows), C.c_size_t(cols), _ptr(perm)))
    return perm


class OfdmDemodulator:
    """pu_ofdm: batched drop-in for ultra::OFDMDemodulator's presynced path (include/ultra/ofdm.hpp:58-127)."""
    DBG_SCALARS = 10

    def __init__(self, ctx, cfg):
        self.ctx = ctx
        self.cfg = cfg
        self._h = C.c_void_p()
        check(lib().pu_ofdm_create(ctx._h, C.byref(cfg), C.byref(self._h)))
        self.symbol_samples = lib().pu_ofdm_symbol_samples(self._h)
        self.n_data = lib().pu_ofdm_data_carriers(self._h)
        self.n_pilot = lib().pu_ofdm_pilot_carriers(self._h)
        self.bits_per_symbol = lib().pu_ofdm_bits_per_symbol(self._h)

    def close(self):
        if self._h:
            lib().pu_ofdm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    KERNELS = {0: "none", 1: "ofdm_presynced_kernel", 2: "ofdm_diff_kernel", 3: "ofdm_diff512_kernel",
               4: "ofdm_presynced_warp_kernel", 5: "ofdm_fast512_kernel", 6: "ofdm_presynced_warp_fast_kernel"}

    @property
    def last_kernel(self):
        """Name of the kernel the last launch on this handle used (pu_ofdm_last_kernel)."""
        return self.KERNELS[lib().pu_ofdm_last_kernel(self._h)]

    def carrier_bins(self):
        buf = (C.c_int32 * 128)()
        n = lib().pu_ofdm_carrier_bins(self._h, buf, 128)
        return np.array(buf[:n], dtype=np.int32)

    def set_precision(self, mode):
        """'exact' (default: FFT bins bit-identical to the reference) or 'fast' (FMA butterflies, LLRs within 1e-4):
        pu_ofdm_set_precision."""
        check(lib().pu_ofdm_set_precision(self._h, {"exact": 0, "fast": 1}[mode]))

    @property
    def precision(self):
        return {0: "exact", 1: "fast"}[lib().pu_ofdm_get_precision(self._h)]

    def set_deinterleave(self, bits_per_symbol, total_bits=648):
        check(lib().pu_ofdm_set_deinterleave(self._h, C.c_size_t(bits_per_symbol), C.c_size_t(total_bits)))

    def set_tx_interleave(self, bits_per_symbol):
        """pu_ofdm_set_tx_interleave: ChannelInterleaver(bits_per_symbol, 648) on every codeword of tx_batch / frame_tx_batch; 0 = off."""
        check(lib().pu_ofdm_set_tx_interleave(self._h, C.c_size_t(bits_per_symbol)))

    def n_llr(self, L, training=2):
        return max(0, L // self.symbol_samples - training) * self.bits_per_symbol

    def presynced_batch(self, samples, training=2, cfo_hz=None, cfo_phase=None, llr_stride=None, llr=None,
                        snr_db=None, final_cfo=None, want_aux=True):
        """samples [B, L] float32 (numpy => host, torch.cuda => device) -> (llr [B, llr_stride], snr_db, final_cfo)."""
        tor = _is_torch(samples)
        if tor:
            import torch
            assert samples.dtype == torch.float32 and samples.dim() == 2 and samples.is_contiguous()
            B, L = samples.shape
        else:
            samples = np.ascontiguousarray(samples, dtype=np.float32)
            if samples.ndim == 1:
                samples = samples.reshape(1, -1)
            B, L = samples.shape
        if llr_stride is None:
            llr_stride = self.n_llr(L, training) if llr is None else llr.shape[1]
        if tor:
            import torch
            if llr is None:
                llr = torch.zeros((B, llr_stride), dtype=torch.float32, device=samples.device)
            if want_aux and snr_db is None:
                snr_db = torch.empty(B, dtype=torch.float32, device=samples.device)
            if want_aux and final_cfo is None:
                final_cfo = torch.empty(B, dtype=torch.float32, device=samples.device)
        else:
            if llr is None:
                llr = np.zeros((B, llr_stride), np.float32)
            if want_aux and snr_db is None:
                snr_db = np.zeros(B, np.float32)
            if want_aux and final_cfo is None:
                final_cfo = np.zeros(B, np.float32)
            if cfo_hz is not None:
                cfo_hz = np.ascontiguousarray(cfo_hz, dtype=np.float32)
            if cfo_phase is not None:
                cfo_phase = np.ascontiguousarray(cfo_phase, dtype=np.float32)
        sp = _space(samples, llr, cfo_hz, cfo_phase, snr_db, final_cfo)
        check(lib().pu_ofdm_presynced_batch(self._h, _ptr(samples), C.c_size_t(B), C.c_size_t(L), int(training),
                                            _ptr(cfo_hz), _ptr(cfo_phase), _ptr(llr), C.c_size_t(llr_stride),
                                            _ptr(snr_db), _ptr(final_cfo), sp, _stream(sp)))
        return llr, snr_db, final_cfo

    def training_cfo_batch(self, samples, training=2):
        """pu_ofdm_training_cfo_batch: estimateCFOFromTraining of every row of samples [B, L] -> cfo_hz [B]."""
        samples = _frames(samples)
        B, L = samples.shape
        out = _like(samples, (B,), np.float32, "float32")
        sp = _space(samples, out)
        check(lib().pu_ofdm_training_cfo_batch(self._h, _ptr(samples), C.c_size_t(B), C.c_size_t(L), int(training), _ptr(out), sp, _stream(sp)))
        return out

    def tx_frame_len(self, ldpc, layout=0):
        n = C.c_size_t(0)
        check(lib().pu_ofdm_tx_batch(self._h, ldpc._h, None, C.c_size_t(0), C.c_size_t(0), C.c_size_t(0), int(layout), C.c_float(0.0),
                                     None, C.c_size_t(0), C.byref(n), 0, None))
        return int(n.value)

    def tx_batch(self, ldpc, payload, layout=0, peak=0.0, out=None):
        """pu_ofdm_tx_batch: payload [B, payload_bytes] uint8 (numpy or torch.cuda) -> frames [B, L] float32: LDPC encode (the
        rate of `ldpc`) + training symbols / Schmidl-Cox preamble + modulate, optionally rescaled to `peak`."""
        tor = _is_torch(payload)
        B, nbytes = payload.shape
        L = self.tx_frame_len(ldpc, layout)
        if tor:
            import torch
            assert payload.dtype == torch.uint8 and payload.dim() == 2
            stride = payload.stride(0)
            if out is None:
                out = torch.empty((B, L), dtype=torch.float32, device=payload.device)
        else:
            payload = np.ascontiguousarray(payload, dtype=np.uint8)
            stride = payload.shape[1]
            if out is None:
                out = np.zeros((B, L), np.float32)
        n = C.c_size_t(0)
        sp = _space(payload, out)
        ostride = out.stride(0) if tor else out.shape[1]
        check(lib().pu_ofdm_tx_batch(self._h, ldpc._h, _ptr(payload), C.c_size_t(stride), C.c_size_t(nbytes), C.c_size_t(B), int(layout),
                                     C.c_float(peak), _ptr(out), C.c_size_t(ostride), C.byref(n), sp, _stream(sp)))
        return out

    def frame_tx_batch(self, ldpc, frames, layout=0, peak=0.0, out=None):
        """pu_frame_tx_batch: frames [B, frame_bytes] uint8 (numpy or torch.cuda) -> waveforms [B, L] float32: v2::encodeFrameWithLDPC at the
        rate of `ldpc` + training symbols / Schmidl-Cox preamble + every codeword modulated back to back, optionally rescaled to `peak`.
        `out` may be wider than L (its padding is left as it is).  Returns (out, n_codewords)."""
        tor = _is_torch(frames)
        B, nbytes = frames.shape
        L, ncw = C.c_size_t(0), C.c_size_t(0)
        check(lib().pu_frame_tx_batch(self._h, ldpc._h, None, C.c_size_t(nbytes), C.c_size_t(nbytes), C.c_size_t(0), int(layout), C.c_float(0.0),
                                      None, C.c_size_t(0), C.byref(L), C.byref(ncw), 0, None))
        if tor:
            import torch
            assert frames.dtype == torch.uint8 and frames.dim() == 2 and frames.stride(1) == 1
            stride = frames.stride(0)
            if out is None:
                out = torch.empty((B, L.value), dtype=torch.float32, device=frames.device)
        else:
            frames = np.ascontiguousarray(frames, dtype=np.uint8)
            stride = frames.shape[1]
            if out is None:
                out = np.zeros((B, L.value), np.float32)
        assert out.shape[0] == B and out.shape[1] >= L.value
        sp = _space(frames, out)
        ostride = out.stride(0) if tor else out.strides[0] // 4
        check(lib().pu_frame_tx_batch(self._h, ldpc._h, _ptr(frames), C.c_size_t(stride), C.c_size_t(nbytes), C.c_size_t(B), int(layout),
                                      C.c_float(peak), _ptr(out), C.c_size_t(ostride), C.byref(L), C.byref(ncw), sp, _stream(sp)))
        return out, int(ncw.value)

    def chirp_receive_batch(self, samples, threshold=0.15, llr_stride=648, want_llr=True):
        """pu_ofdm_chirp_receive_batch: dual-chirp detectSync + setFrequencyOffset + process + getSoftBits for every row of
        samples [B, L] -> (llr [B, llr_stride], n_llr [B], sync_info [B, 4] int32, sync_values [B, 4] float32, snr_db [B])."""
        tor = _is_torch(samples)
        if tor:
            import torch
            assert samples.dtype == torch.float32 and samples.dim() == 2 and samples.is_contiguous()
            B, L = samples.shape
            dev = samples.device
            llr = torch.zeros((B, llr_stride), dtype=torch.float32, device=dev) if want_llr else None
            n = torch.zeros(B, dtype=torch.int32, device=dev)
            info = torch.zeros((B, 4), dtype=torch.int32, device=dev)
            val = torch.zeros((B, 4), dtype=torch.float32, device=dev)
            snr = torch.zeros(B, dtype=torch.float32, device=dev)
        else:
            samples = np.ascontiguousarray(samples, dtype=np.float32)
            if samples.ndim == 1:
                samples = samples.reshape(1, -1)
            B, L = samples.shape
            llr = np.zeros((B, llr_stride), np.float32) if want_llr else None
            n = np.zeros(B, np.int32)
            info = np.zeros((B, 4), np.int32)
            val = np.zeros((B, 4), np.float32)
            snr = np.zeros(B, np.float32)
        sp = _space(samples, n, info, val, snr)
        check(lib().pu_ofdm_chirp_receive_batch(self._h, _ptr(samples), C.c_size_t(B), C.c_size_t(L), C.c_float(threshold), _ptr(llr),
                                                C.c_size_t(llr_stride), _ptr(n), _ptr(info), _ptr(val), _ptr(snr), sp, _stream(sp)))
        return llr, n, info, val, snr

    def acquire_batch(self, samples, chunk=960, sync_threshold=0.0):
        """pu_ofdm_acquire_batch: samples [B, L] (numpy or torch.cuda) -> (sync_info [B, 4] int32 = {synced, sync offset,
        samples consumed before the first data symbol, process() calls}, coarse_cfo_hz [B])."""
        tor = _is_torch(samples)
        if tor:
            import torch
            assert samples.dtype == torch.float32 and samples.dim() == 2 and samples.is_contiguous()
            B, L = samples.shape
            info = torch.zeros((B, 4), dtype=torch.int32, device=samples.device)
            cfo = torch.zeros(B, dtype=torch.float32, device=samples.device)
        else:
            samples = np.ascontiguousarray(samples, dtype=np.float32)
            if samples.ndim == 1:
                samples = samples.reshape(1, -1)
            B, L = samples.shape
            info = np.zeros((B, 4), np.int32)
            cfo = np.zeros(B, np.float32)
        sp = _space(samples, info, cfo)
        check(lib().pu_ofdm_acquire_batch(self._h, _ptr(samples), C.c_size_t(B), C.c_size_t(L), C.c_size_t(chunk),
                                          C.c_float(sync_threshold), _ptr(info), _ptr(cfo), sp, _stream(sp)))
        return info, cfo

    def process_batch(self, samples, chunk=960, llr_stride=648, sync_threshold=0.0):
        """pu_ofdm_process_batch: OFDMDemodulator::process fed in chunk-sample pieces + getSoftBits() for every row of
        samples [B, L] -> (llr [B, llr_stride], n_llr [B], sync_info [B, 4], coarse_cfo_hz [B], snr_db [B])."""
        tor = _is_torch(samples)
        if tor:
            import torch
            assert samples.dtype == torch.float32 and samples.dim() == 2 and samples.is_contiguous()
            B, L = samples.shape
            dev = samples.device
            llr = torch.zeros((B, llr_stride), dtype=torch.float32, device=dev)
            n = torch.zeros(B, dtype=torch.int32, device=dev)
            info = torch.zeros((B, 4), dtype=torch.int32, device=dev)
            cfo = torch.zeros(B, dtype=torch.float32, device=dev)
            snr = torch.zeros(B, dtype=torch.float32, device=dev)
        else:
            samples = np.ascontiguousarray(samples, dtype=np.float32)
            if samples.ndim == 1:
                samples = samples.reshape(1, -1)
            B, L = samples.shape
            llr = np.zeros((B, llr_stride), np.float32)
            n = np.zeros(B, np.int32)
            info = np.zeros((B, 4), np.int32)
            cfo = np.zeros(B, np.float32)
            snr = np.zeros(B, np.float32)
        sp = _space(samples, llr, n, info, cfo, snr)
        check(lib().pu_ofdm_process_batch(self._h, _ptr(samples), C.c_size_t(B), C.c_size_t(L), C.c_size_t(chunk),
                                          C.c_float(sync_threshold), _ptr(llr), C.c_size_t(llr_stride), _ptr(n), _ptr(info),
                                          _ptr(cfo), _ptr(snr), sp, _stream(sp)))
        return llr, n, info, cfo, snr

    def presynced_debug(self, samples, training=2, cfo_hz=0.0, cfo_phase=0.0):
        x = np.ascontiguousarray(samples, dtype=np.float32)
        L = len(x)
        nds = max(0, L // self.symbol_samples - training)
        nd, nu = self.n_data, self.n_data + self.n_pilot
        rec = 4 * nu + 3 * nd + self.DBG_SCALARS
        records = np.zeros(max(nds, 1) * rec, np.float32)
        cap = max(self.n_llr(L, training), 1)
        llr = np.zeros(cap, np.float32)
        n = C.c_int(0)
        check(lib().pu_ofdm_presynced_debug(self._h, _ptr(x), C.c_size_t(L), int(training), C.c_float(cfo_hz),
                                            C.c_float(cfo_phase), _ptr(llr), C.c_size_t(cap), _ptr(records),
                                            C.c_size_t(len(records)), C.byref(n)))
        r = records[: nds * rec].reshape(nds, rec)
        cplx = lambda a: np.ascontiguousarray(a).view(np.complex64)
        return dict(n_sym=nds, carriers=self.carrier_bins(), llr=llr[: self.n_llr(L, training)],
                    bins=cplx(r[:, : 2 * nu]), h=cplx(r[:, 2 * nu: 4 * nu]), eq=cplx(r[:, 4 * nu: 4 * nu + 2 * nd]),
                    nv=r[:, 4 * nu + 2 * nd: 4 * nu + 3 * nd].copy(), scalars=r[:, 4 * nu + 3 * nd:].copy())


# ------------------------------------------------------------------------------------------------ DPSK waveforms
class DpskConfig(C.Structure):
    """pu_dpsk_config: POD mirror of ultra::DPSKConfig (src/psk/dpsk.hpp:42-50).  modulation 0 DBPSK, 1 DQPSK, 2 D8PSK."""
    _fields_ = [("sample_rate", C.c_float), ("carrier_freq", C.c_float), ("samples_per_symbol", C.c_uint32),
                ("modulation", C.c_uint32)]


class McDpskConfig(C.Structure):
    """pu_mcdpsk_config: POD mirror of ultra::MultiCarrierDPSKConfig (src/psk/multi_carrier_dpsk.hpp:26-89)."""
    _fields_ = [("sample_rate", C.c_float), ("freq_low", C.c_float), ("freq_high", C.c_float), ("num_carriers", C.c_uint32),
                ("samples_per_symbol", C.c_uint32), ("bits_per_symbol", C.c_uint32), ("training_symbols", C.c_uint32)]


def dpsk_config(mod=1, sps=384, fc=1500.0, fs=48000.0):
    return DpskConfig(fs, fc, sps, mod)


def mcdpsk_config(nc=8, bits=2, sps=512, f_lo=500.0, f_hi=2500.0, fs=48000.0, training=8):
    return McDpskConfig(fs, f_lo, f_hi, nc, sps, bits, training)


def _tx_call(fn, *args):
    n = C.c_size_t(0)
    fn(*args, None, C.c_size_t(0), C.byref(n))
    out = np.zeros(n.value, np.float32)
    check(fn(*args, _ptr(out), C.c_size_t(len(out)), C.byref(n)))
    return out


def dpsk_tx(cfg, data, layout=0):
    """pu_dpsk_tx: DPSKModulator on the host (layout 0 Barker preamble + data, 1 reference symbol + data, 2 data only)."""
    d = np.ascontiguousarray(data, dtype=np.uint8)
    return _tx_call(lib().pu_dpsk_tx, C.byref(cfg), int(layout), _ptr(d), C.c_size_t(len(d)))


def mcdpsk_tx(cfg, data):
    """pu_mcdpsk_tx: training sequence + reference symbol + data (MultiCarrierDPSKModulator, host)."""
    d = np.ascontiguousarray(data, dtype=np.uint8)
    return _tx_call(lib().pu_mcdpsk_tx, C.byref(cfg), _ptr(d), C.c_size_t(len(d)))


def _frames(samples):
    if _is_torch(samples):
        import torch
        assert samples.dtype == torch.float32 and samples.dim() == 2 and samples.is_contiguous()
        return samples
    s = np.ascontiguousarray(samples, dtype=np.float32)
    return s.reshape(1, -1) if s.ndim == 1 else s


def _like(samples, shape, dtype_np, dtype_torch_name):
    if _is_torch(samples):
        import torch
        return torch.zeros(shape, dtype=getattr(torch, dtype_torch_name), device=samples.device)
    return np.zeros(shape, dtype_np)


def _psk_tx_batch(fn, h, ldpc, payload, peak, out):
    """Shared body of DpskDemodulator.tx_batch / McDpskDemodulator.tx_batch (pu_dpsk_tx_batch / pu_mcdpsk_tx_batch)."""
    n = C.c_size_t(0)
    check(fn(h, ldpc._h, None, C.c_size_t(0), C.c_size_t(0), C.c_size_t(0), C.c_float(0.0), None, C.c_size_t(0), C.byref(n), 0, None))
    L = n.value
    tor = _is_torch(payload)
    if tor:
        import torch
        assert payload.dtype == torch.uint8 and payload.dim() == 2
        B = payload.shape[0]
        out = torch.empty((B, L), dtype=torch.float32, device=payload.device) if out is None else out
        stride = payload.stride(0)
    else:
        payload = np.ascontiguousarray(payload, dtype=np.uint8)
        B = payload.shape[0]
        out = np.zeros((B, L), np.float32) if out is None else out
        stride = payload.shape[1]
    sp = _space(payload, out)
    check(fn(h, ldpc._h, _ptr(payload), C.c_size_t(stride), C.c_size_t(payload.shape[1]), C.c_size_t(B), C.c_float(peak), _ptr(out),
             C.c_size_t(L), C.byref(n), sp, _stream(sp)))
    return out


class DpskDemodulator:
    """pu_dpsk: batched drop-in for ultra::DPSKDemodulator::demodulateSoft with external timing."""

    def __init__(self, ctx, cfg):
        self.ctx, self.cfg = ctx, cfg
        self._h = C.c_void_p()
        check(lib().pu_dpsk_create(ctx._h, C.byref(cfg), C.byref(self._h)))
        self.bits_per_symbol = lib().pu_dpsk_bits_per_symbol(self._h)

    def close(self):
        if self._h:
            lib().pu_dpsk_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def tx_batch(self, ldpc, payload, peak=0.0, out=None):
        """pu_dpsk_tx_batch: LDPC encode + Barker preamble + DPSK modulate for every row of payload [B, bytes] on the GPU."""
        return _psk_tx_batch(lib().pu_dpsk_tx_batch, self._h, ldpc, payload, peak, out)

    def n_llr(self, L, data_start):
        return max(0, (L - data_start) // self.cfg.samples_per_symbol) * self.bits_per_symbol

    def receive_batch(self, samples, llr_stride=648, want_llr=True):
        """pu_dpsk_receive_batch: findPreamble + demodulateSoft (tools/test_dpsk_snr.cpp:66-73) for every row of samples [B, L]
        -> (llr [B, llr_stride], n_llr [B], data_start [B], est_cfo_hz [B], phase_offset [B])."""
        tor = _is_torch(samples)
        if tor:
            import torch
            assert samples.dtype == torch.float32 and samples.dim() == 2 and samples.is_contiguous()
            B, L = samples.shape
            dev = samples.device
            llr = torch.zeros((B, llr_stride), dtype=torch.float32, device=dev) if want_llr else None
            n = torch.zeros(B, dtype=torch.int32, device=dev)
            ds = torch.zeros(B, dtype=torch.int32, device=dev)
            cfo = torch.zeros(B, dtype=torch.float32, device=dev)
            ph = torch.zeros(B, dtype=torch.float32, device=dev)
        else:
            samples = np.ascontiguousarray(samples, dtype=np.float32)
            if samples.ndim == 1:
                samples = samples.reshape(1, -1)
            B, L = samples.shape
            llr = np.zeros((B, llr_stride), np.float32) if want_llr else None
            n = np.zeros(B, np.int32)
            ds = np.zeros(B, np.int32)
            cfo = np.zeros(B, np.float32)
            ph = np.zeros(B, np.float32)
        sp = _space(samples, n, ds, cfo, ph)
        check(lib().pu_dpsk_receive_batch(self._h, _ptr(samples), C.c_size_t(B), C.c_size_t(L), _ptr(llr), C.c_size_t(llr_stride), _ptr(n),
                                          _ptr(ds), _ptr(cfo), _ptr(ph), sp, _stream(sp)))
        return llr, n, ds, cfo, ph

    def demod_soft_batch(self, samples, data_start, ref_mode=1, est_cfo=None, phase_off=None, llr_stride=None, llr=None):
        x = _frames(samples)
        B, L = x.shape
        if llr_stride is None:
            llr_stride = max(self.n_llr(L, data_start), 1) if llr is None else llr.shape[1]
        if llr is None:
            llr = _like(x, (B, llr_stride), np.float32, "float32")
        if not _is_torch(x):
            est_cfo = None if est_cfo is None else np.ascontiguousarray(est_cfo, dtype=np.float32)
            phase_off = None if phase_off is None else np.ascontiguousarray(phase_off, dtype=np.float32)
        sp = _space(x, llr, est_cfo, phase_off)
        check(lib().pu_dpsk_demod_soft_batch(self._h, _ptr(x), C.c_size_t(B), C.c_size_t(L), C.c_size_t(data_start), int(ref_mode),
                                             _ptr(est_cfo), _ptr(phase_off), _ptr(llr), C.c_size_t(llr_stride), sp, _stream(sp)))
        return llr


class McDpskDemodulator:
    """pu_mcdpsk: batched drop-in for ultra::MultiCarrierDPSKDemodulator (setReference + demodulateSoft, external timing)."""

    def __init__(self, ctx, cfg):
        self.ctx, self.cfg = ctx, cfg
        self._h = C.c_void_p()
        check(lib().pu_mcdpsk_create(ctx._h, C.byref(cfg), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().pu_mcdpsk_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def tx_batch(self, ldpc, payload, peak=0.0, out=None):
        """pu_mcdpsk_tx_batch: LDPC encode + training + reference + MC-DPSK modulate for every row of payload [B, bytes] on the GPU."""
        return _psk_tx_batch(lib().pu_mcdpsk_tx_batch, self._h, ldpc, payload, peak, out)

    def set_tx_interleave(self, bits_per_symbol):
        """pu_mcdpsk_set_tx_interleave: ChannelInterleaver(bits_per_symbol, 648) on the codeword of tx_batch; 0 = off."""
        check(lib().pu_mcdpsk_set_tx_interleave(self._h, C.c_size_t(bits_per_symbol)))

    def n_llr(self, L):
        c = self.cfg
        return max(0, L // c.samples_per_symbol - c.training_symbols - 1) * c.num_carriers * c.bits_per_symbol

    def got_chirp_batch(self, samples, chirp_cfo_hz, llr_stride=648):
        """pu_mcdpsk_got_chirp_batch: setChirpDetected(cfo) -> process(training + ref + data) -> getSoftBits for every row of
        samples [B, L] -> (llr [B, llr_stride], n_llr [B], cfo_after_hz [B])."""
        tor = _is_torch(samples)
        if tor:
            import torch
            assert samples.dtype == torch.float32 and samples.dim() == 2 and samples.is_contiguous()
            B, L = samples.shape
            dev = samples.device
            cfo = torch.as_tensor(chirp_cfo_hz, dtype=torch.float32, device=dev).contiguous()
            llr = torch.zeros((B, llr_stride), dtype=torch.float32, device=dev)
            n = torch.zeros(B, dtype=torch.int32, device=dev)
            after = torch.zeros(B, dtype=torch.float32, device=dev)
        else:
            samples = np.ascontiguousarray(samples, dtype=np.float32)
            if samples.ndim == 1:
                samples = samples.reshape(1, -1)
            B, L = samples.shape
            cfo = np.ascontiguousarray(chirp_cfo_hz, dtype=np.float32)
            llr = np.zeros((B, llr_stride), np.float32)
            n = np.zeros(B, np.int32)
            after = np.zeros(B, np.float32)
        assert len(cfo) == B
        sp = _space(samples, cfo, llr, n, after)
        check(lib().pu_mcdpsk_got_chirp_batch(self._h, _ptr(samples), C.c_size_t(B), C.c_size_t(L), _ptr(cfo), _ptr(llr),
                                              C.c_size_t(llr_stride), _ptr(n), _ptr(after), sp, _stream(sp)))
        return llr, n, after

    def chirp_receive_batch(self, samples, threshold=0.15, llr_stride=648):
        """pu_mcdpsk_chirp_receive_batch: dual-chirp detectSync + setFrequencyOffset + process + getSoftBits for every row of samples
        [B, L] -> (llr [B, llr_stride], n_llr [B], sync_info [B, 4], sync_values [B, 4], cfo_after_hz [B])."""
        x = _frames(samples)
        B, L = x.shape
        llr = _like(x, (B, llr_stride), np.float32, "float32")
        n = _like(x, (B,), np.int32, "int32")
        info = _like(x, (B, 4), np.int32, "int32")
        val = _like(x, (B, 4), np.float32, "float32")
        after = _like(x, (B,), np.float32, "float32")
        sp = _space(x, llr, n, info, val, after)
        check(lib().pu_mcdpsk_chirp_receive_batch(self._h, _ptr(x), C.c_size_t(B), C.c_size_t(L), C.c_float(threshold), _ptr(llr),
                                                  C.c_size_t(llr_stride), _ptr(n), _ptr(info), _ptr(val), _ptr(after), sp, _stream(sp)))
        return llr, n, info, val, after

    def demod_soft_batch(self, samples, llr_stride=None, llr=None, want_cfo=True):
        x = _frames(samples)
        B, L = x.shape
        if llr_stride is None:
            llr_stride = max(self.n_llr(L), 1) if llr is None else llr.shape[1]
        if llr is None:
            llr = _like(x, (B, llr_stride), np.float32, "float32")
        cfo = _like(x, (B,), np.float32, "float32") if want_cfo else None
        sp = _space(x, llr, cfo)
        check(lib().pu_mcdpsk_demod_soft_batch(self._h, _ptr(x), C.c_size_t(B), C.c_size_t(L), _ptr(llr), C.c_size_t(llr_stride),
                                               _ptr(cfo), sp, _stream(sp)))
        return llr, cfo


# ---------------------------------------------------------------------------------------------- sweep driver (pu_linksim_run)
WF_OFDM, WF_OFDM_SC, WF_OFDM_CHIRP, WF_DPSK, WF_DPSK_ACQ, WF_MCDPSK, WF_MCDPSK_CHIRP = range(7)
CHANNELS = {"awgn": 0, "good": 1, "moderate": 2, "poor": 3, "flutter": 4,
            "itu_good": 5, "itu_moderate": 6, "itu_poor": 7, "itu_flutter": 8}


class SweepMode(C.Structure):
    """pu_sweep_mode: one row of the mode table (waveform x modulation x code rate x channel x SNR grid)."""
    _fields_ = [("waveform", C.c_uint32), ("ofdm", ModemConfig), ("dpsk", DpskConfig), ("mcdpsk", McDpskConfig),
                ("code_rate", C.c_uint32), ("payload_bytes", C.c_uint32), ("channel", C.c_uint32), ("n_snr", C.c_uint32),
                ("snr_first_db", C.c_float), ("snr_step_db", C.c_float), ("peak", C.c_float), ("precision", C.c_uint32),
                ("chunk", C.c_uint32), ("cost", C.c_float), ("lead_samples", C.c_uint32), ("tail_samples", C.c_uint32),
                ("cfo_hz", C.c_float), ("fresh_payloads", C.c_uint32), ("frame_payload_bytes", C.c_uint32), ("interleave_bps", C.c_uint32)]

    @property
    def snr_points(self):
        return [self.snr_first_db + i * self.snr_step_db for i in range(self.n_snr)]


class SweepDesc(C.Structure):
    _fields_ = [("modes", C.POINTER(SweepMode)), ("n_modes", C.c_uint32), ("pool", C.c_uint32), ("trials_per_point", C.c_uint64),
                ("block_trials", C.c_uint32), ("max_iter", C.c_uint32), ("base_seed", C.c_uint64), ("rank", C.c_uint32),
                ("world", C.c_uint32), ("batch_bytes", C.c_uint64), ("manifest_dir", C.c_char_p), ("max_units", C.c_uint64),
                ("run_id", C.c_uint64)]


class SweepStats(C.Structure):
    _fields_ = [("units_total", C.c_uint64), ("units_resumed", C.c_uint64), ("units_run", C.c_uint64), ("frames_run", C.c_uint64),
                ("seconds", C.c_double), ("setup_seconds", C.c_double), ("wait_seconds", C.c_double), ("fill_seconds", C.c_double),
                ("enqueue_seconds", C.c_double), ("busy_cost", C.c_double), ("total_cost", C.c_double)]


def sweep_mode(waveform, cfg, code_rate, payload_bytes, channel, snr_first, snr_step, n_snr, peak=0.0, precision="exact", chunk=0, cost=0.0,
               lead_samples=0, tail_samples=0, cfo_hz=0.0, fresh_payloads=False, frame_payload_bytes=0, interleave_bps=0):
    """One pu_sweep_mode.  frame_payload_bytes > 0 makes every trial a protocol-v2 DATA frame of that many payload bytes (OFDM waveforms;
    payload_bytes is then unused) with whole-frame counters (linksim.FRAME_COUNTER_NAMES).  interleave_bps > 0 passes every codeword
    through ChannelInterleaver(interleave_bps, 648) (OFDM and MC-DPSK waveforms)."""
    m = SweepMode()
    m.waveform = waveform
    if isinstance(cfg, ModemConfig):
        m.ofdm = cfg
    elif isinstance(cfg, DpskConfig):
        m.dpsk = cfg
    else:
        m.mcdpsk = cfg
    m.code_rate, m.payload_bytes, m.channel, m.n_snr = int(code_rate), int(payload_bytes), CHANNELS[channel] if isinstance(channel, str) else int(channel), int(n_snr)
    m.snr_first_db, m.snr_step_db, m.peak = float(snr_first), float(snr_step), float(peak or 0.0)
    m.precision, m.chunk, m.cost = {"exact": 0, "fast": 1}[precision], int(chunk), float(cost)
    m.lead_samples, m.tail_samples, m.cfo_hz, m.fresh_payloads = int(lead_samples), int(tail_samples), float(cfo_hz), int(bool(fresh_payloads))
    m.frame_payload_bytes = int(frame_payload_bytes)
    m.interleave_bps = int(interleave_bps)
    return m


class Sweep:
    """Host view of a pu_sweep_desc: keeps the mode array alive and wraps pu_sweep_* / pu_linksim_run."""

    def __init__(self, modes, trials_per_point, block_trials=4096, pool=64, rank=0, world=1, base_seed=0xB200, max_iter=50,
                 batch_bytes=0, manifest_dir=None, max_units=0, run_id=0):
        self.modes = list(modes)
        self._arr = (SweepMode * len(self.modes))(*self.modes)
        self._dir = manifest_dir.encode() if manifest_dir else None
        self.desc = SweepDesc(self._arr, len(self.modes), pool, trials_per_point, block_trials, max_iter, base_seed, rank, world,
                              batch_bytes, self._dir, max_units, run_id)
        L = lib()
        L.pu_sweep_unit_count.restype = C.c_uint64
        L.pu_sweep_point_count.restype = C.c_uint32
        self.n_units = int(L.pu_sweep_unit_count(C.byref(self.desc)))
        self.n_points = int(L.pu_sweep_point_count(C.byref(self.desc)))
        if self.n_units == 0:
            raise PuError("invalid sweep description")

    def partition(self, done=None):
        owner = np.zeros(self.n_units, np.uint32)
        cost = np.zeros(self.n_units, np.float64)
        d = None if done is None else np.ascontiguousarray(done, dtype=np.uint8)
        check(lib().pu_sweep_partition(C.byref(self.desc), _ptr(d), _ptr(owner), _ptr(cost)))
        return owner, cost

    def unit(self, u):
        m, s, t0, nt = C.c_uint32(), C.c_uint32(), C.c_uint64(), C.c_uint32()
        check(lib().pu_sweep_unit(C.byref(self.desc), C.c_uint64(u), C.byref(m), C.byref(s), C.byref(t0), C.byref(nt)))
        return m.value, s.value, t0.value, nt.value

    def payload(self, mode, index):
        """Payload of TX pool waveform `index` of mode `mode` (the DATA frame's payload in frame modes)."""
        m = self.modes[mode]
        out = np.zeros(m.frame_payload_bytes or m.payload_bytes, np.uint8)
        lib().pu_sweep_payload(C.c_uint64(self.desc.base_seed), C.c_uint32(mode), C.c_uint32(index), _ptr(out), C.c_size_t(len(out)))
        return out

    def run(self, ctx, raw=False):
        """pu_linksim_run -> (counters [n_points, 6] uint64 on the host, SweepStats); raw=True: pu_linksim_run_raw -> (counters, stats,
        raw [n_points, 4] uint64 = linksim.RAW_COUNTER_NAMES of the soft bits the decoder was given)."""
        counters = np.zeros((self.n_points, 6), np.uint64)
        st = SweepStats()
        if not raw:
            check(lib().pu_linksim_run(ctx._h, C.byref(self.desc), _ptr(counters), C.byref(st)))
            return counters, st
        table = np.zeros((self.n_points, 4), np.uint64)
        check(lib().pu_linksim_run_raw(ctx._h, C.byref(self.desc), _ptr(counters), _ptr(table), C.byref(st)))
        return counters, st, table

    def point_rows(self, counters):
        """[(mode index, snr_db, counter row)] in counter-table order."""
        rows, at = [], 0
        for mi, m in enumerate(self.modes):
            for s in m.snr_points:
                rows.append((mi, s, counters[at]))
                at += 1
        return rows


def wilson_interval(errors, n, z=1.96):
    lo, hi = C.c_double(), C.c_double()
    lib().pu_wilson_interval(C.c_uint64(int(errors)), C.c_uint64(int(n)), C.c_double(z), C.byref(lo), C.byref(hi))
    return lo.value, hi.value

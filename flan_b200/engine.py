"""Thin Python driver over the C ABI for the tests and bench.py.

torch is plumbing here: it owns device memory and the CUDA stream the kernels are enqueued on; all
arithmetic happens in libflan_b200.so. Method names follow the reference's (Audio::convert_to_PV,
PV::convert_to_audio, Audio::convert_to_mid_side; src/flan/Conversions/AudioPV.cpp).
"""
import ctypes

import numpy as np
import torch

from . import capi


class Engine:
    def __init__(self, device=0, lib_path=None):
        if not torch.cuda.is_available():
            raise RuntimeError("flan_b200 needs a CUDA device (no CPU fallback)")
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        self.ctx = capi.Context(device, lib_path)
        self.lib = self.ctx.lib

    # -- helpers ---------------------------------------------------------------------------------
    def _bind_stream(self):
        self.ctx.call("flan_b200_set_stream", ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))

    @staticmethod
    def _chk(t, dtype=torch.float32):
        assert t.is_cuda and t.dtype == dtype and t.is_contiguous(), "need a contiguous CUDA %s tensor" % dtype
        return ctypes.c_void_p(t.data_ptr())

    def num_frames(self, n, hop):
        return int(self.lib.flan_b200_num_frames(n, hop))

    def analysis_rate(self, sr, hop):
        return float(self.lib.flan_b200_analysis_rate(sr, hop))

    def hop_from_rates(self, sr, ar):
        return int(self.lib.flan_b200_hop_from_rates(sr, ar))

    def launch_count(self):
        return int(self.lib.flan_b200_launch_count(self.ctx.h))

    KERNEL_KINDS = {"analysis": 0, "phase_seg": 1, "phase_scan": 2, "synthesis": 3, "aux": 4,
                    "repitch": 5, "stretch": 6, "modify_tables": 7, "io_codec": 8}

    def set_timing(self, enabled):
        self.ctx.call("flan_b200_set_timing", int(enabled))

    def kernel_time(self, kind):
        """(total_ms, launches) of one kernel kind since the last query (synchronises the stream)."""
        ms, n = ctypes.c_double(0), ctypes.c_int64(0)
        self._bind_stream()
        self.ctx.call("flan_b200_kernel_time", self.KERNEL_KINDS[kind], ctypes.byref(ms), ctypes.byref(n))
        return ms.value, n.value

    def synchronize(self):
        self.ctx.call("flan_b200_synchronize")

    # -- Audio::convert_to_PV --------------------------------------------------------------------
    def convert_to_pv(self, audio, sr, W, hop, N, out=None, for_resynthesis=False):
        """audio: cuda float32 [C, n] -> pv: cuda float32 [C, F, N/2+1, 2] of (m, f).
        for_resynthesis: the rows will be resynthesised as they are (flan_b200_hint_resynthesis): the kernel also leaves
        their phase summaries, and convert_to_audio(..., unchanged=True) does not read the rows a second time."""
        C, n = audio.shape
        F = self.num_frames(n, hop)
        if out is None:
            out = torch.empty((C, F, N // 2 + 1, 2), dtype=torch.float32, device=self.device)
        self._bind_stream()
        if for_resynthesis:
            self.ctx.call("flan_b200_hint_resynthesis")
        self.ctx.call("flan_b200_convert_to_pv", self._chk(audio), C, n, sr, W, hop, N, self._chk(out), None)
        return out

    def convert_to_pv_range(self, audio_local, audio_offset, n_total, sr, W, hop, N, frame_begin, frame_end, out=None,
                            for_resynthesis=False):
        C, n_local = audio_local.shape
        rows = frame_end - frame_begin
        B = N // 2 + 1
        if out is None:
            out = torch.empty((C, rows, B, 2), dtype=torch.float32, device=self.device)
        self._bind_stream()
        if for_resynthesis:
            self.ctx.call("flan_b200_hint_resynthesis")
        self.ctx.call("flan_b200_convert_to_pv_range", self._chk(audio_local), n_local, audio_offset, n_local, C, n_total,
                      sr, W, hop, N, frame_begin, frame_end, self._chk(out), rows * B)
        return out

    # -- PV::convert_to_audio --------------------------------------------------------------------
    def convert_to_audio(self, pv, sr, ar, W, out=None, check_nan=False, unchanged=False):
        """unchanged: pv has not been written since the call that produced it (flan_b200_promise_unchanged): phase
        summaries that call left behind, if any, are used instead of a second read of the rows."""
        C, F, B, _ = pv.shape
        hop = self.hop_from_rates(sr, ar)
        if out is None:
            out = torch.empty((C, F * hop), dtype=torch.float32, device=self.device)
        flag = ctypes.c_int(0)
        self._bind_stream()
        if unchanged:
            self.ctx.call("flan_b200_promise_unchanged", self._chk(pv))
        self.ctx.call("flan_b200_convert_to_audio", self._chk(pv), C, F, B, sr, ar, W, self._chk(out), None,
                      ctypes.byref(flag) if check_nan else None)
        return (out, bool(flag.value)) if check_nan else out

    def phase_summary(self, pv_rows, frame_begin, sr, ar, W, unchanged=False):
        C, rows, B, _ = pv_rows.shape
        state = torch.empty((C, B, 4), dtype=torch.float64, device=self.device)
        self._bind_stream()
        if unchanged:
            self.ctx.call("flan_b200_promise_unchanged", self._chk(pv_rows))
        self.ctx.call("flan_b200_phase_summary", self._chk(pv_rows), rows * B, C, frame_begin, frame_begin + rows, B,
                      sr, ar, W, self._chk(state, torch.float64))
        return state

    def phase_carry(self, all_states, rank):
        R, C, B, _ = all_states.shape
        carry = torch.empty((C, B, 4), dtype=torch.float64, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_phase_carry", self._chk(all_states, torch.float64), rank, C, B, self._chk(carry, torch.float64))
        return carry

    def convert_to_audio_range(self, pv_rows, frame_begin, frames_total, sr, ar, W, carry, out_offset, out_len, out=None,
                               reuse_summary=False):
        C, rows, B, _ = pv_rows.shape
        if out is None:
            out = torch.empty((C, out_len), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_convert_to_audio_range", self._chk(pv_rows), rows * B, C, frame_begin, frame_begin + rows,
                      frames_total, B, sr, ar, W, None if carry is None else self._chk(carry, torch.float64),
                      int(reuse_summary), self._chk(out), out_len, out_offset, out_len)
        return out

    def convert_to_audio_range_head(self, pv_rows, frame_begin, frames_total, sr, ar, W, carry, out_offset, out_len, head_event,
                                    out=None, reuse_summary=False):
        """convert_to_audio_range with the frames that reach into the previous shard launched first; head_event (a
        torch.cuda.Event that has been recorded once, so that its handle exists) is recorded right after them."""
        C, rows, B, _ = pv_rows.shape
        if out is None:
            out = torch.empty((C, out_len), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_convert_to_audio_range_head", self._chk(pv_rows), rows * B, C, frame_begin, frame_begin + rows,
                      frames_total, B, sr, ar, W, None if carry is None else self._chk(carry, torch.float64),
                      int(reuse_summary), self._chk(out), out_len, out_offset, out_len,
                      ctypes.c_void_p(head_event.cuda_event) if head_event is not None else None)
        return out

    def add(self, dst, src):
        assert dst.numel() == src.numel()
        self._bind_stream()
        self.ctx.call("flan_b200_add", self._chk(dst), self._chk(src), dst.numel())

    def empty_like_audio(self, C, n):
        return torch.empty((C, n), dtype=torch.float32, device=self.device)

    def add_into(self, dst_view, src):
        """dst_view[c, :] += src[c, :] for a (possibly strided-by-channel) view of an audio tensor."""
        for c in range(dst_view.shape[0]):
            self.add(dst_view[c], src[c])

    # -- Audio::convert_to_mid_side ---------------------------------------------------------------
    def mid_side(self, audio):
        assert audio.shape[0] == 2
        out = torch.empty_like(audio)
        self._bind_stream()
        self.ctx.call("flan_b200_mid_side", self._chk(audio), self._chk(out), audio.shape[1])
        return out

    # -- PV-domain chain: PV::repitch / modify_frequency / stretch / modify_time (PV/PVModify.cpp:196-385) ----
    def _table(self, table, F, B):
        """Strided view of a frame x bin table: cuda float32 [F, B] (full), [B] (one row for every frame),
        [F, 1] (one column for every bin) or a Python / numpy scalar (a constant Function)."""
        if not torch.is_tensor(table):
            table = torch.full((1,), float(table), dtype=torch.float32, device=self.device)
        shape = tuple(table.shape)
        if shape == (F, B):
            fs, bs = B, 1
        elif shape == (B,):
            fs, bs = 0, 1
        elif shape == (F, 1):
            fs, bs = 1, 0
        elif table.numel() == 1:
            fs, bs = 0, 0
        else:
            raise ValueError("table shape %s does not fit a %d x %d grid" % (shape, F, B))
        return table, self._chk(table), fs, bs

    def repitch(self, pv, sr, factor, interp=0, out=None):
        C, F, B, _ = pv.shape
        t, tp, fs, bs = self._table(factor, F, B)
        if out is None:
            out = torch.empty_like(pv)
        self._bind_stream()
        self.ctx.call("flan_b200_repitch", self._chk(pv), C, F, B, sr, tp, fs, bs, interp, self._chk(out))
        return out

    def modify_frequency(self, pv, sr, mod_hz, in_mod, interp=0, out=None):
        C, F, B, _ = pv.shape
        t, tp, fs, bs = self._table(mod_hz, F, B)
        assert tuple(in_mod.shape) == (C, F, B)
        if out is None:
            out = torch.empty_like(pv)
        self._bind_stream()
        self.ctx.call("flan_b200_modify_frequency", self._chk(pv), C, F, B, sr, tp, fs, bs, self._chk(in_mod), interp, self._chk(out))
        return out

    def stretch_map(self, F, B, sr, ar, factor):
        t, tp, fs, bs = self._table(factor, F, B)
        out = torch.empty((F, B) if bs else (F, 1), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_stretch_map", tp, fs, bs, F, B, sr, ar, self._chk(out))
        return out

    def modify_time(self, pv, sr, ar, seconds, interp=0, summary_window=0):
        C, F, B, _ = pv.shape
        t, tp, fs, bs = self._table(seconds, F, B)
        frames = ctypes.c_int64(0)
        self._bind_stream()
        self.ctx.call("flan_b200_modify_time_frames", tp, fs, bs, F, B, sr, ar, ctypes.byref(frames))
        n = max(int(frames.value), 0)
        out = torch.empty((C, n, B, 2), dtype=torch.float32, device=self.device)
        self.ctx.call("flan_b200_modify_time", self._chk(pv), C, F, B, sr, ar, tp, fs, bs, interp, frames.value,
                      self._chk(out) if n else None, summary_window)
        return out

    def stretch(self, pv, sr, ar, factor, interp=0, summary_window=0):
        """summary_window: the PV's window size; the kernel then also leaves the phase summaries of its output behind, and
        convert_to_audio(..., unchanged=True) right after it skips the second read of the rows."""
        C, F, B, _ = pv.shape
        return self.modify_time(pv, sr, ar, self.stretch_map(F, B, sr, ar, factor), interp, summary_window)

    # -- expression Functions (flan_b200_fx_*): a capi.FxProgram sampled on the grid or evaluated at every MF -------
    def fx_sample(self, prog, F, B, time_step, bin_width):
        """The program over the F x B grid, in the view its dependence selects: [F, B], [F, 1], [B] or [1]."""
        ut, uf = ctypes.c_int(), ctypes.c_int()
        if self.lib.flan_b200_fx_check(ctypes.byref(prog), ctypes.byref(ut), ctypes.byref(uf)) != capi.OK:
            raise capi.FlanB200Error(capi.INVALID, self.lib.flan_b200_fx_last_error().decode())
        shape = {(1, 1): (F, B), (1, 0): (F, 1), (0, 1): (B,), (0, 0): (1,)}[(ut.value, uf.value)]
        out = torch.empty(shape, dtype=torch.float32, device=self.device)
        fs, bs = ctypes.c_int64(), ctypes.c_int()
        self._bind_stream()
        self.ctx.call("flan_b200_fx_sample", ctypes.byref(prog), F, B, time_step, bin_width, self._chk(out),
                      ctypes.byref(fs), ctypes.byref(bs))
        return out

    def fx_at_pv(self, prog, pv, frame_rate):
        """program( float(x) / frame_rate, pv[c, x, b].f ) for every MF: cuda float32 [C, F, B]."""
        C, F, B, _ = pv.shape
        out = torch.empty((C, F, B), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_fx_at_pv", ctypes.byref(prog), self._chk(pv), C, F, B, frame_rate, self._chk(out))
        return out

    # -- file formats either side of the path (PVBuffer::save / load, AudioBuffer::save / load) -----------------
    def flan_encode(self, pv, sr):
        C, F, B, _ = pv.shape
        out = torch.empty((C * F * B * 6,), dtype=torch.uint8, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_flan_encode", self._chk(pv), C * F * B, float((B - 1) * 2), sr, self._chk(out, torch.uint8))
        return out

    def flan_decode(self, data, shape, sr):
        C, F, B = shape
        out = torch.empty((C, F, B, 2), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_flan_decode", self._chk(data, torch.uint8), C * F * B, float((B - 1) * 2), sr, self._chk(out))
        return out

    def save_flan(self, path, pv, sr, ar, W):
        C, F, B, _ = pv.shape
        self._bind_stream()
        self.ctx.call("flan_b200_save_flan", path.encode(), self._chk(pv), C, F, B, sr, ar, W)

    def load_flan(self, path):
        """Returns (pv, sample_rate, rate_field, window_size); rate_field is what the reference's load stores as the
        analysis rate (the hop that save wrote, PVBuffer.cpp:134 vs :245)."""
        C, F, B, W = ctypes.c_int(), ctypes.c_int64(), ctypes.c_int(), ctypes.c_int()
        sr, rf = ctypes.c_float(), ctypes.c_float()
        self.ctx.call("flan_b200_flan_info", path.encode(), ctypes.byref(C), ctypes.byref(F), ctypes.byref(B),
                      ctypes.byref(sr), ctypes.byref(rf), ctypes.byref(W))
        pv = torch.empty((C.value, F.value, B.value, 2), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_load_flan", path.encode(), self._chk(pv), pv.numel() // 2)
        return pv, sr.value, rf.value, W.value

    def pcm24_encode(self, audio):
        C, n = audio.shape
        out = torch.empty((C * n * 3,), dtype=torch.uint8, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_pcm24_encode", self._chk(audio), C, n, self._chk(out, torch.uint8))
        return out

    def pcm24_decode(self, data, C, n):
        out = torch.empty((C, n), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_pcm24_decode", self._chk(data, torch.uint8), C, n, self._chk(out))
        return out

    def pcm_encode(self, audio, subtype):
        """audio: cuda float32 [C, n] -> interleaved sample bytes of a WAV sample type (capi.WAV_*)."""
        C, n = audio.shape
        out = torch.empty((C * n * capi.WAV_WIDTH[subtype],), dtype=torch.uint8, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_pcm_encode", self._chk(audio), C, n, subtype, self._chk(out, torch.uint8))
        return out

    def pcm_decode(self, data, C, n, subtype):
        out = torch.empty((C, n), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_pcm_decode", self._chk(data, torch.uint8), C, n, subtype, self._chk(out))
        return out

    def save_wav(self, path, audio, sr, subtype=capi.WAV_PCM_24):
        C, n = audio.shape
        self._bind_stream()
        self.ctx.call("flan_b200_save_wav_as", path.encode(), self._chk(audio), C, n, sr, subtype)

    def wav_format(self, path):
        """The sample type (capi.WAV_*) of a WAV file's data."""
        t = ctypes.c_int()
        self.ctx.call("flan_b200_wav_format", path.encode(), ctypes.byref(t))
        return t.value

    def load_wav(self, path):
        C, n, sr = ctypes.c_int(), ctypes.c_int64(), ctypes.c_float()
        self.ctx.call("flan_b200_wav_info", path.encode(), ctypes.byref(C), ctypes.byref(n), ctypes.byref(sr))
        audio = torch.empty((C.value, n.value), dtype=torch.float32, device=self.device)
        self._bind_stream()
        self.ctx.call("flan_b200_load_wav", path.encode(), self._chk(audio), audio.numel())
        return audio, sr.value

    # -- host-buffer forms (the call the reference-facing C++ layer makes) -------------------------
    def convert_to_pv_host(self, audio_np, sr, W, hop, N, mid_side=False, out=None):
        audio_np = np.ascontiguousarray(audio_np, np.float32)
        C, n = audio_np.shape
        F = self.num_frames(n, hop)
        if out is None:
            out = np.empty((C, F, N // 2 + 1, 2), np.float32)
        self._bind_stream()
        self.ctx.call("flan_b200_convert_to_pv_host", ctypes.c_void_p(audio_np.ctypes.data), C, n, sr, W, hop, N,
                      int(mid_side), ctypes.c_void_p(out.ctypes.data), None)
        return out

    def convert_to_audio_host(self, pv_np, sr, ar, W, left_right=False, out=None):
        pv_np = np.ascontiguousarray(pv_np, np.float32)
        C, F, B, _ = pv_np.shape
        hop = self.hop_from_rates(sr, ar)
        if out is None:
            out = np.empty((C, F * hop), np.float32)
        flag = ctypes.c_int(0)
        self._bind_stream()
        self.ctx.call("flan_b200_convert_to_audio_host", ctypes.c_void_p(pv_np.ctypes.data), C, F, B, sr, ar, W,
                      int(left_right), ctypes.c_void_p(out.ctypes.data), None, ctypes.byref(flag))
        return out, bool(flag.value)

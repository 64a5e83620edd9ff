"""Render engine: host planning (plan.py) -> device-resident job tables -> the kernel sequence.

`render(params, progress=None)` is the drop-in for reference `render` (main_v2.py:588-792): same
arguments, same `(float64[out_n, 2], meta)` result, same progress call shapes, exceptions propagate.
`BatchRenderer` / `render_batch` run many independent renders (the reference's batch loop,
main_v2.py:1578-1593) as one batched launch sequence on one GPU; `parallel.py` shards a batch over
the GPUs of a box.

Stage order (one batched launch sequence for all renders):
  synth (PCG64 + ziggurat normals, closed-form modes)            ms_synth_normal / ms_synth_dust
  [tilted-noise modes: rfft -> power-law tilt -> irfft, finish]  ms_spectral_* / ms_synth_tilt_finish
  grain spectral op: low-pass -> stretch -> multiband            ms_spectral_*
  overlap-add placement + ADSR                                   ms_overlap_add
  reflection cloud (+) impulse response as one FIR, overlap-save ms_fir_*
  stereo diffusion, soft clip, normalise                         ms_post
  [... and for renders with `export_sr`: resampled to that rate]  ms_post_export
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _abi, plan as P


# --------------------------------------------------------------------------- device abstraction
class CudaDevice:
    """torch-backed device memory on one GPU.  The only device the product ships."""

    def __init__(self, index=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("audio_suite_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.torch = torch
        self.index = torch.cuda.current_device() if index is None else int(index)
        # the library allocates its twiddle / chirp tables with cudaMalloc on the CURRENT device and caches them per
        # process, so a process drives exactly one GPU (one process per GPU, as torchrun launches them)
        owner = CudaDevice._owner
        if owner is not None and owner != self.index:
            raise RuntimeError(f"audio_suite_b200: this process already renders on cuda:{owner}; use one process per GPU")
        CudaDevice._owner = self.index
        torch.cuda.set_device(self.index)
        self.dev = torch.device("cuda", self.index)
        self.lib = _abi.lib()
        self.uploaded = 0

    _owner = None

    def stream_ptr(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.dev).cuda_stream)

    def empty(self, n, dtype):
        t = {np.float32: self.torch.float32, np.float64: self.torch.float64, np.uint8: self.torch.uint8,
             np.int32: self.torch.int32, np.uint64: self.torch.int64}[dtype]
        n = max(1, int(n))
        s = self._slot
        if s is not None:                       # carve from the slot's arena (no allocator call on the streamed path)
            nbytes = n * np.dtype(dtype).itemsize
            a = (s["off"] + 255) & ~255
            s["off"] = a + nbytes               # virtual offset: also counts what did not fit, to size the next arena
            if a + nbytes <= s["cap"]:
                return s["buf"][a:a + nbytes].view(t)
        return self.torch.empty(n, dtype=t, device=self.dev)

    # ---- arenas for streamed batches: slot k is one device buffer that the k-th live renderer carves all of
    #      its tensors from; it is sized from what the previous user of the slot needed and only ever grows.
    _slot = None

    def slot_begin(self, key):
        slots = self.__dict__.setdefault("_slots", {})
        s = slots.setdefault(key, {"buf": None, "cap": 0, "off": 0})
        if s["off"] > s["cap"]:
            s["buf"] = None
            s["cap"] = int(s["off"] * 1.2) + (64 << 20)
            s["buf"] = self.torch.empty(s["cap"], dtype=self.torch.uint8, device=self.dev)
        s["off"] = 0
        self._slot = s

    def slot_end(self):
        self._slot = None

    def zeros(self, n, dtype):
        b = self.empty(n, dtype)
        b.zero_()
        return b

    def upload(self, arr):
        """numpy array (any dtype) -> device bytes, staged through a ring of pinned blocks owned by the device
        object.  (`tensor.pin_memory()` per upload costs 10-20 ms a call whenever other processes on the box
        are busy -- measured on the B200 hosts with the planning workers running -- so nothing on the
        streamed path allocates pinned memory.)"""
        a = np.ascontiguousarray(arr)
        self.uploaded += a.nbytes
        flat = a.view(np.uint8).reshape(-1) if a.size else np.zeros(1, np.uint8)
        n = flat.size
        dst = self.empty(n, np.uint8)
        if n > self._RING_BLOCK:
            return dst.copy_(self.torch.from_numpy(np.array(flat, copy=True)).pin_memory(), non_blocking=True)
        if not self._ring:
            self._ring = [[self.torch.empty(self._RING_BLOCK, dtype=self.torch.uint8).pin_memory(), None] for _ in range(self._RING_N)]
            self._ring_np = [blk[0].numpy() for blk in self._ring]
            self._ring_cur, self._ring_off = 0, 0
        if self._ring_off + n > self._RING_BLOCK:
            self._ring_cur, self._ring_off = (self._ring_cur + 1) % self._RING_N, 0
            ev = self._ring[self._ring_cur][1]
            if ev is not None:
                ev.synchronize()              # long complete in steady state: the ring holds several slices of tables
        blk, off = self._ring[self._ring_cur], self._ring_off
        self._ring_np[self._ring_cur][off:off + n] = flat
        dst.copy_(blk[0][off:off + n], non_blocking=True)
        if blk[1] is None:
            blk[1] = self.torch.cuda.Event()
        blk[1].record(self.torch.cuda.current_stream(self.dev))
        self._ring_off = off + ((n + 255) & ~255)
        return dst

    _RING_BLOCK, _RING_N = 32 << 20, 4
    _ring = None

    def ptr(self, buf):
        return C.c_void_p(buf.data_ptr())

    def download(self, buf, offset, count):
        """slice of a device buffer -> numpy"""
        return buf[offset:offset + count].cpu().numpy()

    def synchronize(self):
        self.torch.cuda.synchronize(self.dev)


def _check(dev, rc):
    if rc != 0:
        raise RuntimeError("microsound_b200: " + (dev.lib.ms_last_error() or b"unknown error").decode())


def choose_precision(plans=None):
    """'auto' precision rule: float64.

    The kernels exist in float32 and float64 (B200 runs FP64 FMAs at half the FP32 rate, so f64 costs
    about 2x, not 30x).  float32 keeps every stage within ~3e-7 of that stage's *peak*, but render()
    ends with two amplifiers of small-signal error that the 1e-5 max-abs bar does not survive in
    general: (1) soft clip after the FIR stage -- with an impulse response or reflection cloud the
    pre-clip peak is routinely 1e2..1e3 and tanh has unit slope at every zero crossing; (2) peak
    normalisation -- when only the quiet start of a grain is placed (short outputs, slow ADSR attack:
    the factory default is a 1.25 ms grain under a 20 ms attack) the audible peak is <1 % of the grain
    peak and normalize() scales the float32 floor up with it.  float32 stays available as an explicit
    choice (`precision="f32"`); parity tests pin where it is within tolerance (C1, C1b, C2)."""
    return "f64"


class _SpectralStage:
    def __init__(self, dev, api, jobs, src, dst):
        """jobs: numpy record array of ms_spec_job (tables.pair_jobs)."""
        self.dev, self.api, self.handle, self.njobs = dev, api, C.c_void_p(None), len(jobs)
        if not len(jobs):
            return
        jobs = np.ascontiguousarray(jobs)
        need = api.ms_spectral_workspace_bytes(jobs.ctypes.data, len(jobs))
        if need == 0:
            _check(dev, -1)
        self.ws = dev.empty(need, np.uint8)
        _check(dev, api.ms_spectral_create(jobs.ctypes.data, len(jobs), dev.ptr(src), dev.ptr(dst),
                                           dev.ptr(self.ws), need, dev.stream_ptr(), C.byref(self.handle)))

    def run(self):
        if self.njobs:
            _check(self.dev, self.api.ms_spectral_run(self.handle, self.dev.stream_ptr()))

    def forward(self):
        if self.njobs:
            _check(self.dev, self.api.ms_spectral_forward(self.handle, self.dev.stream_ptr()))

    def inverse(self):
        if self.njobs:
            _check(self.dev, self.api.ms_spectral_inverse(self.handle, self.dev.stream_ptr()))

    def z_table(self):
        """(byte offset of the spectra inside the workspace, per-job offsets in complex elements, input order)"""
        offs = np.zeros(self.njobs, np.int64)
        base = C.c_size_t(0)
        _check(self.dev, self.api.ms_spectral_z_table(self.handle, offs.ctypes.data, C.byref(base)))
        return int(base.value), offs

    def close(self):
        if self.handle:
            self.api.ms_spectral_destroy(self.handle)
            self.handle = C.c_void_p(None)


class BatchRenderer:
    """Plans a batch of independent renders once, keeps every table resident on the device and
    re-runs the kernel sequence on demand (`run()`), e.g. for benchmarking or repeated renders."""

    def __init__(self, params_list=None, device=None, precision="auto", workers=None, tables=None):
        import time as _time
        from . import tables as T
        self.dev = device or CudaDevice()
        t0 = _time.perf_counter()
        if tables is not None:
            self.tables, self.plans = tables, None                            # already planned (tables.plan_stream)
        else:
            self.tables, self.plans = T.plan_and_pack(params_list, workers)  # plans is None for pooled batches
        self.t_plan = _time.perf_counter() - t0
        self.precision = choose_precision(self.plans) if precision == "auto" else precision
        self.api = _abi.Api(self.dev.lib, self.precision)
        self.real = np.float32 if self.precision == "f32" else np.float64
        up0 = getattr(self.dev, "uploaded", 0) + self.dev.lib.ms_h2d_bytes()
        t0 = _time.perf_counter()
        self._upload(T)
        self.t_pack = _time.perf_counter() - t0
        self.h2d_bytes = getattr(self.dev, "uploaded", 0) + self.dev.lib.ms_h2d_bytes() - up0

    # ---- device buffers + native plans -----------------------------------------------------------------
    cep_stages, plock_stage, imprint_stage = (), None, None          # batches without these stages

    def _upload(self, T):
        import os as _os, time as _time
        dev, t, real = self.dev, self.tables, self.real
        _tr = [] if _os.environ.get("MS_TRACE") else None
        _t0 = _time.perf_counter()

        def _mark(name):
            if _tr is not None:
                _tr.append((name, _time.perf_counter() - _t0))
        self.n_renders, self.n_evt, self.frames = len(t.post), len(t.sy1), t.frames
        self.max_out_n, self.max_h = t.max_out_n, t.max_h
        self.any_dust, self.any_tilt = t.dust_pos.size > 0, len(t.tilt) > 0
        self.n_fir = len(t.fir)
        self.pool = dev.empty(t.pool_n, real)
        self.mono = dev.zeros(t.mono_n, real)
        self.out = dev.empty(2 * t.frames, np.float32)
        self.maxbits = dev.zeros(self.n_renders, np.uint64)
        _mark("alloc")
        # one CTA per event, dispatched in table order: longest events first, so the tail of the launch is short ones
        sy1 = t.sy1[np.argsort(-t.sy1["n"].astype(np.int64), kind="stable")] if len(t.sy1) > 1 else t.sy1
        # dust / tilted-noise kernels launch 64 CTAs per table entry: hand them compact tables of just their events
        dust = sy1[sy1["mode"] == P.MODE_DUST]
        tilt = t.sy2[(t.sy2["mode"] == P.MODE_NOISE) | (t.sy2["mode"] == P.MODE_SKEW)]
        self.n_dust_evt, self.n_tilt_evt = len(dust), len(tilt)
        normal = sy1[(sy1["mode"] != P.MODE_DUST) & (sy1["mode"] < P.MODE_WAVELET)]      # the modes that draw normals
        stick = sy1[sy1["mode"] == P.MODE_STICK]
        if len(stick):                            # stick-slip: its normals (one per sample) go to the scratch at `aux` first
            pre = stick.copy()
            pre["out"] = stick["aux"]
            normal = np.concatenate([normal, pre])
        tab = sy1[sy1["mode"] > P.MODE_WAVELET]                                           # IR fragment / scan line / silence
        self.n_tab_evt = len(tab)
        self.d_sy_tab = dev.upload(tab) if self.n_tab_evt else None
        self.n_normal_evt = len(normal)
        self.d_sy1 = dev.upload(normal) if self.n_normal_evt else None
        self.d_sy_dust = dev.upload(dust) if self.n_dust_evt else None
        self.d_sy_tilt = dev.upload(tilt) if self.n_tilt_evt else None
        wav = sy1[sy1["mode"] == P.MODE_WAVELET]
        self.n_wav_evt = len(wav)
        if self.n_wav_evt:
            self.d_sy_wav = dev.upload(wav)
            self.d_atoms, self.d_atom_shift = dev.upload(t.atoms), dev.upload(t.atom_shift)
        self.d_ola_r, self.d_ola_e = dev.upload(t.ola_r), dev.upload(t.ola_e)
        self.n_env = len(t.env_reps)
        self.envpool = dev.empty(max(1, t.env_n), real)
        self.d_env_reps = dev.upload(t.env_reps) if self.n_env else None
        # export_sr: the renders that have one run ms_post_export instead of ms_post, on the maxbits after the plain ones
        self.n_export = len(t.export)
        if self.n_export:
            exporting = np.zeros(self.n_renders, bool)
            exporting[t.export_of] = True
            plain = t.post[~exporting]
            self.n_plain, self.max_n_plain = len(plain), int(plain["n"].max()) if len(plain) else 0
            self.d_post = dev.upload(plain) if len(plain) else None
            self.d_post_export, self.d_export = dev.upload(t.post[t.export_of]), dev.upload(t.export)
            self.d_bank = dev.upload(t.bank.astype(real))
            self.max_n_export = int(t.post["n"][t.export_of].max())
            self.max_out_export = int((t.export["out_end"] - t.export["out"]).max())
        else:
            self.d_post = dev.upload(t.post)
        if self.any_dust:
            self.d_dpos, self.d_dval = dev.upload(t.dust_pos), dev.upload(t.dust_val.astype(real))
        _mark("uploads")
        stage = lambda jobs, buf: _SpectralStage(dev, self.api, jobs, buf, buf)     # noqa: E731
        self.tilt_stage = stage(T.pair_jobs(t.tilt), self.pool)
        self.grain_stage = stage(T.pair_jobs(t.grain), self.pool)
        self.rot_stage = stage(T.pair_jobs(t.rot), self.mono)
        # resonator bank / waveguide (time domain) and the multiband unfold that follows them
        self.n_res, self.n_wg = len(t.res), len(t.wg)
        if self.n_wg:
            self.d_wg_evt, self.d_wg_lines = dev.upload(t.wg), dev.upload(t.wg_lines)
        self.post_stage = stage(T.pair_jobs(t.post_grain), self.pool)
        if self.n_res:
            self.d_res_evt, self.d_res_modes, self.h_res_evt = dev.upload(t.res), dev.upload(t.res_modes), t.res
        # cepstral warp: three stages of single-signal jobs around the elementwise steps of ms_cepstral; the outer one
        # transforms the grain, the inner two work in a scratch of [spectrum | cepstrum | warped cepstrum] per grain
        self.n_cep = len(t.cep)
        if self.n_cep:
            ev = t.cep.copy()
            n = ev["n"].astype(np.int64)
            xp_len, cep_len = (2 * (n // 2 + 1) + 3) // 4 * 4, (n + 3) // 4 * 4
            base = np.concatenate([[0], np.cumsum(xp_len + 2 * cep_len)])
            ev["xp"], ev["cep"], ev["cep2"] = base[:-1], base[:-1] + xp_len, base[:-1] + xp_len + cep_len
            self.cep_scratch = dev.empty(int(base[-1]), real)
            inner = np.zeros(self.n_cep, T.SPEC_ITEM)
            inner["n"] = n
            self.cep_stages = [stage(T.single_jobs(t.cep_items), self.pool)]
            for at in (ev["cep"], ev["cep2"]):                       # inverse only, forward only
                inner["src"] = inner["dst"] = at
                self.cep_stages.append(stage(T.single_jobs(inner), self.cep_scratch))
            self.cep_zb = []
            for name, st_ in zip(("z1", "z2", "z3"), self.cep_stages):
                b0, ev[name] = st_.z_table()
                self.cep_zb.append(b0)
            self.d_cep_evt, self.cep_max_n, self.h_cep_evt = dev.upload(ev), int(n.max()), ev
        # partial lock: single-signal jobs from the event's raw transient; low-pass / warp are evaluated by the
        # lock kernel on the forward spectrum, the inverse applies what follows it (multiband)
        self.n_plock = len(t.plock)
        if self.n_plock:
            self.plock_stage = stage(T.single_jobs(t.plock_items), self.pool)
            ev = t.plock.copy()
            self.plock_zbase, ev["z"] = self.plock_stage.z_table()
            bins = ev["n"].astype(np.int64) // 2 + 1
            scr = np.concatenate([[0], np.cumsum((3 * bins + 3) // 4 * 4)])       # 16-byte aligned complex scratch per grain
            ev["scratch"] = scr[:-1]
            self.d_plock_evt = dev.upload(ev)
            self.plock_scratch = dev.empty(int(scr[-1]), real)
        # event feedback (+ imprint): the events of a render depend on each other, so they are processed rank by rank
        # (rank e of all renders together): feedback kernel, then -- with the imprint on -- forward / one-grain step /
        # inverse on a spectral stage of that rank's grains; the step keeps one moving average per render (its slot)
        self.seq_ranks = []
        if len(t.seq):
            sq = t.seq
            renders, slot = np.unique(sq["render"], return_inverse=True)
            self.seq_max_bins = int(sq["fb"]["n_cur"].max()) // 2 + 1
            self.seq_mem = dev.zeros(len(renders) * self.seq_max_bins, real)
            self.seq_prev_bins = dev.zeros(len(renders), np.int32)
            for e in np.unique(sq["rank"]):
                at = sq["rank"] == e
                fb = sq["fb"][at & (sq["fb"]["dst"] >= 0)]
                item = {"n_fb": len(fb), "n_imp": 0}
                if len(fb):
                    item["d_fb"], item["fb_max_n"] = dev.upload(fb), int(fb["n_cur"].max())
                at &= sq["imp_item"]["dst"] >= 0
                if at.any():
                    stg = stage(T.single_jobs(sq["imp_item"][at]), self.pool)
                    iv = sq["imp"][at]
                    zbase, iv["z"] = stg.z_table()
                    iv["slot"] = slot[at]
                    item.update(n_imp=len(iv), stage=stg, zbase=zbase, d_imp=dev.upload(iv), h_imp=iv)
                self.seq_ranks.append(item)
        # spectral imprint: single-signal jobs (Z = the grain's DFT), forward -> per-render moving average -> inverse
        self.n_imprint_renders = len(t.imprint_r)
        if len(t.imprint):
            self.imprint_stage = stage(T.single_jobs(t.imprint_items), self.pool)
            ev = t.imprint.copy()
            self.imprint_zbase, ev["z"] = self.imprint_stage.z_table()
            self.d_imp_evt, self.d_imp_render = dev.upload(ev), dev.upload(t.imprint_r)
            self.h_imp_evt, self.h_imp_render = ev, t.imprint_r
            self.imprint_max_bins = int(ev["n"].max()) // 2 + 1
        _mark("spectral_create")
        self.fir_handle = C.c_void_p(None)
        if self.n_fir:
            fir = np.ascontiguousarray(t.fir)
            self.d_fir = dev.upload(fir)
            self.d_tap_off = dev.upload(t.tap_off if t.tap_off.size else np.zeros(1, np.int32))
            self.d_tap_gain = dev.upload((t.tap_gain if t.tap_gain.size else np.zeros(1)).astype(real))
            self.d_ir = dev.upload(t.irs.astype(real))
            need = self.api.ms_fir_workspace_bytes(fir.ctypes.data, len(fir))
            if need == 0:
                _check(dev, -1)
            self.fir_ws = dev.empty(need, np.uint8)
            _check(dev, self.api.ms_fir_create(fir.ctypes.data, len(fir), dev.ptr(self.d_ir), dev.ptr(self.d_tap_off),
                                               dev.ptr(self.d_tap_gain), dev.ptr(self.mono), dev.ptr(self.mono),
                                               dev.ptr(self.fir_ws), need, dev.stream_ptr(), C.byref(self.fir_handle)))
        _mark("fir_create")
        if _tr is not None:
            import sys as _sys
            print("  _upload: " + " ".join("%s %.1f" % (n, 1e3 * v) for n, v in _tr), file=_sys.stderr, flush=True)

    # ---- execution -------------------------------------------------------------------------------------
    def run(self, mark=None, probe=None):
        """Launch the whole kernel sequence on the current stream.  `mark(name)` (optional) is called
        after each stage has been enqueued (bench.py records a CUDA event there).  `probe(name, item)` (tests only)
        is called around the stages whose output the reference itself does not determine to rounding (cepstral warp,
        spectral imprint, resonator sign): the stage-level parity tests read the device buffers there and feed the
        oracle the SAME input (tests/kernel_checks.py: check_stages)."""
        dev, lib = self.dev, self.api
        st = dev.stream_ptr()
        mark = mark or (lambda name: None)
        probe = probe or (lambda name, item=None: None)
        if self.n_evt:
            if self.n_normal_evt:
                _check(dev, lib.ms_synth_normal(dev.ptr(self.d_sy1), self.n_normal_evt, dev.ptr(self.pool), st))
            if self.n_dust_evt:
                _check(dev, lib.ms_synth_dust(dev.ptr(self.d_sy_dust), self.n_dust_evt, dev.ptr(self.d_dpos), dev.ptr(self.d_dval),
                                              dev.ptr(self.pool), st))
            if self.n_tab_evt:
                dv = dev.ptr(self.d_dval) if self.any_dust else C.c_void_p(None)
                _check(dev, lib.ms_synth_table(dev.ptr(self.d_sy_tab), self.n_tab_evt, dv, dev.ptr(self.pool), st))
            if self.n_wav_evt:
                _check(dev, lib.ms_synth_wavelet(dev.ptr(self.d_sy_wav), self.n_wav_evt, dev.ptr(self.d_atoms),
                                                 dev.ptr(self.d_atom_shift), dev.ptr(self.pool), st))
            mark("synth")
            if self.any_tilt:
                self.tilt_stage.run()
                _check(dev, lib.ms_synth_tilt_finish(dev.ptr(self.d_sy_tilt), self.n_tilt_evt, dev.ptr(self.pool), st))
                mark("tilt_spectral")
            self.grain_stage.run()
            mark("grain_spectral")
            if self.n_cep:
                s1, s2, s3 = self.cep_stages
                zp = [C.c_void_p(dev.ptr(s_.ws).value + b0) for s_, b0 in zip(self.cep_stages, self.cep_zb)]
                args = (dev.ptr(self.d_cep_evt), self.n_cep, self.cep_max_n, zp[0], zp[1], zp[2], dev.ptr(self.cep_scratch), st)
                s1.forward()
                _check(dev, lib.ms_cepstral(0, *args))
                probe("cep_x")
                s2.inverse()
                _check(dev, lib.ms_cepstral(1, *args))
                s3.forward()
                _check(dev, lib.ms_cepstral(2, *args))
                probe("cep_y")
                s1.inverse()
                mark("cepstral_warp")
            if self.n_plock:
                self.plock_stage.forward()
                zptr = C.c_void_p(dev.ptr(self.plock_stage.ws).value + self.plock_zbase)
                _check(dev, lib.ms_partial_lock(dev.ptr(self.d_plock_evt), self.n_plock, zptr, dev.ptr(self.plock_scratch), st))
                self.plock_stage.inverse()
                mark("partial_lock")
            if self.n_res:
                probe("res_x")
                _check(dev, lib.ms_resonator(dev.ptr(self.d_res_evt), self.n_res, dev.ptr(self.d_res_modes), dev.ptr(self.pool), st))
            if self.n_res:
                probe("res_y")
            if self.n_wg:
                _check(dev, lib.ms_waveguide(dev.ptr(self.d_wg_evt), self.n_wg, dev.ptr(self.d_wg_lines), dev.ptr(self.pool), st))
            if self.n_res or self.n_wg:
                self.post_stage.run()
                mark("resonator_waveguide")
            if self.seq_ranks:
                self.seq_prev_bins.fill_(-1) if hasattr(self.seq_prev_bins, "fill_") else self.seq_prev_bins.fill(-1)
                for item in self.seq_ranks:
                    if item["n_fb"]:
                        _check(dev, lib.ms_feedback(dev.ptr(item["d_fb"]), item["n_fb"], item["fb_max_n"], dev.ptr(self.pool), st))
                    if item["n_imp"]:
                        stg = item["stage"]
                        stg.forward()
                        zptr = C.c_void_p(dev.ptr(stg.ws).value + item["zbase"])
                        probe("seq_imprint_x", item)
                        _check(dev, lib.ms_imprint_step(dev.ptr(item["d_imp"]), item["n_imp"], self.seq_max_bins, zptr,
                                                        dev.ptr(self.seq_mem), dev.ptr(self.seq_prev_bins), st))
                        probe("seq_imprint_y", item)
                        stg.inverse()
                mark("event_feedback")
            if self.imprint_stage is not None:
                self.imprint_stage.forward()
                zptr = C.c_void_p(dev.ptr(self.imprint_stage.ws).value + self.imprint_zbase)
                probe("imprint_x")
                _check(dev, lib.ms_imprint(dev.ptr(self.d_imp_evt), dev.ptr(self.d_imp_render), self.n_imprint_renders,
                                           self.imprint_max_bins, zptr, st))
                probe("imprint_y")
                self.imprint_stage.inverse()
                mark("spectral_imprint")
        if self.n_env:
            _check(dev, lib.ms_adsr_tables(dev.ptr(self.d_env_reps), self.n_env, self.max_out_n, dev.ptr(self.envpool), st))
        _check(dev, lib.ms_overlap_add(dev.ptr(self.d_ola_r), self.n_renders, self.max_out_n, dev.ptr(self.d_ola_e),
                                       dev.ptr(self.pool), dev.ptr(self.envpool), dev.ptr(self.mono), st))
        mark("overlap_add")
        if self.n_fir:
            _check(dev, lib.ms_fir_run(self.fir_handle, st))
            mark("fir_overlap_save")
        if len(self.tables.odd):
            base, isz = dev.ptr(self.mono).value, np.dtype(self.real).itemsize
            for (y_at, scratch, n, dr) in self.tables.odd.tolist():
                _check(dev, lib.ms_roll(C.c_void_p(base + isz * y_at), C.c_void_p(base + isz * scratch), n, dr, st))
            self.rot_stage.run()
        if not self.n_export:
            _check(dev, lib.ms_post(dev.ptr(self.d_post), self.n_renders, self.max_out_n, dev.ptr(self.mono),
                                    dev.ptr(self.maxbits), dev.ptr(self.out), st))
        else:
            if self.n_plain:
                _check(dev, lib.ms_post(dev.ptr(self.d_post), self.n_plain, self.max_n_plain, dev.ptr(self.mono),
                                        dev.ptr(self.maxbits), dev.ptr(self.out), st))
            mb = C.c_void_p(dev.ptr(self.maxbits).value + 8 * self.n_plain)
            _check(dev, lib.ms_post_export(dev.ptr(self.d_post_export), dev.ptr(self.d_export), self.n_export, self.max_n_export,
                                           self.max_out_export, dev.ptr(self.mono), mb, dev.ptr(self.d_bank), dev.ptr(self.out), st))
        mark("post")

    # ---- CUDA graph ------------------------------------------------------------------------------------
    def capture(self):
        """Capture the launch sequence of run() into a CUDA graph (the ~50 launches of a step become one graph launch:
        small slices stop being launch-bound).  The tables are resident and nothing in run() allocates or synchronises,
        so the sequence is capturable once it has run eagerly (kernel attributes and library tables are then in place)."""
        torch = self.dev.torch
        self.run()
        self.dev.synchronize()
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(self.dev.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev.dev))
        n0 = self.dev.lib.ms_launch_count()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                self.run()
        torch.cuda.current_stream(self.dev.dev).wait_stream(side)
        self.graph, self.graph_launches = g, int(self.dev.lib.ms_launch_count() - n0)      # kernel nodes one replay launches
        return g

    graph, graph_launches = None, 0

    def replay(self):
        """run() through the captured graph (capture() first)."""
        if self.graph is None:
            self.capture()
        self.graph.replay()

    # ---- results ---------------------------------------------------------------------------------------
    def output(self, r):
        """float32 [out_n, 2] of render r (host copy; out_n frames at its export rate, if any)."""
        n = int(self.tables.out_n[r])
        return self.dev.download(self.out, 2 * int(self.tables.out_at[r]), 2 * n).reshape(n, 2)

    def output_f64(self, r):
        """float64 [out_n, 2] of render r -- the float32 samples widened ON THE DEVICE (exact), as the reference returns them
        (`stereo.astype(np.float64)`, M:792).  For the 57.6 M frames of C4 the host-side astype alone cost 0.3 s."""
        if not hasattr(self.dev, "torch"):
            return self.output(r).astype(np.float64)
        n, a = int(self.tables.out_n[r]), 2 * int(self.tables.out_at[r])
        return self.out[a:a + 2 * n].double().cpu().numpy().reshape(n, 2)

    def outputs_device(self):
        return self.out

    def meta(self, r):
        t = self.tables
        m = dict(out_sr=int(t.srs[r, 0]), design_sr_base=int(t.srs[r, 1]), micro_last=None, grain_last=None)
        at = np.flatnonzero(t.export_of == r)
        if at.size:                                  # export_sr = base_sr * up / down, exactly
            up, down = t.export["rate"][at[0], :2].tolist()
            m["out_sr"] = m["out_sr"] * up // down
        micro, grain, n = t.last[r].tolist()
        if n > 0:
            m["micro_last"] = np.asarray(self.dev.download(self.pool, micro, n)).astype(np.float64)
            m["grain_last"] = np.asarray(self.dev.download(self.pool, grain, n)).astype(np.float64)
        return m

    def close(self):
        for s in (self.tilt_stage, self.grain_stage, self.rot_stage, self.imprint_stage, self.plock_stage, self.post_stage) + \
                tuple(self.cep_stages) + tuple(it["stage"] for it in getattr(self, "seq_ranks", []) if it["n_imp"]):
            if s is not None:
                s.close()
        if self.fir_handle:
            self.api.ms_fir_destroy(self.fir_handle)
            self.fir_handle = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- plan cache of render(): the Render button pressed again on unchanged settings (the reference re-renders from scratch,
#      M:1431-1456).  A small LRU of planned renderers keyed by the parameter VALUES: a hit re-runs the whole kernel sequence
#      (from the second hit on as one CUDA-graph launch) -- nothing about the audio is cached, only the host planning and
#      the table uploads are skipped.  Array-valued entries (`_ir_audio`, `_img_gray`) enter the key by identity, shape and a
#      strided checksum, so an array edited in place is seen as new.  Only renders up to _CACHE_MAX_FRAMES frames are kept.
_RENDER_CACHE = {}
_CACHE_ENTRIES, _CACHE_MAX_FRAMES = 8, 4_000_000


_array_key = P.array_signature


def _cache_key(params, dev, precision):
    try:
        items = tuple(sorted((k, v) for k, v in params.items() if not k.startswith("_")))
        hash(items)
    except TypeError:
        return None
    return (items, _array_key(params.get("_ir_audio")), _array_key(params.get("_img_gray")), id(dev), precision)


def clear_render_cache():
    for br, _ in _RENDER_CACHE.values():
        br.close()
    _RENDER_CACHE.clear()


def render(params, progress=None, device=None, precision="auto", cache=True):
    """Drop-in for reference render() (main_v2.py:588-792).  `cache=False` plans from scratch every time."""
    key = _cache_key(params, device, precision) if (cache and device is None or (cache and hasattr(device, "torch"))) else None
    hit = _RENDER_CACHE.pop(key, None) if key is not None else None
    if hit is not None:
        br, uses = hit
    else:
        br, uses = BatchRenderer([params], device=device, precision=precision), 0
    if progress:
        rp = br.plans[0] if br.plans else P.plan_render(params)        # (the native planner keeps no per-event records)
        progress(0, f"Output SR {rp.base_sr} Hz | Design SR {rp.design_sr_base} Hz")
    if uses >= 1 and hasattr(br.dev, "torch"):
        br.replay()                                                    # captured on the first hit, replayed afterwards
    else:
        br.run()
    if progress:
        n_evt = len(rp.events)
        for ev in rp.events:
            if ev.placed and ev.index % 50 == 0:
                progress(int(5 + 70 * (ev.index / max(1, n_evt))), f"Events {ev.index}/{n_evt}  {ev.note}".strip())      # M:758
    audio = br.output_f64(0)
    meta = br.meta(0)
    if key is not None and br.tables.frames <= _CACHE_MAX_FRAMES:
        _RENDER_CACHE[key] = (br, uses + 1)                            # most recent last
        while len(_RENDER_CACHE) > _CACHE_ENTRIES:
            old, _ = _RENDER_CACHE.pop(next(iter(_RENDER_CACHE)))
            old.close()
    else:
        br.close()
    if progress:
        progress(100, "Done.")
    return audio, meta


def _prefetch(gen, depth=2):
    """Runs a generator in a helper thread, `depth` items ahead: the parent's pipe reads / unpickling / merging of
    slice k+1 (tables.plan_stream) overlap its table uploads and kernel launches for slice k."""
    import queue
    import threading
    q = queue.Queue(maxsize=depth)
    end = object()

    def pump():
        try:
            for item in gen:
                q.put(item)
            q.put(end)
        except BaseException as e:          # re-raised in the consumer
            q.put(e)
    threading.Thread(target=pump, daemon=True).start()
    while True:
        item = q.get()
        if item is end:
            return
        if isinstance(item, BaseException):
            raise item
        yield item


def render_batch(params_list, device=None, precision="auto", host_out=None, chunk=384, depth=3, workers=None, piece=32, ramp=True):
    """See _render_batch.  The cyclic garbage collector is paused for the duration of the call: a full collection over a
    few thousand parameter dicts costs ~35 ms (measured: every fifth 100 ms sweep took 135 ms) and nothing here makes cycles."""
    import gc
    import sys
    was = gc.isenabled()
    gc.disable()
    # the launching thread shares the interpreter with the planning threads: with the default 5 ms switch interval every
    # return from a ctypes / CUDA call could wait that long for the lock (measured: 5-7 ms per slice set-up instead of 2)
    si = sys.getswitchinterval()
    sys.setswitchinterval(float(_os_env("MS_SWITCH") or 1e-4))
    try:
        return _render_batch(params_list, device, precision, host_out, chunk, depth, workers, piece, ramp)
    finally:
        sys.setswitchinterval(si)
        if was:
            gc.enable()


def _os_env(name):
    import os
    return os.environ.get(name, "")


def _render_batch(params_list, device=None, precision="auto", host_out=None, chunk=384, depth=3, workers=None, piece=32, ramp=True):
    """Independent renders (the reference's batch loop, main_v2.py:1578-1593) streamed through the GPU.

    The batch is cut into slices of `chunk` renders.  Worker processes plan slice k+1 (numpy Generators,
    integer segment maps) while the GPU renders slice k and slice k-1 drains to host memory on a copy
    stream, so planning, kernels and the device->host transfer overlap.  Returns a list of float32
    [out_n, 2] arrays, one per render, in order -- views into `host_out` (a pinned 1-D float32 torch tensor
    of at least 2 * total frames) when it is given, else into a pinned buffer allocated here."""
    from collections import deque
    import os as _os, time as _time
    from . import tables as T
    t_start = t_prev = _time.perf_counter()
    dev = device or CudaDevice()
    if isinstance(chunk, int) and ramp and len(params_list) >= 8 * piece:
        # short first slices: the GPU and the drain start early; short LAST slices: what is left after the host has enqueued
        # its last slice (that slice's kernels + its device->host copy) is short too.  Small batches (a rank's share of a
        # multi-GPU sweep) are still cut into about eight slices so that planning, kernels and the drain overlap.
        n = len(params_list)
        c = max(piece, min(int(chunk), (n // 8) // piece * piece))
        # (measured on B200, 4096 renders, c = 512: heads 128,256 -> 86.7 ms; 64,128,256 -> 80.8; 32,64,128,256 -> 82.9;
        #  128,384 -> 77.1: every slice costs 1-2 ms of host work, and the host is what paces the first third of the sweep)
        head = [max(piece, c // 4), max(piece, 3 * c // 4)]
        tail = [max(piece, c // 2), max(piece, c // 4), max(piece, c // 4)]
        if _os_env("MS_RAMP"):                     # development switch: "head sizes / tail sizes", e.g. "64,128,256/256,128,64"
            h_, t_ = _os_env("MS_RAMP").split("/")
            head, tail = [int(x) for x in h_.split(",") if x], [int(x) for x in t_.split(",") if x]
        body = max(0, n - sum(head) - sum(tail))
        chunk = head + [c] * (body // c) + ([body % c] if body % c else []) + tail
    if not hasattr(dev, "torch"):                   # host emulator device (tests): one slice after the other
        outs = []
        for tb in T.plan_stream(params_list, chunk, workers=workers or 1, piece=piece):
            br = BatchRenderer(device=dev, precision=precision, tables=tb)
            br.run()
            outs += [br.output(r) for r in range(br.n_renders)]
            br.close()
        return outs
    torch = dev.torch
    # frames of the whole batch (main_v2.py:590; at the export rate of renders with `export_sr`), memoised per distinct
    # (duration, rate, export rate): a sweep repeats a few values
    import operator
    frames_of, get_dur = {}, operator.itemgetter("out_dur_s", "base_sr")
    total = 0
    for p in params_list:
        key = get_dur(p) + (p.get("export_sr"),)
        f = frames_of.get(key)
        if f is None:
            f = frames_of[key] = P.export_frames(int(max(1, round(float(key[0]) * int(key[1])))), P.export_ratio(p))
        total += f
    if host_out is None:
        host_out = torch.empty(2 * total, dtype=torch.float32).pin_memory()
    if host_out.numel() < 2 * total:
        raise ValueError("host_out is smaller than 2 * total frames")
    main = torch.cuda.current_stream(dev.dev)
    copy = torch.cuda.Stream(dev.dev)
    live, views, at = deque(), [], 0
    h2d = 0
    trace = [] if _os.environ.get("MS_TRACE") else None
    if trace is not None:
        trace.append("  set-up before the first slice is asked for: %.1f ms" % (1e3 * (_time.perf_counter() - t_start)))
    k = 0
    for tb in _prefetch(T.plan_stream(params_list, chunk, workers=workers, piece=piece)):
        t_got = _time.perf_counter()
        dev.slot_begin(k % (depth + 1))        # the previous user of this slot has retired (see below)
        try:
            br = BatchRenderer(device=dev, precision=precision, tables=tb)
        finally:
            dev.slot_end()
        k += 1
        t_ctor = _time.perf_counter()
        br.run()
        h2d += br.h2d_bytes
        rendered = torch.cuda.Event()
        rendered.record(main)
        with torch.cuda.stream(copy):
            copy.wait_event(rendered)
            host_out[at:at + 2 * tb.frames].copy_(br.out[:2 * tb.frames], non_blocking=True)
            drained = torch.cuda.Event()
            drained.record(copy)
        for a, n in zip(tb.out_at.tolist(), tb.out_n.tolist()):
            views.append((at + 2 * a, n))
        at += 2 * tb.frames
        live.append((br, drained))
        t_enq = _time.perf_counter()
        while len(live) >= depth + 1:
            old, ev = live.popleft()
            ev.synchronize()
            old.close()
        if trace is not None:
            now = _time.perf_counter()
            trace.append("  slice %d: wait_plan %.1f ctor %.1f enqueue %.1f retire %.1f | t=%.1f ms" % (
                k - 1, 1e3 * (t_got - t_prev), 1e3 * (t_ctor - t_got), 1e3 * (t_enq - t_ctor), 1e3 * (now - t_enq), 1e3 * (now - t_start)))
            t_prev = now
    while live:
        old, ev = live.popleft()
        ev.synchronize()
        old.close()
    render_batch.last_h2d_bytes = h2d
    if trace is not None:
        import sys as _sys
        print("\n".join(trace) + "\n  drained at t=%.1f ms" % (1e3 * (_time.perf_counter() - t_start)), file=_sys.stderr, flush=True)
    flat = host_out.numpy()
    return [flat[a:a + 2 * n].reshape(n, 2) for a, n in views]

"""Per-frame characterization session: the reference driver's hot loop (test_fullframework.py:288-641)
for B independent clips advanced in lock-step, entirely on the GPU.

One `step()` = encode the clips' new pose windows -> context feature -> nearest-neighbour match ->
CVAE sample (autoregressive on the previous character feature) -> AdaIN decode -> to_mot ->
de-normalise -> root integration / blending / foot-lock IK. All buffers are pre-allocated, so the
whole step can be captured once into a CUDA graph (`capture()`) and replayed per frame.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, kinematics, packing
from .balltree import BallTree


@dataclass
class NormStats:
    """Normalisation tables the driver loads from norm.npz / cnt_norm.npz / cvae_norm.npz
    (test_fullframework.py:64-99), already divided by std_weight where the driver does (:89-92)."""
    Y_mean: np.ndarray          # [24,15]  (joint rows 1: of the [25,15] table)
    Y_std: np.ndarray
    cnt_mean: np.ndarray        # [90,256]
    cnt_std: np.ndarray
    src_cnt_mean: np.ndarray
    src_cnt_std: np.ndarray
    cha_encoded_mean: np.ndarray
    cha_encoded_std: np.ndarray


class CharacterizationSession:
    def __init__(self, gen_sd, cvae_sd, cfg, stats: NormStats, cha_encoded, cha_cnt_nm, batch: int,
                 device="cuda", precision="fp32", with_cm_path=False, match_tensor_cores=None, post_params=None,
                 lanes: int = 1, admission: bool = False, source_bank=None, result_bank=None):
        """gen_sd / cvae_sd: reference-layout state dicts. cha_encoded [N,90,256] and cha_cnt_nm [N,23040]
        (already (cnt-mean)/std scaled): the target character's feature DB, CUDA or CPU tensors.

        admission=True: clips start in any slot on any frame. Every frame takes one more input, the uint8 [B] row
        `start` (step_host(start=...), or a "start" entry of pinned_inputs()); a slot whose byte is 1 runs that frame as
        frame 0 of a new clip: its matched DB row seeds the autoregression (its CVAE output is not used) and its
        post-process state starts from the raw pose. All other slots run a steady-state frame in the same launches, so
        one captured graph serves every frame, and capture() may run before the first one. Everything a clip carries
        from frame to frame (prev_cha, the post-process states) is per slot and rewritten by a start, so a reused slot
        behaves exactly like a fresh one. A slot whose clip has ended keeps computing on whatever finite inputs the
        caller leaves in its rows; its outputs are meaningless until it is started again, and nothing of an idle or
        previous occupant reaches a started clip. Slots that never started compute on the zero-initialised buffers.

        source_bank (a SourceBank; needs admission=True): every slot's X, side and contacts are built on the device from
        the bank by mocha_source_windows, the first launch of the frame. The per-frame inputs become the `start` row,
        an int32 [B] `clip` row (the bank's clip id of each starting slot, read only where start is set) and eps
        (step_bank(), or pinned_inputs() for submit / collect). A started slot serves its clip's windows one per frame
        and repeats the last one once the clip has ended; an idle slot (never started, or started with an id the bank
        does not hold) gets zero inputs.

        result_bank (a ResultBank of the same source_bank): the last launch of each lane's frame, mocha_record_frames,
        records every serving slot's post-IK pose, integrated source root and matched DB row into the clip's record
        rows (the `post` path; the reference exports no other). serve() runs a list of bank clips through the slots and
        returns each clip's bvh.save payload, built on the device."""
        if source_bank is not None and not admission:
            raise _lib.MochaError("source_bank needs CharacterizationSession(admission=True)")
        if result_bank is not None and source_bank is None:
            raise _lib.MochaError("result_bank needs CharacterizationSession(..., source_bank=...)")
        if result_bank is not None and result_bank.bank is not source_bank:
            raise _lib.MochaError("result_bank records another source bank than this session's source_bank")
        self.lib = _lib.load()
        _lib.check(self.lib.mocha_check_device(), "mocha_check_device")
        dev = torch.device(device)
        self.dev, self.B = dev, batch
        self.prec = _lib.precision_code(precision)
        self.gen = packing.PackedGenerator(gen_sd, cfg, dev)
        self.cvae = packing.PackedCVAE(cvae_sd, 90, 256, 2, 4, 512, dev)
        d = self.gen.dims
        self.T, self.V, self.Cin, self.D, self.ntok = d.T, d.V, d.Cin, d.D, self.gen.ntok
        f32 = dict(dtype=torch.float32, device=dev)

        def tab(a):
            return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).to(dev).contiguous()

        self.Y_mean, self.Y_std = tab(stats.Y_mean), tab(stats.Y_std)
        self.cnt_mean, self.cnt_std = tab(stats.cnt_mean), tab(stats.cnt_std)
        self.m0, self.s0 = tab(stats.src_cnt_mean), tab(stats.src_cnt_std)
        self.m1, self.s1 = tab(stats.cha_encoded_mean), tab(stats.cha_encoded_std)
        self.cha_encoded = torch.as_tensor(cha_encoded, dtype=torch.float32).to(dev).contiguous()
        if isinstance(cha_cnt_nm, BallTree):      # a ready tree (e.g. BallTree.from_feature_db)
            self.tree = cha_cnt_nm
        else:
            self.tree = BallTree(torch.as_tensor(cha_cnt_nm, dtype=torch.float32).to(dev), device=dev,
                                 use_tensor_cores=match_tensor_cores)
        # matcher choice is fixed here: the tensor-core path needs the bf16 DB packed (which fixes the origin,
        # tree.center, of the bf16 query the encode stage emits) before the first frame runs
        t = self.tree
        use_tc = t.use_tensor_cores
        if use_tc is None or use_tc == "auto":
            # throughput mode: tensor-core coarse pass + fp64 re-rank (split-K when the DB is small);
            # parity mode (fp32) keeps the brute-force fp64 kernel unless the problem is large
            use_tc = batch * t.N >= t.TC_THRESHOLD_PAIRS or (
                self.prec == _lib.MOCHA_BF16 and batch >= 16 and t.D % 8 == 0 and t.D >= 1024)
        self._use_tc = bool(use_tc)
        if self._use_tc:
            t._ensure_bf16()
        self.with_cm_path = with_cm_path
        B, n, D = batch, self.ntok, self.D
        # static I/O buffers (graph-capturable)
        self.X = torch.zeros((B, d.T, d.V, d.Cin), **f32)
        self.src_hips_vel = torch.zeros((B, d.T, 3), **f32)
        self.src_rvel = torch.zeros((B, 3), **f32)
        self.src_rang = torch.zeros((B, 3), **f32)
        self.contacts = torch.zeros((B, 2), dtype=torch.uint8, device=dev)
        self.eps = torch.zeros((B, D), **f32)
        self.admission = bool(admission)
        if self.admission:
            self.start = torch.zeros((B,), dtype=torch.uint8, device=dev)     # 1 = the slot starts a new clip this frame
        self._input_names = ("X", "side", "contacts", "eps") + (("start",) if self.admission else ())
        self.bank = source_bank
        if source_bank is not None:
            if source_bank.dev != dev or source_bank.T != d.T or source_bank.J != d.V + 1:
                raise _lib.MochaError(f"source_bank holds windows of {source_bank.T} frames x {source_bank.J} joints on "
                                      f"{source_bank.dev}; this session needs {d.T} x {d.V + 1} on {dev}")
            self.clip = torch.zeros((B,), dtype=torch.int32, device=dev)       # bank clip id of each starting slot
            self.slot_clip = torch.full((B,), -1, dtype=torch.int32, device=dev)
            self.slot_cursor = torch.zeros((B,), dtype=torch.int32, device=dev)
            self._input_names = ("start", "clip", "eps")
        self.results = result_bank
        if result_bank is not None:
            self.slot_count = torch.zeros((B,), dtype=torch.int32, device=dev)   # windows recorded by each slot's clip
        # intermediates
        self.tokens = torch.empty((B, n, D), **f32)
        self.encoded = torch.empty((B, n, D), **f32)
        self.cnt = torch.empty((B, n, D), **f32)
        self.cnt_nm = torch.empty((B, n * D), **f32)
        self.cnt_nm16 = torch.empty((B, n * D), dtype=torch.bfloat16, device=dev)   # tensor-core matcher operand
        self.match_idx = torch.zeros((B, 1), dtype=torch.int64, device=dev)
        self.match_dist = torch.zeros((B, 1), dtype=torch.float64, device=dev)
        self.cond = torch.empty((B, 2 * n, D), **f32)
        self.cvae_out = torch.empty((B, n, D), **f32)
        self.prev_cha = torch.zeros((B, n, D), **f32)      # prev_cha_encoded (de-normalised)
        self.decoded = torch.empty((B, n, D), **f32)
        self.Y = torch.empty((B, d.T, d.V, d.Cin), **f32)
        self.cm_cha = torch.empty((B, n, D), **f32)
        self.cm_Y = torch.empty((B, d.T, d.V, d.Cin), **f32)
        self.post = kinematics.PostProcessor(B, dev, post_params)
        self.cm_post = kinematics.PostProcessor(B, dev, post_params) if with_cm_path else None
        dims = C.byref(self.gen.struct.dims)
        with _lib.workspace_precision(self.prec):
            nbytes = max(self.lib.mocha_embed_workspace_bytes(dims, B), self.lib.mocha_encoder_workspace_bytes(dims, B),
                         self.lib.mocha_decoder_workspace_bytes(dims, B), self.lib.mocha_to_mot_workspace_bytes(dims, B),
                         self.lib.mocha_cvae_workspace_bytes(C.byref(self.cvae.struct), B, 2 * n),
                         self.lib.mocha_match_exact_workspace_bytes(B, self.tree.N, 1),
                         self.lib.mocha_match_tc_workspace_bytes(B, self.tree.N, self.tree.D, self.tree.kc))
        self.ws = torch.empty(nbytes + 4096, dtype=torch.uint8, device=dev)
        # Sub-batch lanes: clips are independent, so the batch can be cut into `lanes` contiguous groups whose frames
        # run concurrently on separate streams (forked / joined inside the captured graph). Most kernels of the frame
        # are latency-bound on <= 148 CTAs with idle SMs in their ramps and tails; a second lane fills them.
        lanes = max(1, min(int(lanes), batch))
        cuts = [round(i * batch / lanes) for i in range(lanes + 1)]
        self.parts = [(cuts[i], cuts[i + 1]) for i in range(lanes) if cuts[i + 1] > cuts[i]]
        self.lane_ws = [self.ws] + [torch.empty_like(self.ws) for _ in self.parts[1:]]
        self.lane_streams = [torch.cuda.Stream(device=dev) for _ in self.parts[1:]]
        # The matcher's result is only read at the init frame (it seeds the autoregression) and by the optional cm_trans
        # decode; in the steady state it is a side branch of the frame, so it runs on its own stream (own workspace)
        # concurrently with the CVAE / decoder chain and is joined at the end of the frame. Its kernels are small
        # (split-K coarse pass, re-rank) and fit next to the 90-CTA block tails.
        mbytes = max(self.lib.mocha_match_exact_workspace_bytes(B, self.tree.N, 1),
                     self.lib.mocha_match_tc_workspace_bytes(B, self.tree.N, self.tree.D, self.tree.kc))
        self.match_ws = [torch.empty(mbytes + 4096, dtype=torch.uint8, device=dev) for _ in self.parts]
        self.match_streams = [torch.cuda.Stream(device=dev) for _ in self.parts]
        self.frame = 0
        self.graph = None
        self.deterministic = False
        # pinned host staging for the end-to-end path
        self.h_X = torch.zeros(self.X.shape, dtype=torch.float32).pin_memory()
        self.h_side = torch.zeros((B, d.T * 3 + 3 + 3), dtype=torch.float32).pin_memory()
        self.h_contacts = torch.zeros((B, 2), dtype=torch.uint8).pin_memory()
        self.h_eps = torch.zeros((B, D), dtype=torch.float32).pin_memory()
        if self.admission:
            self.h_start = torch.zeros((B,), dtype=torch.uint8).pin_memory()
        if self.bank is not None:
            self.h_clip = torch.zeros((B,), dtype=torch.int32).pin_memory()
        self.h_out = torch.zeros(self.post.out.shape, dtype=torch.uint8).pin_memory()
        self.side = torch.zeros((B, d.T * 3 + 3 + 3), **f32)

    # ---------------------------------------------------------------------------------------------
    def _s(self):
        return _lib.stream_ptr()

    def _ws(self, ws=None):
        ws = self.ws if ws is None else ws
        return _lib.ptr(ws), ws.numel()

    def encode(self, X, tokens, encoded, cnt, cnt_nm, cnt_nm16=None, ws=None):
        lib, g = self.lib, C.byref(self.gen.struct)
        B = X.shape[0]
        wp, wn = self._ws(ws)
        _lib.check(lib.mocha_embed_fwd(g, _lib.ptr(X), B, _lib.ptr(tokens), 1, self.prec, wp, wn, self._s()), "embed")
        _lib.check(lib.mocha_encoder_fwd(g, _lib.ptr(tokens), B, _lib.ptr(encoded), self.prec, wp, wn, self._s()), "encoder")
        _lib.check(lib.mocha_cnt_features(_lib.ptr(encoded), B, self.ntok, self.D, 1e-5, _lib.ptr(cnt),
                                          _lib.ptr(self.cnt_mean), _lib.ptr(self.cnt_std), _lib.ptr(cnt_nm),
                                          None if cnt_nm16 is None else _lib.ptr(cnt_nm16),
                                          None if (cnt_nm16 is None or self.tree.center is None) else _lib.ptr(self.tree.center),
                                          self._s()), "cnt_features")

    def _decode(self, src_encoded, cha, decoded, Y, ws=None):
        lib, g = self.lib, C.byref(self.gen.struct)
        wp, wn = self._ws(ws)
        B = src_encoded.shape[0]
        _lib.check(lib.mocha_decoder_fwd(g, _lib.ptr(src_encoded), _lib.ptr(cha), B, _lib.ptr(decoded), self.prec,
                                         wp, wn, self._s()), "decoder")
        _lib.check(lib.mocha_to_mot_fwd(g, _lib.ptr(decoded), B, None, _lib.ptr(self.Y_mean), _lib.ptr(self.Y_std),
                                        _lib.ptr(Y), self.prec, wp, wn, self._s()), "to_mot")

    def _match(self, lo=0, hi=None, ws=None):
        lib, t = self.lib, self.tree
        hi = self.B if hi is None else hi
        wp, wn = self._ws(ws)
        q, q16 = self.cnt_nm[lo:hi], self.cnt_nm16[lo:hi]
        idx, dist = self.match_idx[lo:hi], self.match_dist[lo:hi]
        if self._use_tc:
            t._ensure_bf16()
            _lib.check(lib.mocha_match_tc(_lib.ptr(q), _lib.ptr(q16), hi - lo, _lib.ptr(t._db16),
                                          _lib.ptr(t.data), _lib.ptr(t._norm), t.N, t.D, 1, t.kc, 0,
                                          _lib.ptr(idx), _lib.ptr(dist), wp, wn, self._s()),
                       "match_tc")
        else:
            _lib.check(lib.mocha_match_exact(_lib.ptr(q), hi - lo, _lib.ptr(t.data), t.N, t.D, 1, 0,
                                             _lib.ptr(idx), _lib.ptr(dist), wp, wn, self._s()),
                       "match_exact")

    def _cvae_step(self, lo: int, hi: int, ws):
        """condition + CVAE sample of clips [lo, hi): prev_cha becomes this frame's de-normalised character feature."""
        lib = self.lib
        sl = slice(lo, hi)
        Bp = hi - lo
        _lib.check(lib.mocha_cvae_condition(_lib.ptr(self.cnt[sl]), _lib.ptr(self.prev_cha[sl]), _lib.ptr(self.m0),
                                            _lib.ptr(self.s0), _lib.ptr(self.m1), _lib.ptr(self.s1),
                                            _lib.ptr(self.cond[sl]), Bp, self.ntok, self.D, self._s()), "condition")
        wp, wn = self._ws(ws)
        _lib.check(lib.mocha_cvae_sample(C.byref(self.cvae.struct), _lib.ptr(self.cond[sl]), Bp, 2 * self.ntok,
                                         None if self.deterministic else _lib.ptr(self.eps[sl]),
                                         _lib.ptr(self.cvae_out[sl]), None, None, _lib.ptr(self.m1), _lib.ptr(self.s1),
                                         _lib.ptr(self.prev_cha[sl]), self.prec, wp, wn, self._s()), "cvae_sample")

    def _admission_part(self, lo: int, hi: int, ws):
        """One lane of an admission-mode frame: every clip runs a steady-state frame, and the clips whose start byte is
        set run their frame 0 inside the same launches (seeded prev_cha, masked post-process)."""
        sl = slice(lo, hi)
        if self.bank is not None:
            self.bank.windows(self.start[sl], self.clip[sl], self.slot_clip[sl], self.slot_cursor[sl], self.X[sl],
                              self.side[sl], self.contacts[sl])
        self.encode(self.X[sl], self.tokens[sl], self.encoded[sl], self.cnt[sl], self.cnt_nm[sl], self.cnt_nm16[sl], ws)
        k = next(i for i, pr in enumerate(self.parts) if pr[0] == lo)
        side = self.match_streams[k]
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self._match(lo, hi, self.match_ws[k])
        self._cvae_step(lo, hi, ws)
        torch.cuda.current_stream().wait_stream(side)       # join: a started clip's decoder needs its match
        # started clips: the matched DB row replaces the CVAE output (test_fullframework.py:298, :437)
        _lib.check(self.lib.mocha_seed_rows(_lib.ptr(self.start[sl]), _lib.ptr(self.match_idx[sl]), 1,
                                            _lib.ptr(self.cha_encoded), self.cha_encoded.shape[0], self.ntok * self.D,
                                            _lib.ptr(self.prev_cha[sl]), hi - lo, self._s()), "seed_rows")
        if self.with_cm_path:
            torch.index_select(self.cha_encoded, 0, self.match_idx[sl, 0], out=self.cm_cha[sl])
        self._decode(self.encoded[sl], self.prev_cha[sl], self.decoded[sl], self.Y[sl], ws)
        self.post.step_packed(self.Y[sl], self.side[sl], self.contacts[sl], lo=lo, start=self.start[sl])
        if self.results is not None:
            self.results.record(self.post.out.view(self.B, -1)[sl].view(-1), self.match_idx[sl], self.start[sl],
                                self.slot_clip[sl], self.slot_count[sl])
        if self.with_cm_path:
            self._decode(self.encoded[sl], self.cm_cha[sl], self.decoded[sl], self.cm_Y[sl], ws)
            self.cm_post.step_packed(self.cm_Y[sl], self.side[sl], self.contacts[sl], lo=lo, start=self.start[sl])

    def _frame_part(self, init: bool, lo: int, hi: int, ws):
        """One lane: clips [lo, hi) from the input buffers to the FrameOut buffer, on the current stream."""
        if self.admission:
            self._admission_part(lo, hi, ws)
            return
        sl = slice(lo, hi)
        self.encode(self.X[sl], self.tokens[sl], self.encoded[sl], self.cnt[sl], self.cnt_nm[sl], self.cnt_nm16[sl], ws)
        side = None
        if not init and not self.with_cm_path:
            k = next(i for i, pr in enumerate(self.parts) if pr[0] == lo)
            side = self.match_streams[k]
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._match(lo, hi, self.match_ws[k])
        else:
            self._match(lo, hi, ws)
        if init or self.with_cm_path:
            torch.index_select(self.cha_encoded, 0, self.match_idx[sl, 0], out=self.cm_cha[sl])
        if init:
            # frame 0: the NN result seeds the autoregression (test_fullframework.py:298, :437)
            self.prev_cha[sl].copy_(self.cm_cha[sl])
        else:
            self._cvae_step(lo, hi, ws)
        self._decode(self.encoded[sl], self.prev_cha[sl], self.decoded[sl], self.Y[sl], ws)
        # the kernel reads the packed `side` rows in place (no slicing copies inside the captured frame)
        self.post.step_packed(self.Y[sl], self.side[sl], self.contacts[sl], lo=lo, init=init)
        if side is not None:
            torch.cuda.current_stream().wait_stream(side)       # join: match_idx / match_dist are frame outputs
        if self.with_cm_path:
            self._decode(self.encoded[sl], self.cm_cha[sl], self.decoded[sl], self.cm_Y[sl], ws)
            self.cm_post.step_packed(self.cm_Y[sl], self.side[sl], self.contacts[sl], lo=lo, init=init)

    def _frame_body(self, init: bool):
        """Everything between the input buffers and the FrameOut buffer (graph-capturable): the lanes' frames, forked
        onto their streams and joined back into the current one."""
        cur = torch.cuda.current_stream()
        for s in self.lane_streams:
            s.wait_stream(cur)
        for k, (lo, hi) in enumerate(self.parts):
            if k == 0:
                self._frame_part(init, lo, hi, self.lane_ws[0])
            else:
                with torch.cuda.stream(self.lane_streams[k - 1]):
                    self._frame_part(init, lo, hi, self.lane_ws[k])
        for s in self.lane_streams:
            cur.wait_stream(s)
        self.post.started = True
        if self.cm_post:
            self.cm_post.started = True

    def capture(self):
        """Capture the steady-state frame (i >= 1) into a CUDA graph. Call after the first frame; in admission mode the
        captured frame is the only frame body (starts are per slot, from the `start` row), so any time will do."""
        if self.frame == 0 and not self.admission:
            raise _lib.MochaError("capture() needs the init frame to have run (state must exist)")
        state_backup = (self.prev_cha.clone(), self.post.state.clone(),
                        self.cm_post.state.clone() if self.cm_post else None)
        slots_backup = (self.slot_clip.clone(), self.slot_cursor.clone()) if self.bank is not None else None
        rec_backup = ((self.slot_count.clone(), self.results.clip_done.clone(), self.results.clip_built.clone())
                      if self.results is not None else None)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._frame_body(False)   # warm-up on a side stream (lazy attribute setting, allocator)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._frame_body(False)
        # capture does not execute; restore the state the warm-up advanced
        self.prev_cha.copy_(state_backup[0])
        self.post.state.copy_(state_backup[1])
        if self.cm_post:
            self.cm_post.state.copy_(state_backup[2])
        if slots_backup is not None:
            self.slot_clip.copy_(slots_backup[0])
            self.slot_cursor.copy_(slots_backup[1])
        if rec_backup is not None:      # record rows the warm-up wrote are rewritten by the next real frame
            self.slot_count.copy_(rec_backup[0])
            self.results.clip_done.copy_(rec_backup[1])
            self.results.clip_built.copy_(rec_backup[2])
        self.graph = g

    # ---------------------------------------------------------------------------------------------
    def step_device(self):
        """Advance one frame from the static device input buffers (X, side, contacts, eps; and start in admission
        mode)."""
        init = self.frame == 0 and not self.admission
        if self.graph is not None and not init:
            self.graph.replay()
        else:
            self._frame_body(init)
        self.frame += 1

    def step_host(self, X, src_hips_vel, src_rvel, src_rang, contacts, eps=None, start=None):
        """End-to-end call with HOST (numpy) inputs: pinned staging -> H2D -> frame -> D2H.
        start (admission mode only): uint8 [B], 1 = the slot starts a new clip on this frame; None = no slot starts.
        Returns the frame outputs as a dict of float64 numpy arrays [B, ...]."""
        B, T = self.B, self.T
        if self.bank is not None:
            raise _lib.MochaError("a session with a source bank takes step_bank(start, clip, eps)")
        if self.admission:
            self.h_start.numpy()[...] = 0 if start is None else np.asarray(start, dtype=np.uint8)
            self.start.copy_(self.h_start, non_blocking=True)
        elif start is not None:
            raise _lib.MochaError("a start row needs CharacterizationSession(admission=True)")
        self.h_X.numpy()[...] = X
        hs = self.h_side.numpy()
        hs[:, :T * 3] = np.asarray(src_hips_vel, dtype=np.float32).reshape(B, T * 3)
        hs[:, T * 3:T * 3 + 3] = src_rvel
        hs[:, T * 3 + 3:] = src_rang
        self.h_contacts.numpy()[...] = contacts
        self.X.copy_(self.h_X, non_blocking=True)
        self.side.copy_(self.h_side, non_blocking=True)
        self.contacts.copy_(self.h_contacts, non_blocking=True)
        if eps is not None:
            self.h_eps.numpy()[...] = eps
            self.eps.copy_(self.h_eps, non_blocking=True)
        elif not self.deterministic:
            self.eps.normal_()
        self.step_device()
        self.h_out.copy_(self.post.out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._decode_out(self.h_out.numpy())

    def step_bank(self, start, clip, eps=None):
        """End-to-end call of a session with a source bank: host (numpy) start row uint8 [B] (None = no slot starts),
        clip row int32 [B] (bank clip ids, read where start is set; None = all 0) and optionally eps [B, D].
        Returns the frame outputs as a dict of float64 numpy arrays [B, ...]."""
        if self.bank is None:
            raise _lib.MochaError("step_bank() needs CharacterizationSession(..., source_bank=...)")
        self.h_start.numpy()[...] = 0 if start is None else np.asarray(start, dtype=np.uint8)
        self.h_clip.numpy()[...] = 0 if clip is None else np.asarray(clip, dtype=np.int32)
        self.start.copy_(self.h_start, non_blocking=True)
        self.clip.copy_(self.h_clip, non_blocking=True)
        if eps is not None:
            self.h_eps.numpy()[...] = eps
            self.eps.copy_(self.h_eps, non_blocking=True)
        elif not self.deterministic:
            self.eps.normal_()
        self.step_device()
        self.h_out.copy_(self.post.out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._decode_out(self.h_out.numpy())

    # ---------------------------------------------------------------------------------------------
    # pipelined end-to-end streaming: the H2D copy of frame i+1 overlaps the kernels of frame i
    # ---------------------------------------------------------------------------------------------
    def pinned_inputs(self):
        """A set of pinned host tensors a caller fills for one frame (shapes of step_host's arguments,
        with src_hips_vel/src_rvel/src_rang packed as `side` [B, T*3+6]; admission mode adds the uint8 [B] `start` row).
        A session with a source bank takes `start`, `clip` (int32 [B]) and `eps` only."""
        return {k: torch.zeros(getattr(self, k).shape, dtype=getattr(self, k).dtype).pin_memory()
                for k in self._input_names}

    def _pipe_init(self):
        dev = self.dev
        self._copy_stream = torch.cuda.Stream(device=dev)
        self._slots = []
        for _ in range(2):
            slot = {k: torch.empty_like(getattr(self, k)) for k in self._input_names}
            slot.update({"h_out": torch.zeros(self.post.out.shape, dtype=torch.uint8).pin_memory(),
                         "h2d": torch.cuda.Event(), "consumed": torch.cuda.Event(), "done": torch.cuda.Event(),
                         "used": False})
            self._slots.append(slot)
        self._ticket = 0

    def submit(self, pinned: dict) -> int:
        """Enqueue one frame from pinned host inputs (see pinned_inputs()); returns a ticket for collect().
        The caller must not modify `pinned` until the next-but-one submit."""
        t, s = self._enqueue(pinned, self._input_names)
        main = torch.cuda.current_stream()
        s["h_out"].copy_(self.post.out, non_blocking=True)
        s["done"].record(main)
        return t

    def _enqueue(self, pinned: dict, names):
        """H2D of the inputs `names` from pinned host tensors on the copy stream (double-buffered device staging), then
        one frame on the current stream. Returns (ticket, pipeline slot)."""
        if not hasattr(self, "_slots"):
            self._pipe_init()
        t = self._ticket
        s = self._slots[t % 2]
        main = torch.cuda.current_stream()
        if s["used"]:
            self._copy_stream.wait_event(s["consumed"])
        with torch.cuda.stream(self._copy_stream):
            for k in names:
                s[k].copy_(pinned[k], non_blocking=True)
            s["h2d"].record(self._copy_stream)
        main.wait_event(s["h2d"])
        for k in names:
            getattr(self, k).copy_(s[k])
        s["consumed"].record(main)
        s["used"] = True            # the next fill of this staging slot waits until this frame has read it
        self._ticket += 1
        self.step_device()
        return t, s

    def serve(self, clip_ids, eps=None) -> dict:
        """Run the source bank's clips `clip_ids` through the slots and return {clip_id: payload}, each payload a dict
        of numpy arrays {src_rotations, src_positions [nwin,24,3] float32, ours_rotations, ours_positions [nwin,24,3]
        float64, match [nwin] int64}: what characterize() returns for one clip (test_fullframework.py:672-721).

        Clips are placed by serving_schedule (first free slot, FIFO) and start on the frame their slot frees up. Per
        frame only the start / clip rows (and eps) go to the device, from pinned double-buffered host rows on a copy
        stream; the host never waits for a frame, only for the copy of the buffer it refills. Before the first of them,
        one extra frame starts every slot idle (start = 1, clip = -1), so that no slot keeps recording a clip of an
        earlier call into the bank's rows; it costs one frame per call and resets every slot's state. After the frame on which
        clips end, one mocha_clip_payload launch on a side stream converts them, and their rows download into pinned
        memory while later frames run. The returned arrays are views of one host buffer per call.

        eps None: eps.normal_() every frame, as step_bank does (the draws then depend on the schedule). Otherwise
        {clip_id: array [nwin-1, D]} in characterize()'s eps_seq layout: window w >= 1 of the clip uses row w-1,
        wherever and whenever it runs; clips without a table draw standard-normal rows on the host.
        """
        from .result_bank import PAYLOAD_KEYS, serving_schedule
        if self.results is None:
            raise _lib.MochaError("serve() needs CharacterizationSession(..., result_bank=...)")
        ids = [int(c) for c in clip_ids]
        if len(set(ids)) != len(ids):
            raise _lib.MochaError("serve(): duplicate clip ids (one clip cannot run in two slots at once)")
        if not ids:
            return {}
        self.results._check_ids(ids)
        bank, B, D = self.bank, self.B, self.D
        nwins = np.array([bank.clip_nwin[c] for c in ids], dtype=np.int64)
        tables, rng = None, None
        if eps is not None:
            tables = {}
            for c in ids:
                if c in eps:
                    e = np.asarray(eps[c], dtype=np.float32)
                    if e.shape != (bank.clip_nwin[c] - 1, D):
                        raise _lib.MochaError(f"serve(): eps of clip {c} must be [{bank.clip_nwin[c] - 1}, {D}], got {e.shape}")
                    tables[c] = e
            rng = np.random.default_rng()
        start_rows, clip_rows, place = serving_schedule(nwins, B)
        nframes = start_rows.shape[0]
        ends = place[:, 1] + nwins - 1
        order = np.argsort(ends, kind="stable")           # clips in the order they end
        ends_sorted = ends[order]
        dev = self.dev
        ids_dev = torch.tensor([ids[k] for k in order], dtype=torch.int32, device=dev)
        # host payload buffers: clip k at rows off[k] .. + nwin
        off = np.concatenate([[0], np.cumsum(nwins)[:-1]])
        total = int(nwins.sum())
        host = [torch.empty((total,) + tuple(t.shape[1:]), dtype=t.dtype).pin_memory()
                for t in self.results.payload_arrays()]
        names = ("start", "clip") + (("eps",) if tables is not None else ())
        pins = [{k: torch.zeros(getattr(self, k).shape, dtype=getattr(self, k).dtype).pin_memory() for k in names}
                for _ in range(2)]
        pin_ready = [None, None]
        side = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream()
        ids_np = np.asarray(ids, dtype=np.int32)
        slot_clip = np.full(B, -1, dtype=np.int64)        # schedule index of each slot's clip
        slot_first = np.zeros(B, dtype=np.int64)
        self.start.fill_(1)                              # drop whatever the slots held: start them idle
        self.clip.fill_(-1)
        self.step_device()
        self.start.zero_()
        j = 0
        for f in range(nframes):
            p = pins[f % 2]
            if pin_ready[f % 2] is not None:
                pin_ready[f % 2].synchronize()           # the copy of frame f-2 out of this buffer has finished
            st = start_rows[f]
            p["start"].numpy()[...] = st
            p["clip"].numpy()[...] = ids_np[clip_rows[f]]
            new = np.nonzero(st)[0]
            slot_clip[new], slot_first[new] = clip_rows[f][new], f
            if tables is not None:
                er = p["eps"].numpy()
                er[...] = 0.0
                for b in range(B):
                    k = slot_clip[b]
                    if k < 0:
                        continue
                    w = f - slot_first[b]
                    if 1 <= w < nwins[k]:
                        e = tables.get(ids[k])
                        er[b] = e[w - 1] if e is not None else rng.standard_normal(D, dtype=np.float32)
            elif not self.deterministic:
                self.eps.normal_()
            _, s = self._enqueue(p, names)
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
            pin_ready[f % 2] = ev
            if j < len(order) and ends_sorted[j] == f:
                j1 = j
                while j1 < len(order) and ends_sorted[j1] == f:
                    j1 += 1
                done_ev = torch.cuda.Event()
                done_ev.record(main)
                side.wait_event(done_ev)
                with torch.cuda.stream(side):
                    ks = order[j:j1]
                    self.results.payload_device(ids_dev[j:], j1 - j, int(nwins[ks].max()))
                    for k in ks:
                        first, n = bank.clip_start[ids[k]], int(nwins[k])
                        for h, t in zip(host, self.results.payload_arrays()):
                            h[off[k]:off[k] + n].copy_(t[first:first + n], non_blocking=True)
                j = j1
        side.synchronize()
        main.synchronize()
        hv = [h.numpy() for h in host]
        return {ids[k]: {name: a[off[k]:off[k] + int(nwins[k])] for name, a in zip(PAYLOAD_KEYS, hv)}
                for k in range(len(ids))}

    def collect(self, ticket: int) -> dict:
        """Wait for a submitted frame and return its outputs (dict of float64 numpy arrays [B, ...])."""
        s = self._slots[ticket % 2]
        s["done"].synchronize()
        return self._decode_out(s["h_out"].numpy())

    def h2d_bytes(self):
        if self.bank is not None:
            return self.h_start.numel() + self.h_clip.numel() * 4 + self.h_eps.numel() * 4
        return (self.h_X.numel() * 4 + self.h_side.numel() * 4 + self.h_contacts.numel() + self.h_eps.numel() * 4
                + (self.h_start.numel() if self.admission else 0))

    def d2h_bytes(self):
        return self.h_out.numel()

    @staticmethod
    def _decode_out(raw):
        dt = np.dtype([("pos", "f8", (25, 3)), ("rot", "f8", (25, 4)), ("vel", "f8", (25, 3)), ("ang", "f8", (25, 3)),
                       ("blend_pos", "f8", (25, 3)), ("ik_pos", "f8", (25, 3)), ("ik_rot", "f8", (25, 4)),
                       ("src_root_pos", "f8", (3,)), ("src_root_rot", "f8", (4,)), ("src_root_vel", "f8", (3,)),
                       ("src_root_ang", "f8", (3,))])
        rec = raw.view(dt)
        return {k: rec[k].copy() for k in dt.names}

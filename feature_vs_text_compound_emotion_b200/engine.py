"""Device-side engines: packed weights resident in HBM + ctypes calls into libcer_b200.so.

PyTorch is used for device memory (torch.empty), the current stream and nothing else; every
FLOP of the path runs in the hand-written kernels behind the C-ABI.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch

from . import _capi
from ._capi import FusionWeights, Ir50Weights, IrSe, IrUnit, TcnBlock, VggConv, VggFc, VggishStep, VggishWeights, check, lib


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class Ir50Engine:
    """IR frame encoder plan (cer_ir50_*): IR-50/100/152, plain or IR-SE (packed units carrying "se" weights run
    through cer_ir50_create_se).  ``frames_per_pass`` bounds the workspace: inputs longer than that are
    processed in passes inside one C call."""

    def __init__(self, packed: dict, device: torch.device, frames_per_pass: int = 512):
        _capi.require_gpu()
        self.device = torch.device(device)
        self.frames_per_pass = int(frames_per_pass)
        dev = lambda t: t.to(self.device).contiguous()
        self._keep: List[torch.Tensor] = []

        def put(t):
            d = dev(t)
            self._keep.append(d)
            return d.data_ptr()

        units = packed["units"]
        self._units = (IrUnit * len(units))()
        for i, u in enumerate(units):
            self._units[i] = IrUnit(u["cin"], u["depth"], u["stride"], u["has_proj"], put(u["w1"]), put(u["bias1"]),
                                    put(u["alpha"]), put(u["w2"]), put(u["bias2"]))
        self._w = Ir50Weights(packed["in_hw"], packed["in_hw"], put(packed["stem_w"]), put(packed["stem_bias"]),
                              put(packed["stem_alpha"]), len(units), self._units, packed["fc_in"], packed["emb_dim"],
                              put(packed["fc_w"]), put(packed["fc_bias"]))
        self.se = "se" in units[0]
        if any(("se" in u) != self.se for u in units):
            raise ValueError("either every unit or no unit carries SE weights")
        self._se = None
        if self.se:
            self._se = (IrSe * len(units))()
            for i, u in enumerate(units):
                self._se[i] = IrSe(u["se"]["fc1"].shape[0], 0, put(u["se"]["fc1"]), put(u["se"]["fc2"]))
        self.emb_dim = packed["emb_dim"]
        self.in_hw = packed["in_hw"]
        self.unit_shapes = []
        # per conv op in plan order (conv1, conv2 per unit, the FC, then the SE plan's projection convs): geometry and
        # algorithmic FLOPs per frame (bench accounting; identity columns of a MaxPool(1, 2) shortcut are not counted)
        self.conv_ops = []
        proj_ops = []
        hw = self.in_hw
        for u in units:
            hin = hw
            hw = (hw - 1) // u["stride"] + 1
            self.unit_shapes.append((hw, hw, u["depth"]))
            self.conv_ops.append({"cin": u["cin"], "cout": u["depth"], "h_in": hin, "h_out": hin, "stride": 1, "proj_cin": 0,
                                  "flop": 2.0 * hin * hin * u["depth"] * 9 * u["cin"]})
            kproj = u["cin"] if u["has_proj"] else 0
            if self.se and kproj:
                proj_ops.append({"cin": u["cin"], "cout": u["depth"], "h_in": hin, "h_out": hw, "stride": u["stride"],
                                 "proj_cin": 0, "flop": 2.0 * hw * hw * u["depth"] * kproj})
                kproj = 0
            kflop = 0 if u.get("identity_sc") else kproj
            self.conv_ops.append({"cin": u["depth"], "cout": u["depth"], "h_in": hin, "h_out": hw, "stride": u["stride"],
                                  "proj_cin": kproj, "flop": 2.0 * hw * hw * u["depth"] * (9 * u["depth"] + kflop)})
        self.conv_ops.append({"cin": packed["fc_in"], "cout": packed["emb_dim"], "h_in": 1, "h_out": 1, "stride": 1, "proj_cin": 0,
                              "flop": 2.0 * packed["fc_in"] * packed["emb_dim"]})
        self.conv_ops += proj_ops
        with torch.cuda.device(self.device):
            nbytes = lib().cer_ir50_workspace_bytes_se(C.byref(self._w), self._se, self.frames_per_pass)
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            h = C.c_void_p()
            check(lib().cer_ir50_create_se(C.byref(h), C.byref(self._w), self._se, self.frames_per_pass, self._ws.data_ptr(),
                                           nbytes), "cer_ir50_create_se")
        self._h = h

    def forward(self, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x: [N,3,H,W] fp32 on the engine's device -> [N, emb_dim] fp32, unit norm."""
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] != self.in_hw or x.shape[3] != self.in_hw:
            raise ValueError(f"expected [N,3,{self.in_hw},{self.in_hw}], got {tuple(x.shape)}")
        if x.device != self.device or x.dtype != torch.float32:
            raise ValueError("input must be fp32 on the engine's CUDA device")
        x = x.contiguous()
        n = x.shape[0]
        if out is None:
            out = torch.empty(n, self.emb_dim, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib().cer_ir50_forward(self._h, x.data_ptr(), n, out.data_ptr(), _capi.current_stream_ptr(self.device)),
                  "cer_ir50_forward")
        return out

    def debug_activation(self, x: torch.Tensor, unit_index: int) -> torch.Tensor:
        """bf16 NHWC output of unit ``unit_index`` (-1: stem) for the first frames_per_pass frames."""
        x = x.contiguous()
        n = x.shape[0]
        H, W, Cc = (self.in_hw, self.in_hw, 64) if unit_index < 0 else self.unit_shapes[unit_index]
        dst = torch.empty(n, H, W, Cc, dtype=torch.bfloat16, device=self.device)
        with torch.cuda.device(self.device):
            r = lib().cer_ir50_debug_activation(self._h, x.data_ptr(), n, unit_index, dst.data_ptr(),
                                                _capi.current_stream_ptr(self.device))
        check(int(r), "cer_ir50_debug_activation")
        return dst

    def launches(self, n_frames: int) -> int:
        return int(lib().cer_ir50_launches(self._h, n_frames))

    @property
    def n_conv_ops(self) -> int:
        return len(self.conv_ops)

    def op_variant(self, op_index: int, n_frames: int) -> str:
        """Kernel instantiation the plan launches for conv op ``op_index`` (conv1, conv2 of each unit, the FC, then
        the SE plan's projection convs)."""
        buf = C.create_string_buffer(96)
        check(lib().cer_ir50_op_variant(self._h, op_index, n_frames, buf, 96), "cer_ir50_op_variant")
        return buf.value.decode()

    def run_ops(self, x: Optional[torch.Tensor], frames: int, first_op: int, last_op: int) -> None:
        """Profiling aid: launch ops [first_op, last_op] of one pass (0 = stem, 1.. = unit convs, last = FC) over the
        activations a previous forward of the same frames left in the plan's buffers."""
        with torch.cuda.device(self.device):
            check(lib().cer_ir50_run_ops(self._h, None if x is None else x.data_ptr(), frames, first_op, last_op,
                                         _capi.current_stream_ptr(self.device)), "cer_ir50_run_ops")

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                lib().cer_ir50_destroy(h)
            except Exception:
                pass
            self._h = None


class VggishEngine:
    """VGGish plan (cer_vggish_*): [N,96,64] fp32 log-mel examples -> [N,128] fp32."""

    def __init__(self, packed: dict, device: torch.device, patches_per_pass: int = 1200):
        _capi.require_gpu()
        self.device = torch.device(device)
        self.patches_per_pass = int(patches_per_pass)
        self._keep: List[torch.Tensor] = []

        def put(t):
            d = t.to(self.device).contiguous()
            self._keep.append(d)
            return d.data_ptr()

        self._convs = (VggConv * len(packed["convs"]))()
        for i, c in enumerate(packed["convs"]):
            self._convs[i] = VggConv(c["cin"], c["cout"], c["pool_after"], put(c["w"]), put(c["bias"]))
        self._fcs = (VggFc * len(packed["fcs"]))()
        for i, f in enumerate(packed["fcs"]):
            self._fcs[i] = VggFc(f["in_dim"], f["out_dim"], f["relu"], put(f["w"]), put(f["bias"]))
        self._w = VggishWeights(packed["in_h"], packed["in_w"], packed["c1"], put(packed["conv1_w"]),
                                put(packed["conv1_bias"]), len(packed["convs"]), self._convs, len(packed["fcs"]),
                                self._fcs, put(packed["zeros"]))
        self.in_h, self.in_w, self.emb_dim = packed["in_h"], packed["in_w"], packed["emb_dim"]
        with torch.cuda.device(self.device):
            nbytes = lib().cer_vggish_workspace_bytes(C.byref(self._w), self.patches_per_pass)
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            h = C.c_void_p()
            check(lib().cer_vggish_create(C.byref(h), C.byref(self._w), self.patches_per_pass, self._ws.data_ptr(), nbytes),
                  "cer_vggish_create")
        self._h = h
        n_steps = check(lib().cer_vggish_steps(h, None, 0), "cer_vggish_steps")
        desc = (VggishStep * n_steps)()
        check(lib().cer_vggish_steps(h, desc, n_steps), "cer_vggish_steps")
        # per plan step after the stem (cer_vggish_step): kind "conv" / "pool" / "fc", the index into packed["convs"] or
        # packed["fcs"] (a pool: of the conv it follows), the per-patch output shape and dtype, and whether a conv's
        # epilogue applied the following max-pool
        self.step_shapes = [{"kind": ("conv", "pool", "fc")[d.kind], "layer": d.layer, "shape": (d.h, d.w, d.c),
                             "dtype": torch.float32 if d.out_fp32 else torch.bfloat16, "pool_fused": bool(d.pool_fused)}
                            for d in desc]

    def forward(self, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if x.dim() != 3 or x.shape[1] != self.in_h or x.shape[2] != self.in_w:
            raise ValueError(f"expected [N,{self.in_h},{self.in_w}], got {tuple(x.shape)}")
        if x.device != self.device or x.dtype != torch.float32:
            raise ValueError("input must be fp32 on the engine's CUDA device")
        x = x.contiguous()
        n = x.shape[0]
        if out is None:
            out = torch.empty(n, self.emb_dim, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib().cer_vggish_forward(self._h, x.data_ptr(), n, out.data_ptr(), _capi.current_stream_ptr(self.device)),
                  "cer_vggish_forward")
        return out

    def launches(self, n: int) -> int:
        return int(lib().cer_vggish_launches(self._h, n))

    def debug_activation(self, x: torch.Tensor, step: int) -> torch.Tensor:
        """Output [n, h, w, c] of plan step ``step`` (-1: the stem's pooled bf16 map) for one pass over x's n <=
        patches_per_pass patches; shape and dtype as in step_shapes."""
        x = x.contiguous()
        n = x.shape[0]
        if step < 0:
            shape, dtype = (self.in_h // 2, self.in_w // 2, self._w.c1), torch.bfloat16
        else:
            shape, dtype = self.step_shapes[step]["shape"], self.step_shapes[step]["dtype"]
        dst = torch.empty(n, *shape, dtype=dtype, device=self.device)
        with torch.cuda.device(self.device):
            r = lib().cer_vggish_debug_activation(self._h, x.data_ptr(), n, step, dst.data_ptr(),
                                                  _capi.current_stream_ptr(self.device))
        check(int(r), "cer_vggish_debug_activation")
        return dst

    def op_variant(self, step: int, n_patches: int) -> str:
        """Kernel instantiation plan step ``step`` launches (-1: the stem) when a pass holds min(n_patches,
        patches_per_pass) patches."""
        buf = C.create_string_buffer(96)
        check(lib().cer_vggish_op_variant(self._h, step, n_patches, buf, 96), "cer_vggish_op_variant")
        return buf.value.decode()

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                lib().cer_vggish_destroy(h)
            except Exception:
                pass
            self._h = None


class TcnEngine:
    """A stack of TemporalBlocks, time-major [B,T,C] fp32.

    precision="tf32" (default): tcgen05 kind::tf32 tensor-core kernel, two launches per block
    (cer_tcn_block_tc_forward).  precision="fp32": the CUDA-core fused kernel, one launch per
    block (cer_tcn_block_forward) -- exact fp32 FMA, ~10x slower, kept for numerics work."""

    def __init__(self, blocks: Sequence[dict], device: torch.device, precision: str = "tf32"):
        _capi.require_gpu()
        if precision not in ("tf32", "fp32"):
            raise ValueError(precision)
        self.device = torch.device(device)
        self.precision = precision
        self._keep: List[torch.Tensor] = []
        self.blocks: List[TcnBlock] = []
        self.c_in = blocks[0]["c_in"]                    # what the caller passes
        self.c_out = blocks[-1]["c_out"]

        def put(t):
            if t is None:
                return None
            d = t.to(self.device).contiguous()
            self._keep.append(d)
            return d.data_ptr()

        if precision == "tf32":
            from .packing import tcn_block_to_kmajor
            blocks = [tcn_block_to_kmajor(b) for b in blocks]
        for b in blocks:
            self.blocks.append(TcnBlock(b["c_in"], b["c_out"], b["kernel_size"], b["dilation"], put(b["w1"]), put(b["b1"]),
                                        put(b["w2"]), put(b["b2"]), put(b["wd"]), put(b["bd"]), put(b["post_scale"]),
                                        put(b["post_shift"])))
        self._ws: Optional[torch.Tensor] = None
        self._retired: List[torch.Tensor] = []

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 3 or x.shape[2] != self.c_in:
            raise ValueError(f"expected [B,T,{self.c_in}], got {tuple(x.shape)}")
        if x.device != self.device or x.dtype != torch.float32:
            raise ValueError("input must be fp32 on the engine's CUDA device")
        if self.blocks[0].c_in != self.c_in:             # channels padded to the kernel's 32-channel chunks
            x = torch.nn.functional.pad(x, (0, self.blocks[0].c_in - self.c_in))
        x = x.contiguous()
        B, T, _ = x.shape
        stream = _capi.current_stream_ptr(self.device)
        cur = x
        with torch.cuda.device(self.device):
            if self.precision == "tf32":
                need = max(B * T * blk.c_out * 4 for blk in self.blocks)
                if self._ws is None or self._ws.numel() < need:
                    # CUDA graphs captured for smaller shapes (LFAN.forward_features) have the old block's
                    # address baked into their kernel nodes: retired workspaces stay alive with the engine
                    if self._ws is not None:
                        self._retired.append(self._ws)
                    self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
            for blk in self.blocks:
                y = torch.empty(B, T, blk.c_out, dtype=torch.float32, device=self.device)
                if self.precision == "tf32":
                    check(lib().cer_tcn_block_tc_forward(C.byref(blk), cur.data_ptr(), y.data_ptr(), B, T,
                                                         self._ws.data_ptr(), self._ws.numel(), stream),
                          "cer_tcn_block_tc_forward")
                else:
                    check(lib().cer_tcn_block_forward(C.byref(blk), cur.data_ptr(), y.data_ptr(), B, T, None, 0, stream),
                          "cer_tcn_block_forward")
                cur = y
        return cur

    @property
    def launches(self) -> int:
        return len(self.blocks) * (2 if self.precision == "tf32" else 1)


class FusionEngine:
    """Cross-modal attention + LayerNorm (+ classifier) (cer_fusion_head_forward)."""

    def __init__(self, fw: dict, device: torch.device):
        _capi.require_gpu()
        self.device = torch.device(device)
        self._keep: List[torch.Tensor] = []

        def put(t):
            d = t.to(self.device).contiguous()
            self._keep.append(d)
            return d.data_ptr()

        w = FusionWeights()
        w.n_modals = fw["n_modals"]
        for i, d in enumerate(fw["dim"]):
            w.dim[i] = d
            w.wqkv[i] = put(fw["wqkv"][i])
            w.bqkv[i] = put(fw["bqkv"][i])
        w.modal_dim, w.num_heads, w.n_out = fw["modal_dim"], fw["num_heads"], fw["n_out"]
        w.wo, w.bo, w.ln_g, w.ln_b = put(fw["wo"]), put(fw["bo"]), put(fw["ln_g"]), put(fw["ln_b"])
        w.wr, w.br = put(fw["wr"]), put(fw["br"])
        self._w = w
        self.dims = list(fw["dim"])
        self.n_out = fw["n_out"]
        self.E = fw["modal_dim"] * fw["n_modals"]
        self.num_heads, self.head_dim = fw["num_heads"], fw["modal_dim"] // fw["num_heads"]
        # the fused kernel stages every weight in shared memory (~150 KB at the reference's sizes);
        # larger configurations run the same arithmetic as separate kernels
        fused_floats = (sum(self.dims) * 3 * fw["modal_dim"] + self.E * self.E + (self.dims[0] + self.E) * self.n_out
                        + fw["n_modals"] * 3 * fw["modal_dim"] + 3 * self.E + 16
                        + 4 * 4 * (sum(self.dims) + fw["n_modals"] * 3 * fw["modal_dim"] + self.E))
        self.composed = fused_floats * 4 > 227 * 1024 - 64 or self.E > 128 or self.n_out > 16
        if self.composed:
            d = lambda t: t.to(self.device).contiguous()
            self._c = {"wqkv": [d(t) for t in fw["wqkv_oi"]], "bqkv": [d(t) for t in fw["bqkv"]], "wo": d(fw["wo_oi"]),
                       "bo": d(fw["bo"]), "g": d(fw["ln_g"]), "b": d(fw["ln_b"]), "wr": d(fw["wr_oi"]), "br": d(fw["br"])}

    def forward(self, feats: Sequence[torch.Tensor], want_fused: bool = False):
        """feats[m]: [rows, D_m] fp32 -> logits [rows, n_out] (and fused [rows, E])."""
        rows = feats[0].shape[0]
        keep = []
        ptrs = (C.c_void_p * len(feats))()
        for i, f in enumerate(feats):
            if f.dim() != 2 or f.shape[0] != rows or f.shape[1] != self.dims[i]:
                raise ValueError(f"modality {i}: expected [{rows},{self.dims[i]}], got {tuple(f.shape)}")
            if f.device != self.device or f.dtype != torch.float32:
                raise ValueError("inputs must be fp32 on the engine's CUDA device")
            f = f.contiguous()
            keep.append(f)
            ptrs[i] = f.data_ptr()
        if self.composed:
            return self._forward_composed(keep, rows, want_fused)
        logits = torch.empty(rows, self.n_out, dtype=torch.float32, device=self.device)
        fused = torch.empty(rows, self.E, dtype=torch.float32, device=self.device) if want_fused else None
        with torch.cuda.device(self.device):
            check(lib().cer_fusion_head_forward(C.byref(self._w), ptrs, rows, logits.data_ptr(), _ptr(fused),
                                                _capi.current_stream_ptr(self.device)), "cer_fusion_head_forward")
        return (logits, fused) if want_fused else logits


class PreprocEngine:
    """The reference's eval video transform on the device (cer_preproc_*): uint8 [N,H,W,3] stored
    crops -> fp32 [N,3,crop,crop] in [-1,1], bit-exact with PIL resize + crop + normalise."""

    def __init__(self, in_h: int, in_w: int, device: torch.device, resize: int = 48, crop: int = 40):
        _capi.require_gpu()
        self.device = torch.device(device)
        self.in_h, self.in_w, self.crop = int(in_h), int(in_w), int(crop)
        with torch.cuda.device(self.device):
            nbytes = lib().cer_preproc_workspace_bytes()
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            h = C.c_void_p()
            check(lib().cer_preproc_create(C.byref(h), self.in_h, self.in_w, resize, crop, self._ws.data_ptr(), nbytes),
                  "cer_preproc_create")
        self._h = h

    def forward(self, frames: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if frames.dim() != 4 or tuple(frames.shape[1:]) != (self.in_h, self.in_w, 3) or frames.dtype != torch.uint8:
            raise ValueError(f"expected uint8 [N,{self.in_h},{self.in_w},3], got {frames.dtype} {tuple(frames.shape)}")
        if frames.device != self.device:
            raise ValueError("frames must be on the engine's CUDA device")
        frames = frames.contiguous()
        n = frames.shape[0]
        if out is None:
            out = torch.empty(n, 3, self.crop, self.crop, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib().cer_preproc_forward(self._h, frames.data_ptr(), n, out.data_ptr(), _capi.current_stream_ptr(self.device)),
                  "cer_preproc_forward")
        return out

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                lib().cer_preproc_destroy(h)
            except Exception:
                pass
            self._h = None


class LogMelEngine:
    """Waveform -> VGGish input examples on the device (cer_logmel_forward + cer_frame_examples).
    ``examples(wave, window_sec, hop_sec)`` mirrors vggish_input.waveform_to_examples for mono
    16 kHz input (hop_sec = 1/fps gives one [96,64] example per video frame, audio.py:126-127)."""

    def __init__(self, device: torch.device, cfg: Optional[dict] = None):
        _capi.require_gpu()
        from . import packing
        self.cfg = dict(cfg or packing.LOGMEL)
        self.device = torch.device(device)
        self._tables = packing.logmel_tables(self.cfg).to(self.device)

    def log_mel(self, wave: torch.Tensor) -> torch.Tensor:
        """wave fp32 [n_samples] on the device -> log-mel fp32 [n_frames, n_mel]."""
        if wave.dim() != 1 or wave.dtype != torch.float32 or wave.device != self.device:
            raise ValueError("wave must be a 1-D fp32 tensor on the engine's CUDA device")
        wave = wave.contiguous()
        c = self.cfg
        n = int(lib().cer_logmel_num_frames(wave.numel(), c["win"], c["hop"]))
        out = torch.empty(n, c["n_mel"], dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib().cer_logmel_forward(wave.data_ptr(), wave.numel(), self._tables.data_ptr(), c["win"], c["hop"], c["fft"],
                                           c["n_mel"], c["log_offset"], out.data_ptr(), _capi.current_stream_ptr(self.device)),
                  "cer_logmel_forward")
        return out

    def examples(self, wave: torch.Tensor, window_sec: float = 0.96, hop_sec: float = 0.96) -> torch.Tensor:
        lm = self.log_mel(wave)
        rate = 1.0 / (self.cfg["hop"] / self.cfg["sample_rate"])
        win = int(round(window_sec * rate))
        hop = hop_sec * rate
        import math
        n = 1 + int(math.floor((lm.shape[0] - win) / hop)) if lm.shape[0] >= win else 0
        starts = torch.tensor([round(hop * i) for i in range(n)], dtype=torch.int32).to(self.device)   # Python round, as my_frame
        out = torch.empty(n, win, self.cfg["n_mel"], dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(lib().cer_frame_examples(lm.data_ptr(), starts.data_ptr(), n, win, self.cfg["n_mel"], out.data_ptr(),
                                           _capi.current_stream_ptr(self.device)), "cer_frame_examples")
        return out


def _fusion_forward_composed(self, feats, rows, want_fused):
    """qkv_proj -> modal attention -> o_proj -> LayerNorm -> cat -> regressor as separate kernels."""
    c = self._c
    qkv = [linear(f, c["wqkv"][i], c["bqkv"][i]) for i, f in enumerate(feats)]
    ptrs = (C.c_void_p * len(qkv))(*[t.data_ptr() for t in qkv])
    vals = torch.empty(rows, self.E, dtype=torch.float32, device=self.device)
    with torch.cuda.device(self.device):
        check(lib().cer_modal_attention_forward(ptrs, rows, len(qkv), self.num_heads, self.head_dim, vals.data_ptr(),
                                                _capi.current_stream_ptr(self.device)), "cer_modal_attention_forward")
    fused = add_layernorm(linear(vals, c["wo"], c["bo"]), None, c["g"], c["b"])
    cat = torch.empty(rows, self.dims[0] + self.E, dtype=torch.float32, device=self.device)
    cat[:, :self.dims[0]].copy_(feats[0])
    cat[:, self.dims[0]:].copy_(fused)
    logits = linear(cat, c["wr"], c["br"])
    return (logits, fused) if want_fused else logits


FusionEngine._forward_composed = _fusion_forward_composed


def stitch_windows(win_logits: torch.Tensor, win_start: torch.Tensor, length: int) -> torch.Tensor:
    """win_logits [n_win, win_len, n_out] fp32, win_start int32 [n_win] -> [length, n_out] mean over
    the windows covering each frame (trainer.py:864-890)."""
    _capi.require_gpu()
    n_win, win_len, n_out = win_logits.shape
    out = torch.empty(length, n_out, dtype=torch.float32, device=win_logits.device)
    with torch.cuda.device(win_logits.device):
        check(lib().cer_stitch_windows(win_logits.contiguous().data_ptr(), win_start.contiguous().data_ptr(), n_win,
                                       win_len, n_out, length, out.data_ptr(), _capi.current_stream_ptr()),
              "cer_stitch_windows")
    return out


def conv_forward(src: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, ksize: int, stride: int, pad: int,
                 alpha: Optional[torch.Tensor] = None, res: Optional[torch.Tensor] = None, out_fp32: bool = False,
                 n_frames: Optional[int] = None) -> torch.Tensor:
    """One convolution through the tcgen05 implicit-GEMM kernel (cer_conv_forward).
    src bf16 [N,H,W,Cin]; weight bf16 [Cout, k*k*Cin]; bias fp32 [1|9, Cout] -> [n,Ho,Wo,Cout]."""
    _capi.require_gpu()
    n_alloc, H, W, cin = src.shape
    n = n_alloc if n_frames is None else n_frames
    cout = weight.shape[0]
    ho, wo = (H + 2 * pad - ksize) // stride + 1, (W + 2 * pad - ksize) // stride + 1
    dst = torch.empty(n, ho, wo, cout, dtype=torch.float32 if out_fp32 else torch.bfloat16, device=src.device)
    bias = bias.reshape(-1, cout).contiguous()
    with torch.cuda.device(src.device):
        check(lib().cer_conv_forward(src.contiguous().data_ptr(), n, n_alloc, H, W, cin, weight.contiguous().data_ptr(),
                                     cout, ksize, stride, pad, bias.data_ptr(), bias.shape[0], _ptr(alpha), _ptr(res),
                                     dst.data_ptr(), int(out_fp32), _capi.current_stream_ptr()), "cer_conv_forward")
    return dst


# ----------------------------------------------------------------------------------------------
# fp32 building blocks of the CAN / JMT / MT heads (cer_linear_forward, cer_softmax_gate,
# cer_sdpa_forward, cer_add_layernorm).  All tensors are row-major 2-D views [rows, features].
# ----------------------------------------------------------------------------------------------
ACT = {None: 0, "leaky_relu": 1, "relu": 2}


def linear(x: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], act: Optional[str] = None,
           out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """y = act(x W^T + b).  x [rows, in] (row stride may exceed in), w [out, in] contiguous; ``out`` may be
    a column slice of a wider buffer (concat without a copy)."""
    rows, k = x.shape
    n = w.shape[0]
    if x.stride(1) != 1 or w.stride() != (k, 1) or w.shape[1] != k:
        raise ValueError("linear: x must be unit-stride in features and w contiguous [out, in]")
    if out is None:
        out = torch.empty(rows, n, dtype=torch.float32, device=x.device)
    if out.stride(1) != 1 or out.shape != (rows, n):
        raise ValueError("linear: bad output view")
    with torch.cuda.device(x.device):
        check(lib().cer_linear_forward(x.data_ptr(), rows, k, x.stride(0), w.data_ptr(), _ptr(b), n, ACT[act], out.data_ptr(),
                                       out.stride(0), _capi.current_stream_ptr()), "cer_linear_forward")
    return out


def softmax_gate(gate: torch.Tensor, feat: torch.Tensor) -> torch.Tensor:
    out = torch.empty_like(feat)
    with torch.cuda.device(feat.device):
        check(lib().cer_softmax_gate(gate.contiguous().data_ptr(), feat.contiguous().data_ptr(), feat.shape[0], feat.shape[1],
                                     out.data_ptr(), _capi.current_stream_ptr()), "cer_softmax_gate")
    return out


def sdpa(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, batch: int, len_q: int, len_k: int,
         precision: str = "tf32") -> torch.Tensor:
    """Single-head attention.  q [batch*len_q, E], k / v [batch*len_k, E] (column slices of a packed
    projection are fine) -> [batch*len_q, E].  precision="tf32": tensor-core flash attention
    (cer_sdpa_tc_forward, E in {64, 128}); "fp32": the exact CUDA-core kernel (cer_sdpa_forward)."""
    e = q.shape[1]
    out = torch.empty(batch * len_q, e, dtype=torch.float32, device=q.device)
    tc = precision == "tf32" and e in (64, 128) and all(t.stride(0) % 4 == 0 and t.data_ptr() % 16 == 0 for t in (q, k, v))
    fn, name = (lib().cer_sdpa_tc_forward, "cer_sdpa_tc_forward") if tc else (lib().cer_sdpa_forward, "cer_sdpa_forward")
    with torch.cuda.device(q.device):
        check(fn(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), batch, len_q, len_k, e,
                 out.data_ptr(), e, _capi.current_stream_ptr()), name)
    return out


def add_layernorm(x: torch.Tensor, res: Optional[torch.Tensor], gamma: torch.Tensor, beta: torch.Tensor,
                  eps: float = 1e-5) -> torch.Tensor:
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        check(lib().cer_add_layernorm(x.contiguous().data_ptr(), None if res is None else res.contiguous().data_ptr(),
                                      x.shape[0], x.shape[1], gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr(),
                                      _capi.current_stream_ptr()), "cer_add_layernorm")
    return out


def tanh_(y: torch.Tensor) -> torch.Tensor:
    """In-place tanh on a contiguous fp32 CUDA tensor (cer_tanh_inplace)."""
    if not y.is_contiguous() or y.dtype != torch.float32:
        raise ValueError("tanh_: contiguous fp32 tensor expected")
    with torch.cuda.device(y.device):
        check(lib().cer_tanh_inplace(y.data_ptr(), y.numel(), _capi.current_stream_ptr()), "cer_tanh_inplace")
    return y


def add_(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a += b on contiguous fp32 CUDA tensors of equal size (cer_add_inplace)."""
    if not (a.is_contiguous() and b.is_contiguous()) or a.numel() != b.numel() or a.dtype != torch.float32 or b.dtype != torch.float32:
        raise ValueError("add_: contiguous fp32 tensors of equal size expected")
    with torch.cuda.device(a.device):
        check(lib().cer_add_inplace(a.data_ptr(), b.data_ptr(), a.numel(), _capi.current_stream_ptr()), "cer_add_inplace")
    return a

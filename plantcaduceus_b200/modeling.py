"""Drop-in for the object the reference obtains from
``AutoModelForMaskedLM.from_pretrained(model_dir, trust_remote_code=True, torch_dtype=...)``
(reference src/zero_shot_score.py:91) and calls as ``model(input_ids=ids).logits`` (:115-116) or
``model(input_ids=ids, output_hidden_states=True).hidden_states[-1]`` (src/train_XGBoost.py:104-105).

All arithmetic happens in libpcad.so (hand-written sm_100a kernels, C ABI in include/pcad.h); torch is
used for device memory and streams only.  There is no CPU path: ``.to("cpu")`` forward calls raise.
"""
from __future__ import annotations

import ctypes as C
import json
import numbers
import os
from dataclasses import dataclass
from typing import Dict, Iterable, List, Optional, Tuple, Union

import numpy as np
import torch

from . import _lib
from .configuration import CaduceusConfig, preset
from .tokenizer import CharDNATokenizer
from .weights import random_init_state_dict


@dataclass
class MaskedLMOutput:
    logits: Optional[torch.Tensor] = None
    hidden_states: Optional[Tuple[torch.Tensor, ...]] = None
    loss: Optional[torch.Tensor] = None


_TORCH_TO_PCAD = {torch.float32: _lib.PCAD_F32, torch.bfloat16: _lib.PCAD_BF16, torch.float16: _lib.PCAD_F16}


def hidden_layer_indices(layers: Union[str, Iterable[int]], n_layer: int) -> List[int]:
    """Indices into the reference's ``hidden_states`` tuple (``n_layer + 1`` entries: 0 the embedding, k in [1, n_layer) layer
    k-1's mixer output, n_layer the final normed state) in the caller's order, negative ones counted from the end as Python
    does.  ``"all"`` is every index.  Raises ValueError for anything else than "all" or a non-empty iterable of ints, for an
    index outside [-(n_layer + 1), n_layer], and for an index requested twice."""
    n = n_layer + 1
    if isinstance(layers, str):
        if layers != "all":
            raise ValueError(f"hidden layers must be 'all' or an iterable of ints, not {layers!r}")
        return list(range(n))
    try:
        items = list(layers)
    except TypeError:
        raise ValueError(f"hidden layers must be 'all' or an iterable of ints, not {layers!r}") from None
    if not items:
        raise ValueError("no hidden layer requested")
    out = []
    for k in items:
        if isinstance(k, (bool, np.bool_)) or not isinstance(k, numbers.Integral):
            raise ValueError(f"hidden layer index {k!r} is not an int")
        k = int(k)
        if not -n <= k < n:
            raise ValueError(f"hidden layer index {k} out of range for {n} hidden states (n_layer = {n_layer})")
        k %= n
        if k in out:
            raise ValueError(f"hidden layer index {k} requested twice (after counting negative indices from the end)")
        out.append(k)
    return out


def hidden_mean_ranges(ranges, B: int, L: int) -> torch.Tensor:
    """Per-window ranges [s_b, e_b) for ``hidden_mean`` as int32 [B, 2] (on ``ranges``' device).  Raises ValueError unless
    ``ranges`` is [B, 2] integers (a tensor, an array or nested sequences).  Values are clamped to [-1, L + 1], which keeps
    every valid range and keeps every invalid one invalid, so that no int64 value wraps into a valid int32 range."""
    try:
        r = ranges if isinstance(ranges, torch.Tensor) else torch.as_tensor(np.asarray(ranges))
    except (TypeError, ValueError, RuntimeError) as e:
        raise ValueError(f"ranges must be [B, 2] integers: {e}") from None
    if r.dtype not in (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8):
        raise ValueError(f"ranges must be [B, 2] integers, not {r.dtype}")
    if tuple(r.shape) != (B, 2):
        raise ValueError(f"ranges must be [B, 2] = [{B}, 2], not {list(r.shape)}")
    return r.to(torch.int64).clamp(-1, L + 1).to(torch.int32).contiguous()


class CaduceusForMaskedLM:
    """Inference-only Caduceus masked LM backed by libpcad."""

    def __init__(self, config: CaduceusConfig, state_dict: Dict[str, torch.Tensor],
                 torch_dtype: torch.dtype = torch.bfloat16, tokenizer: Optional[CharDNATokenizer] = None):
        config.validate_supported()
        if torch_dtype == torch.float16:
            # The reference picks fp16 only on pre-Ampere GPUs (zero_shot_score.py:80-82); not a B200 case.
            raise ValueError("float16 is not supported by the B200 engine; use bfloat16 or float32")
        if torch_dtype not in (torch.bfloat16, torch.float32):
            raise ValueError(f"unsupported torch_dtype {torch_dtype}")
        self.config = config
        self.dtype = torch_dtype
        self.device = torch.device("cpu")
        self._sd = state_dict
        self._handle = None
        self._tokenizer = tokenizer or CharDNATokenizer()
        self._lib = _lib.load()  # fail loudly if the extension is missing

    # ---- construction -------------------------------------------------------------------------
    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path: Union[str, Dict[str, torch.Tensor]],
                        config: Optional[CaduceusConfig] = None, torch_dtype: torch.dtype = torch.bfloat16,
                        trust_remote_code: bool = True, **_kw) -> "CaduceusForMaskedLM":
        """Accepts a state dict (+config), or a local checkpoint directory holding ``config.json`` and
        ``model.safetensors`` / ``pytorch_model.bin``.  Hub names cannot be resolved offline."""
        if isinstance(pretrained_model_name_or_path, dict):
            if config is None:
                raise ValueError("config is required when loading from a state dict")
            return cls(config, pretrained_model_name_or_path, torch_dtype)
        path = str(pretrained_model_name_or_path)
        if os.path.isdir(path):
            with open(os.path.join(path, "config.json")) as f:
                cfg = CaduceusConfig.from_dict(json.load(f))
            st = os.path.join(path, "model.safetensors")
            if os.path.exists(st):
                from safetensors.torch import load_file
                sd = load_file(st)
            else:
                sd = torch.load(os.path.join(path, "pytorch_model.bin"), map_location="cpu", weights_only=True)
            # safetensors checkpoints are saved with tied tensors de-duplicated: restore both names of every tie, as HF's
            # tie_weights does after loading (embedding <-> LM head, mamba_fwd <-> mamba_rev in/out projections)
            from .weights import restore_tied_names
            restore_tied_names(sd, cfg.n_layer)
            return cls(cfg, sd, torch_dtype, CharDNATokenizer.from_pretrained(path))
        raise FileNotFoundError(
            f"{path!r} is not a local checkpoint directory (no network here). Use from_random('{path}') for "
            f"random-initialised weights of that architecture.")

    @classmethod
    def from_random(cls, name_or_config: Union[str, CaduceusConfig], seed: int = 0,
                    torch_dtype: torch.dtype = torch.bfloat16) -> "CaduceusForMaskedLM":
        cfg = preset(name_or_config) if isinstance(name_or_config, str) else name_or_config
        return cls(cfg, random_init_state_dict(cfg, seed), torch_dtype)

    def state_dict(self) -> Dict[str, torch.Tensor]:
        return self._sd

    # ---- nn.Module-like surface -------------------------------------------------------------------
    def eval(self) -> "CaduceusForMaskedLM":
        return self

    def to(self, *args, **kwargs) -> "CaduceusForMaskedLM":
        device = kwargs.get("device")
        dtype = kwargs.get("dtype")
        for a in args:
            if isinstance(a, torch.dtype):
                dtype = a
            elif a is not None:
                device = a
        new_device = torch.device(device) if device is not None else self.device
        new_dtype = dtype if dtype is not None else self.dtype
        if new_dtype not in (torch.bfloat16, torch.float32):
            raise ValueError(f"unsupported dtype {new_dtype}")
        if new_device.type == "cuda" and new_device.index is None:
            new_device = torch.device("cuda", torch.cuda.current_device())
        changed = (new_device != self.device) or (new_dtype != self.dtype)
        self.device, self.dtype = new_device, new_dtype
        if changed or (self._handle is None and new_device.type == "cuda"):
            self._release()
            if new_device.type == "cuda":
                self._build_handle()
        return self

    def cuda(self, index: Optional[int] = None):
        return self.to(torch.device("cuda", torch.cuda.current_device() if index is None else index))

    def parameters(self):
        seen = set()
        for v in self._sd.values():
            if v.data_ptr() not in seen:
                seen.add(v.data_ptr())
                yield v

    def _release(self):
        if self._handle is not None:
            self._lib.pcad_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _build_handle(self):
        cfg = self.config
        pc = _lib.PcadConfig()
        pc.d_model, pc.n_layer, pc.vocab_size = cfg.d_model, cfg.n_layer, cfg.vocab_size
        pc.d_state, pc.d_conv, pc.expand, pc.dt_rank = cfg.d_state, cfg.d_conv, cfg.expand, cfg.dt_rank
        pc.norm_eps = float(cfg.norm_epsilon)
        pc.residual_in_fp32 = int(bool(cfg.residual_in_fp32))
        pc.dtype = _TORCH_TO_PCAD[self.dtype]
        pc.mixer = _lib.PCAD_MIXER_MAMBA2 if cfg.is_mamba2 else _lib.PCAD_MIXER_MAMBA1
        pc.headdim, pc.ngroups = cfg.headdim, cfg.ngroups
        for i in range(16):
            pc.complement_map[i] = int(cfg.complement_map.get(i, i)) if i < cfg.vocab_size else i
        h = C.c_void_p()
        _lib.check(self._lib.pcad_create(C.byref(pc), self.device.index, C.byref(h)))
        self._handle = h
        try:
            comp_want = [int(cfg.complement_map.get(i, i)) for i in range(cfg.vocab_size)]
            for name, t in self._sd.items():
                src = t.detach()
                # HF checkpoints carry the RCPS modules' persistent integer buffers ([EXT] RCPSEmbedding / RCPSLMHead
                # register_buffer("complement_map")): not weights.  They must agree with config.complement_map, which
                # is what the engine was created with.
                if name.endswith("complement_map"):
                    got = [int(x) for x in src.flatten().tolist()]
                    if got[:cfg.vocab_size] != comp_want[:len(got)]:
                        raise ValueError(f"{name} = {got} disagrees with config.complement_map = {comp_want}")
                    continue
                if not src.is_floating_point():
                    continue
                # Weights are rounded to the model dtype exactly as from_pretrained(torch_dtype=...) would.
                # (that cast covers A_log and D too; Mamba then reads them back with .float()).
                if src.dtype != self.dtype and src.is_floating_point():
                    src = src.to(self.dtype)
                src = src.contiguous()
                shape = (C.c_int64 * src.dim())(*src.shape)
                _lib.check(self._lib.pcad_set_weight(h, name.encode(), C.c_void_p(src.data_ptr()), shape, src.dim(),
                                                     _TORCH_TO_PCAD[src.dtype]), h)
            _lib.check(self._lib.pcad_finalize(h), h)
            self.set_tokenizer(self._tokenizer)
        except Exception:
            self._release()
            raise

    def set_tokenizer(self, tok: CharDNATokenizer):
        """Hands the tokenizer's byte LUT / mask id / a,c,g,t ids to the engine (device tokenisation)."""
        self._tokenizer = tok
        if self._handle is None:
            return
        lut = (C.c_uint8 * 256)(*[int(x) for x in tok.lut])
        v = tok.get_vocab()
        acgt = (C.c_int32 * 4)(v["a"], v["c"], v["g"], v["t"])
        _lib.check(self._lib.pcad_set_tokenizer(self._handle, lut, tok.mask_token_id, acgt), self._handle)

    # ---- forward -----------------------------------------------------------------------------------
    def _require_handle(self):
        if self._handle is None:
            raise RuntimeError("model is not on a CUDA device; the B200 engine has no CPU path (call .to('cuda:0'))")

    def _stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def __call__(self, input_ids: Optional[torch.Tensor] = None, output_hidden_states: bool = False,
                 return_dict: bool = True, hidden_layers: Union[None, str, Iterable[int]] = None, **unused) -> MaskedLMOutput:
        return self.forward(input_ids=input_ids, output_hidden_states=output_hidden_states, hidden_layers=hidden_layers)

    def forward(self, input_ids: torch.Tensor, output_hidden_states: bool = False,
                compute_logits: bool = True, hidden_layers: Union[None, str, Iterable[int]] = None) -> MaskedLMOutput:
        """``hidden_layers`` ("all", or indices into the reference's hidden_states, negative ones from the end) implies
        ``output_hidden_states`` and returns the reference's full tuple of ``n_layer + 1`` entries, [B, L, 2*d_model] each,
        the requested ones filled and the others None.  With ``compute_logits=False`` the forward then stops after the layer
        that produces the deepest requested entry.  Without it, hidden_states holds the final normed state only."""
        self._require_handle()
        if input_ids is None or input_ids.dim() != 2:
            raise ValueError("input_ids must be a [batch, length] integer tensor")
        want, idx, _ = self._tap_indices(hidden_layers)
        ids = input_ids.to(device=self.device, dtype=torch.int64).contiguous()
        B, L = ids.shape
        with torch.cuda.device(self.device):
            logits = torch.empty((B, L, self.config.vocab_size), dtype=torch.float32, device=self.device) \
                if compute_logits else None
            taps = [torch.empty((B, L, 2 * self.config.d_model), dtype=self.dtype, device=self.device) for _ in want] \
                if output_hidden_states or hidden_layers is not None else []
            if B > 0 and L > 0:
                lg = C.c_void_p(logits.data_ptr()) if logits is not None else None
                if hidden_layers is None:   # the C drop-in for model(ids): the launches of pcad_forward_taps([n_layer])
                    _lib.check(self._lib.pcad_forward(self._handle, C.c_void_p(ids.data_ptr()), B, L, lg,
                                                      C.c_void_p(taps[0].data_ptr()) if taps else None, self._stream()),
                               self._handle)
                else:
                    ptrs = (C.c_void_p * len(want))(*[t.data_ptr() for t in taps])
                    _lib.check(self._lib.pcad_forward_taps(self._handle, C.c_void_p(ids.data_ptr()), B, L, lg, len(want), idx,
                                                           ptrs, self._stream()), self._handle)
                self._raise_on_bad_ids(True)
        if hidden_layers is None:
            # hidden_states: only the final (normed) state is materialised; hidden_states[-1] is what the
            # reference's callers read (train_XGBoost.py:105, notebooks/examples.ipynb:183).
            return MaskedLMOutput(logits=logits, hidden_states=tuple(taps) or None)
        hidden: List[Optional[torch.Tensor]] = [None] * (self.config.n_layer + 1)
        for k, t in zip(want, taps):
            hidden[k] = t
        return MaskedLMOutput(logits=logits, hidden_states=tuple(hidden))

    def _tap_indices(self, layers: Union[None, str, Iterable[int]]) -> Tuple[List[int], C.Array, Optional[List[int]]]:
        """``layers`` as ``forward``'s ``hidden_layers`` (None: the final normed state) in the form the engine takes them:
        (the indices in increasing order, the same as a ctypes int32 array, and the permutation that puts results stacked
        in that order back into the caller's order, or None where the two orders agree).  Raises ValueError as
        ``hidden_layer_indices``."""
        n_layer = self.config.n_layer
        layers = [n_layer] if layers is None else hidden_layer_indices(layers, n_layer)
        want = sorted(layers)
        back = None if want == layers else [want.index(k) for k in layers]
        return want, (C.c_int32 * len(want))(*want), back

    def _raise_on_bad_ids(self, sync: bool):
        """Token ids outside [0, vocab_size) raise IndexError, as the reference's nn.Embedding lookup would
        (the engine validates on the device; ``sync`` waits for the stream so the answer covers this call)."""
        rc = self._lib.pcad_take_id_error(self._handle, self._stream(), int(sync))
        if rc != 0:
            msg = self._lib.pcad_last_error(self._handle)
            raise IndexError(msg.decode() if msg else "token id out of range")

    def score_masked(self, ids_u8: torch.Tensor, positions: torch.Tensor, check_ids: bool = True) -> torch.Tensor:
        """ids_u8: uint8 [B, L] token ids (already masked) on the device; positions: int32 [B, n_mask], or a Python int when every
        window is scored at the same index (the reference's tokenIdx; lets the engine prune the last layer).
        Returns float32 [B, n_mask, 4] logits in a,c,g,t order (extract_logits / _masked_probs gather).
        ``check_ids=False`` keeps the call asynchronous: an out-of-range id is then reported by the next checking call."""
        self._require_handle()
        ids = ids_u8.to(device=self.device, dtype=torch.uint8).contiguous()
        B, L = ids.shape
        if isinstance(positions, int):
            # the reference's own case: one scored index shared by every window (extract_logits, tokenIdx) -> [B, 1, 4]
            with torch.cuda.device(self.device):
                out = torch.empty((B, 1, 4), dtype=torch.float32, device=self.device)
                if B > 0 and L > 0:
                    _lib.check(self._lib.pcad_score_masked_at(self._handle, C.c_void_p(ids.data_ptr()), int(positions), B, L,
                                                              C.c_void_p(out.data_ptr()), self._stream()), self._handle)
                    self._raise_on_bad_ids(check_ids)
            return out
        pos = positions.to(device=self.device, dtype=torch.int32).contiguous()
        if pos.dim() == 1:
            pos = pos[:, None]
        n_mask = pos.shape[1]
        with torch.cuda.device(self.device):
            out = torch.empty((B, n_mask, 4), dtype=torch.float32, device=self.device)
            if B > 0 and L > 0 and n_mask > 0:
                _lib.check(self._lib.pcad_score_masked(self._handle, C.c_void_p(ids.data_ptr()), C.c_void_p(pos.data_ptr()),
                                                       B, L, n_mask, C.c_void_p(out.data_ptr()), self._stream()), self._handle)
                self._raise_on_bad_ids(check_ids)
        return out

    def hidden_at(self, ids_u8: torch.Tensor, positions: torch.Tensor,
                  layers: Union[None, str, Iterable[int]] = None) -> torch.Tensor:
        """``hidden_states[-1][b, positions[b, i], :]`` for uint8 ids [B, L]: [B, n_pos, 2*d_model] in the model dtype,
        without materialising the full hidden state (reference extract_embeddings, train_XGBoost.py:104-105).  With
        ``layers`` ("all", or indices into hidden_states as ``forward``'s ``hidden_layers``): [len(layers), B, n_pos,
        2*d_model], entry i from hidden_states[layers[i]]; the forward stops after the deepest requested layer."""
        self._require_handle()
        want, idx, back = self._tap_indices(layers)
        ids = ids_u8.to(device=self.device, dtype=torch.uint8).contiguous()
        pos = positions.to(device=self.device, dtype=torch.int32).contiguous()
        B, L = ids.shape
        if pos.dim() == 1:
            pos = pos[:, None]
        n_pos = pos.shape[1]
        with torch.cuda.device(self.device):
            out = torch.empty((len(want), B, n_pos, 2 * self.config.d_model), dtype=self.dtype, device=self.device)
            if B > 0 and L > 0 and n_pos > 0:
                _lib.check(self._lib.pcad_hidden_at_layers(self._handle, C.c_void_p(ids.data_ptr()), C.c_void_p(pos.data_ptr()),
                                                           B, L, n_pos, len(want), idx, C.c_void_p(out.data_ptr()),
                                                           self._stream()), self._handle)
                self._raise_on_bad_ids(True)
            if back is not None:
                out = out[back]
        return out[0] if layers is None else out

    def hidden_mean(self, ids_u8: torch.Tensor, ranges=None, layers: Union[None, str, Iterable[int]] = None) -> torch.Tensor:
        """Mean over each window's positions of a ``hidden_states`` entry, float32, without [B, L, 2*d_model] buffers:
        ``out[b] = hidden_states[k][b, s_b:e_b].float().mean(0)`` in the engine's fixed summation order (pcad.h,
        pcad_hidden_mean_at_layers).  ``ranges``: [B, 2] integers (s_b, e_b), or None for every position; a window whose
        range is invalid (s < 0, e > L or s >= e) gets a NaN row.  ``layers=None``: [B, 2*d_model] from the final normed
        state; otherwise ("all", or indices as ``forward``'s ``hidden_layers``) [len(layers), B, 2*d_model] in the caller's
        order.  The forward stops after the deepest requested layer.  Raises ValueError for ranges that are not [B, 2]
        integers."""
        self._require_handle()
        want, idx, back = self._tap_indices(layers)
        ids = ids_u8.to(device=self.device, dtype=torch.uint8).contiguous()
        B, L = ids.shape
        rng = None if ranges is None else hidden_mean_ranges(ranges, B, L).to(self.device)
        with torch.cuda.device(self.device):
            out = torch.empty((len(want), B, 2 * self.config.d_model), dtype=torch.float32, device=self.device)
            if B > 0 and L > 0:
                _lib.check(self._lib.pcad_hidden_mean_at_layers(
                    self._handle, C.c_void_p(ids.data_ptr()), C.c_void_p(rng.data_ptr()) if rng is not None else None, B, L,
                    len(want), idx, C.c_void_p(out.data_ptr()), self._stream()), self._handle)
                self._raise_on_bad_ids(True)
            else:
                out.fill_(float("nan"))   # L = 0: no range is valid
            if back is not None:
                out = out[back]
        return out[0] if layers is None else out

    def score_windows_host(self, ascii_windows: Union[np.ndarray, torch.Tensor], token_idx: int,
                           out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """End-to-end host call: uint8 ASCII [B, L] in (ideally pinned) host memory -> float32 [B, 4] host logits
        (a,c,g,t) at the masked position.  H2D copy, device tokenise + mask, forward, D2H copy, sync."""
        self._require_handle()
        a = torch.from_numpy(ascii_windows) if isinstance(ascii_windows, np.ndarray) else ascii_windows
        if a.dtype != torch.uint8 or a.dim() != 2 or a.device.type != "cpu" or not a.is_contiguous():
            raise ValueError("ascii_windows must be a contiguous uint8 [B, L] host array")
        B, L = a.shape
        if out is None:
            out = torch.empty((B, 4), dtype=torch.float32).pin_memory() if B > 0 else torch.empty((0, 4))
        if B > 0:
            with torch.cuda.device(self.device):
                _lib.check(self._lib.pcad_score_windows_host(self._handle, C.c_void_p(a.data_ptr()), B, L, int(token_idx),
                                                             C.c_void_p(out.data_ptr()), self._stream()), self._handle)
        return out

    def extract_windows_device(self, chrom_dev: torch.Tensor, pos0: torch.Tensor, token_idx: int = 255,
                               length: int = 512) -> torch.Tensor:
        """Windows for variants at 0-based positions ``pos0`` of a chromosome resident on the device: uint8 [B, length],
        byte-identical to ``genome_io.extract_window`` (the reference's seq_from_vcf slice-and-pad rule)."""
        self._require_handle()
        chrom = chrom_dev.to(device=self.device, dtype=torch.uint8).contiguous()
        pos = pos0.to(device=self.device, dtype=torch.int64).contiguous()
        B = pos.numel()
        with torch.cuda.device(self.device):
            out = torch.empty((B, length), dtype=torch.uint8, device=self.device)
            if B > 0:
                _lib.check(self._lib.pcad_extract_windows(self._handle, C.c_void_p(chrom.data_ptr()), chrom.numel(),
                                                          C.c_void_p(pos.data_ptr()), B, length, int(token_idx),
                                                          C.c_void_p(out.data_ptr()), self._stream()), self._handle)
        return out

    def score_windows_device(self, ascii_dev: torch.Tensor, token_idx: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``score_windows_host`` for windows already on the device: uint8 [B, L] -> float32 [B, 4] (device, async;
        written into ``out`` when given: a contiguous float32 [B, 4] device tensor)."""
        self._require_handle()
        a = ascii_dev.to(device=self.device, dtype=torch.uint8).contiguous()
        B, L = a.shape
        with torch.cuda.device(self.device):
            if out is None:
                out = torch.empty((B, 4), dtype=torch.float32, device=self.device)
            elif out.shape != (B, 4) or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.device:
                raise ValueError("out must be a contiguous float32 [B, 4] tensor on the model's device")
            if B > 0:
                _lib.check(self._lib.pcad_score_windows_dev(self._handle, C.c_void_p(a.data_ptr()), B, L, int(token_idx),
                                                            C.c_void_p(out.data_ptr()), self._stream()), self._handle)
        return out

    def tokenize_device(self, ascii_dev: torch.Tensor) -> torch.Tensor:
        self._require_handle()
        a = ascii_dev.to(device=self.device, dtype=torch.uint8).contiguous()
        out = torch.empty_like(a)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.pcad_tokenize(self._handle, C.c_void_p(a.data_ptr()), a.numel(),
                                               C.c_void_p(out.data_ptr()), self._stream()), self._handle)
        return out

    # ---- introspection -----------------------------------------------------------------------------
    def workspace_bytes(self, B: int, L: int) -> int:
        self._require_handle()
        n = C.c_size_t()
        _lib.check(self._lib.pcad_workspace_bytes(self._handle, B, L, C.byref(n)), self._handle)
        return int(n.value)

    def set_profiling(self, enabled: bool):
        self._require_handle()
        _lib.check(self._lib.pcad_set_profiling(self._handle, int(enabled)), self._handle)

    def get_profile(self) -> Dict[str, Dict[str, float]]:
        self._require_handle()
        ms = (C.c_float * len(_lib.STAGES))()
        n = (C.c_int64 * len(_lib.STAGES))()
        _lib.check(self._lib.pcad_get_profile(self._handle, ms, n), self._handle)
        return {s: {"ms": float(ms[i]), "launches": int(n[i])} for i, s in enumerate(_lib.STAGES)}

    def launch_count(self) -> int:
        self._require_handle()
        return int(self._lib.pcad_launch_count(self._handle))


def AutoModelForMaskedLM_from_pretrained(name_or_path, **kw) -> CaduceusForMaskedLM:
    """Spelling used in INTEGRATION.md for swapping the reference's loader line."""
    return CaduceusForMaskedLM.from_pretrained(name_or_path, **kw)

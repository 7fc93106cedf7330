"""Engine: the batched GPU operations behind the drop-in sketch objects.

PyTorch is used only to own device memory and streams; every operation is one or a few calls
into the C ABI (include/dandd_b200.h) on torch's current stream, so `torch.cuda.Event` timing
and stream semantics work as usual.  One Engine per process / per GPU."""
import ctypes as C
import os
from dataclasses import dataclass
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import DD_COVER_PART_BYTES, DD_HIST_BINS, DD_PACK_FLAG_FASTQ, DD_PACK_FLAG_OVERFLOW, DandDError, check


class FastqInput(DandDError):
    """The packed text holds a line beginning with '+': FASTQ.  The caller rewrites the text with
    Engine.fastq_to_fasta (kseq's walk of the records, on the host) and packs that instead."""


def kmask_of(ks: Iterable[int]) -> int:
    m = 0
    for k in ks:
        k = int(k)
        if not 1 <= k <= 32:
            raise ValueError(f"k={k} outside 1..32 (HLL estimation supports k<=32; reference README.md:82)")
        m |= 1 << (k - 1)
    if m == 0:
        raise ValueError("no k values given")
    return m


def ks_of(kmask: int) -> List[int]:
    return [k for k in range(1, 33) if (kmask >> (k - 1)) & 1]


@dataclass
class PackedSeq:
    """A FASTA packed into the 2-bit symbol stream (layout: include/dandd_b200.h, K1)."""
    codes: torch.Tensor       # uint8 storage holding the u32 code words
    invalid: torch.Tensor     # uint8 storage holding the u32 break-bit words
    state: torch.Tensor       # 32 bytes: dd_pack_state
    cap_symbols: int
    text_bytes: int
    _nsym: Optional[int] = None

    @property
    def nsym(self) -> int:
        """Number of symbols (reads the device state: synchronises)."""
        if self._nsym is None:
            st = self.state.cpu().numpy().view(np.uint64)
            if int(st[3]) & DD_PACK_FLAG_OVERFLOW:
                raise DandDError("packed stream overflowed its capacity")
            if int(st[3]) & DD_PACK_FLAG_FASTQ:
                raise FastqInput("FASTQ text (a line begins with '+') must go through Engine.fastq_to_fasta first")
            self._nsym = int(st[0])
        return self._nsym

    def check(self) -> "PackedSeq":
        """Raise if the packer flagged the text (overflow, FASTQ).  Synchronises."""
        self.nsym  # noqa: B018
        return self


class Engine:
    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise DandDError("no CUDA device visible to torch; dandd_b200 has no CPU fallback")
        check(self.lib.dd_init(int(device)), "dd_init")
        self.device = torch.device("cuda", int(device))
        torch.cuda.set_device(self.device)
        sm, maj, mnr, l2, mem = C.c_int(), C.c_int(), C.c_int(), C.c_size_t(), C.c_size_t()
        check(self.lib.dd_device_info(int(device), C.byref(sm), C.byref(maj), C.byref(mnr), C.byref(l2), C.byref(mem)))
        self.sm_count, self.cc, self.l2_bytes, self.total_mem = sm.value, (maj.value, mnr.value), l2.value, mem.value
        self._ws = {}
        # SURVEY.md A.6 (UNVERIFIED encoder quirk): opt-in emulation, for every entry point of this engine
        self.polyt_sentinel = os.environ.get("DANDD_B200_POLYT_SENTINEL", "0") not in ("", "0")
        check(self.lib.dd_set_option(b"polyt_sentinel", int(self.polyt_sentinel)), "dd_set_option")

    # ---- plumbing ---------------------------------------------------------------------------
    def bind_thread(self) -> None:
        """Make this engine's GPU the calling thread's current device.  The CUDA runtime's current
        device is per host thread: an engine created on one thread (the command line starts it in the
        background) must be bound again on every other thread that launches through it."""
        torch.cuda.set_device(self.device)

    @property
    def stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _buf(self, nbytes: int, tag: str) -> torch.Tensor:
        """Grow-only scratch tensors keyed by role (uint8)."""
        t = self._ws.get(tag)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.device)
            self._ws[tag] = t
        return t

    def _dev_u8(self, data) -> torch.Tensor:
        if isinstance(data, torch.Tensor):
            return data.to(self.device, dtype=torch.uint8).contiguous().view(-1)
        if isinstance(data, (bytes, bytearray, memoryview)):
            data = np.frombuffer(data, dtype=np.uint8)
        arr = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        if arr.size == 0:
            return torch.empty(0, dtype=torch.uint8, device=self.device)
        return torch.from_numpy(arr.copy() if not arr.flags.writeable else arr).to(self.device, non_blocking=False)

    # ---- K1 ---------------------------------------------------------------------------------
    @staticmethod
    def skip_preamble(text) -> int:
        """Offset of the first '>' or '@' (kseq ignores everything before the first record marker,
        SURVEY.md A.1); len if there is none."""
        if isinstance(text, torch.Tensor) and text.is_cuda:
            n = int(text.numel())
            block = 1 << 26
            for off in range(0, n, block):            # the marker is almost always in the first block
                part = text[off:off + block]
                hit = ((part == 62) | (part == 64)).nonzero()
                if hit.numel():
                    return off + int(hit[0])
            return n
        if isinstance(text, torch.Tensor):
            ptr, n = text.data_ptr(), int(text.numel())
        else:
            arr = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) else \
                np.ascontiguousarray(text, dtype=np.uint8).reshape(-1)
            ptr, n = arr.ctypes.data, int(arr.size)
        return int(_lib.load().dd_fasta_first_record_host(ptr, n)) if n else 0

    @staticmethod
    def fastq_to_fasta(text) -> bytes:
        """kseq_read()'s walk over FASTA/FASTQ text, written back as plain FASTA (host side, no GPU):
        what the packer must be given when it reports DD_PACK_FLAG_FASTQ."""
        arr = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) else \
            np.ascontiguousarray(text, dtype=np.uint8).reshape(-1)
        out = np.empty(arr.size + 16, dtype=np.uint8)
        n = _lib.load().dd_fastq_to_fasta_host(arr.ctypes.data, arr.size, out.ctypes.data) if arr.size else 0
        return out[:n].tobytes()

    def pack(self, text, chunk_bytes: Optional[int] = None, start: Optional[int] = None, ws_tag: str = "pack") -> PackedSeq:
        """FASTA text (bytes / numpy / torch uint8) -> PackedSeq.  `chunk_bytes` packs in several
        chunks through the carried state (used by the tests to exercise streaming).  `start` = offset
        of the first '>' if the caller knows it (device-resident text is otherwise scanned for it)."""
        if start is None and not isinstance(text, torch.Tensor):
            start = self.skip_preamble(text)          # on the host, before the upload
        d_text = self._dev_u8(text)
        if start is None:
            start = self.skip_preamble(d_text) if d_text.numel() else 0
        off = min(int(start), int(d_text.numel()))
        n = int(d_text.numel()) - off
        if off % 16 and n > 0:
            d_text = d_text[off:].clone()   # keep the 128-bit loads aligned
        elif off:
            d_text = d_text[off:]
        cb, ib = self.lib.dd_pack_codes_bytes(max(n, 1)), self.lib.dd_pack_invalid_bytes(max(n, 1))
        codes = torch.empty(cb, dtype=torch.uint8, device=self.device)
        invalid = torch.empty(ib, dtype=torch.uint8, device=self.device)
        state = torch.empty(32, dtype=torch.uint8, device=self.device)
        st = self.stream
        check(self.lib.dd_pack_reset(codes.data_ptr(), cb, invalid.data_ptr(), ib, state.data_ptr(), st), "dd_pack_reset")
        chunk = int(chunk_bytes) if chunk_bytes else max(n, 1)
        wsb = self.lib.dd_pack_workspace_bytes(min(chunk, max(n, 1)))
        ws = self._buf(wsb, ws_tag)   # one scratch buffer per stream in flight
        pos = 0
        while pos < n:
            ln = min(chunk, n - pos)
            part = d_text[pos:pos + ln]
            if part.data_ptr() % 16:
                part = part.clone()
            check(self.lib.dd_pack_fasta(part.data_ptr(), ln, codes.data_ptr(), invalid.data_ptr(), max(n, 1),
                                         state.data_ptr(), ws.data_ptr(), ws.numel(), st), "dd_pack_fasta")
            if self.polyt_sentinel:
                check(self.lib.dd_pack_polyt_sentinel(codes.data_ptr(), invalid.data_ptr(), state.data_ptr(), 0, 0, ln, st),
                      "dd_pack_polyt_sentinel")
            pos += ln
        return PackedSeq(codes, invalid, state, max(n, 1), n)

    # ---- K2 (+K4 for the leaf cardinalities) ------------------------------------------------------
    def sketch(self, seq: PackedSeq, ks: Sequence[int], p: int = 20, canon: bool = True,
               out: Optional[torch.Tensor] = None, ranges=None, floor_every: Optional[int] = None,
               hist_out: Optional[torch.Tensor] = None, ws_tag: str = "sketch"):
        """All-k HLL sketch of one packed sequence.  Returns (regs [nk, 2^p] uint8, cards [nk] f64),
        both on the device.  `ranges` (list of (begin, end) symbol ranges) forces chunked updates.
        With `hist_out` ([nk, 64] int32) the register histograms go there and the estimator is left to
        a later batched mle() call (cards is then None): one MLE launch per batch, not per genome."""
        kmask = kmask_of(ks)
        nk = bin(kmask).count("1")
        m = 1 << p
        wsb = self.lib.dd_sketch_workspace_bytes(nk, p)
        ws = self._buf(wsb, ws_tag)
        st = self.stream
        regs = out if out is not None else torch.empty((nk, m), dtype=torch.uint8, device=self.device)
        assert regs.is_contiguous() and regs.numel() == nk * m
        defer = hist_out is not None
        hist = hist_out if defer else torch.empty((nk, DD_HIST_BINS), dtype=torch.int32, device=self.device)
        assert hist.is_contiguous() and hist.numel() == nk * DD_HIST_BINS
        cards = None if defer else torch.empty(nk, dtype=torch.float64, device=self.device)
        check(self.lib.dd_sketch_begin(ws.data_ptr(), ws.numel(), nk, p, st), "dd_sketch_begin")
        if ranges is None and floor_every:
            n = seq.nsym                      # needs the symbol count on the host: one sync
            ranges = [(b, min(n, b + floor_every)) for b in range(0, n, floor_every)]
        if ranges is None:
            # whole stream in one launch; the symbol count stays on the device (no host sync)
            self._update_from_state(seq, kmask, p, canon, ws, st)
        else:
            seen = 0
            for (b, e) in ranges:
                check(self.lib.dd_sketch_update_range(seq.codes.data_ptr(), seq.invalid.data_ptr(), int(b), int(e), kmask,
                                                      p, int(canon), ws.data_ptr(), ws.numel(), st), "dd_sketch_update_range")
                seen += e - b
                if floor_every and seen >= (16 << p):
                    check(self.lib.dd_sketch_refresh_floor(ws.data_ptr(), ws.numel(), kmask, p, st), "dd_sketch_refresh_floor")
        check(self.lib.dd_sketch_end(ws.data_ptr(), ws.numel(), nk, p, regs.data_ptr(), hist.data_ptr(),
                                     None if defer else cards.data_ptr(), st), "dd_sketch_end")
        return regs, cards

    def mle(self, hist: torch.Tensor, p: int) -> torch.Tensor:
        """Ertl-MLE cardinalities from register histograms [..., 64] (int32, device)."""
        flat = hist.contiguous().view(-1, DD_HIST_BINS)
        out = torch.empty(flat.shape[0], dtype=torch.float64, device=self.device)
        check(self.lib.dd_mle_from_hist(flat.data_ptr(), flat.shape[0], p, out.data_ptr(), self.stream), "dd_mle_from_hist")
        return out.view(hist.shape[:-1])

    def _update_from_state(self, seq, kmask, p, canon, ws, st):
        # the pack state says [prev_nsym, nsym); for a whole-stream sketch rewind prev_nsym to 0
        state = seq.state.clone()
        state.view(torch.int64)[1] = 0
        # (dd_sketch_update_sched == dd_sketch_update for streams shorter than 16 x 2^p symbols; longer ones
        # are cut at the floor schedule's boundaries with a refresh at each)
        check(self.lib.dd_sketch_update_sched(seq.codes.data_ptr(), seq.invalid.data_ptr(), state.data_ptr(), 0, 0,
                                              seq.text_bytes, 0, kmask, p, int(canon), ws.data_ptr(), ws.numel(), st),
              "dd_sketch_update_sched")
        self._keep = state  # keep alive until the stream has consumed it

    def sketch_fasta_host(self, text: bytes, ks: Sequence[int], p: int = 20, canon: bool = True,
                          want_regs: bool = True, pinned_regs: Optional[torch.Tensor] = None,
                          out_dev: Optional[torch.Tensor] = None, cards_out: Optional[torch.Tensor] = None,
                          ws_tag: str = "host", sync: bool = True):
        """The host-buffer C-ABI path: FASTA bytes in host memory -> (regs numpy [nk, 2^p] or None,
        cards numpy [nk]).  H2D, pack, sketch, estimate, D2H all inside the one call.  `out_dev`
        (uint8 [nk, 2^p] on the device) additionally keeps the registers resident in HBM.
        sync=False enqueues on the current stream and returns (dd_sketch_fasta_host_async): give every
        stream in flight its own `ws_tag` and a pinned `cards_out` (float64 [nk]), and synchronise
        the stream before reading the results."""
        kmask = kmask_of(ks)
        nk = bin(kmask).count("1")
        m = 1 << p
        if isinstance(text, torch.Tensor):
            h_ptr, n = text.data_ptr(), text.numel()
        else:
            arr = np.frombuffer(text, dtype=np.uint8)
            h_ptr, n = arr.ctypes.data, arr.size
        wsb = self.lib.dd_sketch_fasta_host_workspace_bytes(n, nk, p)
        ws = self._buf(wsb, ws_tag)
        if cards_out is not None:
            assert cards_out.dtype == torch.float64 and cards_out.numel() == nk and cards_out.is_contiguous()
            cards, c_ptr = cards_out, cards_out.data_ptr()
        else:
            cards = np.empty(nk, dtype=np.float64)
            c_ptr = cards.ctypes.data
        regs = None
        r_ptr = None
        if want_regs:
            if pinned_regs is not None:
                regs, r_ptr = pinned_regs, pinned_regs.data_ptr()
            else:
                regs = np.empty((nk, m), dtype=np.uint8)
                r_ptr = regs.ctypes.data
        d_ptr = None
        if out_dev is not None:
            assert out_dev.is_contiguous() and out_dev.numel() == nk * m and out_dev.dtype == torch.uint8
            d_ptr = out_dev.data_ptr()
        fn = self.lib.dd_sketch_fasta_host if sync else self.lib.dd_sketch_fasta_host_async
        check(fn(h_ptr, n, kmask, p, int(canon), r_ptr, c_ptr, d_ptr, ws.data_ptr(), ws.numel(), self.stream),
              "dd_sketch_fasta_host")
        return regs, cards

    # ---- K4 ---------------------------------------------------------------------------------
    def cards(self, regs: torch.Tensor, p: int) -> torch.Tensor:
        """Ertl-MLE cardinality of each sketch in regs [..., 2^p] (uint8, device)."""
        m = 1 << p
        flat = regs.contiguous().view(-1, m)
        nsk = flat.shape[0]
        hist = torch.empty((nsk, DD_HIST_BINS), dtype=torch.int32, device=self.device)
        out = torch.empty(nsk, dtype=torch.float64, device=self.device)
        check(self.lib.dd_card_ertl_mle(flat.data_ptr(), nsk, p, out.data_ptr(), hist.data_ptr(), self.stream), "dd_card_ertl_mle")
        return out.view(regs.shape[:-1])

    # ---- K3 ---------------------------------------------------------------------------------
    def union(self, sketches: Sequence[torch.Tensor]) -> torch.Tensor:
        """Register-wise max of equally sized uint8 device tensors (`dashing union`)."""
        n = sketches[0].numel()
        keep = [s.contiguous() for s in sketches]
        ptrs = torch.tensor([s.data_ptr() for s in keep], dtype=torch.int64).to(self.device)
        out = torch.empty_like(keep[0])
        check(self.lib.dd_union_max(ptrs.data_ptr(), len(keep), n, out.data_ptr(), self.stream), "dd_union_max")
        self._keep = (keep, ptrs)
        return out

    def prefix_union_cards(self, regs: torch.Tensor, orders, p: int, final_only: bool = False,
                           materialize: bool = False):
        """regs [n_genomes, nk, 2^p]; orders [n_ord, n_steps] genome indices (-1 = skip).
        Returns cards [n_ord, n_steps or 1, nk] f64 (and the unions if materialize)."""
        n_g, nk, m = regs.shape
        assert m == 1 << p and regs.is_contiguous()
        order = torch.as_tensor(np.asarray(orders, dtype=np.int32)).to(self.device).contiguous()
        n_ord, n_steps = order.shape
        osteps = 1 if final_only else n_steps
        hist = torch.empty((n_ord, osteps, nk, DD_HIST_BINS), dtype=torch.int32, device=self.device)
        cards = torch.empty((n_ord, osteps, nk), dtype=torch.float64, device=self.device)
        unions = torch.empty((n_ord, osteps, nk, m), dtype=torch.uint8, device=self.device) if materialize else None
        ws = None
        if not materialize and p >= 12:   # scratch for the bit-plane kernel (transposed sketches + identical-prefix table)
            ws = self._buf(self.lib.dd_prefix_union_workspace_bytes(n_ord, n_steps, n_g, nk, p), "prefix")
        check(self.lib.dd_prefix_union_card(regs.data_ptr(), order.data_ptr(), n_ord, n_steps, n_g, nk, p, int(final_only),
                                            cards.data_ptr(), hist.data_ptr(), unions.data_ptr() if materialize else None,
                                            ws.data_ptr() if ws is not None else None, ws.numel() if ws is not None else 0,
                                            self.stream), "dd_prefix_union_card")
        self._keep = order
        return (cards, unions) if materialize else cards

    # ---- bit planes (K3/K6 on sketches that are unioned many times) -------------------------------
    def to_planes(self, regs: torch.Tensor, p: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """regs [..., 2^p] uint8 -> bit planes [n_sketches, 6, 2^p/32] int32 (dd_to_planes), once;
        prefix_union_cards_planes / pairwise_cards(planes=...) then never transpose again."""
        m = 1 << p
        flat = regs.contiguous().view(-1, m)
        nsk = flat.shape[0]
        if out is None:
            out = torch.empty((nsk, 6, m // 32), dtype=torch.int32, device=self.device)
        assert out.is_contiguous() and out.numel() * 4 == self.lib.dd_planes_bytes(nsk, p)
        check(self.lib.dd_to_planes(flat.data_ptr(), nsk, p, out.data_ptr(), self.stream), "dd_to_planes")
        return out

    def prefix_union_cards_planes(self, planes: torch.Tensor, n_genomes: int, nk: int, orders, p: int,
                                  final_only: bool = False) -> torch.Tensor:
        """prefix_union_cards on sketches already transposed by to_planes ([n_genomes * nk, 6, 2^p/32])."""
        order = torch.as_tensor(np.asarray(orders, dtype=np.int32)).to(self.device).contiguous()
        n_ord, n_steps = order.shape
        osteps = 1 if final_only else n_steps
        hist = torch.empty((n_ord, osteps, nk, DD_HIST_BINS), dtype=torch.int32, device=self.device)
        cards = torch.empty((n_ord, osteps, nk), dtype=torch.float64, device=self.device)
        ws = self._buf(self.lib.dd_prefix_union_workspace_bytes(n_ord, n_steps, 0, 0, p), "prefix_dedup")
        check(self.lib.dd_prefix_union_card_planes(planes.data_ptr(), order.data_ptr(), n_ord, n_steps, n_genomes, nk, p,
                                                   int(final_only), cards.data_ptr(), hist.data_ptr(), ws.data_ptr(),
                                                   ws.numel(), self.stream), "dd_prefix_union_card_planes")
        self._keep = order
        return cards

    def union_sets(self, member_ptrs, p: int, final_only: bool = True, materialize: bool = False):
        """member_ptrs: int64 [n_sets, n_steps] device addresses of 2^p-byte sketches (0 = skip).
        Returns cards [n_sets, n_steps or 1] f64 (and unions [n_sets, n_steps or 1, 2^p] if asked).
        The caller keeps the member tensors alive until the stream has run."""
        ptrs = torch.as_tensor(np.ascontiguousarray(member_ptrs, dtype=np.int64)).to(self.device)
        n_sets, n_steps = ptrs.shape
        osteps = 1 if final_only else n_steps
        m = 1 << p
        hist = torch.empty((n_sets, osteps, DD_HIST_BINS), dtype=torch.int32, device=self.device)
        cards = torch.empty((n_sets, osteps), dtype=torch.float64, device=self.device)
        unions = torch.empty((n_sets, osteps, m), dtype=torch.uint8, device=self.device) if materialize else None
        check(self.lib.dd_union_sets_card(ptrs.data_ptr(), n_sets, n_steps, p, int(final_only), cards.data_ptr(),
                                          hist.data_ptr(), unions.data_ptr() if materialize else None, self.stream),
              "dd_union_sets_card")
        self._keep = ptrs
        return (cards, unions) if materialize else cards

    def pairwise_cards(self, regs: Optional[torch.Tensor], pairs, p: int, planes: Optional[torch.Tensor] = None,
                       n_genomes: Optional[int] = None, nk: Optional[int] = None,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """card(A u B) for every listed pair and every k: [n_pairs, nk] f64.  Either `regs`
        [n_genomes, nk, 2^p] (transposed into scratch on every call) or `planes` from to_planes()
        with n_genomes / nk given (tiles of a big pair matrix share one transpose)."""
        if isinstance(pairs, torch.Tensor):
            pr = pairs.to(self.device, dtype=torch.int32).contiguous().view(-1, 2)
        else:
            pr = torch.as_tensor(np.asarray(pairs, dtype=np.int32).reshape(-1, 2)).to(self.device).contiguous()
        n_pairs = pr.shape[0]
        if planes is None:
            n_genomes, nk, m = regs.shape
        hist = self._buf(n_pairs * nk * DD_HIST_BINS * 4, "pair_hist")
        cards = out if out is not None else torch.empty((n_pairs, nk), dtype=torch.float64, device=self.device)
        assert cards.is_contiguous() and cards.numel() == n_pairs * nk and cards.dtype == torch.float64
        if planes is not None:
            check(self.lib.dd_pairwise_union_card_planes(planes.data_ptr(), n_genomes, nk, p, pr.data_ptr(), n_pairs,
                                                         cards.data_ptr(), hist.data_ptr(), self.stream),
                  "dd_pairwise_union_card_planes")
        else:
            ws = self._buf(self.lib.dd_prefix_union_workspace_bytes(0, 0, n_genomes, nk, p), "prefix") if p >= 12 else None
            check(self.lib.dd_pairwise_union_card(regs.data_ptr(), n_genomes, nk, p, pr.data_ptr(), n_pairs, cards.data_ptr(),
                                                  hist.data_ptr(), ws.data_ptr() if ws is not None else None,
                                                  ws.numel() if ws is not None else 0, self.stream), "dd_pairwise_union_card")
        self._keep = pr
        return cards

    # ---- K10 --------------------------------------------------------------------------------
    def leave_out_hist(self, regs: torch.Tensor, group, n_groups: int, p: int, reg_range: Optional[tuple] = None,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Register histograms int32 [nk, 1 + n_groups, 64] on the device: row 0 of the union of all genomes of regs
        [n, nk, 2^p], row 1 + g of the union of every genome whose group[g'] != g (group: n ids in [0, n_groups)).
        One read of the registers (K10).  reg_range=(begin, end): only those registers of every k (multiples of 16);
        histograms of disjoint ranges add up.  out: an int32 [nk, 1 + n_groups, 64] tensor to ADD into."""
        n, nk, m = regs.shape
        assert m == 1 << p and regs.is_contiguous() and regs.dtype == torch.uint8
        begin, end = reg_range if reg_range is not None else (0, m)
        group = np.asarray(group, dtype=np.int32).reshape(-1)
        if group.size != n:
            raise DandDError("leave_out_hist: %d group ids for %d genomes" % (group.size, n))
        d_group = torch.from_numpy(group).to(self.device)
        if out is None:
            out = torch.zeros((nk, 1 + int(n_groups), DD_HIST_BINS), dtype=torch.int32, device=self.device)
        assert out.is_contiguous() and out.dtype == torch.int32 and out.numel() == nk * (1 + int(n_groups)) * DD_HIST_BINS
        ws = self._buf(self.lib.dd_leave_out_workspace_bytes(n, nk), "leave_out")
        check(self.lib.dd_leave_out_hist(regs.data_ptr(), n, nk, p, d_group.data_ptr(), int(n_groups), int(begin), int(end),
                                         out.data_ptr(), ws.data_ptr(), ws.numel(), self.stream), "dd_leave_out_hist")
        return out

    # ---- K11 --------------------------------------------------------------------------------
    def cards_hist(self, regs: torch.Tensor, p: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(cards float64 [...], histograms int32 [..., 64]) of the sketches regs [..., 2^p] on the device (K4)."""
        flat = regs.contiguous().view(-1, 1 << p)
        hist = torch.empty((flat.shape[0], DD_HIST_BINS), dtype=torch.int32, device=self.device)
        out = torch.empty(flat.shape[0], dtype=torch.float64, device=self.device)
        check(self.lib.dd_card_ertl_mle(flat.data_ptr(), flat.shape[0], p, out.data_ptr(), hist.data_ptr(), self.stream),
              "dd_card_ertl_mle")
        return out.view(regs.shape[:-1]), hist.view(tuple(regs.shape[:-1]) + (DD_HIST_BINS,))

    def greedy_dense_hist(self, regs: torch.Tensor, union: torch.Tensor, union_hist: torch.Tensor, cand, p: int):
        """(hist int32 [C, nk, 64], live int32 [C, nk]) on the device: the histogram of max(union, regs[g]) and the
        number of registers where regs[g] > union, for the C distinct genome indices `cand` (host), every k.  regs
        [n, nk, 2^p], union [nk, 2^p], union_hist [nk, 64] (cards_hist of union).  Reads every register (K11 dense)."""
        n, nk, m = regs.shape
        assert m == 1 << p and regs.is_contiguous() and union.is_contiguous() and union_hist.is_contiguous()
        cand = np.ascontiguousarray(cand, dtype=np.int32)
        hist = torch.empty((cand.size, nk, DD_HIST_BINS), dtype=torch.int32, device=self.device)
        live = torch.empty((cand.size, nk), dtype=torch.int32, device=self.device)
        ws = self._buf(self.lib.dd_greedy_workspace_bytes(cand.size), "greedy")
        check(self.lib.dd_greedy_dense_hist(regs.data_ptr(), n, nk, p, union.data_ptr(), union_hist.data_ptr(),
                                            cand.ctypes.data, cand.size, hist.data_ptr(), live.data_ptr(), ws.data_ptr(),
                                            ws.numel(), self.stream), "dd_greedy_dense_hist")
        return hist, live

    def greedy_compact(self, regs: torch.Tensor, union: torch.Tensor, cand, seg_off, p: int) -> dict:
        """The live registers (regs[g] > union) of the candidates `cand` as u32 entries `j << 6 | value` in segments
        g * nk + k whose capacities are the host offsets seg_off [n * nk + 1] (K11 compaction).  Returns the sparse
        state {"entries", "seg_off", "seg_len"} that greedy_sparse_hist reads and updates."""
        n, nk, m = regs.shape
        assert m == 1 << p and regs.is_contiguous() and union.is_contiguous()
        cand = np.ascontiguousarray(cand, dtype=np.int32)
        seg_off = np.ascontiguousarray(seg_off, dtype=np.int64)
        assert seg_off.size == n * nk + 1
        total = int(seg_off[-1])
        state = {"entries": torch.empty(max(total, 1), dtype=torch.int32, device=self.device), "n_entries": total,
                 "seg_off": torch.empty(n * nk + 1, dtype=torch.int64, device=self.device),
                 "seg_len": torch.empty(n * nk, dtype=torch.int32, device=self.device), "n": n}
        ws = self._buf(self.lib.dd_greedy_workspace_bytes(cand.size), "greedy")
        check(self.lib.dd_greedy_compact(regs.data_ptr(), n, nk, p, union.data_ptr(), cand.ctypes.data, cand.size,
                                         seg_off.ctypes.data, state["seg_off"].data_ptr(), state["seg_len"].data_ptr(),
                                         state["entries"].data_ptr(), total, ws.data_ptr(), ws.numel(), self.stream),
              "dd_greedy_compact")
        return state

    def greedy_sparse_hist(self, state: dict, union: torch.Tensor, union_hist: torch.Tensor, cand, p: int):
        """greedy_dense_hist from the sparse state of greedy_compact (K11 sparse): the entries no longer above union
        are dropped for good, so every call must follow the previous one's union update."""
        nk = union.shape[0]
        assert union.shape[1] == 1 << p and union.is_contiguous() and union_hist.is_contiguous()
        cand = np.ascontiguousarray(cand, dtype=np.int32)
        hist = torch.empty((cand.size, nk, DD_HIST_BINS), dtype=torch.int32, device=self.device)
        live = torch.empty((cand.size, nk), dtype=torch.int32, device=self.device)
        ws = self._buf(self.lib.dd_greedy_workspace_bytes(cand.size), "greedy")
        check(self.lib.dd_greedy_sparse_hist(state["entries"].data_ptr(), state["n_entries"], state["seg_off"].data_ptr(),
                                             state["seg_len"].data_ptr(), state["n"], nk, p, union.data_ptr(),
                                             union_hist.data_ptr(), cand.ctypes.data, cand.size, hist.data_ptr(),
                                             live.data_ptr(), ws.data_ptr(), ws.numel(), self.stream),
              "dd_greedy_sparse_hist")
        return hist, live

    # ---- K5 ---------------------------------------------------------------------------------
    def exact_counts(self, seqs: Sequence[PackedSeq], k: int, canon: bool = True, capacity: Optional[int] = None,
                     shard: Optional[tuple] = None) -> List[int]:
        """Insert the sequences one after another into one k-mer set and return the number of
        distinct (canonical) k-mers after each: [|S1|, |S1 u S2|, ...] (exact, KMC semantics).
        shard=(rank, world): only the k-mers of this rank's key range are stored and counted; the
        ranks' results add up to the unsharded counts (dandd_b200.dist.sum_counts)."""
        nsyms = [s.nsym for s in seqs]
        srank, sworld = (int(shard[0]), int(shard[1])) if shard is not None else (0, 1)
        if capacity is None:
            capacity = 1024
            while capacity < 2 * max(1, sum(nsyms)) // sworld + 1024:
                capacity *= 2
        wsb = self.lib.dd_exact_workspace_bytes(k, capacity)
        ws = self._buf(wsb, "exact")
        st = self.stream
        counts = torch.zeros(len(seqs), dtype=torch.int64, device=self.device)
        check(self.lib.dd_exact_begin(ws.data_ptr(), ws.numel(), k, capacity, st), "dd_exact_begin")
        for i, (s, n) in enumerate(zip(seqs, nsyms)):
            check(self.lib.dd_exact_insert_shard(s.codes.data_ptr(), s.invalid.data_ptr(), 0, n, k, int(canon), ws.data_ptr(),
                                                 ws.numel(), capacity, srank, sworld, st), "dd_exact_insert_shard")
            check(self.lib.dd_exact_count(ws.data_ptr(), ws.numel(), k, capacity, counts[i:].data_ptr(), st), "dd_exact_count")
        out = counts.cpu().numpy().astype(np.uint64)
        if (out == np.uint64(0xFFFFFFFFFFFFFFFF)).any():
            raise DandDError("exact k-mer table overflowed; pass a larger capacity")
        return [int(v) for v in out]

    # ---- K7 ---------------------------------------------------------------------------------
    def exact_pair_intersections(self, seqs: Sequence[PackedSeq], k: int, canon: bool = True,
                                 singles: Optional[Sequence[int]] = None, shard: Optional[tuple] = None) -> np.ndarray:
        """|A n B| for every pair of `seqs` at k: uint64 [n(n-1)/2], pairs (0,1), (0,2) .. (n-2,n-1).
        `singles` = |A| per sequence (exact_counts; with `shard`, this rank's shard of them) sizes the job
        and picks the path: presence bitmaps and a popcount per pair where almost every genome holds
        almost every k-mer (dense_pairs), else co-occurrence lists (sparse).  shard=(rank, world): only
        this rank's key range, the ranks' results add up (dandd_b200.dist.sum_counts)."""
        world = int(shard[1]) if shard is not None else 1
        if singles is None:
            singles = [self.exact_counts([s], k, canon, shard=shard)[0] for s in seqs]
        if dense_pairs(k, singles, world):
            return self.exact_pairs_dense(seqs, k, canon, shard=shard)
        return self.exact_pairs_sparse(seqs, k, canon, singles, shard=shard)

    def _pairs_budget(self) -> int:
        """Share of the device memory a pass may take: what is free plus what torch holds cached but unused."""
        free, _ = torch.cuda.mem_get_info(self.device)
        cached = torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        return int((free + cached) * PAIR_BUDGET_SHARE)

    def exact_pairs_sparse(self, seqs: Sequence[PackedSeq], k: int, canon: bool, singles: Sequence[int],
                           shard: Optional[tuple] = None, passes: Optional[int] = None) -> np.ndarray:
        """The co-occurrence-list path of exact_pair_intersections, in `passes` key-range passes (default:
        as few as fit the memory budget, plan_pair_passes)."""
        n = len(seqs)
        if n < 2:
            return np.zeros(n * (n - 1) // 2, dtype=np.uint64)
        if k > 64 and n > 65536:
            raise DandDError("exact pairs above k = 64 take at most 65536 genomes per job")

        def launch(ws, cap, nodes, part):
            check(self.lib.dd_exact_pairs_accumulate(ws.data_ptr(), ws.numel(), k, cap, nodes, n, n, part, self.stream),
                  "dd_exact_pairs_accumulate")

        out, _ = self._list_job(seqs, k, canon, singles, shard, passes, n * (n - 1) // 2, False, launch,
                                "exact pair table or node array overflowed; the single counts given understate the genomes")
        return out

    def _list_job(self, seqs: Sequence[PackedSeq], k: int, canon: bool, sizes: Sequence[int], shard: Optional[tuple],
                  passes: Optional[int], cells: int, node_counts: bool, launch, overflow: str, after=None):
        """One job over the K7 co-occurrence lists, in key-range passes (plan_pair_passes over `sizes`: the exact
        singles, or length bounds that never understate them).  Every pass, each genome pushes itself onto the list
        of every key of the pass it holds (genome g = seqs[g]); then launch(workspace, capacity, max_nodes, out_ptr)
        adds the pass's result into `cells` zeroed int64 cells on the device, and one copy brings them to the host.
        An all-ones cell means the table or node array overflowed: DandDError(overflow).  Returns (the cells summed
        over the passes, uint64; with node_counts, |A_g| per genome, uint64 [n], else None): the list-node counter is
        read after every genome's insert (dd_exact_pairs_node_count), and its growth over genome g is
        |A_g n the pass's key range|.  after(workspace, capacity, max_nodes, got), if given, runs at the end of every pass
        while its lists are still in the workspace; got is the pass's copy (uint64 [cells | node counter after genome g])."""
        n = len(seqs)
        srank, sworld = (int(shard[0]), int(shard[1])) if shard is not None else (0, 1)
        nsyms = [s.nsym for s in seqs]
        # [cells | node counter after genome g]
        part = torch.zeros(cells + (n if node_counts else 0), dtype=torch.int64, device=self.device)
        out = np.zeros(cells, dtype=np.uint64)
        singles = np.zeros(n, dtype=np.uint64) if node_counts else None
        plan = plan_pair_passes(sizes, k, lambda c, m: int(self.lib.dd_exact_pairs_workspace_bytes(k, c, m, n)),
                                self._pairs_budget(), passes)
        self.last_pair_plan = dict(plan, path="sparse")
        cap, nodes = plan["capacity"], plan["max_nodes"]
        ws = self._buf(plan["ws_bytes"], "exact_pairs")
        st = self.stream
        try:
            for p in range(plan["passes"]):
                sr, sw = pass_shard(srank, sworld, p, plan["passes"])
                check(self.lib.dd_exact_pairs_begin(ws.data_ptr(), ws.numel(), k, cap, nodes, n, st), "dd_exact_pairs_begin")
                for g, (s, ns) in enumerate(zip(seqs, nsyms)):
                    check(self.lib.dd_exact_pairs_insert_shard(s.codes.data_ptr(), s.invalid.data_ptr(), 0, ns, k, int(canon), g,
                                                               ws.data_ptr(), ws.numel(), cap, nodes, n, sr, sw, st),
                          "dd_exact_pairs_insert_shard")
                    if node_counts:
                        check(self.lib.dd_exact_pairs_node_count(ws.data_ptr(), ws.numel(), part.data_ptr() + 8 * (cells + g),
                                                                 st), "dd_exact_pairs_node_count")
                part[:cells].zero_()
                launch(ws, cap, nodes, part.data_ptr())
                got = part.cpu().numpy().view(np.uint64)
                if (got[:cells] == np.uint64(0xFFFFFFFFFFFFFFFF)).any():
                    raise DandDError(overflow)
                out += got[:cells]
                if after is not None:
                    after(ws, cap, nodes, got)
                if node_counts:
                    singles += np.diff(got[cells:], prepend=np.uint64(0))
            return out, singles
        finally:
            del ws
            self._ws.pop("exact_pairs", None)     # a pass may take half the device: not kept for later stages

    def _first_rank_launch(self, k: int, n: int, ranks: np.ndarray):
        """The K8 launch of _list_job for the rank table `ranks` [R, n] (uint16 on the host; copied to the device here)."""
        d_ranks = torch.from_numpy(ranks.view(np.int16)).to(self.device)
        return lambda ws, cap, nodes, part: check(
            self.lib.dd_exact_first_rank_hist(ws.data_ptr(), ws.numel(), k, cap, nodes, n, n, d_ranks.data_ptr(), ranks.shape[0],
                                              part, self.stream), "dd_exact_first_rank_hist")

    # ---- K8 ---------------------------------------------------------------------------------
    def exact_first_rank_hist(self, seqs: Sequence[PackedSeq], k: int, canon: bool, ranks,
                              singles: Optional[Sequence[int]] = None, shard: Optional[tuple] = None,
                              passes: Optional[int] = None) -> np.ndarray:
        """hist uint64 [R, n] for a rank table `ranks` [R, n] (uint16; 0xFFFF = genome not in the row): hist[r][m] =
        distinct k-mers of seqs whose minimum rank over the genomes holding them is m under row r.  A progressive
        ordering's row holds each genome's position (prefix i: cumsum(hist[r])[i - 1]); a set's row holds 0 for its
        members (its union: hist[r][0]).  One K7 list job at k (every genome read once per pass) and one K8 launch
        per pass.  singles / shard / passes as for exact_pairs_sparse."""
        n = len(seqs)
        ranks = np.ascontiguousarray(ranks, dtype=np.uint16).reshape(-1, n)
        rows = ranks.shape[0]
        if n == 0 or rows == 0:
            return np.zeros((rows, n), dtype=np.uint64)
        if n > 65535:
            raise DandDError("first-rank histograms take at most 65535 genomes per job (ranks are 16-bit)")
        if singles is None:
            singles = [self.exact_counts([s], k, canon, shard=shard)[0] for s in seqs]
        hist, _ = self._list_job(seqs, k, canon, singles, shard, passes, rows * n, False, self._first_rank_launch(k, n, ranks),
                                 "exact k-mer table or node array overflowed; the single counts given understate the genomes")
        return hist.reshape(rows, n)

    def exact_family_counts(self, seqs: Sequence[PackedSeq], k: int, canon: bool, ranks, shard: Optional[tuple] = None,
                            passes: Optional[int] = None):
        """(singles uint64 [n], hist uint64 [R, n]) in one job at k: hist as exact_first_rank_hist gives it for the rank
        table `ranks` [R, n], and singles[g] = |A_g| (this rank's key range under `shard`).  Unlike
        exact_first_rank_hist nothing is counted up front: the job is sized from the sequence lengths (length_bounds,
        never below the real counts), and the singles come from the list-node counter -- every genome pushes one node
        per key it holds, so the counter's growth over its insert is its count (dd_exact_pairs_node_count, summed
        over passes).  One K7 list job and one K8 launch per pass, one device->host copy per pass."""
        n = len(seqs)
        ranks = np.ascontiguousarray(ranks, dtype=np.uint16).reshape(-1, n) if n else np.zeros((len(ranks), 0), np.uint16)
        rows = ranks.shape[0]
        if n == 0:
            return np.zeros(n, dtype=np.uint64), np.zeros((rows, n), dtype=np.uint64)
        if n > 65535:
            raise DandDError("family counts take at most 65535 genomes per job (ranks are 16-bit)")
        world = int(shard[1]) if shard is not None else 1
        bounds = length_bounds([s.nsym for s in seqs], k, world)
        # with no row, one row that holds no genome: K8 still reports a full table or node array
        table = ranks if rows else np.full((1, n), 0xFFFF, dtype=np.uint16)
        launch = self._first_rank_launch(k, n, table)
        hist, singles = self._list_job(seqs, k, canon, bounds, shard, passes, table.size, True, launch,
                                       "exact k-mer table or node array overflowed; the length bounds understate the genomes")
        return singles, hist.reshape(-1, n)[:rows]

    # ---- K9 ---------------------------------------------------------------------------------
    def exact_spectrum(self, seqs: Sequence[PackedSeq], k: int, canon: bool, shard: Optional[tuple] = None,
                       passes: Optional[int] = None):
        """(hist, singles, priv), uint64 [n] each, in one job at k: hist[c - 1] = distinct k-mers held by exactly c of
        seqs, singles[g] = |A_g|, priv[g] = k-mers held by seqs[g] alone (this rank's key range under `shard`).  Sized
        from the sequence lengths and with the singles from the list-node counter, as exact_family_counts; one K7 list
        job, one K9 launch and one device->host copy per pass."""
        n = len(seqs)
        if n == 0:
            return tuple(np.zeros(n, dtype=np.uint64) for _ in range(3))
        if k > 64 and n > 65536:
            raise DandDError("the exact spectrum above k = 64 takes at most 65536 genomes per job")
        world = int(shard[1]) if shard is not None else 1
        bounds = length_bounds([s.nsym for s in seqs], k, world)

        def launch(ws, cap, nodes, part):      # cells [hist | priv]
            check(self.lib.dd_exact_occupancy_hist(ws.data_ptr(), ws.numel(), k, cap, nodes, n, n, part, part + 8 * n,
                                                   self.stream), "dd_exact_occupancy_hist")

        got, singles = self._list_job(seqs, k, canon, bounds, shard, passes, 2 * n, True, launch,
                                      "exact k-mer table or node array overflowed; the length bounds understate the genomes")
        return got[:n], singles, got[n:]

    # ---- K13 --------------------------------------------------------------------------------
    def exact_query_counts(self, seqs: Sequence[PackedSeq], n_refs: int, k: int, canon: bool, shard: Optional[tuple] = None,
                           passes: Optional[int] = None):
        """(singles uint64 [R + Q], inter uint64 [Q, R], shared uint64 [Q], union_R int) in one job at k, where seqs[:n_refs]
        are the R references and seqs[n_refs:] the Q queries: singles[g] = |A_g|, inter[q, r] = |A_q n A_r| (query q is
        seqs[R + q]), shared[q] = |A_q n U_R| and union_R = |U_R|, U_R the union of the references (this rank's key range
        under `shard`).  So |U_R u A_q| = union_R + |A_q| - shared[q].  Sized from the sequence lengths and with the
        singles from the list-node counter, as exact_family_counts; one K7 list job, one K13 launch and one
        device->host copy per pass."""
        n, R = len(seqs), int(n_refs)
        Q = n - R
        if R < 1 or Q < 1:
            raise DandDError("query counts need at least one reference and one query, got %d and %d" % (R, Q))
        if k > 64 and n > 65536:
            raise DandDError("query counts above k = 64 take at most 65536 genomes per job")
        world = int(shard[1]) if shard is not None else 1
        bounds = length_bounds([s.nsym for s in seqs], k, world)
        cells = Q * R

        def launch(ws, cap, nodes, part):      # cells [inter | shared | union_R]
            check(self.lib.dd_exact_query_counts(ws.data_ptr(), ws.numel(), k, cap, nodes, n, R, Q, part, part + 8 * cells,
                                                 part + 8 * (cells + Q), self.stream), "dd_exact_query_counts")

        got, singles = self._list_job(seqs, k, canon, bounds, shard, passes, cells + Q + 1, True, launch,
                                      "exact k-mer table or node array overflowed; the length bounds understate the genomes")
        return singles, got[:cells].reshape(Q, R), got[cells:cells + Q], int(got[-1])

    # ---- K12 --------------------------------------------------------------------------------
    def exact_cover_index(self, seqs: Sequence[PackedSeq], k: int, canon: bool, shard: Optional[tuple] = None,
                          passes: Optional[int] = None) -> dict:
        """The greedy cover index of seqs at k (K12), one part per key-range pass, resident on the device:
        {"k", "n", "parts": [{"offsets", "holders", "key_of_node", "covered", "n_keys", "n_nodes", "node_start"}],
        "singles": uint64 [n] (|A_g|), "keys": distinct keys (|union of all|), "bytes": device bytes of the parts}
        (this rank's key range under `shard`).  One K7 list job: after every pass's inserts, a count of its keys and
        nodes is read back and the pass's index is allocated to exactly that and emitted from the lists; node_start
        [n + 1] (host) holds the node counter before every genome's insert, so genome g's keys in the part are
        key_of_node[node_start[g]:node_start[g + 1]].  Raises DandDError for a full table or node array, and torch's
        OutOfMemoryError when the index does not fit."""
        n = len(seqs)
        if not 1 <= n <= 65535:
            raise DandDError("the exact cover index takes 1..65535 genomes per job (holders are 16-bit), got %d" % n)
        world = int(shard[1]) if shard is not None else 1
        bounds = length_bounds([s.nsym for s in seqs], k, world)
        parts = []

        def count(ws, cap, nodes, part):      # cells [distinct keys, nodes]
            check(self.lib.dd_exact_cover_count(ws.data_ptr(), ws.numel(), k, cap, nodes, n, part, self.stream),
                  "dd_exact_cover_count")

        def emit(ws, cap, nodes, got):
            n_keys, n_nodes = int(got[0]), int(got[1])
            dev = self.device
            part = {"offsets": torch.empty(n_keys + 1, dtype=torch.int32, device=dev),
                    "holders": torch.empty(max(n_nodes, 1), dtype=torch.int16, device=dev),
                    "key_of_node": torch.empty(max(n_nodes, 1), dtype=torch.int32, device=dev),
                    "covered": torch.zeros(max(n_keys, 1), dtype=torch.uint8, device=dev),
                    "n_keys": n_keys, "n_nodes": n_nodes,
                    "node_start": np.concatenate([[0], got[2:]]).astype(np.uint64)}
            status = torch.empty(2, dtype=torch.int64, device=dev)
            check(self.lib.dd_exact_cover_emit(ws.data_ptr(), ws.numel(), k, cap, nodes, n, n, n_keys, n_nodes,
                                               part["offsets"].data_ptr(), part["holders"].data_ptr(),
                                               part["key_of_node"].data_ptr(), status.data_ptr(), self.stream),
                  "dd_exact_cover_emit")
            if status.cpu().numpy().view(np.uint64).tolist() != [n_keys, n_nodes]:
                raise DandDError("exact cover index at k=%d: the lists did not match their count" % k)
            parts.append(part)

        got, singles = self._list_job(seqs, k, canon, bounds, shard, passes, 2, True, count,
                                      "exact k-mer table or node array overflowed; the length bounds understate the genomes",
                                      after=emit)
        nbytes = sum(sum(part[t].numel() * part[t].element_size() for t in ("offsets", "holders", "key_of_node", "covered"))
                     for part in parts)
        return {"k": int(k), "n": n, "parts": parts, "singles": singles, "keys": int(got[0]), "bytes": nbytes}

    def exact_cover_step(self, indices: Sequence[dict], genome: int, lost: torch.Tensor) -> None:
        """Genome `genome` joins the union (K12): for every part of every index (one per k, from exact_cover_index), the
        keys of the genome not covered yet are covered and add 1 to lost[c][h] of every genome h holding them, c the
        index's position.  lost: int64 [len(indices), n] on the device, added to.  One launch, no synchronisation."""
        n = int(indices[0]["n"])
        assert lost.dtype == torch.int64 and lost.is_contiguous() and tuple(lost.shape) == (len(indices), n)
        table = np.zeros((sum(len(ix["parts"]) for ix in indices), DD_COVER_PART_BYTES // 8), dtype=np.uint64)
        i = 0
        for c, ix in enumerate(indices):
            for part in ix["parts"]:
                table[i] = [part["offsets"].data_ptr(), part["holders"].data_ptr(), part["key_of_node"].data_ptr(),
                            part["covered"].data_ptr(), lost[c].data_ptr(), part["n_keys"], part["n_nodes"],
                            part["node_start"].ctypes.data]
                i += 1
        ws = self._buf(table.shape[0] * DD_COVER_PART_BYTES, "cover_step")
        check(self.lib.dd_exact_cover_step(table.ctypes.data, table.shape[0], n, int(genome), ws.data_ptr(), ws.numel(),
                                           self.stream), "dd_exact_cover_step")

    def exact_pairs_dense(self, seqs: Sequence[PackedSeq], k: int, canon: bool, shard: Optional[tuple] = None,
                          block: Optional[int] = None) -> np.ndarray:
        """The bitmap path of exact_pair_intersections (k <= DD_EXACT_BITMAP_MAXK): one K5 presence bitmap
        per genome, popc(A & B) per pair.  Genomes go through in blocks of `block` (default: as many as
        two blocks of bitmaps fit the memory budget)."""
        n = len(seqs)
        if n < 2:
            return np.zeros(n * (n - 1) // 2, dtype=np.uint64)
        srank, sworld = (int(shard[0]), int(shard[1])) if shard is not None else (0, 1)
        stride = (int(self.lib.dd_exact_workspace_bytes(k, 0)) + 255) // 256 * 256
        if block is None:
            block = max(1, min(n, self._pairs_budget() // (2 * stride)))
        block = min(int(block), n)
        nb = (n + block - 1) // block
        self.last_pair_plan = {"path": "dense", "passes": 1, "block": block, "bitmap_bytes": stride}
        rows = self._buf(block * stride, "pairs_rows")
        cols = self._buf(block * stride, "pairs_cols") if nb > 1 else rows
        out = torch.zeros(n * (n - 1) // 2, dtype=torch.int64, device=self.device)
        st = self.stream

        def fill(buf, g0):
            for i, g in enumerate(range(g0, min(n, g0 + block))):
                ws = buf.data_ptr() + i * stride
                s = seqs[g]
                check(self.lib.dd_exact_begin(ws, stride, k, 0, st), "dd_exact_begin")
                check(self.lib.dd_exact_insert_shard(s.codes.data_ptr(), s.invalid.data_ptr(), 0, s.nsym, k, int(canon), ws, stride,
                                                     0, srank, sworld, st), "dd_exact_insert_shard")

        for bi in range(nb):
            r0 = bi * block
            fill(rows, r0)
            nr = min(n, r0 + block) - r0
            for bj in range(bi, nb):
                c0 = bj * block
                if bj != bi:
                    fill(cols, c0)
                cbuf = rows if bj == bi else cols
                check(self.lib.dd_exact_pair_popc(rows.data_ptr(), r0, nr, cbuf.data_ptr(), c0, min(n, c0 + block) - c0, stride, k, n,
                                                  out.data_ptr(), st), "dd_exact_pair_popc")
        result = out.cpu().numpy().view(np.uint64).copy()
        del rows, cols
        for tag in ("pairs_rows", "pairs_cols"):
            self._ws.pop(tag, None)
        return result


# Exact all pairs (K7): the bitmap path wins where 4^k bits per genome are cheap next to the number of k-mers a
# genome holds -- then almost every genome holds almost every k-mer and the co-occurrence lists would hold
# sum(occ^2) ~ n^2 4^k / 2 entries.  DENSE_BITS_PER_KMER is the crossover: 4^k / DENSE_BITS_PER_KMER <= mean |A|.
DENSE_BITS_PER_KMER = 32
PAIR_BUDGET_SHARE = 0.5      # share of the free device memory one pass of the pair job may take


def dense_pairs(k: int, singles: Sequence[int], world: int = 1) -> bool:
    """Whether exact_pair_intersections takes the bitmap path.  `singles` may be one key-range shard of the
    counts (shard world `world`): the rule looks at whole genomes."""
    if k > _lib.DD_EXACT_BITMAP_MAXK or not len(singles):
        return False
    mean = float(np.mean(np.asarray(singles, dtype=np.float64))) * world
    return 4 ** k / DENSE_BITS_PER_KMER <= mean


def length_bounds(nsyms: Sequence[int], k: int, world: int = 1) -> List[int]:
    """Upper bounds of the single counts |A_g| from the sequence lengths, to size a job that has not counted them:
    a genome holds at most one distinct k-mer per symbol and at most 4^k of them; a key-range shard of `world`
    holds its share of those (the share's fluctuation is what plan_pair_passes' margin covers, as for passes)."""
    cap = 4 ** int(k) if int(k) < 32 else None
    return [-(-(min(int(s), cap) if cap else int(s)) // int(world)) for s in nsyms]


def pass_shard(rank: int, world: int, p: int, passes: int) -> tuple:
    """Key range of pass p of rank `rank`: the ranks split the keys, every rank splits its range again over its
    passes -- shard (rank + world * p) of (world * passes), so every key is handled by exactly one (rank, pass)."""
    return rank + world * p, world * passes


def plan_pair_passes(singles: Sequence[int], k: int, ws_bytes, budget: int, passes: Optional[int] = None) -> dict:
    """Table capacity, node count and number of key-range passes for the sparse pair job.  singles: |A| per
    genome in the key range to cover; ws_bytes(capacity, max_nodes) -> workspace bytes.  A pass holds about
    1/passes of the keys: the table must take every distinct key of its range (at most sum |A|, at most 4^k)
    at load <= 1/2, the node array one node per (genome, key).  Hash shares fluctuate: a margin is added."""
    total = int(sum(int(s) for s in singles))
    distinct = min(total, 4 ** k) if k < 32 else total
    p = int(passes) if passes else 1
    while True:
        keys = -(-distinct // p)
        capacity = 1024
        while capacity < 2 * (keys + keys // 16) + 1024:
            capacity *= 2
        max_nodes = -(-total // p) + total // (16 * p) + 4096
        need = ws_bytes(capacity, max_nodes)
        if passes or (need <= budget and max_nodes < 0xFFFFFFFE) or p >= 1 << 16:   # (node indices are u32)
            return {"passes": p, "capacity": capacity, "max_nodes": max_nodes, "ws_bytes": need}
        p *= 2


_default_engine = None


def get_engine() -> Engine:
    """Process-wide engine on LOCAL_RANK's GPU (torchrun) or device 0."""
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    return _default_engine


def set_engine(engine) -> None:
    """Install a different engine object (another device; tests install an oracle-backed double
    here to exercise the host logic on machines without a GPU)."""
    global _default_engine
    _default_engine = engine

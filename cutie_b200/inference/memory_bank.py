"""Token-major memory arena that replaces the reference's dict-of-tensors store.

The reference grows every key/value/shrinkage/selection/usage tensor with torch.cat on each memory
frame and re-concatenates on every eviction (cutie/inference/kv_memory_store.py:6-16, :194-204): an
O(N) copy of the whole bank per memory frame, with values kept channel-major [B, CV, N] so a top-k
gather touches 30 x 256 scattered 4-byte words per query.  Here:

  * every array is preallocated [B, capacity, C] *token-major* (one memory token = one contiguous row:
    256 B of key, 1 KB of value per object), so the readout gather reads whole rows;
  * non-permanent working memory is a ring: all evictions in the reference remove the OLDEST temporary
    tokens (FIFO kv_memory_store.py:206-207, consolidation memory_manager.py:317-320,
    clear kv:321-324), i.e. they advance a head pointer -- zero bytes moved;
  * permanent memory is a second append-only region; long-term memory is a linear region that is
    compacted (gathered) only when obsolete features are evicted (kv:209-242).

KeyValueMemoryStore keeps the reference class's public surface (size/perm_size/non_perm_size/engaged/
num_objects/buckets/key/value/shrinkage/selection/get_v_size/__contains__), the channel-major
properties being materialised on demand for inspection only.
"""
from collections import defaultdict
from typing import Dict, List, Literal, Optional, Tuple

import torch

from cutie_b200 import kernels as K_
from cutie_b200.kernels import BankSegment


class TokenArena:
    """A set of same-length token-major arrays [B, capacity, C_i] with ring semantics."""

    def __init__(self, ring: bool):
        self.ring = ring
        self.arrays: Dict[object, torch.Tensor] = {}
        self.widths: Dict[object, int] = {}
        self.cap = 0
        self.head = 0
        self.count = 0
        self.hint = 0
        self.B = None
        self.device = None
        # tcgen05 operand image of the 'key'/'shr' arrays (kernels.bank_key_image) + physical runs not yet imaged
        self.key_image: Optional[torch.Tensor] = None
        self.image_mu: Optional[torch.Tensor] = None
        self.dirty: List[Tuple[int, int]] = []
        # logical-order bookkeeping for readers that remember token indices across frames (threshold seeds): tokens ever
        # pushed / dropped from the front, and a generation that changes whenever the order changes any other way
        self.total_pushed = 0
        self.total_dropped = 0
        self.generation = 0

    # -- allocation ------------------------------------------------------------------------
    def declare(self, name, width: int, B: int, device):
        if self.B is None:
            self.B, self.device = B, device
        assert self.B == B
        if name not in self.widths:
            self.widths[name] = width
            if self.cap:
                self.arrays[name] = self._alloc(width, self.cap)

    def _alloc(self, width: int, cap: int) -> torch.Tensor:
        shape = (self.B, cap) if width == 0 else (self.B, cap, width)
        return torch.zeros(shape, dtype=torch.float32, device=self.device)

    def set_capacity_hint(self, tokens: int):
        self.hint = max(self.hint, int(tokens))

    def reserve(self, extra: int):
        need = self.count + extra
        if need <= self.cap:
            return
        new_cap = max(need, self.hint, 2 * self.cap)
        old, pieces = self.arrays, self.pieces()
        self.arrays = {}
        for name, width in self.widths.items():
            t = self._alloc(width, new_cap)
            if name in old:
                pos = 0
                for s, n in pieces:
                    t[:, pos:pos + n] = old[name][:, s:s + n]
                    pos += n
            self.arrays[name] = t
        self.cap, self.head = new_cap, 0
        self.key_image = None                          # re-linearised: rebuild the image of what was kept
        self.dirty = [(0, self.count)] if self.count else []

    def forget(self, name):
        self.arrays.pop(name, None)
        self.widths.pop(name, None)

    # -- ring bookkeeping ------------------------------------------------------------------
    def pieces(self, start: int = 0, length: Optional[int] = None) -> List[Tuple[int, int]]:
        """Physical (offset, len) runs covering logical tokens [start, start+length)."""
        if length is None:
            length = self.count - start
        if length <= 0:
            return []
        p = (self.head + start) % self.cap if self.cap else 0
        first = min(length, self.cap - p)
        out = [(p, first)]
        if first < length:
            out.append((0, length - first))
        return out

    def push(self, n: int) -> List[Tuple[int, int]]:
        """Reserve n new tokens at the tail; returns the physical runs to fill."""
        self.reserve(n)
        runs = self.pieces(self.count, n) if self.ring else [(self.head + self.count, n)]
        if not self.ring:
            assert self.head == 0
        self.count += n
        self.total_pushed += n
        self.dirty += runs                   # the caller fills these rows next; imaged lazily by flush_key_image
        return runs

    def drop_oldest(self, n: int):
        n = min(n, self.count)
        if n <= 0:
            return
        self.total_dropped += n
        if self.ring:
            self.head = (self.head + n) % self.cap
            self.count -= n
            if self.count == 0:
                self.head = 0
        else:                      # linear region: only a full clear is ever requested
            assert n == self.count
            self.count = 0

    def view(self, name, run: Tuple[int, int]) -> torch.Tensor:
        s, n = run
        return self.arrays[name][:, s:s + n]

    def flush_key_image(self, mu: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        """Bring the operand image up to date with every row written since the last call (new memory frames:
        one small launch; after a re-allocation or compaction: the whole arena).  `mu` [B, 64]: the bucket's key centre
        (the image holds k - mu); one image is only ever built with one centre."""
        if 'key' not in self.arrays or self.widths.get('key') != 64:
            return None
        if self.key_image is None:
            self.key_image = torch.zeros(self.B, K_.key_image_tiles(self.cap), K_.KEY_IMAGE_FLOATS,
                                         dtype=torch.float32, device=self.device)
            self.image_mu = mu
        assert (mu is None) == (self.image_mu is None) and (mu is None or mu.data_ptr() == self.image_mu.data_ptr()), \
            'a key image is tied to the centre it was first built with'
        for s, n in self.dirty:
            if n > 0:
                K_.bank_key_image(self.arrays['key'], self.arrays['shr'], s, n, self.key_image, mu)
        self.dirty = []
        return self.key_image


class _Bucket:
    def __init__(self, ring_temp: bool):
        self.objects: List[int] = []
        self.perm = TokenArena(ring=False)
        self.temp = TokenArena(ring=ring_temp)
        self.perm_chunks: List[int] = []      # appended chunk sizes (the reference prepends: logical order is reversed)


class KeyValueMemoryStore:
    """Arena-backed equivalent of cutie/inference/kv_memory_store.py:19-352."""

    def __init__(self, save_selection: bool = False, save_usage: bool = False, ring: bool = True,
                 key_centres: Optional[Dict[int, torch.Tensor]] = None):
        self.save_selection = save_selection
        self.save_usage = save_usage
        self.ring = ring
        # bucket id -> key centre [B, 64] of the tcgen05 operand images (shared between the working and the long-term
        # store of one MemoryManager: their segments are read in ONE affinity call and must agree on it)
        self.key_centres: Dict[int, torch.Tensor] = {} if key_centres is None else key_centres
        self.global_bucket_id = 0
        self._b: Dict[int, _Bucket] = {}
        self.perm_end_pt: Dict[int, int] = defaultdict(int)
        self._objs: Dict[int, int] = {}          # object id -> bucket id
        self.temp_hint = 0                       # capacity hints (tokens) applied to every bucket's arenas
        self.perm_hint = 0

    # -- reference surface: sizes ----------------------------------------------------------
    @property
    def buckets(self) -> Dict[int, List[int]]:
        return {b: bk.objects for b, bk in self._b.items()}

    def size(self, bucket_id: int) -> int:
        bk = self._b.get(bucket_id)
        return 0 if bk is None else bk.perm.count + bk.temp.count

    def perm_size(self, bucket_id: int) -> int:
        return self.perm_end_pt[bucket_id]

    def non_perm_size(self, bucket_id: int) -> int:
        return self.size(bucket_id) - self.perm_size(bucket_id)

    def engaged(self, bucket_id: Optional[int] = None) -> bool:
        return len(self._b) > 0 if bucket_id is None else bucket_id in self._b

    @property
    def num_objects(self) -> int:
        return len(self._objs)

    def get_v_size(self, obj_id: int) -> int:
        return self.size(self._objs[obj_id])

    def __contains__(self, obj_id) -> bool:
        return obj_id in self._objs

    # -- insertion (kv_memory_store.py:55-149) ---------------------------------------------
    def _declare(self, bk: _Bucket, B, CK, CV, device, objs):
        bk.perm.set_capacity_hint(self.perm_hint)
        bk.temp.set_capacity_hint(self.temp_hint)
        for arena, is_temp in ((bk.perm, False), (bk.temp, True)):
            arena.declare('key', CK, B, device)
            arena.declare('shr', 0, B, device)
            if is_temp and self.save_selection:
                arena.declare('sel', CK, B, device)
            if is_temp and self.save_usage:
                arena.declare('use', 0, B, device)
                arena.declare('life', 0, B, device)
            for o in objs:
                arena.declare(('val', o), CV, B, device)

    def slots_for_add(self, obj_ids: List[int], ne: int, B: int, CK: int, CV: int, device,
                      supposed_bucket_id: int = -1,
                      as_permanent: Literal['no', 'first', 'all'] = 'no'):
        """Bucket assignment + permanence rules of KeyValueMemoryStore.add; reserves `ne` token slots in
        every enabled bucket and returns [(bucket_id, arena, runs, is_permanent)] for the caller to fill
        (directly from the producer: a transpose kernel or the consolidation kernel)."""
        assert as_permanent in ('no', 'first', 'all')
        if supposed_bucket_id >= 0:
            if supposed_bucket_id not in self._b:
                self._b[supposed_bucket_id] = _Bucket(self.ring)
            bk = self._b[supposed_bucket_id]
            for o in obj_ids:
                if o not in self._objs:
                    self._objs[o] = supposed_bucket_id
                assert self._objs[o] == supposed_bucket_id
            bk.objects = list(obj_ids)
            enabled = [supposed_bucket_id]
        else:
            new_bucket = None
            enabled = []
            for o in obj_ids:
                if o in self._objs:
                    b = self._objs[o]
                else:
                    if new_bucket is None:
                        new_bucket = self.global_bucket_id
                        self.global_bucket_id += 1
                        self._b[new_bucket] = _Bucket(self.ring)
                    b = new_bucket
                    self._b[b].objects.append(o)
                    self._objs[o] = b
                if b not in enabled:
                    enabled.append(b)
        out = []
        for b in enabled:
            bk = self._b[b]
            permanent = False
            if as_permanent == 'all':
                self.perm_end_pt[b] += ne
                permanent = True
            elif as_permanent == 'first' and self.perm_end_pt[b] == 0:
                self.perm_end_pt[b] = ne
                permanent = True
            self._declare(bk, B, CK, CV, device, bk.objects)
            arena = bk.perm if permanent else bk.temp
            runs = arena.push(ne)
            if permanent:
                bk.perm_chunks.append(ne)
            elif self.save_usage:
                for r in runs:                                   # kv:132-134
                    arena.view('use', r).zero_()
                    arena.view('life', r).fill_(1e-7)
            out.append((b, arena, runs, permanent))
        return out

    def add(self, key: torch.Tensor, values: Dict[int, torch.Tensor], shrinkage: torch.Tensor,
            selection: Optional[torch.Tensor], supposed_bucket_id: int = -1,
            as_permanent: Literal['no', 'first', 'all'] = 'no') -> None:
        """Reference-shaped insert: key [B,CK,n], values {obj: [B,CV,n]}, shrinkage [B,1,n],
        selection [B,CK,n] (channel-major, as the encoders emit them)."""
        B, CK, ne = key.shape
        assert shrinkage.dim() == 3 and (not self.save_selection or selection.dim() == 3)
        objs = list(values.keys())
        CV = values[objs[0]].shape[1]
        for b, arena, runs, permanent in self.slots_for_add(objs, ne, B, CK, CV, key.device,
                                                            supposed_bucket_id, as_permanent):
            pos = 0
            for r in runs:
                n = r[1]
                K_.bank_append(key[:, :, pos:pos + n].contiguous(), arena.view('key', r))
                arena.view('shr', r).copy_(shrinkage[:, 0, pos:pos + n])
                if not permanent and self.save_selection:
                    K_.bank_append(selection[:, :, pos:pos + n].contiguous(), arena.view('sel', r))
                for o in self._b[b].objects:
                    if o in values:
                        K_.bank_append(values[o][:, :, pos:pos + n].contiguous(), arena.view(('val', o), r))
                pos += n

    # -- read-side views -------------------------------------------------------------------
    def segments(self, bucket_id: int, obj_ids: Optional[List[int]] = None, *, perm: bool = True,
                 temp_start: int = 0, temp_len: Optional[int] = None) -> List[BankSegment]:
        """Physical runs in read order (permanent region, then temporary oldest->newest)."""
        bk = self._b[bucket_id]
        objs = bk.objects if obj_ids is None else obj_ids
        out = []
        regions = []
        if perm and bk.perm.count:
            regions.append((bk.perm, bk.perm.pieces()))
        if bk.temp.count:
            regions.append((bk.temp, bk.temp.pieces(temp_start, temp_len)))
        mu = self.key_centre(bucket_id, regions)
        for arena, runs in regions:
            image = arena.flush_key_image(mu)
            for r in runs:
                out.append(BankSegment(arena.view('key', r), arena.view('shr', r),
                                       tuple(arena.view(('val', o), r) for o in objs), image, r[0],
                                       mu if image is not None else None))
        return out

    def key_centre(self, bucket_id: int, regions=None) -> Optional[torch.Tensor]:
        """The bucket's key centre: the mean key of the first tokens it ever served (the permanent first frame), fixed
        for the bucket's life.  Any vector is valid -- the energies do not depend on it -- it only tightens the FP16
        filter's error bound (network-derived keys sit on a large common mean)."""
        mu = self.key_centres.get(bucket_id)
        if mu is None and regions:
            arena, runs = regions[0]
            if runs and runs[0][1] > 0 and arena.widths.get('key') == 64:
                mu = arena.view('key', runs[0]).mean(dim=1).contiguous()
                self.key_centres[bucket_id] = mu
        return mu

    def temp_runs(self, bucket_id: int, start: int = 0, length: Optional[int] = None):
        bk = self._b[bucket_id]
        return bk.temp, bk.temp.pieces(start, length)

    # -- usage (kv:151-162, :244-250) --------------------------------------------------------
    def update_bucket_usage(self, bucket_id: int, usage_acc: torch.Tensor, acc_offset: int) -> None:
        """usage_acc: fixed-point per-token accumulators for the whole read; `acc_offset` is where this
        store's TEMPORARY tokens start inside it."""
        if not self.save_usage:
            return
        arena, runs = self.temp_runs(bucket_id)
        pos = acc_offset
        for r in runs:
            K_.usage_commit(arena.view('use', r), arena.view('life', r), usage_acc, pos)
            pos += r[1]

    def get_usage(self, bucket_id: int) -> torch.Tensor:
        if not self.save_usage:
            raise RuntimeError('I did not count usage!')
        arena, runs = self.temp_runs(bucket_id)
        use = torch.cat([arena.view('use', r) for r in runs], 1)
        life = torch.cat([arena.view('life', r) for r in runs], 1)
        return use / life

    # -- eviction --------------------------------------------------------------------------
    def sieve_by_range(self, bucket_id: int, start: int, end: int, min_size: int) -> None:
        """kv:164-204 restricted to what the reference ever asks for: start == 0 (drop the oldest
        temporary tokens, keep the last -end); buckets with <= min_size temporary tokens are untouched."""
        assert start == 0 and end <= 0
        bk = self._b[bucket_id]
        n = bk.temp.count
        if n <= min_size:
            return
        bk.temp.drop_oldest(n if end == 0 else max(n + end, 0))

    def remove_old_memory(self, bucket_id: int, max_len: int) -> None:
        self.sieve_by_range(bucket_id, 0, -max_len, max_len)

    def clear_non_permanent_memory(self) -> None:
        for b in self._b:
            self.sieve_by_range(b, 0, 0, 0)

    def remove_obsolete_features(self, bucket_id: int, max_size: int) -> None:
        """kv:209-242 (long-term store): keep the max_size most used tokens, in descending-usage order."""
        bk = self._b[bucket_id]
        assert self.perm_end_pt[bucket_id] == 0 and not bk.temp.ring
        usage = self.get_usage(bucket_id)
        keep = torch.topk(usage, k=max_size, dim=1)[1]                      # [B, max_size], per batch entry
        arena = bk.temp
        run = (0, arena.count)
        fresh = {}
        for name, width in arena.widths.items():
            src = arena.view(name, run)
            dst = torch.zeros_like(arena.arrays[name])
            if width == 0:
                K_.bank_gather([src.unsqueeze(-1)], keep, dst[:, :max_size].unsqueeze(-1))
            else:
                K_.bank_gather([src], keep, dst[:, :max_size])
            fresh[name] = dst
        arena.arrays = fresh
        arena.count = max_size
        arena.generation += 1                # tokens re-ordered by usage: remembered indices are void
        arena.dirty = [(0, max_size)]

    def replace_temp_rows(self, bucket_id: int, rows: Dict[object, torch.Tensor]) -> None:
        """Replace the whole temporary region of a linear (long-term) bucket by `rows` (name -> [B, n, C] or [B, n]): the
        key-sharded form of remove_obsolete_features, whose survivors arrive from other ranks."""
        bk = self._b[bucket_id]
        arena = bk.temp
        assert not arena.ring and set(rows) == set(arena.widths)
        n = next(iter(rows.values())).shape[1]
        for name, t in rows.items():
            dst = torch.zeros_like(arena.arrays[name])
            dst[:, :n] = t
            arena.arrays[name] = dst
        arena.count = n
        arena.generation += 1
        arena.dirty = [(0, n)] if n else []

    # -- object removal (kv:280-307) ---------------------------------------------------------
    def purge_except(self, obj_keep_idx: List[int]) -> None:
        keep = set(obj_keep_idx)
        for b in list(self._b):
            bk = self._b[b]
            for o in [o for o in bk.objects if o not in keep]:
                bk.perm.forget(('val', o))
                bk.temp.forget(('val', o))
                del self._objs[o]
            bk.objects = [o for o in bk.objects if o in keep]
            if not bk.objects:
                del self._b[b]
                self.key_centres.pop(b, None)

    # -- channel-major materialisation (inspection / parity tests; never on the frame path) ----
    def _export(self, bucket_id: int, name, perm: bool, temp: bool = True) -> torch.Tensor:
        bk = self._b[bucket_id]
        parts = []
        if perm and bk.perm.count:
            pos, chunks = 0, []
            for n in bk.perm_chunks:
                chunks.append(bk.perm.view(name, (pos, n)))
                pos += n
            parts += chunks[::-1]                                           # the reference prepends (kv:142)
        if temp:
            parts += [bk.temp.view(name, r) for r in bk.temp.pieces()]
        rows = torch.cat(parts, 1) if parts else None
        if rows is None:
            return None
        if rows.dim() == 2:
            return rows.unsqueeze(1).clone()
        out = torch.empty(rows.shape[0], rows.shape[2], rows.shape[1], device=rows.device)
        K_.bank_export(rows.contiguous(), out)
        return out

    @property
    def key(self) -> Dict[int, torch.Tensor]:
        return {b: self._export(b, 'key', True) for b in self._b}

    @property
    def shrinkage(self) -> Dict[int, torch.Tensor]:
        return {b: self._export(b, 'shr', True) for b in self._b}

    @property
    def selection(self) -> Dict[int, torch.Tensor]:
        return {b: self._export(b, 'sel', False) for b in self._b}

    @property
    def value(self) -> Dict[int, torch.Tensor]:
        return {o: self._export(b, ('val', o), True) for o, b in self._objs.items()}

    # reference attribute aliases (memory_manager / GUI code reads .k/.v/.s/.e in places)
    k, v, s, e = key, value, shrinkage, selection

    def _temp_counter(self, name) -> Dict[int, torch.Tensor]:
        out = {}
        for b, bk in self._b.items():
            parts = [bk.temp.view(name, r) for r in bk.temp.pieces()]
            out[b] = torch.cat(parts, 1) if parts else torch.zeros(bk.temp.B, 0, device=bk.temp.device)
        return out

    @property
    def use_cnt(self) -> Dict[int, torch.Tensor]:
        return self._temp_counter('use')

    @property
    def life_cnt(self) -> Dict[int, torch.Tensor]:
        return self._temp_counter('life')

    def set_capacity_hint(self, temp_tokens: int = 0, perm_tokens: int = 0):
        self.temp_hint, self.perm_hint = int(temp_tokens), int(perm_tokens)

"""Dataset + synthetic multiplexing — drop-in for /root/reference/dquartic/utils/data_loader.py:10-185.

`DIAMSDataset` keeps the reference's constructor, `__len__`, `__getitem__ -> 4 fp32 tensors`, `reset_epoch()`,
the python-`random` pair rejection loop with per-epoch de-duplication (111-125; identical index sequence for an
identical `random.seed`) and the per-pair min-max normalisation arithmetic (70-88, numpy semantics).

`DeviceBatchLoader` is the B200 data path: the slice pool lives in HBM (or in pinned host memory, staged per
batch), the host only draws the pair indices, and one fused kernel chain (csrc/data.cu) does min/max,
normalisation and hands the four tensors to the harness on the device.  It is iterable like a DataLoader and
exposes `.dataset`, so `ModelInterface.train(...)` accepts it unchanged.
"""
import os
import random
from typing import Literal

import numpy as np
import torch
from torch.utils.data import Dataset

from .. import _native as N


class DIAMSDataset(Dataset):
    def __init__(self, parquet_directory=None, ms2_file=None, ms1_file=None,
                 normalize: Literal[None, "minmax"] = None):
        if parquet_directory is None and ms1_file is not None and ms2_file is not None:
            self.ms2_data = np.load(ms2_file, mmap_mode="r")
            self.ms1_data = np.load(ms1_file, mmap_mode="r")
            self.data_type = "npy"
            print(f"Info: Loaded  {len(self.ms2_data)} MS2 slice samples and {len(self.ms1_data)} MS1 slice samples from NPY files.")
        elif parquet_directory is not None and ms1_file is None and ms2_file is None:
            self._load_parquet(parquet_directory)
            self.data_type = "npy"  # staged into arrays once instead of two directory scans per item (reference 161-185)
            print(f"Info: Loaded {len(self.ms2_data)} MS2 slice samples and MS1 slice samples from Parquet files.")
        else:
            raise ValueError(
                "Invalid input data arguments. Please provide either a `parquet_directory` or `ms2_file` and `ms1_file`. "
                f"Got parquet_directory={parquet_directory}, ms2_file={ms2_file}, ms1_file={ms1_file}.")
        self.normalize = normalize
        self.used_pairs = set()
        self.epoch_reset = False

    def _load_parquet(self, parquet_directory):
        """pyarrow reader for the schema written by the reference's create_parquet_data
        (utils/data_generation.py:206-223): ms1_data / ms2_data list<f32> + ms1_shape / ms2_shape."""
        import glob
        import pyarrow.parquet as pq

        ms2, ms1, meta = [], [], []
        cols = ["slice_index", "mz_isolation_target", "ms1_data", "ms2_data", "ms1_shape", "ms2_shape"]
        for f in sorted(glob.glob(os.path.join(parquet_directory, "*.parquet"))):
            tbl = pq.read_table(f, columns=cols).to_pydict()
            for si, mt, a1, a2, s1, s2 in zip(tbl["slice_index"], tbl["mz_isolation_target"], tbl["ms1_data"],
                                              tbl["ms2_data"], tbl["ms1_shape"], tbl["ms2_shape"]):
                ms2.append(np.asarray(a2, dtype=np.float32).reshape(tuple(s2)))
                ms1.append(np.asarray(a1, dtype=np.float32).reshape(tuple(s1)))
                meta.append((int(si), float(mt)))
        if not ms2:
            raise ValueError(f"no parquet slices found under {parquet_directory}")
        self.ms2_data = np.stack(ms2)
        self.ms1_data = np.stack(ms1)
        # the reference's parquet pair rule (data_loader.py:141-142): two rows with the same isolation window AND the
        # same slice index are never paired (the .npy rule is idx_1 != idx_2, which this implies)
        self.pair_meta = meta

    def __len__(self):
        return len(self.ms2_data)

    @property
    def n_train(self):
        """Training pairs are drawn from slices [0, n_train); the rest is held out for validation
        (`dquartic.utils.validation.hold_out`).  Default: every slice."""
        n = getattr(self, "_n_train", None)
        return len(self.ms2_data) if n is None else n

    @n_train.setter
    def n_train(self, n):
        if not 2 <= int(n) <= len(self.ms2_data):
            raise ValueError(f"{n} training slices of {len(self.ms2_data)}: at least 2 are needed to draw a pair")
        self._n_train = int(n)

    def draw_pair(self):
        """The reference's rejection loop (data_loader.py:111-125) over the training slices: returns (idx_1, idx_2)."""
        return self.pair_from(random, 0, self.n_train, self.used_pairs)

    def pair_from(self, rng, lo, hi, used):
        """The rejection loop with the random source `rng` over slices [lo, hi), not repeating an unordered pair in (and
        adding it to) `used`."""
        while True:
            idx_1 = rng.randint(lo, hi - 1)
            idx_2 = rng.randint(lo, hi - 1)
            if idx_1 == idx_2:
                continue
            meta = getattr(self, "pair_meta", None)
            if meta is not None and meta[idx_1] == meta[idx_2]:
                continue
            pair = tuple(sorted((idx_1, idx_2)))
            if pair in used:
                continue
            used.add(pair)
            return idx_1, idx_2

    def __getitem__(self, idx):
        i1, i2 = self.draw_pair()  # idx is ignored, as in the reference
        a, a1, b, b1 = self.ms2_data[i1], self.ms1_data[i1], self.ms2_data[i2], self.ms1_data[i2]
        if self.normalize == "minmax":
            self.ms2_min = np.min([a.min(), b.min()])
            self.ms2_max = np.max([a.max(), b.max()])
            self.ms1_min = np.min([a1.min()])
            self.ms1_max = np.max([a1.max()])
            a = (a - self.ms2_min) / (self.ms2_max - self.ms2_min)
            a1 = (a1 - self.ms1_min) / (self.ms1_max - self.ms1_min)
            b = (b - self.ms2_min) / (self.ms2_max - self.ms2_min)
            b1 = (b1 - self.ms1_min) / (self.ms1_max - self.ms1_min)
        else:
            raise ValueError("Invalid normalization method. Valid options are: None, 'minmax'.")
        return tuple(torch.from_numpy(np.asarray(z).astype(np.float32)) for z in (a, a1, b, b1))

    def reset_epoch(self):
        self.used_pairs.clear()
        self.epoch_reset = True


class DeviceBatchLoader:
    """GPU multiplexing loader.  pool='hbm': the whole pool is uploaded once; pool='pinned': the pool stays in
    pinned host memory and only the drawn slices are copied per batch (async, on the current stream)."""

    def __init__(self, dataset: DIAMSDataset, batch_size: int, device, pool: str = "hbm", batches_per_epoch=None,
                 rank: int = 0, world_size: int = 1):
        if dataset.normalize != "minmax":
            raise ValueError("Invalid normalization method. Valid options are: None, 'minmax'.")
        self.dataset = dataset
        self.batch_size = int(batch_size)
        self.device = torch.device(device)
        self.pool = pool
        n = len(dataset)   # the whole pool lives on the device, held-out slices included (validation mixtures)
        self.batches_per_epoch = batches_per_epoch or (dataset.n_train + self.batch_size - 1) // self.batch_size
        ms2 = np.asarray(dataset.ms2_data)
        ms1 = np.asarray(dataset.ms1_data)
        if ms2.dtype in (np.int32, np.int64, np.int16, np.uint16, np.uint8, np.int8):
            ms2, ms1, self.dtype_code = ms2.astype(np.int32), ms1.astype(np.int32), 0
        else:
            ms2, ms1, self.dtype_code = ms2.astype(np.float32), ms1.astype(np.float32), 1
        self.rt, self.mz = ms2.shape[1], ms2.shape[2]
        ms2_t, ms1_t = torch.from_numpy(np.ascontiguousarray(ms2)), torch.from_numpy(np.ascontiguousarray(ms1))
        if pool == "hbm":
            self.ms2 = ms2_t.to(self.device)
            self.ms1 = ms1_t.to(self.device)
        elif pool == "pinned":
            self.ms2 = ms2_t.pin_memory()
            self.ms1 = ms1_t.pin_memory()
            # two device staging slots (double buffer) filled by per-slice async copies on a side stream: the H2D
            # traffic of batch i+1 overlaps the training step of batch i.  Only the DISTINCT slices of a batch travel.
            nslot = min(2 * self.batch_size, n)
            self._dstage2 = [torch.empty((nslot, self.rt, self.mz), dtype=ms2_t.dtype, device=self.device) for _ in range(2)]
            self._dstage1 = [torch.empty((nslot, self.rt), dtype=ms1_t.dtype, device=self.device) for _ in range(2)]
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._pending = None     # (pairs, slot, event, pidx, bytes)
            self._slot = 0
            self._free_ev = [None, None]   # recorded after the multiplex kernel that last read the slot
        else:
            raise ValueError("pool must be 'hbm' or 'pinned'")
        self.h2d_bytes = 0

    def __len__(self):
        return self.batches_per_epoch

    def draw(self, nb):
        return [self.dataset.draw_pair() for _ in range(nb)]

    def _issue_copies(self, pairs, stream):
        """Async H2D of the distinct slices of `pairs` into the next staging slot; returns (slot, event, pidx, bytes)."""
        slot = self._slot
        self._slot ^= 1
        uniq = sorted({i for p in pairs for i in p})
        pos = {i: k for k, i in enumerate(uniq)}
        pidx_h = torch.tensor([[pos[a], pos[b]] for a, b in pairs], dtype=torch.long).pin_memory()
        with torch.cuda.stream(stream):
            if self._free_ev[slot] is not None:
                stream.wait_event(self._free_ev[slot])
            d2, d1 = self._dstage2[slot], self._dstage1[slot]
            for k, i in enumerate(uniq):
                d2[k].copy_(self.ms2[i], non_blocking=True)
            d1[: len(uniq)].copy_(self.ms1[uniq].pin_memory(), non_blocking=True)
            pidx = pidx_h.to(self.device, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
        nbytes = len(uniq) * (self.rt * self.mz * d2.element_size() + self.rt * d1.element_size()) + pidx_h.numel() * 8
        return slot, ev, pidx, nbytes

    def prefetch(self, pairs):
        """Start the host->device copies of a future batch on the side stream (pool='pinned')."""
        if self.pool != "pinned":
            return
        self._pending = (pairs,) + self._issue_copies(pairs, self._copy_stream)

    def make_batch(self, pairs, want_cond=False, weights=(0.5, 0.5)):
        nb = len(pairs)
        dev = self.device
        slot = None
        if self.pool == "hbm":
            ms2, ms1 = self.ms2, self.ms1
            pidx = torch.tensor(pairs, dtype=torch.long).to(dev, non_blocking=True)
            self.h2d_bytes = pidx.numel() * 8
        else:
            cur = torch.cuda.current_stream(dev)
            if self._pending is not None and self._pending[0] is pairs:
                _, slot, ev, pidx, nbytes = self._pending
            else:
                slot, ev, pidx, nbytes = self._issue_copies(pairs, self._copy_stream)
            self._pending = None
            cur.wait_event(ev)
            ms2, ms1 = self._dstage2[slot], self._dstage1[slot]
            self.h2d_bytes = nbytes
        x0 = torch.empty((nb, self.rt, self.mz), dtype=torch.float32, device=dev)
        other = torch.empty_like(x0)
        cond = torch.empty_like(x0) if want_cond else None
        m1 = torch.empty((nb, self.rt), dtype=torch.float32, device=dev)
        m2 = torch.empty_like(m1)
        stats = torch.empty((nb, 4), dtype=torch.int32, device=dev)
        N.call("dq_multiplex", ms2, ms1, self.dtype_code, pidx, stats, float(weights[0]), float(weights[1]), x0, other,
               cond, m1, m2, nb, self.rt * self.mz, self.rt)
        if slot is not None:
            # pidx was allocated on the copy stream: tell the caching allocator the compute stream reads it, or the
            # block could be handed to the next prefetch() while the multiplex kernel is still queued
            pidx.record_stream(torch.cuda.current_stream(dev))
            ev2 = torch.cuda.Event()
            ev2.record(torch.cuda.current_stream(dev))
            self._free_ev[slot] = ev2
        if want_cond:
            return x0, m1, other, m2, cond
        return x0, m1, other, m2

    def __iter__(self):
        nxt = self.draw(self.batch_size)
        self.prefetch(nxt)
        for b in range(self.batches_per_epoch):
            pairs = nxt
            if b + 1 < self.batches_per_epoch:
                nxt = self.draw(self.batch_size)
            batch = self.make_batch(pairs)
            if b + 1 < self.batches_per_epoch:
                self.prefetch(nxt)     # copies of the next batch overlap the training step of this one
            yield batch

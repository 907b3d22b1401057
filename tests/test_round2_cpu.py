"""CPU: round-2 host-side additions — the parquet slice format (SURVEY.md §8f-1), the secondary loss modes of the
oracle, window sharding, the vendoring recipe of the reference arm and the optimizer-shard layout."""
import os
import random

import numpy as np
import pytest
import torch


def _write_parquet(path, ms2, ms1, files=("runA.sqMass", "runB.sqMass"), dup_meta=False, base=0):
    """One parquet file with the reference's schema (utils/data_generation.py:206-223), all 14 columns."""
    import pyarrow as pa
    import pyarrow.parquet as pq

    schema = pa.schema([
        ("file", pa.string()), ("slice_index", pa.int64()), ("mz_isolation_target", pa.float64()),
        ("mz_start", pa.float64()), ("mz_end", pa.float64()), ("rt_start", pa.float64()), ("rt_end", pa.float64()),
        ("ms1_data", pa.list_(pa.float32())), ("ms2_data", pa.list_(pa.float32())),
        ("ms1_shape", pa.list_(pa.int64())), ("ms2_shape", pa.list_(pa.int64())),
        ("rt_values", pa.list_(pa.float32())), ("mz_values_ms1", pa.list_(pa.float32())),
        ("mz_values_ms2", pa.list_(pa.float32())),
    ])
    rows = []
    for i in range(len(ms2)):
        rows.append({
            "file": files[i % len(files)], "slice_index": (0 if dup_meta else base + i // 2), "mz_isolation_target": 400.0 + (0 if dup_meta else 25.0 * (i % 2)),
            "mz_start": 387.5, "mz_end": 412.5, "rt_start": 10.0 * i, "rt_end": 10.0 * i + 9.0,
            "ms1_data": ms1[i].flatten().astype(np.float32), "ms2_data": ms2[i].flatten().astype(np.float32),
            "ms1_shape": list(ms1[i].shape), "ms2_shape": list(ms2[i].shape),
            "rt_values": np.arange(ms2[i].shape[0], dtype=np.float32), "mz_values_ms1": np.arange(3, dtype=np.float32),
            "mz_values_ms2": np.arange(ms2[i].shape[1], dtype=np.float32),
        })
    pq.write_table(pa.Table.from_pylist(rows, schema=schema), path)


def test_parquet_slices_round_trip_bit_exact(tmp_path):
    from dquartic.utils.data_loader import DIAMSDataset

    rng = np.random.default_rng(7)
    ms2 = (rng.random((6, 5, 16)) * 1e4).astype(np.float32)
    ms1 = (rng.random((6, 5)) * 1e5).astype(np.float32)
    _write_parquet(str(tmp_path / "a.parquet"), ms2[:4], ms1[:4])
    _write_parquet(str(tmp_path / "b.parquet"), ms2[4:], ms1[4:], base=10)
    ds = DIAMSDataset(parquet_directory=str(tmp_path), normalize="minmax")
    assert len(ds) == 6
    assert np.array_equal(np.asarray(ds.ms2_data), ms2) and np.array_equal(np.asarray(ds.ms1_data), ms1)
    # items: same arithmetic as the .npy path on the same arrays
    np.save(tmp_path / "ms2.npy", ms2)
    np.save(tmp_path / "ms1.npy", ms1)
    dn = DIAMSDataset(ms2_file=str(tmp_path / "ms2.npy"), ms1_file=str(tmp_path / "ms1.npy"), normalize="minmax")
    random.seed(3)
    a = [ds[0] for _ in range(5)]
    random.seed(3)
    b = [dn[0] for _ in range(5)]
    for x, y in zip(a, b):
        for u, v in zip(x, y):
            assert torch.equal(u, v)
    with pytest.raises(ValueError):
        DIAMSDataset(parquet_directory=str(tmp_path), ms2_file="x", ms1_file="y")


def test_parquet_pair_rule_same_window_and_slice_never_paired(tmp_path):
    """reference data_loader.py:141-142: rows with equal (mz_isolation_target, slice_index) are rejected as a pair."""
    from dquartic.utils.data_loader import DIAMSDataset

    rng = np.random.default_rng(1)
    ms2 = rng.random((4, 3, 8)).astype(np.float32)
    ms1 = rng.random((4, 3)).astype(np.float32)
    _write_parquet(str(tmp_path / "a.parquet"), ms2[:2], ms1[:2])
    _write_parquet(str(tmp_path / "b.parquet"), ms2[2:], ms1[2:])   # same (slice, window) keys as file a
    ds = DIAMSDataset(parquet_directory=str(tmp_path), normalize="minmax")
    assert ds.pair_meta[0] == ds.pair_meta[2] and ds.pair_meta[1] == ds.pair_meta[3]
    random.seed(0)
    seen = set()
    for _ in range(4):     # 6 index pairs exist, (0, 2) and (1, 3) are forbidden: exactly 4 remain
        i, j = ds.draw_pair()
        assert ds.pair_meta[i] != ds.pair_meta[j]
        seen.add(tuple(sorted((i, j))))
    assert seen == {(0, 1), (0, 3), (1, 2), (2, 3)}


def test_sic_loss_and_modes_are_defined_and_differentiable():
    import dquartic_oracle as O
    from test_oracle_golden import TINY  # noqa: F401  (same tiny config as the golden tests)

    cfg = dict(dim=4, channels=1, dim_mults=[1, 2, 2, 3, 3, 4, 4], conditional=True, init_cond_channels=1,
               attn_cond_channels=1, tfer_dim_mult=620, downsample_dim=320, simple=True)
    P = {k: v.clone().requires_grad_(not k.endswith("freqs")) for k, v in O.det_params(cfg, 3).items()}
    _, _, ab = O.schedule_tables(1000, "cosine")
    g = torch.Generator().manual_seed(5)
    x0 = torch.rand(2, 4, 320, generator=g)
    c2 = torch.rand(2, 4, 320, generator=g)
    c1 = torch.rand(2, 4, generator=g)
    noise = torch.randn(2, 4, 320, generator=g)
    t = torch.tensor([10, 700])
    base, _ = O.train_loss(P, cfg, ab, x0, c2, c1, t, noise)
    l_eps, _ = O.train_loss_modes(P, cfg, ab, x0, c2, c1, t, noise)
    assert torch.allclose(l_eps, base.expand(2))          # eps mode, weight 0: the pinned default path
    l_sic, _ = O.train_loss_modes(P, cfg, ab, x0, c2, c1, t, noise, ms1_loss_weight=0.25)
    assert l_sic.shape == (2,) and torch.isfinite(l_sic).all() and not torch.allclose(l_sic, l_eps)
    l_x0, out = O.train_loss_modes(P, cfg, ab, x0, c2, c1, t, noise, pred_type="x0", pos_output_only=True)
    assert (out >= 0).all()                               # Softplus head
    w = O.loss_weight_table(ab, "x0")[t]
    assert torch.allclose(l_x0 / w, (l_x0 / w)[0].expand(2))
    l_x0.mean().backward()
    assert all(torch.isfinite(v.grad).all() for k, v in P.items() if v.requires_grad)
    xp, eps = O.ddim_update_x0(ab, x0, c2, 500)
    assert torch.allclose(eps, (x0 - torch.sqrt(ab[500]) * c2) / torch.sqrt(1 - ab[500]))


def test_window_sharding_is_a_partition_and_seeds_are_stable():
    from dquartic.model.model import DDIMDiffusionModel as D

    for n in (0, 1, 7, 8, 100000):
        for world in (1, 2, 3, 8):
            blocks = [D.shard_windows(n, r, world) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(blocks, blocks[1:]))
            sizes = [hi - lo for lo, hi in blocks]
            assert max(sizes) - min(sizes) <= 1
    seeds = {D.window_seed(1234, w) for w in range(10000)}
    assert len(seeds) == 10000 and D.window_seed(1234, 5) != D.window_seed(1235, 5)
    assert D.window_seed(7, 3) == 7 * 0x9E3779B97F4A7C15 + 3 * 0xD1B54A32D192ED03 + 0x2545F4914F6CDD1D & 0x7FFFFFFFFFFFFFFF


def test_optimizer_shard_layout_covers_the_buffer_once():
    from dquartic.model.model_interface import FusedAdamW

    class _Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.zeros(4))
            self.n_trainable_flat = 1000

        def flat_params(self):
            return torch.zeros(1008)

    ranges = [(100, 400), (600, 200)]
    world = 4
    cover = np.zeros(1000, dtype=int)
    for rank in range(world):
        opt = FusedAdamW(_Net())
        opt.set_sharding(rank, world, ranges)
        segs = opt._build_segments()
        so = 0
        for o, cnt, s in segs:
            assert s == so
            so += cnt
        own = {100 + rank * 100, 600 + rank * 50}
        for o, cnt, _ in segs:
            if o in own:
                cover[o:o + cnt] += 1
            elif rank == 0:
                cover[o:o + cnt] += 1
        assert so == 1000 - 600 + 150        # replicated 400 + own pieces 100 + 50
    assert (cover == 1).all()


def test_reference_vendoring_recipe_runs_where_the_reference_is(tmp_path):
    """oracle/make_ref.py on a stand-in checkout with the reference's layout: the hot-path modules are copied unmodified,
    package markers and shims are added; without a checkout it is a no-op that succeeds (build() calls it that way)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = os.path.join(root, "oracle", "make_ref.py")
    env = {k: v for k, v in os.environ.items() if k != "DQUARTIC_REFERENCE"}
    r = subprocess.run([sys.executable, script], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    checkout, dst = tmp_path / "reference", tmp_path / "_ref"
    rels = ("model/model.py", "model/model_interface.py", "model/unet1d.py", "model/building_blocks.py",
            "utils/data_loader.py")
    for rel in rels:
        (checkout / "dquartic" / rel).parent.mkdir(parents=True, exist_ok=True)
        (checkout / "dquartic" / rel).write_text(f"# {rel}\n")
    r = subprocess.run([sys.executable, script, str(checkout), str(dst)], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr
    for rel in rels:
        assert (dst / "dquartic" / rel).read_text() == f"# {rel}\n"
    for rel in ("dquartic/__init__.py", "dquartic/model/__init__.py", "dquartic/utils/__init__.py"):
        assert (dst / rel).exists()
    for shim in ("rotary_embedding_torch.py", "duckdb.py"):
        assert (dst / shim).read_bytes() == open(os.path.join(root, "oracle", "_shims", shim), "rb").read()
    r = subprocess.run([sys.executable, script, str(tmp_path / "missing"), str(dst)], capture_output=True, text=True,
                       env=env)
    assert r.returncode != 0


def test_deferred_parameter_gathers_are_awaited_before_the_parameters_are_read():
    """`FusedAdamW.step(defer_gather=True)` leaves the parameter all-gathers in flight; `UNet1d.sync_params` (called by
    `flat_params`, `state_dict`, the bf16 operand refresh and deepcopy) must wait for every one of them exactly once."""
    from dquartic.model.unet1d import UNet1d

    class _Work:
        def __init__(self):
            self.waited = 0

        def wait(self):
            self.waited += 1

    class _Shell:   # the two attributes the methods touch, without building a network
        sync_params = UNet1d.sync_params
        flat_params = UNet1d.flat_params

    sh = _Shell()
    sh._flat = torch.zeros(3)
    works = [_Work(), _Work()]
    sh.__dict__["_pending_param_works"] = list(works)
    assert sh.flat_params() is sh._flat
    assert [w.waited for w in works] == [1, 1] and sh.__dict__["_pending_param_works"] == []
    sh.sync_params()                      # nothing pending: no second wait
    assert [w.waited for w in works] == [1, 1]

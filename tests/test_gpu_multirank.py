"""GPU suite, two ranks over NCCL (skipped with fewer than two visible GPUs): the SAME global pairs sharded two ways give the
aggregate of the single-GPU evaluation bit for bit -- per-sequence means, the mean over sequences
(StarGANv2AdvCon/core/solver.py:352-354) and the pair count; the pooled RMSE to 1e-12 (fp64 sums of fp64 per-pair sums)."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

CLIPS = [9, 4, 1, 7]          # frames per sequence -> 8 + 3 + 0 + 6 pairs; one sequence without pairs
H, W, SEED = 96, 160, 4242


def _global_data(tcl, device):
    pairs = tcl.sharding.pairs_per_sequence(CLIPS)
    P = sum(pairs)
    ff, bf = tcl.synth.make_flows(P, H, W, seed=SEED, max_shift=9.0, device="cpu")
    prev, cur = tcl.synth.make_frames(P, 3, H, W, seed=SEED, kind="white", device="cpu")
    return pairs, tuple(t.to(device) for t in (ff, bf, prev, cur))


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    import tcl_b200 as tcl
    pairs, (ff, bf, prev, cur) = _global_data(tcl, device)
    plan = tcl.plan_shards(pairs, world, rank)
    sl = slice(plan.start, plan.stop)
    seq = torch.tensor(plan.seq_of_pair, dtype=torch.long, device=device)
    out = tcl.evaluate_sharded(ff[sl].contiguous(), bf[sl].contiguous(), prev[sl].contiguous(), cur[sl].contiguous(), seq, len(pairs))
    torch.cuda.synchronize()
    # fewer pairs than GPUs: the same two pairs on both ranks, one horizontal band each (SURVEY.md 8e)
    banded = tcl.evaluate_banded(ff[:2].contiguous(), bf[:2].contiguous(), prev[:2].contiguous(), cur[:2].contiguous())
    out = dict(out, band_sums=banded["pair_sums"], band_rmse=banded["pair_rmse"])
    torch.save({k: v.detach().cpu() for k, v in out.items()}, os.path.join(out_dir, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_two_rank_sharded_evaluation_equals_single_gpu(tcl, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    port = 29600 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    device = torch.device("cuda", 0)
    pairs, (ff, bf, prev, cur) = _global_data(tcl, device)
    seq = torch.tensor([s for s, n in enumerate(pairs) for _ in range(n)], dtype=torch.long, device=device)
    one = {k: v.cpu() for k, v in tcl.evaluate_sharded(ff, bf, prev, cur, seq, len(pairs)).items()}
    for r in range(2):
        got = torch.load(os.path.join(tmp_path, f"r{r}.pt"))
        for key in ("per_sequence_mean", "mean_over_sequences", "mean_over_pairs", "n_pairs"):
            assert torch.equal(got[key], one[key]), (r, key)
        assert torch.allclose(got["pooled_rmse"], one["pooled_rmse"], rtol=1e-12, atol=0.0)
    whole = tcl.fused_forward(bf[:2].contiguous(), prev[:2].contiguous(), cur[:2].contiguous(), ff=ff[:2].contiguous())
    for r in range(2):
        got = torch.load(os.path.join(tmp_path, f"r{r}.pt"))
        assert torch.allclose(got["band_sums"], whole.pair_sums.cpu(), rtol=1e-12, atol=0.0)   # (bands of whole 32-row tile rows)
        assert torch.allclose(got["band_rmse"], whole.pair_vals.cpu(), rtol=1e-6, atol=0.0)
    assert int(one["n_pairs"]) == sum(pairs) and float(one["per_sequence_mean"][2]) == 0.0   # the sequence without pairs

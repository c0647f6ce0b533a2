"""Multi-GPU check (torchrun, one rank per GPU): a trace time-sharded over the ranks with halos must give
the same global median, the same events (global sample indices, ids in time order) and the same CUSUM+
levels as the unsharded run on rank 0.
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P scripts/check_sharded.py
        [--stepfit-samples N | --stepfit-fallback]
With --stepfit-samples the trace holds short single-level pulses instead, the analyzers fit the events shorter than N
samples with the step-response model, and the step-fit columns (type, parameters) are compared as well.  With
--stepfit-fallback the trace holds two-level events and shallow long events (-180 pA, 9 000-90 000 samples, which
CUSUM+ leaves without a sub-level), the analyzers fit those with the step-response fallback, and the step-fit columns
are compared the same way."""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
from cusumtools_b200 import pipeline, synth

ap = argparse.ArgumentParser()
ap.add_argument("--stepfit-samples", type=int, default=0)
ap.add_argument("--stepfit-fallback", action="store_true")
args = ap.parse_args()
sf_samples, sf_fallback = args.stepfit_samples, args.stepfit_fallback
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
S = synth.CHIMERA_SETTINGS
n = 6_291_456
codes, _ = synth.c1_trace(n=n, n_events=1500, seed=5)
block = 1 << 16
kw = dict(threshold=5.0, hysteresis=1.0, baseline_block=block, baseline_min=4700.0, baseline_max=5300.0,
          cusum_delta=400.0, cusum_h=10.0)
if sf_samples:
    codes = synth.device_trace(n, dev, seed=5, levels=((-1000.0, 150),)).cpu().numpy()
    kw["stepfit_samples"] = sf_samples
elif sf_fallback:
    tpl = []
    for L in (9000, 20_000, 45_000, 90_000):
        tpl += [synth.EVENT_LEVELS, ((-180.0, L),)]
    codes = synth.device_trace(n, dev, seed=5, events_per_s=40.0, levels=tpl).cpu().numpy()
    # baseline blocks from samples within 5 sigma of the baseline only: the shallow events must not shift it
    kw.update(stepfit_fallback=True, baseline_min=4900.0, baseline_max=5100.0)
lo, hi = pipeline.shard_bounds(n, world, rank, block)
halo = pipeline.required_halo(1e5, 8, synth.FS, max_event=100_000 + 2 * 100, block=block)    # maxpoints + 2 * event_padding (the analyzer's defaults)
a, b = max(0, lo - halo), min(n, hi + halo)
an = pipeline.TraceAnalyzer(b - a, S, 1e5, 8, lo_halo=lo - a, hi_halo=b - hi, group=dist.group.WORLD, device=dev, **kw)
r = an.run(torch.from_numpy(codes[a:b]).to(dev))
mine = torch.stack((r.events.starts + lo, r.events.ends + lo, r.levels.n_levels.to(torch.int64)), 1)
sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
dist.all_gather(sizes, torch.tensor([mine.shape[0]], dtype=torch.int64, device=dev))
parts = [torch.zeros((int(s.item()), 3), dtype=torch.int64, device=dev) for s in sizes]
dist.all_gather(parts, mine) if len({int(s.item()) for s in sizes}) == 1 else None
if len({int(s.item()) for s in sizes}) != 1:                       # ragged: pad to the maximum
    m = max(int(s.item()) for s in sizes)
    pad = torch.full((m, 3), -1, dtype=torch.int64, device=dev); pad[:mine.shape[0]] = mine
    buf = [torch.zeros((m, 3), dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(buf, pad)
    parts = [bb[:int(s.item())] for bb, s in zip(buf, sizes)]
# the streamed form of the same shard (time sub-shards overlapped with the host->device copy) must agree with it
san = pipeline.StreamingAnalyzer(b - a, S, 1e5, 8, lo_halo=lo - a, hi_halo=b - hi, shards=3, first_blocks=2,
                                 group=dist.group.WORLD, device=dev, **kw)
rs = san.run_from_host(torch.from_numpy(codes[a:b].copy()).pin_memory())
gs, ge = r.events.starts.cpu().numpy(), r.events.ends.cpu().numpy()
stream_ok = (tuple(rs.median_codes) == tuple(r.median_codes) and rs.first_event_id == r.first_event_id
             and rs.total_events == r.total_events and len(rs.tables["starts"]) == len(gs)
             and np.abs(rs.tables["starts"] - gs).max(initial=0) <= 1 and np.abs(rs.tables["ends"] - ge).max(initial=0) <= 1
             and torch.max(torch.abs(rs.filtered - r.filtered)).item() < 0.02)
flag = torch.tensor([int(stream_ok)], dtype=torch.int64, device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
stream_ok = bool(flag.item())
# stage 4 sharded: every rank transforms its contiguous block of Welch segments of the filtered trace (its samples
# filtered here with a warm-up halo and the GLOBAL median), one all_reduce of the L/2+1 sums (SURVEY.md 8e)
from cusumtools_b200 import filters, psd
Lw = 1 << 16
s0, s1, p0, p1 = psd.segment_share(n, Lw, world, rank)
hw = 4096
qa, qb = max(0, p0 - hw), min(n, p1 + hw)
yl = filters.dequant_filtfilt(torch.from_numpy(codes[qa:qb]).to(dev), S, 1e5, 8, median_codes=r.median_codes)[p0 - qa:p1 - qa]
fP, P = psd.welch_sharded(yl, synth.FS, Lw, shift=float(r.pad_value), group=dist.group.WORLD)
sf_parts = pipeline.gather_tables({"types": r.types.to(torch.int64), "params": r.stepfit.params}, dist.group.WORLD) if sf_samples or sf_fallback else None
first = torch.tensor([r.first_event_id, r.total_events], dtype=torch.int64, device=dev)
firsts = [torch.zeros(2, dtype=torch.int64, device=dev) for _ in range(world)]
dist.all_gather(firsts, first)
ok = True
if rank == 0:
    allev = torch.cat(parts).cpu().numpy()
    one = pipeline.TraceAnalyzer(n, S, 1e5, 8, device=dev, **kw)
    ref = one.run(torch.from_numpy(codes).to(dev))
    want = torch.stack((ref.events.starts, ref.events.ends, ref.levels.n_levels.to(torch.int64)), 1).cpu().numpy()
    ids = [int(f[0]) for f in firsts]
    ok = (r.median_codes == ref.median_codes and allev.shape == want.shape and np.array_equal(allev[:, :2], want[:, :2])
          and np.mean(allev[:, 2] == want[:, 2]) > 0.999 and ids == list(np.cumsum([0] + [int(s.item()) for s in sizes[:-1]]))
          and int(firsts[0][1]) == want.shape[0] and stream_ok)
    fW, PW = psd.welch(ref.filtered, synth.FS, Lw)
    psd_ok = bool(np.allclose(fP, fW) and np.all(np.abs(P - PW) <= 2e-5 * PW + 1e-9 * PW.max()))
    ok = ok and psd_ok
    if sf_samples:
        gt, gp = sf_parts["types"].cpu().numpy(), sf_parts["params"].cpu().numpy()
        wt, wp = ref.types.cpu().numpy().astype(np.int64), ref.stepfit.params.cpu().numpy()
        both = (gt == 1) & (wt == 1) if gt.shape == wt.shape else np.zeros(0, bool)
        sf_ok = bool(gt.shape == wt.shape and np.mean(gt == wt) > 0.999 and both.sum() > 0.9 * len(wt)
                     and np.percentile(np.abs(gp[both] - wp[both])[:, 1], 99) < 0.5)
        print(f"stepfit columns over {world} GPUs: {int(both.sum())} fits in both, {'agree' if sf_ok else 'DIFFER'}")
        ok = ok and sf_ok
    elif sf_fallback:
        gt, gp = sf_parts["types"].cpu().numpy(), sf_parts["params"].cpu().numpy()
        wt, wp = ref.types.cpu().numpy().astype(np.int64), ref.stepfit.params.cpu().numpy()
        both = (gt == 1) & (wt == 1) if gt.shape == wt.shape else np.zeros(0, bool)
        sf_ok = bool(gt.shape == wt.shape and np.array_equal(gt, wt) and both.sum() >= 10
                     and np.percentile(np.abs(gp[both] - wp[both])[:, 1], 99) < 0.5)
        print(f"stepfit fallback columns over {world} GPUs: {int(both.sum())} fits in both, {'agree' if sf_ok else 'DIFFER'}")
        ok = ok and sf_ok
    print(f"sharded over {world} GPUs: {allev.shape[0]} events vs {want.shape[0]} unsharded, median {r.median_codes} vs "
          f"{ref.median_codes}, ids {ids}, streamed form {'agrees' if stream_ok else 'DIFFERS'}, sharded PSD {'agrees' if psd_ok else 'DIFFERS'}: {'OK' if ok else 'MISMATCH'}")
dist.destroy_process_group()
sys.exit(0 if ok else 1)

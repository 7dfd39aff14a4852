"""Per-kernel device time of headline train steps (bench.py's Predictor(bias) loop, queries in HBM) from
torch.profiler with CUDA activities.  Warm-up steps run unprofiled; the table lists every kernel of the profiled
steps with its total, per-step time and share.
usage: python scripts/profile_kernels.py [--typed] [--batches 256] [--steps 5] [--out DIR]"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.profiler import ProfilerActivity, profile

import bench


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--typed", action="store_true")
    ap.add_argument("--batches", type=int, default=256)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the table to DIR/kernels_<graph>.txt")
    a = ap.parse_args()
    from rnnlogic_b200 import KnowledgeGraph
    from rnnlogic_b200.predictors import Predictor
    shape, N, R, train, valid, test, rules = bench.build_workload("fb15k237", typed=a.typed)
    batches = bench.make_batches(train, R, seed=1)
    dev = torch.device("cuda:0")
    kg = KnowledgeGraph(entity_size=N, relation_size=R, train=train, valid=valid, test=test)
    model = Predictor(kg, entity_feature="bias")
    model.set_rules([[h] + list(b) for h, b in rules])
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        model.rule_weights.copy_(torch.randn(model.num_rules, generator=g) * 0.1)
    model = model.cuda(dev)
    run = bench.Runner(model, bench.deal_steps(batches, model.compiled, a.batches, a.warmup + a.steps, 1, 0), a.batches, 1, dev)
    run.size_cells()
    run.device_loop(a.warmup, a.steps)                           # warm-up, launch-shape feedback
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run.device_loop(0, a.steps)
        torch.cuda.synchronize()
    tot = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.device_time_total > 0:
            n, t = tot.get(ev.name, (0, 0.0))
            tot[ev.name] = (n + 1, t + ev.device_time_total)
    allt = sum(t for _, t in tot.values())
    lines = ["%s, %d headline steps of %d batches, %s" % ("typed graph" if a.typed else "i.i.d. graph", a.steps, a.batches,
                                                          torch.cuda.get_device_name(0)),
             "%10s %10s %7s %6s  %s" % ("total us", "us/step", "share", "calls", "kernel")]
    for name, (n, t) in sorted(tot.items(), key=lambda kv: -kv[1][1]):
        lines.append("%10.1f %10.1f %6.1f%% %6d  %s" % (t, t / a.steps, 100 * t / allt, n, name[:110]))
    lines.append("%10.1f %10.1f  all kernels" % (allt, allt / a.steps))
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "kernels_%s.txt" % ("typed" if a.typed else "iid")), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

"""Time the AMP update's discriminator data path and print one JSON line (card name and power limit included).

(a) launch: one hl_amp_update_batch launch (AMPUpdateSampler.sample with a normaliser) at each --mb, with a --ring-rows
    replay ring and a --preload-rows preload.  --launches back-to-back calls captured in one CUDA graph, timed with CUDA
    events over --repeats replays (device time per launch, no host launch cost).  Algorithmic bytes per row: read 480
    (two 120 B ring rows, 2 x (48 + 72) B of preload columns), write 960 (four 30-wide states, two 60-wide inputs);
    their sum over the time, as a share of the measured HBM peak.  The gathers are random rows of tables larger than L2
    (240 MB ring, 784 MB preload), so the DRAM traffic is larger than these bytes: a row piece is read as whole 32 B
    sectors.
(b) one update's data path: --minibatches minibatches the reference way -- zip(ReplayBuffer.feed_forward_generator,
    AMPLoader.feed_forward_generator) (host np.random.choice, H2D copy, gather), 4 x normalize_torch, 2 x cat -- against
    AMPUpdateSampler.generator.  Host clock around each, ending in torch.cuda.synchronize(); one unmeasured round, then
    --rounds rounds, alternating the two.
(c) with --with-disc: (b) with a [1024, 512] discriminator's forward on both inputs, the MSE +-1 losses, the gradient
    penalty on the raw expert pair, an Adam step and two Normalizer.update calls in the loop.

    python tools/amp_update_timing.py [--mb 98304 102400 393216] [--with-disc] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.amp_rollout_timing import PEAK_GBS, events_ms, graph_of, power_limit_w  # noqa: E402

READ_B, WRITE_B = 480, 960


def _setup(ring_rows, preload_rows, dev):
    from types import SimpleNamespace
    from isaacgymloco_b200.amp_discriminator import Normalizer
    from isaacgymloco_b200.motion_loader import AMPLoader
    from isaacgymloco_b200.replay_buffer import ReplayBuffer
    g = torch.Generator(device=dev).manual_seed(1)
    rb = ReplayBuffer(30, ring_rows, dev)
    rb.states.copy_(torch.randn(ring_rows, 30, device=dev, generator=g))
    rb.next_states.copy_(torch.randn(ring_rows, 30, device=dev, generator=g))
    rb.num_samples = ring_rows
    # a loader in the preload state: its feed_forward_generator / gather_pairs read only these attributes
    ld = SimpleNamespace(preload_transitions=True, device=dev,
                         preloaded_s=torch.randn(preload_rows, 49, device=dev, generator=g),
                         preloaded_s_next=torch.randn(preload_rows, 49, device=dev, generator=g))
    ld.gather_pairs = lambda idxs: AMPLoader.gather_pairs(ld, idxs)
    ld.feed_forward_generator = lambda k, mb: AMPLoader.feed_forward_generator(ld, k, mb)
    norm = Normalizer(30, device=dev)
    norm.update(torch.randn(4096, 30, device=dev, generator=g))
    return rb, ld, norm


def measure_launch(rb, ld, norm, mb, launches, repeats):
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    sm = AMPUpdateSampler(ld, rb, norm, mb, 7)
    gr = graph_of(sm.sample, launches)
    v = []
    for _ in range(2):
        v.extend(1e3 * t / launches for t in events_ms(gr.replay, repeats))
    med = statistics.median(v)
    nbytes = (READ_B + WRITE_B) * mb
    del gr
    return {"mb": mb, "launches_per_replay": launches, "median_us": med, "min_us": min(v), "max_us": max(v),
            "algorithmic_bytes": nbytes, "algorithmic_gbs": nbytes / (med * 1e-6) / 1e9,
            "share_of_peak": nbytes / (med * 1e-6) / (PEAK_GBS * 1e9)}


class _Disc:
    """HybridPPO.update's discriminator half: forward on both inputs, MSE +-1, gradient penalty, Adam, normaliser."""

    def __init__(self, dev, norm):
        from isaacgymloco_b200.amp_discriminator import AMPDiscriminator
        torch.manual_seed(3)
        self.disc = AMPDiscriminator(60, 2.0, [1024, 512], dev)
        self.opt = torch.optim.Adam(self.disc.parameters(), lr=1e-5)
        self.norm, self.mse = norm, torch.nn.MSELoss()

    def __call__(self, ps, es, esn, xp, xe):
        pd, ed = self.disc(xp), self.disc(xe)
        loss = (self.mse(ed, torch.ones_like(ed)) + self.mse(pd, -torch.ones_like(pd))) / 2
        loss = loss + self.disc.compute_grad_pen(es, esn, lambda_=10)
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        self.norm.update(ps)
        self.norm.update(es)


def measure_update(rb, ld, norm, mb, k, rounds, with_disc):
    from isaacgymloco_b200.amp_update import AMPUpdateSampler
    sm = AMPUpdateSampler(ld, rb, norm, mb, 11)
    disc = _Disc(rb.device, norm) if with_disc else None
    np.random.seed(0)

    def reference():
        for (s, sn), (es, esn) in zip(rb.feed_forward_generator(k, mb), ld.feed_forward_generator(k, mb)):
            xp = torch.cat([norm.normalize_torch(s), norm.normalize_torch(sn)], -1)
            xe = torch.cat([norm.normalize_torch(es), norm.normalize_torch(esn)], -1)
            if disc is not None:
                disc(s, es, esn, xp, xe)

    def sampler():
        for b in sm.generator(k):
            if disc is not None:
                disc(b.policy_state, b.expert_state, b.expert_next_state, b.x_policy, b.x_expert)

    per = {"reference": [], "sampler": []}
    for rnd in range(rounds + 1):
        for name, fn in (("reference", reference), ("sampler", sampler)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            dt = 1e3 * (time.perf_counter() - t0)
            if rnd > 0:                 # round 0: warm-up (allocator, cuBLAS, library handles)
                per[name].append(dt)
    out = {name: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for name, v in per.items()}
    out.update(mb=mb, minibatches=k, rounds=rounds, with_disc=with_disc,
               reference_over_sampler=out["reference"]["median_ms"] / out["sampler"]["median_ms"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mb", type=int, nargs="*", default=[98_304, 102_400, 393_216])
    ap.add_argument("--ring-rows", type=int, default=1_000_000)
    ap.add_argument("--preload-rows", type=int, default=2_000_000)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--minibatches", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--with-disc", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("amp_update_timing.py needs a CUDA device")
    dev = torch.device("cuda:0")
    rb, ld, norm = _setup(args.ring_rows, args.preload_rows, dev)
    res = {"device": torch.cuda.get_device_name(), "power_limit_w": power_limit_w(), "peak_gbs": PEAK_GBS,
           "ring_rows": args.ring_rows, "preload_rows": args.preload_rows,
           "launch": [measure_launch(rb, ld, norm, mb, args.launches, args.repeats) for mb in args.mb],
           "update": [measure_update(rb, ld, norm, mb, args.minibatches, args.rounds, False) for mb in args.mb]}
    if args.with_disc:
        res["update_with_disc"] = [measure_update(rb, ld, norm, mb, args.minibatches, args.rounds, True) for mb in args.mb]
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

"""Per-phase cycle breakdown of the simulation loop (needs a -DMZ_PHASE_TIMERS build: make -C muzero.jl_b200/csrc -B EXTRA=-DMZ_PHASE_TIMERS)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from muzero_jl_b200 import capi

G, S = 4096, 50
names = ["select", "stage", "-", "network(+wait)", "-", "hidden write(+wait)", "expand", "backup"]
for mode, label in ((capi.NN_FP32_EXACT, "fp32_exact"), (capi.NN_BF16_TC, "bf16_tcgen05"), (capi.NN_SPLIT_MMA, "split_mma")):
    ctx = capi.Context(capi.default_config(num_slots=G, num_iters=S, replay_buffer_size=10000, nn_mode=mode))
    ctx.init_weights(1337)
    ctx.self_play(0, G, 1.0)
    sims, moves = ctx.self_play(G, G, 1.0)
    raw = ctx.phase_cycles().astype(float)
    pc = raw[28:46].reshape(2, 9)
    for g, who in ((0, "thread 0 (tree lane / prediction group)"), (1, "thread 128 (dynamics group)")):
        n = pc[g, 8]; rounds = n * S
        if n == 0:
            print(label, who, "no timers in this build"); continue
        tot = pc[g, :8].sum()
        nm = list(names)
        if mode == capi.NN_SPLIT_MMA:      # with a dynamics tail the hidden state is written by the tail team; the workers wait for it before staging
            nm[5] = "tail-done wait + hidden write"
        print("%s %s: %.0f cycles/round; " % (label, who, tot / rounds) + ", ".join("%s %.0f" % (nm[i], pc[g, i] / rounds) for i in range(8) if nm[i] != "-"))
    for o, who in ((12, 'issuing thread, group 0'), (20, 'epilogue thread, group 1')):
        q = raw[o + 6]
        if q > 0:
            lab = ['issue', 'mbarrier wait', 'tcgen05.ld', 'epilogue', 'fence.proxy.async', 'group barrier']
            if mode == capi.NN_SPLIT_MMA:      # epilogue threads only (the issuer is a warp of its own): wait for the MMAs, read, compute + store, fences, arrive
                lab = ['mbarrier wait', 'tcgen05.ld', 'epilogue', 'fences', 'bar.arrive', '-']
            print('%s TC round (%s): %.0f cycles; ' % (label, who, raw[o:o + 6].sum() / q) + ', '.join('%s %.0f' % (lab[i], raw[o + i] / q) for i in range(6)))
    if raw[56] > 0:   # split-precision kernel with a dynamics tail: the issuer of group 1 times each tail (its rounds + the hidden-state write)
        print('%s dynamics tail (off the chain; issuer warp, end of its chain rounds -> tail done): %.0f cycles' % (label, raw[55] / raw[56]))
    if raw[53] > 0:   # kernel-level stamps of thread 0 (split-precision kernel)
        ks = ['set-up', 'stage observations', 'representation', 'root prediction', 'root expansion + noise', 'simulation loop', 'move epilogue + teardown']
        print('%s whole kernel (thread 0, mean cycles per launch): ' % label + ', '.join('%s %.0f' % (ks[i], raw[46 + i] / raw[53]) for i in range(7)) + '; slowest CTA of any launch %.0f vs mean %.0f' % (raw[54], raw[46:53].sum() / raw[53]))
    ctx.close()

"""Timeline of the tcgen05 conv kernel's CTA 0 (tuning build with -DEXP_TRACE):
    python -c "from emphases_b200 import build; build.build(output='emphases_b200/exp_TRACE.so', extra_flags=['-DEXP_TRACE'])"
    EMPHASES_B200_LIB=$PWD/emphases_b200/exp_TRACE.so python tools/conv_trace.py
Events (clock64 of SM 0): 0/1 epilogue slot 0 waits for / sees mma_done, 2 its
operand stores are issued, 3 act_ready arrive; 4/5 MMA warp waits for / sees
act_ready[0], 6 slot 0's MMAs issued, 7 last slot's MMAs issued; 8 + s the
epilogue of slot s sees mma_done[s], i.e. slot s's MMAs have completed;
at the tile boundary of slot 0 (index = round): 12 the next tile's rows are
in registers, 14 the last layer's epilogue and pooling are done, 15 the slot's
warps passed their named barrier, 13 / 16 the next tile's operands are stored /
act_ready is arrived on.

Index = round * layers + layer.  The word decoder launched after the frame stack
writes the same buffer for its few rounds, so the medians skip the first rounds."""
import ctypes, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
import emphases_b200 as emphases
from emphases_b200 import engine, _lib

EVENTS, SLOTS, LAYERS = 17, 4, 7
lengths, times = bench.corpus_layout(3000, 1234)
state = bench.random_state(); emphases.configure(PRECISION='bf16')
model = emphases.Model(); model.load_state_dict(state); model = model.cuda().eval()
dev = torch.device('cuda', 0)
audio, offsets = bench.make_audio(lengths, 99, device=dev)
plan = engine.make_plan([(t, int(n)) for t, n in zip(times, lengths)], None, 'sum')
eng = emphases.get_engine(dev)
views = eng.upload_plan(plan)
for _ in range(3):
    eng.forward_packed(audio, plan, model.packed_weights(), method='sum',
                       location='intermediate', precision=emphases.precision_code(), views=views)
torch.cuda.synchronize()
lib = _lib.load()
host = np.zeros((EVENTS, 512), dtype=np.int64)
lib.emph_conv_trace_read.argtypes = [ctypes.c_void_p]
print('rc', lib.emph_conv_trace_read(host.ctypes.data))
t = host.astype(np.float64)
done = t[8:8 + SLOTS]

# layer steps i -> i + 1 of rounds 10 .. last complete round, all stamps present
last = int(np.max(np.nonzero(t[5])[0])) if t[5].any() else 0
steps = [i for i in range(10 * LAYERS, last)
         if t[5, i + 1] > t[5, i] > 0 and (done[:, i] > 0).all() and done[0, i + 1] > 0]
print('layer steps used:', len(steps), f'(indices {steps[0]} .. {steps[-1]})' if steps else '')


def median(values):
    values = [v for v in values if np.isfinite(v)]
    return float(np.median(values)) if values else float('nan')


epi = [i for i in steps if i % LAYERS != LAYERS - 1 and t[1, i] > 0 and t[3, i] > 0]
rows = [
    ('period (act_ready[0] seen -> next act_ready[0] seen)', [t[5, i + 1] - t[5, i] for i in steps]),
    ('MMA warp waits for act_ready[0]', [t[5, i] - t[4, i] for i in steps]),
    ("act_ready[0] seen -> slot 0's MMAs issued", [t[6, i] - t[5, i] for i in steps]),
    ("slots 1-3's MMAs issued", [t[7, i] - t[6, i] for i in steps]),
    ('slot 0 issued -> its mma_done seen', [done[0, i] - t[6, i] for i in steps]),
    ('epilogue: done seen -> operands stored', [t[2, i] - t[1, i] for i in epi]),
    ('epilogue: stored -> act_ready arrive', [t[3, i] - t[2, i] for i in epi]),
]
# the tensor pipe runs a slot's MMAs once they are issued and the previous
# slot's are done: slot s (s >= 1) runs from done[s-1] to done[s]; slot 0 of
# the next step starts at max(its issue, slot 3's done) and the pipe is idle
# from slot 3's done to slot 0's issue when that comes later
for s in range(1, SLOTS):
    rows.append((f"slot {s}'s 15 MMAs: done[{s - 1}] -> done[{s}]",
                 [done[s, i] - done[s - 1, i] for i in steps]))
rows.append(("slot 0's 15 MMAs: max(issue, done[3] before) -> done[0]",
             [done[0, i + 1] - max(t[5, i + 1], done[SLOTS - 1, i]) for i in steps]))
rows.append(('tensor pipe idle: done[3] -> next act_ready[0] seen',
             [max(0., t[5, i + 1] - done[SLOTS - 1, i]) for i in steps]))
print('| per layer step (clk, median) | value |')
print('|---|---|')
for name, values in rows:
    print(f'| {name} | {median(values):.0f} |')
period = median(rows[0][1])
idle = median(rows[-1][1])
busy = period - idle
print(f'pipe busy {busy:.0f} of {period:.0f} clk per step -> {busy / (SLOTS * 15):.1f} clk per pair MMA '
      f'while busy, {period / (SLOTS * 15):.1f} over the whole step')
# the step that crosses into the next tile (last layer, pooling, the next
# tile's rows) against the steps inside a tile
print('| step from layer (clk) | median period | median act_ready[0] wait | median pipe idle |')
print('|---|---|---|---|')
for layer in range(LAYERS):
    at = [i for i in steps if i % LAYERS == layer]
    print(f'| {layer} -> {layer + 1 if layer + 1 < LAYERS else "next tile 0"} | '
          f'{median([t[5, i + 1] - t[5, i] for i in at]):.0f} | '
          f'{median([t[5, i + 1] - t[4, i + 1] for i in at]):.0f} | '
          f'{median([max(0., t[5, i + 1] - done[SLOTS - 1, i]) for i in at]):.0f} |')
if steps:
    span = t[5, steps[-1] + 1] - t[5, steps[0]]
    print(f'mean period {span / len(steps):.0f} clk over {len(steps)} steps')

# the tile boundary of slot 0, round r -> r + 1
bounds = [r for r in range(10, last // LAYERS - 1)
          if t[12, r] > 0 and t[13, r + 1] > 0 and t[16, r + 1] > 0 and t[5, (r + 1) * LAYERS] > 0]
parts = [
    ('layer 5 act_ready arrive -> next tile rows fetched', lambda r: t[12, r] - t[3, r * LAYERS + LAYERS - 2]),
    ('rows fetched -> last layer mma_done seen', lambda r: done[0, r * LAYERS + LAYERS - 1] - t[12, r]),
    ('mma_done seen -> last layer epilogue + pooling done', lambda r: t[14, r] - done[0, r * LAYERS + LAYERS - 1]),
    ('-> named barrier of the slot passed', lambda r: t[15, r] - t[14, r]),
    ("-> next tile's operands stored", lambda r: t[13, r + 1] - t[15, r]),
    ('-> act_ready arrive', lambda r: t[16, r + 1] - t[13, r + 1]),
    ('-> MMA warp sees act_ready[0]', lambda r: t[5, (r + 1) * LAYERS] - t[16, r + 1]),
]
print(f'| tile boundary of slot 0 (clk, median over {len(bounds)} rounds) | value |')
print('|---|---|')
for name, f in parts:
    print(f'| {name} | {median([f(r) for r in bounds]):.0f} |')

"""A small run of every hot entry point for compute-sanitizer (memcheck / racecheck / initcheck):
   compute-sanitizer --tool memcheck python tools/sanitize_small.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from tarok_b200.env import TarokEnv, pack_records

n = int(sys.argv[1]) if len(sys.argv) > 1 else 5000
env = TarokEnv(n, seed=3, history=True)
for mode in (16, 17, 0):
    env.rollout(mode, first_game_id=10)            # graph-backed
    env.rollout(mode, first_game_id=11)            # odd id: no draw cache
    env.set_graph(False); env.rollout(mode, first_game_id=12); env.set_graph(True)
    env.rollout(mode, first_game_id=12, fused=True)
env.deal(0)
perm = env.export_perm().cpu().numpy()
c = np.full(n, 3, np.uint8); d = (np.arange(n) & 3).astype(np.uint8); k = (np.arange(n) % 4).astype(np.uint8)
rec, bad = pack_records(perm, c, d, k, threads=2)
sc = torch.empty((n, 4), dtype=torch.int16).pin_memory(); st = torch.zeros(32, dtype=torch.int64).pin_memory()
env.rollout_host(perm, c, d, k, sc, st, fused=True); torch.cuda.synchronize(); a = sc.numpy().copy()
env.rollout_records(rec, sc, st); torch.cuda.synchronize(); assert (sc.numpy() == a).all()
env.rollout_host_packed(perm, c, d, k, sc, st, threads=2); torch.cuda.synchronize(); assert (sc.numpy() == a).all()
env.rollout_host(perm, c, d, k, sc, st, fused=False); torch.cuda.synchronize(); assert (sc.numpy() == a).all()
env.close()
from tarok_b200.samoigra import Samoigra
s = Samoigra(512, device=0, seed=1, random_card=[0.1] * 4)
s.odigraj(0); s.zapri()
s = Samoigra(512, device=0, seed=1, random_card=[0.1] * 4, boti=(2, 3))    # tarok_auction_bots / _exchange_bots / _step_bots
s.odigraj(1); s.zapri()
torch.cuda.synchronize()
print("sanitize_small ok")

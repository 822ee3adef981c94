"""Two neural players against two Bot_igralec players at 65,536 envs: the usual yardstick of a self-play net is its score
against uniform-random players.  Players 0 and 1 run their nets; players 2 and 3 are bots whose bids, king call, exchange
and cards are drawn in-kernel.  Prints the score sum of every player (stats[4 + p]) per rollout, and after a training pass
of the neural players."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tarok_b200.samoigra import Samoigra

if __name__ == "__main__":
    n = 65536
    s = Samoigra(n, seed=1, random_card=0.05, boti=(2, 3))
    for it in range(3):
        stats, _ = s.odigraj(first_game_id=it * n)
        print("rollout", it, "score sum by player (neural 0, 1 | bots 2, 3):", stats[4:8].tolist(),
              "finished", int(stats[18]), "errors", int(stats[20]))
        s.nauci(first_game_id=it * n)
    s.zapri()

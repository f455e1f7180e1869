"""Simpler round-2 variant: integer cut on level k11 == 1 only.
  c1* = smallest colB such that at least k strongly-positive k11==1 cells have colB <= c1*   (pure integer prefix scan)
  level-1 strong cells with colB > c1* cannot be in the top-k (LLR strictly decreasing in colB) -> never evaluated;
  every other cell is evaluated as today.  Exact."""
import sys
sys.path.insert(0, __import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.dirname(__import__('os').path.abspath(__file__)))))
from select_model import llr, brute, random_row
import random

def level1_cut(cells, ra, N, k, min_llr, item, self_, Cmax=1024, stats=None):
    hist = [0] * Cmax
    def strong1(b, k11, cb):
        return k11 == 1 and cb < Cmax and 2 * ra * cb < N and not (self_ and b == item)
    for b, k11, cb in cells:
        if strong1(b, k11, cb): hist[cb] += 1
    cut, cum = None, 0
    for c in range(Cmax):
        cum += hist[c]
        if cum >= k:
            cut = c
            break
    out, evals = [], 0
    for b, k11, cb in cells:
        if self_ and b == item: continue
        if cut is not None and strong1(b, k11, cb) and cb > cut: continue      # integer test only
        v = llr(k11, ra, cb, N); evals += 1
        if min_llr is not None and not v >= min_llr: continue
        if v > 0: out.append((-v, b, k11))
    out.sort()
    if stats is not None:
        stats['evals'] = stats.get('evals', 0) + evals; stats['cells'] = stats.get('cells', 0) + len(cells)
    return [(b, -nv, k11) for nv, b, k11 in out[:k]]

if __name__ == '__main__':
    rng = random.Random(11)
    for t in range(3000):
        cells, ra, N = random_row(rng)
        k = rng.choice([1, 5, 50, 50, 200]); min_llr = rng.choice([None, None, 0.5, 5.0])
        item = rng.randrange(0, 5000); self_ = rng.random() < 0.3
        assert brute(cells, ra, N, k, min_llr, item, self_) == level1_cut(cells, ra, N, k, min_llr, item, self_), t
    print('3000 random rows identical')

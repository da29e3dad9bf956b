import sys, os, numpy as np
a, b = sys.argv[1], sys.argv[2]
fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
assert fa == fb, (fa, fb)
bad = [f for f in fa if not np.array_equal(np.load(os.path.join(a, f)), np.load(os.path.join(b, f)))]
print("dump files", len(fa), "differing", bad)

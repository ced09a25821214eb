# CPU convolutions and matrix products (oneDNN / MKL) split their sums by the number of intra-op threads, so
# the CPU oracle's last bits depend on it: tests/golden/ was generated with this many, and the tests use it too.
GOLDEN_THREADS = 8

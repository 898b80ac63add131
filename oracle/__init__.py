"""CPU oracle for the batched env engine -- TEST INFRASTRUCTURE, never a product path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import, call, link or execute anything in this package.  The product package
(custom_gymnasium_environments_b200) never imports it and fails loudly when its CUDA
library is missing.

Contents
  philox.py        the engine's counter-based RNG contract, restated in numpy
  replay.py        ReplayRandom: feeds that stream into the reference's module-level `random`
  ref_loader.py    imports the UNMODIFIED reference from /root/reference behind stub
                   gymnasium/pygame modules (build container only; the reference cannot travel)
  snake_port.py    pure-Python restatement of SnakeEnvClassic (the CPU-baseline "port")
  c/               plain-C restatement (fast checker for GPU-scale parity), built into oracle/_c/
  gen_golden.py    drives the real reference and writes tests/golden/*.npz
  golden_files.py  reads and writes tests/golden/*.npz (one env's vectors split over files of at most 1 MB)

Parity pin: the reference holds no golden vectors (SURVEY.md section 4: zero asserts).
The pin is tests/golden/*.npz, produced by gen_golden.py from the reference itself run
in the build container; every oracle restatement is checked against those files.
"""

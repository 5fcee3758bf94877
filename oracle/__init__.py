"""
oracle/ -- TEST INFRASTRUCTURE ONLY.

CPU restatement of the genesis-forge manager step (the path named by BASELINE.json's north_star)
plus the harness that runs the UNMODIFIED reference package from /root/reference under stub
third-party modules.  Nothing in the product package (genesis_forge_b200/) imports from here; only
tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs do, and there
only as the checker or the timed CPU baseline -- never as the thing shipped.

Modules
-------
geom.py           restated genesis.utils.geom arithmetic (third-party, PARITY UNPINNED, see header)
shim.py           stub modules (genesis, gstaichi, gymnasium, tensordict, hid, skrl) so that the
                  unmodified reference imports in a container without Genesis
ref_harness.py    builds the reference's own ManagedEnvironment + managers from a term-table spec
                  (needs /root/reference; used here to pin the port and to generate tests/golden/)
manager_port.py   the oracle proper: torch-CPU, op-for-op restatement of the reference managers,
                  driven by the same term-table spec; travels to the GPU box
specs.py          the five BASELINE.json configs as term-table specs
make_golden.py    regenerates tests/golden/ from the unmodified reference; load() reads a trace
"""

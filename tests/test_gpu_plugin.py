"""GPU tests of the drop-in boundary proper: the B200 Platform plugin (libOpenMMB200.so, plugin/) loaded into the
UNMODIFIED reference OpenMM (oracle/_ref/libOpenMM.so) through Platform::loadPluginLibrary, driven through the
reference's public API (System / NonbondedForce / Context / LangevinIntegrator), compared with the Reference platform
in the same process -- plus the reference's own test bodies (tests/Test<X>.h) built against the B200 platform."""
import os
import subprocess
import numpy as np
import pytest
from conftest import relative_force_error, ROOT

pytestmark = pytest.mark.gpu
PLUGIN = os.path.join(ROOT, "oracle", "_ref", "plugins", "libOpenMMB200.so")
REFTESTS = os.path.join(ROOT, "oracle", "_ref", "tests")


@pytest.fixture(scope="module")
def omm():
    from oracle import omm
    if not omm.available() or not os.path.exists(PLUGIN):
        pytest.fail("oracle/_ref or the plugin is not built: run __graft_entry__.build() where the reference sources exist")
    omm.load_plugin(PLUGIN)
    assert "B200" in omm.platforms()
    return omm


def test_plugin_forces_energy_match_reference_platform(omm):
    from openmm_b200 import systems
    for d in (systems.water_box(7, cutoff=0.9).rounded(), systems.water_box(7, cutoff=0.9, rigid=False).rounded(),
              systems.random_ions(894, 3.0, cutoff=1.0, triclinic=True).rounded(), systems.cluster(70).rounded()):
        pme = d.pme_parameters() if d.method == systems.NB_PME else None
        a = omm.Simulation(d, "B200", pme=pme)
        b = omm.Simulation(d, "Reference", pme=pme)
        assert a.platform() == "B200"
        fa, ea = a.forces_energy()
        fb, eb = b.forces_energy()
        assert relative_force_error(fa, fb) < 1e-4
        assert abs(ea - eb)/max(1.0, abs(eb)) < 1e-4
        if pme is not None:
            assert a.pme_parameters()[1:] == tuple(pme[1:])


def test_plugin_force_groups_direct_vs_reciprocal(omm):
    from openmm_b200 import systems
    d = systems.water_box(7, cutoff=0.9).rounded()
    pme = d.pme_parameters()
    a = omm.Simulation(d, "B200", pme=pme, recip_group=1)
    b = omm.Simulation(d, "Reference", pme=pme, recip_group=1)
    ftot = b.forces_energy(3)[0]
    scale = np.maximum(1.0, np.linalg.norm(ftot, axis=1))[:, None]
    for groups in (1, 2, 3):
        fa, ea = a.forces_energy(groups)
        fb, eb = b.forces_energy(groups)
        # each group against the reference's SAME group; the error is measured on the scale of the TOTAL force of
        # the atom (the reciprocal part alone is a small difference of large fp32 grid terms)
        assert np.abs((fa - fb)/scale).max() < 1e-4 and abs(ea - eb)/max(1.0, abs(eb)) < 1e-4


def test_plugin_langevin_dynamics_and_constraints(omm):
    from openmm_b200 import systems
    d = systems.water_box(8, cutoff=0.9).rounded()
    sim = omm.Simulation(d, "B200", integrator=(systems.INT_LANGEVIN, 300.0, 2.0, 0.002), pme=d.pme_parameters())
    sim.set_velocities_to_temperature(300.0, 3)
    sim.step(400)
    st = sim.state(positions=True, energy=True)
    x = st["positions"]
    for i, j, dist in zip(d.con_i[::5], d.con_j[::5], d.con_d[::5]):
        assert abs(np.linalg.norm(x[i]-x[j]) - dist) < 1e-5
    dof = 3*d.natoms - len(d.con_i)
    T = 2*st["kinetic"]/(dof*0.00831446261815324)
    assert 250 < T < 350
    assert abs(sim.L.omm_context_get_time(sim.ctx) - 0.8) < 1e-9


def test_plugin_deterministic_verlet_follows_reference(omm):
    from openmm_b200 import systems
    d = systems.water_box(6, cutoff=0.9).rounded()
    v = np.random.default_rng(3).standard_normal((d.natoms, 3))*0.3
    a = omm.Simulation(d, "B200", integrator=(systems.INT_VERLET, 0, 0, 0.001), pme=d.pme_parameters())
    b = omm.Simulation(d, "Reference", integrator=(systems.INT_VERLET, 0, 0, 0.001), pme=d.pme_parameters())
    for s in (a, b):
        s.set_velocities(v)
        s.step(10)
    sa, sb = a.state(positions=True, energy=True), b.state(positions=True, energy=True)
    assert np.abs(sa["positions"] - sb["positions"]).max() < 5e-6
    assert abs(sa["potential"] - sb["potential"])/abs(sb["potential"]) < 1e-4
    assert abs(sa["kinetic"] - sb["kinetic"])/sb["kinetic"] < 1e-3


def test_plugin_checkpoint(omm):
    from openmm_b200 import systems
    d = systems.water_box(5, cutoff=0.75).rounded()
    sim = omm.Simulation(d, "B200", integrator=(systems.INT_LANGEVIN, 300.0, 1.0, 0.002), pme=d.pme_parameters())
    sim.step(5)
    sim.checkpoint_roundtrip()
    sim.step(5)
    assert np.isfinite(sim.state(positions=True)["positions"]).all()


REFERENCE_TEST_BINARIES = ["TestB200NonbondedForce", "TestB200Ewald", "TestB200Settle", "TestB200LangevinIntegrator", "TestB200LangevinMiddleIntegrator",
                           "TestB200VerletIntegrator", "TestB200HarmonicBondForce", "TestB200HarmonicAngleForce", "TestB200PeriodicTorsionForce",
                           "TestB200CMMotionRemover", "TestB200LocalEnergyMinimizer"]


@pytest.mark.parametrize("name", REFERENCE_TEST_BINARIES)
def test_reference_own_test_bodies_pass_on_b200_platform(name):
    """tests/Test<X>.h of the reference compiled against our platform (plugin/tests/shim.cpp lists which functions)."""
    exe = os.path.join(REFTESTS, name)
    if not os.path.exists(exe):
        pytest.fail("%s not built (make -C plugin reftests where the reference sources exist)" % exe)
    env = dict(os.environ, B200_PLUGIN=PLUGIN)
    for attempt in range(2):
        # the reference's statistical assertions (ASSERT_USUALLY_*: "This test is stochastic and may occasionally fail")
        # get one rerun, as devtools/run-ctest.py:86-118 does for the reference's own CI
        p = subprocess.run([exe], capture_output=True, text=True, timeout=600, env=env)
        if p.returncode == 0 and "Done" in p.stdout:
            break
        if "stochastic" not in p.stdout:
            break
    assert p.returncode == 0 and "Done" in p.stdout, p.stdout[-2000:] + p.stderr[-2000:]


_PME_HOOK_SCRIPT = r"""
import sys, os, ctypes, numpy as np
root = os.environ["B200MD_ROOT"]
sys.path.insert(0, root)
from openmm_b200 import systems
from oracle import omm
omm.load_plugin(os.path.join(root, "oracle", "_ref", "libOpenMMCPU.so"))
plug = os.path.join(root, "oracle", "_ref", "plugins", "libOpenMMB200Pme.so")
omm.load_plugin(plug)                         # registers "CalcPmeReciprocalForce" on the Reference and CPU platforms
count = ctypes.CDLL(plug).b200pme_exec_count
count.restype = ctypes.c_long
d = systems.water_box(9, cutoff=0.9).rounded()
pme = d.pme_parameters()
ref = omm.Simulation(d, "Reference", pme=pme, recip_group=1)
cpu = omm.Simulation(d, "CPU", pme=pme, recip_group=1)
n0 = count()
fc, ec = cpu.forces_energy(2)                 # reciprocal-space group only
n1 = count()
fr, er = ref.forces_energy(2)
err = np.abs(fc - fr).max(axis=1)/np.maximum(1.0, np.linalg.norm(fr, axis=1))
ft, et = cpu.forces_energy(3)                 # everything: CPU platform direct space + our reciprocal space
frt, ert = ref.forces_energy(3)
errt = np.abs(ft - frt).max(axis=1)/np.maximum(1.0, np.linalg.norm(frt, axis=1))
print("RESULT", n1 - n0, err.max(), abs(ec - er)/abs(er), errt.max(), abs(et - ert)/abs(ert))
"""


@pytest.mark.gpu
def test_standalone_pme_kernel_serves_the_reference_cpu_platform():
    """SURVEY.md 8f rank 3: libOpenMMB200Pme.so (plugin/B200PmePlugin.cpp) registers a "CalcPmeReciprocalForce" kernel (kernels.h:1493-1557, the
    plugins/cpupme pattern).  The UNMODIFIED reference CPU platform then routes reciprocal space through the bespoke
    spread / FFT / convolution / gather (CpuKernels.cpp:620-690) and must still agree with the Reference platform."""
    import sys
    from conftest import ROOT
    env = dict(os.environ, B200MD_ROOT=ROOT)
    out = subprocess.run([sys.executable, "-c", _PME_HOOK_SCRIPT], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    served, ferr, eerr, ferr_all, eerr_all = [l for l in out.stdout.splitlines() if l.startswith("RESULT")][0].split()[1:]
    msg = out.stdout[-400:]
    assert int(served) >= 1, msg               # the hook was taken: our kernel computed the CPU platform's reciprocal space
    # the reciprocal-space force alone is a few kJ/mol/nm per atom in this box, so its floor-1 relative error is the
    # absolute error of the fp32 spectral pipeline (measured 3.9e-4); against the total force it is 3e-6
    assert float(ferr) < 1e-3 and float(eerr) < 1e-7, msg
    assert float(ferr_all) < 1e-4 and float(eerr_all) < 1e-5, msg


def test_cpp_host_application_loads_system_xml_and_pdb(omm, tmp_path):
    """SURVEY.md 8(f) rank 1: a C++ program that uses only the reference's public API (XmlSerializer::deserialize<System>,
    a PDB reader, Platform::loadPluginLibrary, Context, LangevinIntegrator::step) runs the real DHFR System on the B200
    platform (plugin/examples/run_system_xml.cpp)."""
    import json
    import sys
    exe = os.path.join(REFTESTS, "run_system_xml")
    if not os.path.exists(exe):
        pytest.fail("run_system_xml not built (make -C plugin reftests where the reference sources exist)")
    base = str(tmp_path/"dhfr")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "make_system_xml.py"), "dhfr", base], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe, base + ".xml", base + ".pdb", "--plugin", PLUGIN, "--steps", "1000"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stdout + r.stderr
    j = json.loads(r.stdout.strip().splitlines()[-1])
    assert j["platform"] == "B200" and j["atoms"] == 23558
    assert j["ns_per_day"] > 200 and -4.5e5 < j["potential_after"] < -2.0e5


def test_fused_step_graph_through_integrator_step_equals_the_two_call_path(omm):
    """Integrator::step on the plugin replays ONE captured step graph per step (lazy forces + b200md_step, B200Platform.cpp
    integrateStep); B200MD_PLUGIN_FUSED=0 selects b200md_compute + b200md_integrate_only.  Same trajectory either way, and
    getState in between (which flushes the lazy evaluation) must not disturb it."""
    from openmm_b200 import systems
    d = systems.water_box(6, cutoff=0.9).rounded()
    v = np.random.default_rng(4).standard_normal((d.natoms, 3))*0.3
    out = []
    for fused in ("1", "0"):
        os.environ["B200MD_PLUGIN_FUSED"] = fused
        sim = omm.Simulation(d, "B200", integrator=(systems.INT_VERLET, 0, 0, 0.001), pme=d.pme_parameters())
        sim.set_velocities(v)
        sim.step(7)
        f_mid = sim.state(forces=True, energy=True)
        sim.step(13)
        st = sim.state(positions=True, velocities=True, energy=True)
        out.append((st["positions"], st["velocities"], f_mid["forces"], f_mid["potential"]))
        sim.close()
    os.environ.pop("B200MD_PLUGIN_FUSED", None)
    assert np.abs(out[0][0] - out[1][0]).max() < 2e-6
    assert np.abs(out[0][2] - out[1][2]).max() < 1e-3*np.abs(out[1][2]).max() and abs(out[0][3] - out[1][3]) < 1e-6*abs(out[1][3])


def test_context_falls_back_when_the_system_is_not_supported(omm):
    """ContextImpl only falls back to the next platform when contextCreated() throws (ContextImpl.cpp:152-166): a System the
    B200 platform cannot run (Ewald summation here) must be refused THERE, so that a Context without an explicit platform is
    still created (on the Reference platform in this process), and an explicit B200 request fails with a clear message."""
    from openmm_b200 import systems
    d = systems.random_ions(64, 2.5, cutoff=1.0).rounded()
    d.method = 3                                   # NonbondedForce::Ewald
    with pytest.raises(RuntimeError, match="B200 platform"):
        omm.Simulation(d, "B200")

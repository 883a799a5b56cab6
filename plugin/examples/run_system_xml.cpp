// run_system_xml.cpp -- a C++ host application for the real benchmark Systems (SURVEY.md 8(f) rank 1).
//
// What a C++ user of the reference does to run DHFR / ApoA1 on this platform, with nothing but the reference's public
// API: load the System with XmlSerializer::deserialize<System> (serialization/include/openmm/serialization/
// XmlSerializer.h), read the coordinates from a PDB file, load the plugin, create a Context on the "B200" platform and
// call LangevinIntegrator::step.  The System XML is what `XmlSerializer::serialize<System>` writes -- e.g. from
// openmm.app's ForceField.createSystem; tools/make_system_xml.py produces data-equivalent files from data/*.npz (built by
// the reference's own forcefield.py, tools/make_benchmark_systems.py).
//
//   run_system_xml system.xml structure.pdb [--platform B200] [--plugin oracle/_ref/plugins/libOpenMMB200.so] [--steps 2000]
//                  [--dt 0.002] [--temperature 300] [--friction 1] [--device 0]
// prints one JSON line: atoms, platform, ns/day, potential energy before / after.
#include "openmm/Platform.h"
#include "openmm/System.h"
#include "openmm/Context.h"
#include "openmm/State.h"
#include "openmm/LangevinIntegrator.h"
#include "openmm/OpenMMException.h"
#include "openmm/serialization/XmlSerializer.h"
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>
#include <string>
#include <vector>

using namespace OpenMM;

// ATOM / HETATM records, columns 31-54 (x, y, z in Angstrom, PDB format 3.3); CRYST1 is ignored: the box is the System's
static std::vector<Vec3> readPdbPositions(const std::string& path) {
    std::ifstream in(path.c_str());
    if (!in) throw OpenMMException("cannot open " + path);
    std::vector<Vec3> pos;
    std::string line;
    while (std::getline(in, line)) {
        if (line.compare(0, 4, "ATOM") != 0 && line.compare(0, 6, "HETATM") != 0) { if (line.compare(0, 6, "ENDMDL") == 0) break; continue; }
        if (line.size() < 54) throw OpenMMException("short ATOM record in " + path);
        const double x = atof(line.substr(30, 8).c_str()), y = atof(line.substr(38, 8).c_str()), z = atof(line.substr(46, 8).c_str());
        pos.push_back(Vec3(0.1*x, 0.1*y, 0.1*z));
    }
    return pos;
}

int main(int argc, char** argv) {
    if (argc < 3) { fprintf(stderr, "usage: %s system.xml structure.pdb [--platform B200] [--plugin path] [--steps N] [--dt ps] [--temperature K] [--friction 1/ps] [--device i]\n", argv[0]); return 2; }
    std::map<std::string, std::string> opt = {{"--platform", "B200"}, {"--plugin", "oracle/_ref/plugins/libOpenMMB200.so"}, {"--steps", "2000"}, {"--dt", "0.002"},
                                              {"--temperature", "300"}, {"--friction", "1"}, {"--device", "0"}};
    for (int i = 3; i + 1 < argc; i += 2) opt[argv[i]] = argv[i+1];
    try {
        std::ifstream xml(argv[1]);
        if (!xml) throw OpenMMException(std::string("cannot open ") + argv[1]);
        System* system = XmlSerializer::deserialize<System>(xml);
        std::vector<Vec3> positions = readPdbPositions(argv[2]);
        if ((int) positions.size() != system->getNumParticles())
            throw OpenMMException("the PDB file has " + std::to_string(positions.size()) + " atoms, the System " + std::to_string(system->getNumParticles()));
        if (opt["--platform"] == "B200") Platform::loadPluginLibrary(opt["--plugin"]);
        Platform& platform = Platform::getPlatformByName(opt["--platform"]);
        std::map<std::string, std::string> props;
        if (opt["--platform"] == "B200") props["DeviceIndex"] = opt["--device"];
        const double dt = atof(opt["--dt"].c_str());
        LangevinIntegrator integrator(atof(opt["--temperature"].c_str()), atof(opt["--friction"].c_str()), dt);
        integrator.setRandomNumberSeed(7);
        Context context(*system, integrator, platform, props);
        context.setPositions(positions);
        context.applyConstraints(1e-6);
        context.setVelocitiesToTemperature(atof(opt["--temperature"].c_str()), 11);
        const double e0 = context.getState(State::Energy).getPotentialEnergy();
        const int steps = atoi(opt["--steps"].c_str());
        integrator.step(std::min(steps, 200));                       // warm-up (graph capture, list sizing)
        context.getState(State::Energy);
        const auto t0 = std::chrono::steady_clock::now();
        integrator.step(steps);
        const double e1 = context.getState(State::Energy).getPotentialEnergy();     // drains the device, as benchmark.py does
        const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        printf("{\"system\": \"%s\", \"atoms\": %d, \"platform\": \"%s\", \"steps\": %d, \"dt_fs\": %.3f, \"ns_per_day\": %.2f, \"us_per_step\": %.2f, "
               "\"potential_before\": %.3f, \"potential_after\": %.3f}\n", argv[1], system->getNumParticles(), context.getPlatform().getName().c_str(), steps,
               1e3*dt, dt*1e-3*steps*86400.0/sec, 1e6*sec/steps, e0, e1);
        delete system;
    }
    catch (const std::exception& e) { fprintf(stderr, "error: %s\n", e.what()); return 1; }
    return 0;
}

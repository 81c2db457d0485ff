// Compile-and-link check of bemb200::evaluate_field (include/bemb200.hpp).  The call is instantiated, never executed
// (argc is never > 100): its executable twin is bem.evaluate_field, which the GPU tests drive.
#include "bemb200.hpp"
using namespace bemb200;
int main(int argc, char**) {
    if (argc > 100) {
        std::vector<Element> elements;
        std::vector<double> nodes;
        PhysicsParams physics(100.0, 343.0, 1.21, false);
        Context ctx(0);
        StagedMesh mesh(ctx, elements, nodes);
        const std::vector<Complex64> p(mesh.num_dofs()), v;
        const std::vector<Complex64> f = evaluate_field(mesh, {0.0, 0.0, 1.0}, p, v, physics);
        return static_cast<int>(f.size());
    }
    return 0;
}

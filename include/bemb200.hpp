// bemb200.hpp -- C++17 host-side mirror of the reference's operator interface for the dense
// TBEM assemble + GMRES path, over the C ABI of bemb200.h (header only, no CUDA/torch types).
//
// The reference is Rust; where its toolchain is absent this header plays the role of the Rust
// shim (rust/bem-b200-sys): same names, argument meaning and error behaviour as
//   math-bem/src/core/types.rs:16-351            PhysicsParams, ElementType, BoundaryCondition, Element
//   math-bem/src/core/assembly/tbem.rs:13-101    TbemSystem, build_tbem_system{,_with_beta,_scaled,_bounded}
//   math-bem/src/core/assembly/tbem.rs:500-534   apply_row_sum_correction
//   math-bem/src/core/solver/fmm_interface.rs:25-52,378-384  DenseOperator, solve_gmres
//   math-solvers/src/traits.rs:316-385           LinearOperator, IdentityPreconditioner
//   math-solvers/src/preconditioners/diagonal.rs DiagonalPreconditioner
//   math-solvers/src/preconditioners/schwarz.rs  AdditiveSchwarzPreconditioner (built on the device from the operator)
//   math-solvers/src/iterative/gmres.rs:16-585   GmresConfig, GmresSolution, gmres, gmres_with_guess,
//                                                gmres_preconditioned{,_with_guess}
//   math-solvers/src/iterative/bicgstab.rs:19-215  BiCgstabConfig, BiCgstabSolution, bicgstab
//   math-solvers/src/iterative/cgs.rs:12-155       CgsConfig, CgsSolution, cgs (+ solve_cgs / solve_with_ilu wrappers)
//   math-solvers/src/direct/lu.rs:15-161         LuError, lu_solve
//   math-bem/src/core/incident.rs:19-342         IncidentField (plane waves / point sources), compute_rhs{,_with_beta}
//   math-bem/src/core/postprocess/pressure.rs:81-259,438-478  compute_scattered_field, compute_rcs
//   math-bem/src/room_acoustics/solver.rs:412-748  RoomMesh, Source, build_bem_matrix_parallel, solve_bem_system,
//                                                calculate_incident_field_derivative_parallel, calculate_field_pressure_bem_parallel
// Shape mismatches throw std::invalid_argument (the reference panics); library failures throw
// bemb200::Error carrying the BEMB200_E* code and bemb200_last_error().
#pragma once
#include <algorithm>
#include <cmath>
#include <complex>
#include <cstdint>
#include <exception>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "bemb200.h"

namespace bemb200 {

using Complex64 = std::complex<double>;
static_assert(sizeof(Complex64) == 2 * sizeof(double), "std::complex<double> must be two doubles");

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error("libbemb200 error " + std::to_string(c) + ": " + m), code(c) {}
};
inline void check(int rc, const bemb200_ctx* ctx = nullptr) {
    if (rc != BEMB200_OK) {
        const char* m = bemb200_last_error(ctx);
        if ((!m || !*m) && ctx) m = bemb200_last_error(nullptr);
        throw Error(rc, m ? m : "");
    }
}

// ---- types.rs -------------------------------------------------------------------------------
struct PhysicsParams {  // types.rs:16-58
    double speed_of_sound, density, frequency, wave_number, omega, wave_length, harmonic_factor, pressure_factor, tau;
    PhysicsParams(double frequency_, double speed_of_sound_, double density_, bool is_internal)
        : speed_of_sound(speed_of_sound_), density(density_), frequency(frequency_) {
        const double PI = 3.14159265358979323846264338327950288;
        omega = 2.0 * PI * frequency;
        wave_number = omega / speed_of_sound;
        wave_length = speed_of_sound / frequency;
        harmonic_factor = 1.0;
        pressure_factor = density * omega * harmonic_factor;
        tau = is_internal ? -1.0 : 1.0;
    }
    double gamma() const { return 1.0; }  // types.rs:216-218
    Complex64 burton_miller_beta() const { return tau > 0.0 ? Complex64(0.0, harmonic_factor / wave_number) : Complex64(0.0, 0.0); }
    Complex64 burton_miller_beta_scaled(double scale) const {
        return tau > 0.0 ? Complex64(0.0, harmonic_factor * scale / wave_number) : Complex64(0.0, 0.0);
    }
    Complex64 burton_miller_beta_optimal(double element_size) const {
        return tau > 0.0 ? Complex64(0.0, harmonic_factor / (wave_number + 1.0 / element_size)) : Complex64(0.0, 0.0);
    }
    std::pair<Complex64, double> burton_miller_beta_adaptive(double radius) const {  // types.rs:173-195
        if (tau <= 0.0) return {Complex64(0.0, 0.0), 1.0};
        const double ka = wave_number * radius;
        const double scale = ka < 0.5 ? 1.0 : (ka < 1.2 ? 4.0 : (ka < 1.8 ? 8.0 : 16.0));
        return {Complex64(0.0, harmonic_factor * scale / wave_number), scale};
    }
};

enum class ElementType { Tri3, Quad4 };
enum class ElementProperty { Surface = 0, MidFace = 1, Evaluation = 2 };

struct BoundaryCondition {  // types.rs:267-292 (the variants the assembly distinguishes, tbem.rs:234-244)
    enum Kind { Velocity, Pressure, VelocityWithAdmittance, TransferAdmittance, TransferWithSurfaceAdmittance } kind = Velocity;
    std::vector<Complex64> values{Complex64(0.0, 0.0)};
    static BoundaryCondition velocity(std::vector<Complex64> v) { return {Velocity, std::move(v)}; }
    static BoundaryCondition pressure(std::vector<Complex64> p) { return {Pressure, std::move(p)}; }
};

struct Element {  // types.rs:329-351
    std::vector<std::size_t> connectivity;
    ElementType element_type = ElementType::Tri3;
    ElementProperty property = ElementProperty::Surface;
    double normal[3] = {0, 0, 0};
    double center[3] = {0, 0, 0};
    double area = 0.0;
    BoundaryCondition boundary_condition;
    std::size_t group = 0;
    std::vector<std::size_t> dof_addresses;
};

// ---- device context -----------------------------------------------------------------------------
class Context {
public:
    explicit Context(int device = 0) { check(bemb200_ctx_create(device, &h_)); }
    Context(int device, int rank, int nranks, const uint8_t* nccl_id, void* cuda_stream = nullptr) {
        check(bemb200_ctx_create_ex(device, rank, nranks, nccl_id, cuda_stream, &h_));
    }
    ~Context() { bemb200_ctx_destroy(h_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    bemb200_ctx* handle() const { return h_; }
    // frequency-sweep controls (no counterpart in the reference: its sweep is a serial loop, bem_solver.rs:403-432)
    void set_background(int blocks_per_sm) { check(bemb200_ctx_set_background(h_, blocks_per_sm), h_); }
    void set_shared_gpu(bool shared) { check(bemb200_ctx_set_shared_gpu(h_, shared ? 1 : 0), h_); }
    bool peer_exchange_active() const {
        int a = 0;
        check(bemb200_ctx_peer_exchange_active(h_, &a), h_);
        return a != 0;
    }

private:
    bemb200_ctx* h_ = nullptr;
};

// ---- LinearOperator / DenseOperator -----------------------------------------------------------------
struct LinearOperator {  // math-solvers/src/traits.rs:316-364
    virtual ~LinearOperator() = default;
    virtual std::size_t num_rows() const = 0;
    virtual std::size_t num_cols() const = 0;
    virtual std::vector<Complex64> apply(const std::vector<Complex64>& x) const = 0;
    virtual std::vector<Complex64> apply_transpose(const std::vector<Complex64>& x) const = 0;
    virtual std::vector<Complex64> apply_hermitian(const std::vector<Complex64>& x) const {  // traits.rs:331-358
        std::vector<Complex64> xc(x.size());
        for (std::size_t i = 0; i < x.size(); ++i) xc[i] = std::conj(x[i]);
        std::vector<Complex64> y = apply_transpose(xc);
        for (auto& v : y) v = std::conj(v);
        return y;
    }
    bool is_square() const { return num_rows() == num_cols(); }
};

class DenseOperator : public LinearOperator {  // fmm_interface.rs:25-52, device resident
public:
    // DenseOperator::new(matrix): row-major n_rows x n_cols host matrix
    DenseOperator(const Context& ctx, const std::vector<Complex64>& matrix, std::size_t n_rows, std::size_t n_cols) : ctx_(&ctx) {
        if (matrix.size() != n_rows * n_cols) throw std::invalid_argument("DenseOperator: matrix size does not match its shape");
        check(bemb200_matrix_from_host(ctx.handle(), reinterpret_cast<const double*>(matrix.data()), n_rows, n_cols, 0, n_rows, &m_),
              ctx.handle());
    }
    DenseOperator(const Context& ctx, bemb200_matrix* owned) : ctx_(&ctx), m_(owned) {}
    ~DenseOperator() override { bemb200_matrix_free(m_); }
    DenseOperator(const DenseOperator&) = delete;
    DenseOperator& operator=(const DenseOperator&) = delete;
    std::size_t num_rows() const override { return bemb200_num_rows(m_); }
    std::size_t num_cols() const override { return bemb200_num_cols(m_); }
    std::vector<Complex64> apply(const std::vector<Complex64>& x) const override {
        if (x.size() != num_cols()) throw std::invalid_argument("apply: vector length does not match num_cols");
        std::vector<Complex64> y(num_rows());
        check(bemb200_apply(m_, reinterpret_cast<const double*>(x.data()), reinterpret_cast<double*>(y.data())), ctx_->handle());
        return y;
    }
    std::vector<Complex64> apply_transpose(const std::vector<Complex64>& x) const override {
        if (x.size() != num_rows()) throw std::invalid_argument("apply_transpose: vector length does not match num_rows");
        std::vector<Complex64> y(num_cols());
        check(bemb200_apply_transpose(m_, reinterpret_cast<const double*>(x.data()), reinterpret_cast<double*>(y.data())),
              ctx_->handle());
        return y;
    }
    std::vector<Complex64> rows(std::size_t row_begin, std::size_t row_end) const {  // device matrix -> host (row block)
        std::vector<Complex64> out((row_end - row_begin) * num_cols());
        check(bemb200_matrix_download(m_, row_begin, row_end, reinterpret_cast<double*>(out.data())), ctx_->handle());
        return out;
    }
    std::vector<Complex64> diagonal() const {
        std::vector<Complex64> d(num_rows());
        check(bemb200_matrix_diagonal(m_, reinterpret_cast<double*>(d.data())), ctx_->handle());
        return d;
    }
    bemb200_matrix* handle() const { return m_; }
    const Context& context() const { return *ctx_; }

private:
    const Context* ctx_;
    bemb200_matrix* m_ = nullptr;
};

// ---- TbemSystem / assembly ---------------------------------------------------------------------------
struct TbemSystem {  // tbem.rs:13-20; the matrix stays on the device behind the operator
    std::unique_ptr<DenseOperator> matrix;
    std::vector<Complex64> rhs;
    std::size_t num_dofs = 0;
};

// &[Element] + nodes flattened to the SoA arrays of `bemb200_mesh` (owns the storage the view points into)
struct MeshSoA {
    std::vector<uint32_t> conn, dof;
    std::vector<uint8_t> etype, bc_len, is_eval;
    std::vector<double> center, normal, area, bc_val;
    std::vector<int32_t> bc_type;
    std::size_t n_elem = 0, ndof = 0;
    // `nodes`: n_nodes x 3 row-major (Array2<f64>)
    MeshSoA(const std::vector<Element>& elements) {
        const std::size_t n = elements.size();
        n_elem = n;
        conn.assign(4 * n, 0xFFFFFFFFu); dof.assign(n, 0);
        etype.resize(n); bc_len.assign(n, 1); is_eval.assign(n, 0);
        center.resize(3 * n); normal.resize(3 * n); area.resize(n); bc_val.assign(8 * n, 0.0);
        bc_type.assign(n, 0);
        for (std::size_t i = 0; i < n; ++i) {
            const Element& e = elements[i];
            etype[i] = e.element_type == ElementType::Tri3 ? 3 : 4;
            if (e.connectivity.size() != etype[i]) throw std::invalid_argument("element connectivity does not match its type");
            for (std::size_t v = 0; v < e.connectivity.size(); ++v) conn[4 * i + v] = static_cast<uint32_t>(e.connectivity[v]);
            for (int d = 0; d < 3; ++d) { center[3 * i + d] = e.center[d]; normal[3 * i + d] = e.normal[d]; }
            area[i] = e.area;
            // get_bc_type_and_value(): tbem.rs:234-244
            const BoundaryCondition& bc = e.boundary_condition;
            std::vector<Complex64> vals;
            switch (bc.kind) {
                case BoundaryCondition::Velocity: case BoundaryCondition::VelocityWithAdmittance: bc_type[i] = 0; vals = bc.values; break;
                case BoundaryCondition::Pressure: bc_type[i] = 1; vals = bc.values; break;
                default: bc_type[i] = 2; vals = {Complex64(0.0, 0.0)}; break;
            }
            if (vals.empty() || vals.size() > 4) throw std::invalid_argument("boundary condition needs 1..4 values");
            bc_len[i] = static_cast<uint8_t>(vals.size());
            for (std::size_t k = 0; k < vals.size(); ++k) { bc_val[8 * i + 2 * k] = vals[k].real(); bc_val[8 * i + 2 * k + 1] = vals[k].imag(); }
            is_eval[i] = e.property == ElementProperty::Evaluation;
            if (!is_eval[i]) {
                if (e.dof_addresses.empty()) throw std::invalid_argument("boundary element without dof address");
                dof[i] = static_cast<uint32_t>(e.dof_addresses[0]);
                ++ndof;
            }
        }
    }
    bemb200_mesh view(const std::vector<double>& nodes) const {
        return bemb200_mesh{nodes.size() / 3, n_elem, nodes.data(), conn.data(), etype.data(), center.data(), normal.data(), area.data(),
                            bc_type.data(), bc_len.data(), bc_val.data(), dof.data(), is_eval.data()};
    }
};
inline bemb200_physics physics_abi(const PhysicsParams& p) { return bemb200_physics{p.wave_number, p.harmonic_factor, p.tau, p.gamma()}; }

inline TbemSystem tbem_system_from_handle(const Context& ctx, bemb200_matrix* m, std::size_t ndof) {
    TbemSystem sys;
    sys.matrix = std::make_unique<DenseOperator>(ctx, m);
    sys.num_dofs = ndof;
    sys.rhs.resize(ndof);
    check(bemb200_rhs_download_full(m, reinterpret_cast<double*>(sys.rhs.data())), ctx.handle());
    return sys;
}

// `nodes`: n_nodes x 3 row-major (Array2<f64>)
inline TbemSystem build_tbem_system_with_beta(const Context& ctx, const std::vector<Element>& elements,
                                              const std::vector<double>& nodes, const PhysicsParams& physics, Complex64 beta) {
    const MeshSoA soa(elements);
    const bemb200_mesh mesh = soa.view(nodes);
    const bemb200_physics phys = physics_abi(physics);
    bemb200_matrix* m = nullptr;
    check(bemb200_assemble(ctx.handle(), &mesh, &phys, beta.real(), beta.imag(), 0, soa.ndof, &m), ctx.handle());
    return tbem_system_from_handle(ctx, m, soa.ndof);
}

// Frequency-independent device copy of the mesh: staged once, reused by every frequency of a sweep and by the
// right-hand-side / field kernels below (no counterpart in the reference, which re-reads `&[Element]` per call).
class StagedMesh {
public:
    StagedMesh(const Context& ctx, const std::vector<Element>& elements, const std::vector<double>& nodes) : ctx_(&ctx) {
        const MeshSoA soa(elements);
        const bemb200_mesh mesh = soa.view(nodes);
        check(bemb200_mesh_stage(ctx.handle(), &mesh, &h_), ctx.handle());
        num_dofs_ = soa.ndof;
        // DOF address of the j-th non-evaluation element; left empty for the sequential map of every generator
        bool sequential = true;
        std::vector<uint32_t> map;
        std::vector<uint8_t> seen(soa.ndof, 0);
        bool permutation = true;
        for (std::size_t i = 0; i < soa.n_elem; ++i) {
            if (soa.is_eval[i]) continue;
            const uint32_t d = soa.dof[i];
            sequential = sequential && d == map.size();
            if (d >= soa.ndof || seen[d]) permutation = false; else seen[d] = 1;
            map.push_back(d);
        }
        if (!sequential && permutation) enum_to_dof_ = std::move(map);
    }
    // A surface vector as the reference takes it (entry j belongs to the j-th non-evaluation element, pressure.rs:96-113,
    // 452-458) re-addressed to the DOF order of the C ABI; the identity for sequential DOF maps.
    std::vector<Complex64> in_dof_order(const std::vector<Complex64>& values) const {
        if (enum_to_dof_.empty()) return values;
        std::vector<Complex64> out(values.size());
        for (std::size_t j = 0; j < values.size(); ++j) out[enum_to_dof_[j]] = values[j];
        return out;
    }
    ~StagedMesh() { bemb200_staged_mesh_free(h_); }
    StagedMesh(const StagedMesh&) = delete;
    StagedMesh& operator=(const StagedMesh&) = delete;
    bemb200_staged_mesh* handle() const { return h_; }
    const Context& context() const { return *ctx_; }
    std::size_t num_dofs() const { return num_dofs_; }
    double dg_dn_sign(double wave_number) const { return bemb200_dg_dn_sign(h_, wave_number); }  // tbem.rs:108-123

private:
    const Context* ctx_;
    bemb200_staged_mesh* h_ = nullptr;
    std::size_t num_dofs_ = 0;
    std::vector<uint32_t> enum_to_dof_;
};
// build_tbem_system_with_beta on a staged mesh (all rows)
inline TbemSystem build_tbem_system_with_beta(const StagedMesh& mesh, const PhysicsParams& physics, Complex64 beta) {
    const bemb200_physics phys = physics_abi(physics);
    bemb200_matrix* m = nullptr;
    check(bemb200_assemble_staged(mesh.context().handle(), mesh.handle(), &phys, beta.real(), beta.imag(), 0, mesh.num_dofs(), &m),
          mesh.context().handle());
    return tbem_system_from_handle(mesh.context(), m, mesh.num_dofs());
}
// Options of one assembly (bemb200_assembly_options, DESIGN.md 4.8).  admittance: empty, or one Y per boundary element in
// enumeration order (entry j <-> the j-th non-evaluation element), v = vbar + Y p on velocity-BC elements.
struct AssemblyOptions {
    int32_t dg_dn_sign = 0;        // 0: the reference's heuristic; +1 / -1 forced
    bool consistent_beta = false;  // the prescribed-velocity right-hand side takes the assembly's beta
    std::vector<Complex64> admittance;
    static AssemblyOptions sign_consistent(std::vector<Complex64> y = {}) {
        AssemblyOptions o;
        o.dg_dn_sign = 1;
        o.consistent_beta = true;
        o.admittance = std::move(y);
        return o;
    }
};
inline TbemSystem build_tbem_system_with_beta(const StagedMesh& mesh, const PhysicsParams& physics, Complex64 beta,
                                              const AssemblyOptions& options) {
    if (!options.admittance.empty() && options.admittance.size() != mesh.num_dofs())
        throw Error(BEMB200_EINVAL, "admittance needs one entry per boundary element");
    const std::vector<Complex64> y = mesh.in_dof_order(options.admittance);
    const bemb200_assembly_options o{options.dg_dn_sign, options.consistent_beta ? 1 : 0,
                                     y.empty() ? nullptr : reinterpret_cast<const double*>(y.data())};
    const bemb200_physics phys = physics_abi(physics);
    bemb200_matrix* m = nullptr;
    check(bemb200_assemble_staged_opts(mesh.context().handle(), mesh.handle(), &phys, beta.real(), beta.imag(), &o, 0, mesh.num_dofs(), &m),
          mesh.context().handle());
    return tbem_system_from_handle(mesh.context(), m, mesh.num_dofs());
}
inline TbemSystem build_tbem_system(const Context& ctx, const std::vector<Element>& el, const std::vector<double>& nodes,
                                    const PhysicsParams& ph) {  // tbem.rs:45-51
    return build_tbem_system_with_beta(ctx, el, nodes, ph, ph.burton_miller_beta());
}
inline TbemSystem build_tbem_system_scaled(const Context& ctx, const std::vector<Element>& el, const std::vector<double>& nodes,
                                           const PhysicsParams& ph, double scale) {  // tbem.rs:85-93
    return build_tbem_system_with_beta(ctx, el, nodes, ph, ph.burton_miller_beta_scaled(scale));
}
inline TbemSystem build_tbem_system_bounded(const Context& ctx, const std::vector<Element>& el, const std::vector<double>& nodes,
                                            const PhysicsParams& ph, double avg_element_size) {  // tbem.rs:64-72
    return build_tbem_system_with_beta(ctx, el, nodes, ph, ph.burton_miller_beta_optimal(avg_element_size));
}
inline double apply_row_sum_correction(TbemSystem& system) {  // tbem.rs:500-520
    double avg = 0.0;
    check(bemb200_row_sum_correction(system.matrix->handle(), &avg), system.matrix->context().handle());
    return avg;
}

inline std::pair<TbemSystem, double> build_tbem_system_corrected(const Context& ctx, const std::vector<Element>& el,
                                                                 const std::vector<double>& nodes, const PhysicsParams& ph) {  // tbem.rs:526-534
    TbemSystem system = build_tbem_system(ctx, el, nodes, ph);
    const double avg = apply_row_sum_correction(system);
    return {std::move(system), avg};
}

// ---- GMRES -------------------------------------------------------------------------------------------------
struct GmresConfig {  // gmres.rs:16-36
    std::size_t max_iterations = 100;  // restart cycles
    std::size_t restart = 30;
    double tolerance = 1e-6;
    std::size_t print_interval = 0;
};
struct GmresSolution {  // gmres.rs:74-85
    std::vector<Complex64> x;
    std::size_t iterations = 0, restarts = 0;
    double residual = 0.0;
    bool converged = false;
};
inline GmresSolution gmres_with_guess(const DenseOperator& op, const std::vector<Complex64>& b, const std::vector<Complex64>* x0,
                                      const GmresConfig& config) {  // gmres.rs:105
    if (b.size() != op.num_rows() || (x0 && x0->size() != b.size())) throw std::invalid_argument("gmres: vector lengths must match");
    GmresSolution s;
    s.x.resize(b.size());
    bemb200_gmres_info info{};
    check(bemb200_gmres(op.handle(), reinterpret_cast<const double*>(b.data()), x0 ? reinterpret_cast<const double*>(x0->data()) : nullptr,
                        static_cast<uint32_t>(config.max_iterations), static_cast<uint32_t>(config.restart), config.tolerance,
                        reinterpret_cast<double*>(s.x.data()), &info),
          op.context().handle());
    s.iterations = info.iterations; s.restarts = info.restarts; s.residual = info.residual; s.converged = info.converged != 0;
    return s;
}
inline GmresSolution gmres(const DenseOperator& op, const std::vector<Complex64>& b, const GmresConfig& config) {  // gmres.rs:96
    return gmres_with_guess(op, b, nullptr, config);
}
inline GmresSolution solve_gmres(const DenseOperator& op, const std::vector<Complex64>& b, const GmresConfig& config) {
    return gmres(op, b, config);  // fmm_interface.rs:378-384
}

struct IdentityPreconditioner {};  // traits.rs:377-385
struct DiagonalPreconditioner {    // preconditioners/diagonal.rs:20-58
    std::vector<Complex64> inv_diag;
    static DiagonalPreconditioner from_diagonal(const std::vector<Complex64>& diag) {
        DiagonalPreconditioner p;
        p.inv_diag.resize(diag.size());
        for (std::size_t i = 0; i < diag.size(); ++i) {
            const double re = diag[i].real(), im = diag[i].imag(), ns = re * re + im * im;
            p.inv_diag[i] = std::hypot(re, im) > 1e-30 ? Complex64(re / ns, -im / ns) : Complex64(1.0, 0.0);
        }
        return p;
    }
};
inline GmresSolution gmres_preconditioned_impl(const DenseOperator& op, const std::vector<Complex64>* inv_diag,
                                               const std::vector<Complex64>& b, const std::vector<Complex64>* x0,
                                               const GmresConfig& config) {
    if (b.size() != op.num_rows() || (x0 && x0->size() != b.size()) || (inv_diag && inv_diag->size() != b.size()))
        throw std::invalid_argument("gmres_preconditioned: vector lengths must match");
    GmresSolution s;
    s.x.resize(b.size());
    bemb200_gmres_info info{};
    check(bemb200_gmres_preconditioned(op.handle(), inv_diag ? reinterpret_cast<const double*>(inv_diag->data()) : nullptr,
                                       reinterpret_cast<const double*>(b.data()),
                                       x0 ? reinterpret_cast<const double*>(x0->data()) : nullptr,
                                       static_cast<uint32_t>(config.max_iterations), static_cast<uint32_t>(config.restart),
                                       config.tolerance, reinterpret_cast<double*>(s.x.data()), &info),
          op.context().handle());
    s.iterations = info.iterations; s.restarts = info.restarts; s.residual = info.residual; s.converged = info.converged != 0;
    return s;
}
inline GmresSolution gmres_preconditioned(const DenseOperator& op, const IdentityPreconditioner&, const std::vector<Complex64>& b,
                                          const GmresConfig& config) {  // gmres.rs:282
    return gmres_preconditioned_impl(op, nullptr, b, nullptr, config);
}
inline GmresSolution gmres_preconditioned(const DenseOperator& op, const DiagonalPreconditioner& p, const std::vector<Complex64>& b,
                                          const GmresConfig& config) {
    return gmres_preconditioned_impl(op, &p.inv_diag, b, nullptr, config);
}
inline GmresSolution gmres_preconditioned_with_guess(const DenseOperator& op, const DiagonalPreconditioner& p,
                                                     const std::vector<Complex64>& b, const std::vector<Complex64>* x0,
                                                     const GmresConfig& config) {  // gmres.rs:434
    return gmres_preconditioned_impl(op, &p.inv_diag, b, x0, config);
}

// AdditiveSchwarzPreconditioner (math-solvers/src/preconditioners/schwarz.rs:31-417) built on the device from the assembled
// operator: from_csr(matrix, num_subdomains, overlap = 0) = block-Jacobi on the contiguous diagonal blocks, or explicit
// subdomains (global DOF indices; overlapping sets get the reference's weights).
class AdditiveSchwarzPreconditioner {
public:
    static AdditiveSchwarzPreconditioner from_operator(const DenseOperator& op, std::size_t num_subdomains) {  // schwarz.rs:66
        AdditiveSchwarzPreconditioner p(op);
        check(bemb200_schwarz_create(op.handle(), static_cast<uint32_t>(num_subdomains), nullptr, nullptr, &p.h_), op.context().handle());
        return p;
    }
    static AdditiveSchwarzPreconditioner from_subdomains(const DenseOperator& op, const std::vector<std::vector<uint64_t>>& subdomains) {
        AdditiveSchwarzPreconditioner p(op);
        std::vector<uint64_t> ptr(1, 0), idx;
        for (const auto& sd : subdomains) {
            idx.insert(idx.end(), sd.begin(), sd.end());
            ptr.push_back(idx.size());
        }
        check(bemb200_schwarz_create(op.handle(), static_cast<uint32_t>(subdomains.size()), ptr.data(), idx.empty() ? ptr.data() : idx.data(),
                                     &p.h_), op.context().handle());
        return p;
    }
    AdditiveSchwarzPreconditioner(AdditiveSchwarzPreconditioner&& o) noexcept : op_(o.op_), h_(o.h_) { o.h_ = nullptr; }
    AdditiveSchwarzPreconditioner(const AdditiveSchwarzPreconditioner&) = delete;
    AdditiveSchwarzPreconditioner& operator=(const AdditiveSchwarzPreconditioner&) = delete;
    ~AdditiveSchwarzPreconditioner() { if (h_) bemb200_precond_free(h_); }
    std::vector<Complex64> apply(const std::vector<Complex64>& r) const {  // Preconditioner::apply (traits.rs:366-371)
        if (r.size() != op_->num_rows()) throw std::invalid_argument("preconditioner: vector lengths must match");
        std::vector<Complex64> z(r.size());
        check(bemb200_precond_apply(h_, reinterpret_cast<const double*>(r.data()), reinterpret_cast<double*>(z.data())), op_->context().handle());
        return z;
    }
    bemb200_precond_stats stats() const {  // schwarz.rs:135-158
        bemb200_precond_stats st{};
        check(bemb200_precond_stats_get(h_, &st), op_->context().handle());
        return st;
    }
    const bemb200_precond* handle() const { return h_; }

private:
    explicit AdditiveSchwarzPreconditioner(const DenseOperator& op) : op_(&op) {}
    const DenseOperator* op_;
    bemb200_precond* h_ = nullptr;
};
inline GmresSolution gmres_preconditioned_with_guess(const DenseOperator& op, const AdditiveSchwarzPreconditioner& p,
                                                     const std::vector<Complex64>& b, const std::vector<Complex64>* x0,
                                                     const GmresConfig& config) {  // gmres.rs:434
    if (b.size() != op.num_rows() || (x0 && x0->size() != b.size()))
        throw std::invalid_argument("gmres_preconditioned: vector lengths must match");
    GmresSolution s;
    s.x.resize(b.size());
    bemb200_gmres_info info{};
    check(bemb200_gmres_schwarz(op.handle(), p.handle(), reinterpret_cast<const double*>(b.data()),
                                x0 ? reinterpret_cast<const double*>(x0->data()) : nullptr, static_cast<uint32_t>(config.max_iterations),
                                static_cast<uint32_t>(config.restart), config.tolerance, reinterpret_cast<double*>(s.x.data()), &info),
          op.context().handle());
    s.iterations = info.iterations; s.restarts = info.restarts; s.residual = info.residual; s.converged = info.converged != 0;
    return s;
}
inline GmresSolution gmres_preconditioned(const DenseOperator& op, const AdditiveSchwarzPreconditioner& p, const std::vector<Complex64>& b,
                                          const GmresConfig& config) {  // gmres.rs:282
    return gmres_preconditioned_with_guess(op, p, b, nullptr, config);
}

// Any other preconditioner: the reference's `Preconditioner` trait (traits.rs:366-371) as an abstract class.  `apply` runs on
// the host (once for M^-1 b, once per restart cycle, once per Arnoldi step) while the Arnoldi process stays on the device
// (bemb200_gmres_callback); an exception thrown by `apply` ends the solve and is rethrown to the caller.
struct Preconditioner {
    virtual ~Preconditioner() = default;
    virtual std::vector<Complex64> apply(const std::vector<Complex64>& r) const = 0;
};
namespace detail {
struct PrecondCall {
    const Preconditioner* p;
    std::exception_ptr error;
};
inline int precond_trampoline(void* user, const double* r, double* z, uint64_t n) noexcept {
    auto* call = static_cast<PrecondCall*>(user);
    try {
        const auto* rc = reinterpret_cast<const Complex64*>(r);
        std::vector<Complex64> out = call->p->apply(std::vector<Complex64>(rc, rc + n));
        if (out.size() != n) throw std::invalid_argument("Preconditioner::apply: result has the wrong length");
        std::copy(out.begin(), out.end(), reinterpret_cast<Complex64*>(z));
        return 0;
    } catch (...) {
        call->error = std::current_exception();
        return 1;
    }
}
}  // namespace detail
inline GmresSolution gmres_preconditioned_with_guess(const DenseOperator& op, const Preconditioner& p, const std::vector<Complex64>& b,
                                                     const std::vector<Complex64>* x0, const GmresConfig& config) {  // gmres.rs:434
    if (b.size() != op.num_rows() || (x0 && x0->size() != b.size()))
        throw std::invalid_argument("gmres_preconditioned: vector lengths must match");
    GmresSolution s;
    s.x.resize(b.size());
    bemb200_gmres_info info{};
    detail::PrecondCall call{&p, nullptr};
    const int rc = bemb200_gmres_callback(op.handle(), &detail::precond_trampoline, &call, reinterpret_cast<const double*>(b.data()),
                                          x0 ? reinterpret_cast<const double*>(x0->data()) : nullptr,
                                          static_cast<uint32_t>(config.max_iterations), static_cast<uint32_t>(config.restart),
                                          config.tolerance, reinterpret_cast<double*>(s.x.data()), &info, nullptr);
    if (call.error) std::rethrow_exception(call.error);
    check(rc, op.context().handle());
    s.iterations = info.iterations; s.restarts = info.restarts; s.residual = info.residual; s.converged = info.converged != 0;
    return s;
}
inline GmresSolution gmres_preconditioned(const DenseOperator& op, const Preconditioner& p, const std::vector<Complex64>& b,
                                          const GmresConfig& config) {  // gmres.rs:282
    return gmres_preconditioned_with_guess(op, p, b, nullptr, config);
}

// ---- pipelined frequency sweep and the single-process multi-GPU group (bemb200_sweep_*, bemb200_multi_*) -------------------------
// Sweep: the per-frequency loop of math-bem/examples/audio_frequency_sweep.rs with the assembly of frequency f + 1 underneath the
// solve of f.  submit() a frequency, next() returns the oldest one solved; keep two in flight.
class Sweep {
public:
    Sweep(int device, const std::vector<Element>& elements, const std::vector<double>& nodes, bool overlap = true,
          int background_blocks_per_sm = 2) {
        const MeshSoA soa(elements);
        const bemb200_mesh mesh = soa.view(nodes);
        check(bemb200_sweep_create(device, 0, 1, nullptr, &mesh, overlap ? 1 : 0, background_blocks_per_sm, &h_));
        n_ = static_cast<std::size_t>(bemb200_sweep_num_dofs(h_));
    }
    ~Sweep() { bemb200_sweep_destroy(h_); }
    Sweep(const Sweep&) = delete;
    Sweep& operator=(const Sweep&) = delete;
    std::size_t num_dofs() const { return n_; }
    // rhs_extra = IncidentField::compute_rhs_with_beta(...) (added to TbemSystem.rhs); empty = none
    void submit(const PhysicsParams& physics, Complex64 beta, const std::vector<Complex64>& rhs_extra, const GmresConfig& config) {
        if (!rhs_extra.empty() && rhs_extra.size() != n_) throw std::invalid_argument("Sweep::submit: vector lengths must match");
        const bemb200_physics phys = physics_abi(physics);
        check(bemb200_sweep_submit(h_, &phys, beta.real(), beta.imag(),
                                   rhs_extra.empty() ? nullptr : reinterpret_cast<const double*>(rhs_extra.data()),
                                   static_cast<uint32_t>(config.max_iterations), static_cast<uint32_t>(config.restart), config.tolerance));
    }
    // solve every following frequency with gmres_preconditioned + block-Jacobi (AdditiveSchwarzPreconditioner::from_csr(.., S, 0));
    // 0 switches back to plain gmres
    void set_block_jacobi(std::size_t num_subdomains) {
        check(bemb200_sweep_set_block_jacobi(h_, static_cast<uint32_t>(num_subdomains), nullptr, nullptr));
    }
    GmresSolution next() {
        GmresSolution s;
        s.x.resize(n_);
        bemb200_gmres_info info{};
        check(bemb200_sweep_next(h_, reinterpret_cast<double*>(s.x.data()), &info, nullptr, nullptr));
        s.iterations = info.iterations; s.restarts = info.restarts; s.residual = info.residual; s.converged = info.converged != 0;
        return s;
    }

private:
    bemb200_sweep* h_ = nullptr;
    std::size_t n_ = 0;
};

// MultiGpu: ONE process, several devices (the shape of BemSolver::solve, bem_solver.rs:273-322): rows block-partitioned over the
// devices, persistent fused GMRES kernel per device, Krylov vectors and reduction partials through peer-mapped memory.
class MultiGpu {
public:
    explicit MultiGpu(const std::vector<int>& devices) {
        check(bemb200_multi_create(devices.data(), static_cast<int>(devices.size()), &h_));
    }
    ~MultiGpu() { bemb200_multi_destroy(h_); }
    MultiGpu(const MultiGpu&) = delete;
    MultiGpu& operator=(const MultiGpu&) = delete;
    int num_ranks() const { return bemb200_multi_num_ranks(h_); }

    class System {  // the row-sharded TbemSystem; must not outlive its group
    public:
        ~System() { bemb200_multi_matrix_free(m_); }
        System(System&& o) noexcept : g_(o.g_), m_(o.m_), rhs(std::move(o.rhs)), num_dofs(o.num_dofs) { o.m_ = nullptr; }
        System(const System&) = delete;
        System& operator=(const System&) = delete;
        GmresSolution gmres(const std::vector<Complex64>& b, const GmresConfig& config) const {  // gmres.rs:96 on the sharded operator
            if (b.size() != num_dofs) throw std::invalid_argument("gmres: vector lengths must match");
            GmresSolution s;
            s.x.resize(b.size());
            bemb200_gmres_info info{};
            g_->check_group(bemb200_multi_gmres(m_, reinterpret_cast<const double*>(b.data()), nullptr, static_cast<uint32_t>(config.max_iterations),
                                                static_cast<uint32_t>(config.restart), config.tolerance, reinterpret_cast<double*>(s.x.data()), &info));
            s.iterations = info.iterations; s.restarts = info.restarts; s.residual = info.residual; s.converged = info.converged != 0;
            return s;
        }

    private:
        friend class MultiGpu;
        System(const MultiGpu* g, bemb200_multi_matrix* m) : g_(g), m_(m) {}
        const MultiGpu* g_;
        bemb200_multi_matrix* m_;

    public:
        std::vector<Complex64> rhs;
        std::size_t num_dofs = 0;
    };

    // build_tbem_system_with_beta on the group: every device assembles its bemb200_partition row block
    System build_tbem_system_with_beta(const std::vector<Element>& elements, const std::vector<double>& nodes, const PhysicsParams& physics,
                                       Complex64 beta) const {
        const MeshSoA soa(elements);
        const bemb200_mesh mesh = soa.view(nodes);
        const bemb200_physics phys = physics_abi(physics);
        bemb200_multi_matrix* m = nullptr;
        check_group(bemb200_multi_assemble(h_, &mesh, &phys, beta.real(), beta.imag(), &m));
        System sys(this, m);
        sys.num_dofs = static_cast<std::size_t>(bemb200_multi_num_rows(m));
        sys.rhs.resize(sys.num_dofs);
        check_group(bemb200_multi_rhs_download(m, reinterpret_cast<double*>(sys.rhs.data())));
        return sys;
    }

private:
    void check_group(int rc) const {
        if (rc != BEMB200_OK) {
            const char* msg = bemb200_multi_last_error(h_);
            throw Error(rc, msg ? msg : "");
        }
    }
    bemb200_multi* h_ = nullptr;
};

// ---- BiCGSTAB / LU (the solvers of BemSolver::solve_dense_system, bem_solver.rs:435-463) ---------------------
struct BiCgstabConfig {  // bicgstab.rs:19-37
    std::size_t max_iterations = 1000;
    double tolerance = 1e-6;
    std::size_t print_interval = 0;
};
struct BiCgstabSolution {  // bicgstab.rs:40-50
    std::vector<Complex64> x;
    std::size_t iterations = 0;
    double residual = 0.0;
    bool converged = false;
};
inline BiCgstabSolution bicgstab(const DenseOperator& op, const std::vector<Complex64>& b, const BiCgstabConfig& config) {  // bicgstab.rs:46
    if (b.size() != op.num_rows()) throw std::invalid_argument("bicgstab: vector length must match the operator");
    BiCgstabSolution s;
    s.x.resize(b.size());
    bemb200_gmres_info info{};
    check(bemb200_bicgstab(op.handle(), reinterpret_cast<const double*>(b.data()), static_cast<uint32_t>(config.max_iterations),
                           config.tolerance, reinterpret_cast<double*>(s.x.data()), &info),
          op.context().handle());
    s.iterations = info.iterations; s.residual = info.residual; s.converged = info.converged != 0;
    return s;
}

// ---- CGS (solve_cgs / solve_with_ilu / solve_tbem_with_ilu, fmm_interface.rs:360-366,389-447) -----------------
struct CgsConfig {  // cgs.rs:12-30
    std::size_t max_iterations = 1000;
    double tolerance = 1e-6;
    std::size_t print_interval = 0;
};
struct CgsSolution {  // cgs.rs:33-43
    std::vector<Complex64> x;
    std::size_t iterations = 0;
    double residual = 0.0;
    bool converged = false;
};
inline CgsSolution cgs(const DenseOperator& op, const std::vector<Complex64>& b, const CgsConfig& config) {  // cgs.rs:46
    if (b.size() != op.num_rows()) throw std::invalid_argument("cgs: vector length must match the operator");
    CgsSolution s;
    s.x.resize(b.size());
    bemb200_gmres_info info{};
    check(bemb200_cgs(op.handle(), reinterpret_cast<const double*>(b.data()), static_cast<uint32_t>(config.max_iterations),
                      config.tolerance, reinterpret_cast<double*>(s.x.data()), &info),
          op.context().handle());
    s.iterations = info.iterations; s.residual = info.residual; s.converged = info.converged != 0;
    return s;
}
inline CgsSolution solve_cgs(const DenseOperator& op, const std::vector<Complex64>& b, const CgsConfig& c) { return cgs(op, b, c); }  // fmm_interface.rs:360
// the reference's "ILU" wrappers run unpreconditioned CGS on the dense matrix (fmm_interface.rs:389-417, 441-447)
inline CgsSolution solve_with_ilu(const DenseOperator& op, const std::vector<Complex64>& b, const CgsConfig& c) { return cgs(op, b, c); }
inline CgsSolution solve_tbem_with_ilu(const DenseOperator& op, const std::vector<Complex64>& b, const CgsConfig& c) { return cgs(op, b, c); }

inline BiCgstabSolution solve_bicgstab(const DenseOperator& op, const std::vector<Complex64>& b, const BiCgstabConfig& c) {  // fmm_interface.rs:369
    return bicgstab(op, b, c);
}

// ---- several right-hand sides (BASELINE config 5): what the reference does with a loop of gmres() calls ----------
// b_all: nrhs vectors of num_rows, each contiguous; one GmresSolution per right-hand side, semantics of gmres() each
inline std::vector<GmresSolution> gmres_batched(const DenseOperator& op, const std::vector<Complex64>& b_all, std::size_t nrhs,
                                                const GmresConfig& config) {
    const std::size_t n = op.num_rows();
    if (nrhs == 0 || b_all.size() != nrhs * n) throw std::invalid_argument("gmres_batched: b_all must hold nrhs vectors of num_rows");
    std::vector<Complex64> x_all(nrhs * n);
    std::vector<bemb200_gmres_info> infos(nrhs);
    check(bemb200_gmres_batched(op.handle(), reinterpret_cast<const double*>(b_all.data()), static_cast<uint32_t>(nrhs),
                                static_cast<uint32_t>(config.max_iterations), static_cast<uint32_t>(config.restart), config.tolerance,
                                reinterpret_cast<double*>(x_all.data()), infos.data(), nullptr, nullptr),
          op.context().handle());
    std::vector<GmresSolution> out(nrhs);
    for (std::size_t s = 0; s < nrhs; ++s) {
        out[s].x.assign(x_all.begin() + s * n, x_all.begin() + (s + 1) * n);
        out[s].iterations = infos[s].iterations; out[s].restarts = infos[s].restarts;
        out[s].residual = infos[s].residual; out[s].converged = infos[s].converged != 0;
    }
    return out;
}
// Y = A X for nrhs vectors at once (tensor-core block matvec); x_all / result: nrhs contiguous vectors
inline std::vector<Complex64> apply_block(const DenseOperator& op, const std::vector<Complex64>& x_all, std::size_t nrhs) {
    if (nrhs == 0 || x_all.size() != nrhs * op.num_cols()) throw std::invalid_argument("apply_block: x_all must hold nrhs vectors of num_cols");
    std::vector<Complex64> y_all(nrhs * op.num_rows());
    check(bemb200_apply_block(op.handle(), reinterpret_cast<const double*>(x_all.data()), static_cast<uint32_t>(nrhs),
                              reinterpret_cast<double*>(y_all.data()), nullptr),
          op.context().handle());
    return y_all;
}

// ---- incident field, field evaluation, RCS on the staged mesh (incident.rs, postprocess/pressure.rs) ------------------
struct IncidentField {  // incident.rs:19-84: plane waves (unit direction, amplitude) and point sources (position, strength)
    std::vector<int32_t> kinds;
    std::vector<double> vecs, amps;
    static IncidentField plane_wave(const double dir[3], double amplitude = 1.0) {  // incident.rs:62-76 (normalised; zero -> -z)
        const double len = std::sqrt(dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2]);
        IncidentField f;
        f.kinds = {0};
        if (len > 1e-10) f.vecs = {dir[0] / len, dir[1] / len, dir[2] / len};
        else f.vecs = {0.0, 0.0, -1.0};
        f.amps = {amplitude, 0.0};
        return f;
    }
    static IncidentField plane_wave_z() { const double d[3] = {0.0, 0.0, 1.0}; return plane_wave(d, 1.0); }       // incident.rs:46-51
    static IncidentField plane_wave_neg_z() { const double d[3] = {0.0, 0.0, -1.0}; return plane_wave(d, 1.0); }  // incident.rs:54-59
    static IncidentField point_source(const double pos[3], double strength = 1.0) {  // incident.rs:79-84
        IncidentField f;
        f.kinds = {1};
        f.vecs = {pos[0], pos[1], pos[2]};
        f.amps = {strength, 0.0};
        return f;
    }
    // compute_rhs_with_beta (incident.rs:317-342) at the staged collocation points: -(gamma p_inc + beta tau dp_inc/dn)
    std::vector<Complex64> compute_rhs_with_beta(const StagedMesh& mesh, const PhysicsParams& physics, Complex64 beta) const {
        const bemb200_physics phys = physics_abi(physics);
        std::vector<Complex64> rhs(mesh.num_dofs());
        check(bemb200_incident_rhs(mesh.handle(), &phys, beta.real(), beta.imag(), static_cast<uint32_t>(kinds.size()), kinds.data(),
                                   vecs.data(), amps.data(), reinterpret_cast<double*>(rhs.data()), nullptr),
              mesh.context().handle());
        return rhs;
    }
    std::vector<Complex64> compute_rhs(const StagedMesh& mesh, const PhysicsParams& physics, bool use_burton_miller) const {  // incident.rs:293-315
        return compute_rhs_with_beta(mesh, physics, use_burton_miller ? physics.burton_miller_beta() : Complex64(0.0, 0.0));
    }
};
// compute_scattered_field (pressure.rs:81-259): eval_points n_eval x 3 row-major; surface_velocity may be empty
inline std::vector<Complex64> compute_scattered_field(const StagedMesh& mesh, const std::vector<double>& eval_points,
                                                      const std::vector<Complex64>& surface_pressure,
                                                      const std::vector<Complex64>& surface_velocity, const PhysicsParams& physics) {
    if (eval_points.size() % 3 != 0) throw std::invalid_argument("compute_scattered_field: eval_points must be n x 3");
    if (surface_pressure.size() != mesh.num_dofs() || (!surface_velocity.empty() && surface_velocity.size() != mesh.num_dofs()))
        throw std::invalid_argument("compute_scattered_field: surface vectors must have num_dofs entries");
    const bemb200_physics phys = physics_abi(physics);
    std::vector<Complex64> out(eval_points.size() / 3);
    const std::vector<Complex64> ps = mesh.in_dof_order(surface_pressure), vs = mesh.in_dof_order(surface_velocity);
    check(bemb200_scattered_field(mesh.handle(), &phys, out.size(), eval_points.data(), reinterpret_cast<const double*>(ps.data()),
                                  vs.empty() ? nullptr : reinterpret_cast<const double*>(vs.data()),
                                  reinterpret_cast<double*>(out.data())),
          mesh.context().handle());
    return out;
}
// compute_rcs (pressure.rs:438-478) for n x 3 unit directions
inline std::vector<double> compute_rcs(const StagedMesh& mesh, const std::vector<Complex64>& surface_pressure,
                                       const std::vector<double>& directions, const PhysicsParams& physics) {
    if (directions.size() % 3 != 0) throw std::invalid_argument("compute_rcs: directions must be n x 3");
    if (surface_pressure.size() != mesh.num_dofs()) throw std::invalid_argument("compute_rcs: surface_pressure must have num_dofs entries");
    const bemb200_physics phys = physics_abi(physics);
    std::vector<double> out(directions.size() / 3);
    const std::vector<Complex64> ps = mesh.in_dof_order(surface_pressure);  // entry j <-> j-th non-evaluation element
    check(bemb200_compute_rcs(mesh.handle(), &phys, static_cast<uint32_t>(out.size()), directions.data(),
                              reinterpret_cast<const double*>(ps.data()), out.data()),
          mesh.context().handle());
    return out;
}
// Complex far-field amplitude F(d) with the surface-velocity term (bemb200_far_field) for n x 3 unit directions;
// surface_velocity (v = dp/dn) may be empty (rigid).  p_scat(R d) = F(d) exp(i s k R) / R + O(1/R^2).
inline std::vector<Complex64> compute_far_field(const StagedMesh& mesh, const std::vector<Complex64>& surface_pressure,
                                                const std::vector<Complex64>& surface_velocity, const std::vector<double>& directions,
                                                const PhysicsParams& physics) {
    if (directions.empty() || directions.size() % 3 != 0) throw std::invalid_argument("compute_far_field: directions must be n x 3, n >= 1");
    if (surface_pressure.size() != mesh.num_dofs() || (!surface_velocity.empty() && surface_velocity.size() != mesh.num_dofs()))
        throw std::invalid_argument("compute_far_field: surface vectors must have num_dofs entries");
    const bemb200_physics phys = physics_abi(physics);
    std::vector<Complex64> out(directions.size() / 3);
    const std::vector<Complex64> ps = mesh.in_dof_order(surface_pressure), vs = mesh.in_dof_order(surface_velocity);
    check(bemb200_far_field(mesh.handle(), &phys, 1, reinterpret_cast<const double*>(ps.data()),
                            vs.empty() ? nullptr : reinterpret_cast<const double*>(vs.data()), 0, static_cast<uint32_t>(out.size()),
                            directions.data(), reinterpret_cast<double*>(out.data())),
          mesh.context().handle());
    return out;
}
// Accurate scattered pressure (bemb200_evaluate_field) at n x 3 eval_points: whole elements (Quad4: the bilinear map) and
// adaptive quadrature near the surface; surface_velocity (v = dp/dn) may be empty.  Points on the surface are NaN.
inline std::vector<Complex64> evaluate_field(const StagedMesh& mesh, const std::vector<double>& eval_points,
                                             const std::vector<Complex64>& surface_pressure,
                                             const std::vector<Complex64>& surface_velocity, const PhysicsParams& physics) {
    if (eval_points.empty() || eval_points.size() % 3 != 0) throw std::invalid_argument("evaluate_field: eval_points must be n x 3, n >= 1");
    if (surface_pressure.size() != mesh.num_dofs() || (!surface_velocity.empty() && surface_velocity.size() != mesh.num_dofs()))
        throw std::invalid_argument("evaluate_field: surface vectors must have num_dofs entries");
    const bemb200_physics phys = physics_abi(physics);
    std::vector<Complex64> out(eval_points.size() / 3);
    const std::vector<Complex64> ps = mesh.in_dof_order(surface_pressure), vs = mesh.in_dof_order(surface_velocity);
    check(bemb200_evaluate_field(mesh.handle(), &phys, 1, reinterpret_cast<const double*>(ps.data()),
                                 vs.empty() ? nullptr : reinterpret_cast<const double*>(vs.data()), 0, out.size(), eval_points.data(),
                                 reinterpret_cast<double*>(out.data())),
          mesh.context().handle());
    return out;
}
// Gradient of the accurate scattered pressure (bemb200_evaluate_field_gradient) at n x 3 eval_points: n x 3 values
// (d/dx, d/dy, d/dz per point); surface_velocity (v = dp/dn) may be empty.  pressure (may be null) receives the n values of
// evaluate_field.  Points on the surface are NaN.
inline std::vector<Complex64> evaluate_field_gradient(const StagedMesh& mesh, const std::vector<double>& eval_points,
                                                      const std::vector<Complex64>& surface_pressure,
                                                      const std::vector<Complex64>& surface_velocity, const PhysicsParams& physics,
                                                      std::vector<Complex64>* pressure = nullptr) {
    if (eval_points.empty() || eval_points.size() % 3 != 0)
        throw std::invalid_argument("evaluate_field_gradient: eval_points must be n x 3, n >= 1");
    if (surface_pressure.size() != mesh.num_dofs() || (!surface_velocity.empty() && surface_velocity.size() != mesh.num_dofs()))
        throw std::invalid_argument("evaluate_field_gradient: surface vectors must have num_dofs entries");
    const bemb200_physics phys = physics_abi(physics);
    const size_t n = eval_points.size() / 3;
    std::vector<Complex64> grad(3 * n);
    if (pressure) pressure->assign(n, Complex64{});
    const std::vector<Complex64> ps = mesh.in_dof_order(surface_pressure), vs = mesh.in_dof_order(surface_velocity);
    check(bemb200_evaluate_field_gradient(mesh.handle(), &phys, 1, reinterpret_cast<const double*>(ps.data()),
                                          vs.empty() ? nullptr : reinterpret_cast<const double*>(vs.data()), 0, n, eval_points.data(),
                                          pressure ? reinterpret_cast<double*>(pressure->data()) : nullptr,
                                          reinterpret_cast<double*>(grad.data())),
          mesh.context().handle());
    return grad;
}

struct LuError : std::runtime_error {  // lu.rs:15-21
    enum Kind { SingularMatrix, DimensionMismatch } kind;
    LuError(Kind k, const std::string& m) : std::runtime_error(m), kind(k) {}
};
// lu_solve(&a, &b) (lu.rs:139-161): `a` is left intact
inline std::vector<Complex64> lu_solve(const DenseOperator& a, const std::vector<Complex64>& b) {
    if (a.num_rows() != a.num_cols() || b.size() != a.num_rows())
        throw LuError(LuError::DimensionMismatch, "Matrix dimensions mismatch: expected " + std::to_string(a.num_rows()) + ", got " + std::to_string(b.size()));
    std::vector<Complex64> x(b.size());
    const int rc = bemb200_lu_solve(a.handle(), reinterpret_cast<const double*>(b.data()), reinterpret_cast<double*>(x.data()), 0, nullptr);
    if (rc == BEMB200_ESINGULAR) throw LuError(LuError::SingularMatrix, "Matrix is singular or nearly singular");
    check(rc, a.context().handle());
    return x;
}

// ---- room acoustics (math-bem/src/room_acoustics/solver.rs, math-xem-common) ---------------------------------
struct Point3D { double x = 0, y = 0, z = 0; };             // math-xem-common/src/types.rs
struct SurfaceElement { std::vector<std::size_t> nodes; };  // types.rs:154-157 (3 or 4 node indices)
struct RoomMesh {                                           // types.rs:185-192
    std::vector<Point3D> nodes;
    std::vector<SurfaceElement> elements;
};
struct Source {  // source.rs:160-219 with DirectivityPattern (magnitude[n_vertical][n_horizontal], 10 degree grid; empty = omnidirectional)
    Point3D position;
    double amplitude = 1.0;
    std::vector<double> directivity;
    std::size_t n_horizontal = 0, n_vertical = 0;
    double crossover_amplitude = 1.0;  // crossover.amplitude_at_frequency(f), evaluated by the caller per frequency
};
class StagedRoomMesh {
public:
    StagedRoomMesh(const Context& ctx, const RoomMesh& mesh) : ctx_(&ctx) {
        std::vector<double> nodes;
        nodes.reserve(mesh.nodes.size() * 3);
        for (const Point3D& p : mesh.nodes) nodes.insert(nodes.end(), {p.x, p.y, p.z});
        std::vector<uint32_t> conn(mesh.elements.size() * 4, 0xFFFFFFFFu);
        for (std::size_t e = 0; e < mesh.elements.size(); ++e) {
            const auto& nd = mesh.elements[e].nodes;
            if (nd.size() != 3 && nd.size() != 4) throw std::invalid_argument("room elements are triangles or quadrilaterals");
            for (std::size_t v = 0; v < nd.size(); ++v) conn[4 * e + v] = static_cast<uint32_t>(nd[v]);
        }
        check(bemb200_room_mesh_stage(ctx.handle(), nodes.data(), mesh.nodes.size(), conn.data(), mesh.elements.size(), &h_), ctx.handle());
    }
    ~StagedRoomMesh() { bemb200_room_mesh_free(h_); }
    StagedRoomMesh(const StagedRoomMesh&) = delete;
    StagedRoomMesh& operator=(const StagedRoomMesh&) = delete;
    bemb200_room_mesh* handle() const { return h_; }
    const Context& context() const { return *ctx_; }
    std::size_t num_elements() const { return bemb200_room_mesh_num_elements(h_); }

private:
    const Context* ctx_;
    bemb200_room_mesh* h_ = nullptr;
};
inline std::vector<bemb200_room_source> room_sources_abi(const std::vector<Source>& sources) {
    std::vector<bemb200_room_source> out(sources.size());
    for (std::size_t i = 0; i < sources.size(); ++i) {
        out[i].position[0] = sources[i].position.x; out[i].position[1] = sources[i].position.y; out[i].position[2] = sources[i].position.z;
        out[i].amplitude = sources[i].amplitude * sources[i].crossover_amplitude;
        out[i].directivity = sources[i].directivity.empty() ? nullptr : sources[i].directivity.data();
        out[i].n_horizontal = static_cast<uint32_t>(sources[i].n_horizontal);
        out[i].n_vertical = static_cast<uint32_t>(sources[i].n_vertical);
    }
    return out;
}
// build_bem_matrix_parallel (solver.rs:448-493) -> device-resident operator
inline std::unique_ptr<DenseOperator> build_bem_matrix_parallel(const StagedRoomMesh& mesh, double k) {
    bemb200_matrix* m = nullptr;
    check(bemb200_room_assemble(mesh.context().handle(), mesh.handle(), k, 0, mesh.num_elements(), &m, nullptr), mesh.context().handle());
    return std::make_unique<DenseOperator>(mesh.context(), m);
}
inline std::vector<Complex64> calculate_incident_field_derivative_parallel(const StagedRoomMesh& mesh, const std::vector<Source>& sources,
                                                                          double k) {  // solver.rs:638-679
    std::vector<Complex64> rhs(mesh.num_elements());
    auto abi = room_sources_abi(sources);
    check(bemb200_room_incident_rhs(mesh.handle(), k, static_cast<uint32_t>(abi.size()), abi.data(), reinterpret_cast<double*>(rhs.data()), nullptr),
          mesh.context().handle());
    return rhs;
}
// solve_bem_system (solver.rs:412-445): GMRES max_iterations 100, restart 50, tolerance 1e-6; returns solution.x
inline std::vector<Complex64> solve_bem_system(const StagedRoomMesh& mesh, const std::vector<Source>& sources, double k,
                                               GmresSolution* solution_out = nullptr) {
    auto op = build_bem_matrix_parallel(mesh, k);
    GmresSolution s = solve_gmres(*op, calculate_incident_field_derivative_parallel(mesh, sources, k), GmresConfig{100, 50, 1e-6, 0});
    if (solution_out) *solution_out = s;
    return s.x;
}
inline std::vector<Complex64> calculate_field_pressure_bem_parallel(const StagedRoomMesh& mesh, const std::vector<Complex64>& surface_pressure,
                                                                   const std::vector<Source>& sources, const std::vector<Point3D>& field_points,
                                                                   double k) {  // solver.rs:687-748
    if (surface_pressure.size() != mesh.num_elements()) throw std::invalid_argument("surface_pressure must have one entry per element");
    std::vector<double> pts;
    for (const Point3D& p : field_points) pts.insert(pts.end(), {p.x, p.y, p.z});
    std::vector<Complex64> out(field_points.size());
    auto abi = room_sources_abi(sources);
    check(bemb200_room_field_pressure(mesh.handle(), k, static_cast<uint32_t>(abi.size()), abi.data(), field_points.size(), pts.data(),
                                      reinterpret_cast<const double*>(surface_pressure.data()), reinterpret_cast<double*>(out.data())),
          mesh.context().handle());
    return out;
}
inline double pressure_to_spl(Complex64 p) {  // math-xem-common/src/types.rs:280-287
    const double m = std::abs(p);
    return m > 1e-20 ? 20.0 * std::log10(m / 20e-6) : -120.0;
}

}  // namespace bemb200

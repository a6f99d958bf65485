// The checker of sph_gravity_at: the CPU oracle (oracle/sph_oracle.cpp, compiled unchanged into this library) plus one
// entry point.  TEST INFRASTRUCTURE, built by tests/_gravat_oracle.py.
//
// Point k becomes a Particle with s_length = h_k (h_fixed when h is NULL) at x_k that is not part of the tree; the
// oracle's own particle_gravforce_one and potential_one (self = -1: no node is left out) walk the tree of the last
// evaluation, and the sink terms follow sink_gravforces (F:567-576) over the sinks with m > 0 at a distance > 0.
#include "../oracle/sph_oracle.cpp"

extern "C" void orc_gravity_at(orc_ctx* c, int64_t n, const double* px, const double* py, const double* pz, const double* h,
                               double* out) {
  Oracle& o = c->o;
  if (o.nodes.empty()) create_tree(o);
  const double theta = o.p.theta_override ? o.p.theta : 0.5;               // F:825
  for (int64_t k = 0; k < n; ++k) {
    Particle p;
    std::memset(&p, 0, sizeof(p));
    p.s_length = h ? h[k] : o.p.h_fixed;
    p.position[0] = px[k]; p.position[1] = py[k]; p.position[2] = pz[k];
    int64_t opened = 0, accepted = 0;
    particle_gravforce_one(o, 0, p, theta, opened, accepted);
    double phi = 0.0;
    potential_one(o, 0, -1, p, theta, phi);
    double phis = 0.0, gs[3] = {0.0, 0.0, 0.0};
    for (const Sink& s : o.sinks) {
      if (!(s.mass > 0.0)) continue;
      double v[3]; for (int d = 0; d < 3; ++d) v[d] = p.position[d] - s.position[d];
      const double dr = std::sqrt(((v[0] * v[0]) + v[1] * v[1]) + v[2] * v[2]);
      if (!(dr > 0.0)) continue;
      const double dd = dr * dr * dr;
      for (int d = 0; d < 3; ++d) { const double w = G_REF * v[d] / dd; gs[d] = gs[d] - (s.mass * w); }   // F:572-574
      phis -= G_REF * s.mass / dr;
    }
    const double col[9] = {G_REF * phi, p.acceleration[0], p.acceleration[1], p.acceleration[2], phis, gs[0], gs[1], gs[2], (double)accepted};
    for (int q = 0; q < 9; ++q) out[q * n + k] = col[q];
  }
}

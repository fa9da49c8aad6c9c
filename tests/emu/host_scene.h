// host_scene.h — TEST INFRASTRUCTURE ONLY: the DevScene of a scene for the host harnesses of tests/emu, after the
// device code is included.
#pragma once

namespace {
// upload_replica (rtc_api.cu) with host pointers
void host_scene(const RtcScene* s, const rtc::Flattened& f, rtc::DevScene& d) {
    memset(&d, 0, sizeof(d));
    rtc::rows3(s->cam_inv, d.cam_inv);
    d.half_w = s->half_w, d.half_h = s->half_h, d.pixel_size = s->pixel_size;
    d.width = (int)s->width, d.height = (int)s->height;
    d.light_is_rect = s->light_is_rect;
    memcpy(d.light_pos, s->light_pos, 12);
    memcpy(d.light_rgb, s->light_rgb, 12);
    memcpy(d.corner, s->corner, 12);
    memcpy(d.u_vec, s->u_cell, 12);
    memcpy(d.v_vec, s->v_cell, 12);
    d.u_steps = s->u_steps, d.v_steps = s->v_steps, d.cells = s->u_steps * s->v_steps;
    d.jitter_len = (int)s->jitter.size();
    d.seed = s->seed;
    auto at = [](const auto& v) { return v.empty() ? nullptr : v.data(); };
    d.jitter = at(s->jitter), d.samples = at(f.samples), d.head = at(f.head), d.rec = at(f.rec), d.xform = at(f.xform);
    d.tri = at(f.tri), d.bound = at(f.bound), d.bvh = at(f.bvh), d.linear = at(f.linear), d.nodes = at(f.nodes);
    d.csg_ops = at(f.ops), d.materials = at(f.materials), d.patterns = at(f.patterns), d.uvs = at(f.uvs), d.texels = at(f.texels);
    d.small_image = at(f.small_image);
    d.n_linear = (int)f.linear.size(), d.bvh_root = f.bvh_root, d.n_prims = f.n_pos, d.all_cast_shadow = f.all_cast_shadow;
}
}  // namespace

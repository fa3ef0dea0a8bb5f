//! cuda_backend.zig — Zig side of the drop-in boundary (include/rayz_cuda.h).
//!
//! NOT COMPILED OR TESTED: the build image has no zig toolchain.  It is written against the
//! reference's own types (src/ecs.zig, src/camera.zig, src/geom.zig, src/material.zig,
//! src/image.zig as of the surveyed tree, Zig 0.13-era std) and shows exactly what a maintainer
//! adds; the tested stand-ins for it are host/rayz_host.hpp (C++) and rayz_b200/host.py (ctypes).
//!
//! Usage in src/renderer.zig — replace the body of `Tracer.render` (renderer.zig:72-101) with
//!
//!     pub fn render(self: *Tracer) !usize {
//!         return cuda.render(self.allocator, &self.cuda_ctx, &self.camera, &self.pool, &self.img,
//!                            self.samples_per_px, self.max_bounces, self.seed);
//!     }
const std = @import("std");
const vec = @import("./vec.zig");
const ecs = @import("./ecs.zig");
const image = @import("./image.zig");
const Camera = @import("./camera.zig").Camera;

pub const RzScene = extern struct {
    n_spheres: u32,
    n_materials: u32,
    n_textures: u32,
    reserved0: u32 = 0,
    sphere_center: [*]const f64,
    sphere_velocity: [*]const f64,
    sphere_radius: [*]const f64,
    sphere_material: [*]const u32,
    mat_kind: [*]const u32,
    mat_fuzz: [*]const f64,
    mat_ior: [*]const f64,
    mat_texture: [*]const u32,
    mat_method: ?[*]const u32,
    tex_kind: [*]const u32,
    tex_color: [*]const f64,
    tex_scale: [*]const f64,
    tex_even: [*]const u32,
    tex_odd: [*]const u32,
};

pub const RzCamera = extern struct {
    look_from: [3]f64,
    px_du: [3]f64,
    px_dv: [3]f64,
    px_origin: [3]f64,
    defocus_u: [3]f64,
    defocus_v: [3]f64,
    defocus: i32,
    reserved0: i32 = 0,
};

pub const RzRenderParams = extern struct {
    width: u32,
    height: u32,
    spp: u32,
    max_depth: u32,
    seed: u64,
    sample_offset: u32 = 0,
    variant: u32 = 0, // RZ_VARIANT_AUTO
    t_min: f32 = 0,
    shard_index: u32 = 0,
    shard_count: u32 = 1,
    band_rows: u32 = 0,
    collect_stats: u32 = 0,
    flags: u32 = 0, // RZ_RENDER_* bits
};

pub const RzConfig = extern struct {
    n_devices: i32,
    device_ids: [8]i32,
    flags: u32 = 0,
};

pub const RZ_RENDER_MOMENTS: u32 = 2; // sum each path's luminance squared: rayz_cuda_noise
pub const RZ_RENDER_ACCUMULATE: u32 = 4; // add this batch to the previous render's sums (progressive rendering)

pub const RzNoise = extern struct {
    samples: u64,
    n_pixels: u32,
    n_above: u32,
    mean_err: f64,
    rms_err: f64,
    max_err: f64,
};

pub const RzContext = opaque {};

pub extern fn rayz_cuda_create(cfg: ?*const RzConfig, out: *?*RzContext) c_int;
pub extern fn rayz_cuda_destroy(ctx: ?*RzContext) void;
pub extern fn rayz_cuda_reserve(ctx: *RzContext, params: *const RzRenderParams) c_int;
pub extern fn rayz_cuda_upload_scene(ctx: *RzContext, scene: *const RzScene) c_int;
pub extern fn rayz_cuda_render(ctx: *RzContext, cam: *const RzCamera, params: *const RzRenderParams, out_linear_rgba: ?[*]f32, out_rgb8: ?[*]u8, out_paths: ?*u64) c_int;
pub extern fn rayz_cuda_primary_ids(ctx: *RzContext, cam: *const RzCamera, width: u32, height: u32, use_bvh: c_int, out_ids: [*]i32) c_int;
pub extern fn rayz_cuda_noise(ctx: *RzContext, target: f32, out_err: ?[*]f32, out: ?*RzNoise) c_int;
pub extern fn rayz_cuda_render_to_noise(ctx: *RzContext, cam: *const RzCamera, params: *const RzRenderParams, target: f32, max_spp: u32, out_linear_rgba: ?[*]f32, out_rgb8: ?[*]u8, out_paths: ?*u64, out_noise: ?*RzNoise) c_int;
pub extern fn rayz_cuda_last_error() [*:0]const u8;

pub const Error = error{ CudaBackend, OutOfMemory };

fn v3(v: vec.V3) [3]f64 {
    return .{ v.x, v.y, v.z };
}

fn check(rc: c_int) Error!void {
    if (rc != 0) {
        std.debug.print("rayz_cuda: {s}\n", .{rayz_cuda_last_error()});
        return error.CudaBackend;
    }
}

/// Drop-in for the pixel loop of Tracer.render.  Zig structs and tagged unions have no C layout,
/// so the pools are COPIED into flat arrays with a switch (ecs.zig:22-27, material.zig:41-43,162-165).
pub fn render(
    allocator: std.mem.Allocator,
    ctx_slot: *?*RzContext,
    camera: *const Camera,
    pool: *const ecs.MemPool,
    img: *image.Image,
    samples_per_px: usize,
    max_bounces: usize,
    seed: u64,
) Error!usize {
    if (ctx_slot.* == null) {
        var cfg = RzConfig{ .n_devices = 1, .device_ids = .{ 0, 0, 0, 0, 0, 0, 0, 0 } };
        try check(rayz_cuda_create(&cfg, ctx_slot));
    }
    const ctx = ctx_slot.*.?;

    const ns = pool.spheres.items.len;
    const nm = pool.materials.items.len;
    const nt = pool.textures.items.len;
    const sc = try allocator.alloc(f64, 3 * ns);
    const sv = try allocator.alloc(f64, 3 * ns);
    const sr = try allocator.alloc(f64, ns);
    const sm = try allocator.alloc(u32, ns);
    const mk = try allocator.alloc(u32, nm);
    const mf = try allocator.alloc(f64, nm);
    const mi = try allocator.alloc(f64, nm);
    const mt = try allocator.alloc(u32, nm);
    const mm = try allocator.alloc(u32, nm);
    const tk = try allocator.alloc(u32, nt);
    const tc = try allocator.alloc(f64, 3 * nt);
    const ts = try allocator.alloc(f64, nt);
    const te = try allocator.alloc(u32, nt);
    const to = try allocator.alloc(u32, nt);

    for (pool.spheres.items, 0..) |s, i| {
        sc[3 * i + 0] = s.center.origin.x;
        sc[3 * i + 1] = s.center.origin.y;
        sc[3 * i + 2] = s.center.origin.z;
        sv[3 * i + 0] = s.center.dir.x;
        sv[3 * i + 1] = s.center.dir.y;
        sv[3 * i + 2] = s.center.dir.z;
        sr[i] = s.radius;
        sm[i] = @intCast(s.material.idx);
    }
    for (pool.materials.items, 0..) |m, i| {
        mf[i] = 0;
        mi[i] = 1;
        mt[i] = 0;
        mm[i] = 2; // HEMISPHERE
        switch (m) {
            .diffuse => |d| {
                mk[i] = 0;
                mt[i] = @intCast(d.texture.idx);
                mm[i] = @intFromEnum(d.method);
            },
            .metallic => |d| {
                mk[i] = 1;
                mf[i] = d.fuzz;
                mt[i] = @intCast(d.texture.idx);
            },
            .dielectric => |d| {
                mk[i] = 2;
                mi[i] = d.refractive_index;
            },
        }
    }
    for (pool.textures.items, 0..) |t, i| {
        tc[3 * i + 0] = 0;
        tc[3 * i + 1] = 0;
        tc[3 * i + 2] = 0;
        ts[i] = 1;
        te[i] = 0;
        to[i] = 0;
        switch (t) {
            .checker => |c| {
                tk[i] = 0;
                ts[i] = c.scale;
                te[i] = @intCast(c.even.idx);
                to[i] = @intCast(c.odd.idx);
            },
            .solid => |c| {
                tk[i] = 1;
                tc[3 * i + 0] = c.color.x;
                tc[3 * i + 1] = c.color.y;
                tc[3 * i + 2] = c.color.z;
            },
        }
    }
    const scene = RzScene{
        .n_spheres = @intCast(ns),
        .n_materials = @intCast(nm),
        .n_textures = @intCast(nt),
        .sphere_center = sc.ptr,
        .sphere_velocity = sv.ptr,
        .sphere_radius = sr.ptr,
        .sphere_material = sm.ptr,
        .mat_kind = mk.ptr,
        .mat_fuzz = mf.ptr,
        .mat_ior = mi.ptr,
        .mat_texture = mt.ptr,
        .mat_method = mm.ptr,
        .tex_kind = tk.ptr,
        .tex_color = tc.ptr,
        .tex_scale = ts.ptr,
        .tex_even = te.ptr,
        .tex_odd = to.ptr,
    };
    try check(rayz_cuda_upload_scene(ctx, &scene)); // copy semantics: the arena may free the arrays now

    const cam = RzCamera{
        .look_from = v3(camera.look_from),
        .px_du = v3(camera.px_du),
        .px_dv = v3(camera.px_dv),
        .px_origin = v3(camera.px_origin),
        .defocus_u = v3(camera.defocus_u),
        .defocus_v = v3(camera.defocus_v),
        .defocus = if (camera.defocus) 1 else 0,
    };
    const params = RzRenderParams{
        .width = @intCast(img.w),
        .height = @intCast(img.h),
        .spp = @intCast(samples_per_px),
        .max_depth = @intCast(max_bounces),
        .seed = seed,
    };
    const lin = try allocator.alloc(f32, img.w * img.h * 4);
    var rays: u64 = 0;
    try check(rayz_cuda_render(ctx, &cam, &params, lin.ptr, null, &rays));
    // widen back into img.pixels so the unmodified Image.writePPM (image.zig:29-41) keeps working
    for (img.pixels, 0..) |*px, i| {
        px.* = .{ .x = lin[4 * i + 0], .y = lin[4 * i + 1], .z = lin[4 * i + 2] };
    }
    return @intCast(rays);
}

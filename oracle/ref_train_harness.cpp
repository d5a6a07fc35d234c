// TEST INFRASTRUCTURE ONLY -- not part of the product path.
//
// Python module that runs the reference's OWN training-step callers, compiled UNCHANGED from /root/reference:
//   src/training/rasterization/fast_rasterizer_autograd.cpp   gs::training::FastGSRasterize  (C++ autograd Function)
//   src/training/optimizers/fused_adam.cpp                    gs::training::FusedAdam
//   src/training/kernels/ssim.cu + include/kernels/fused_ssim.cuh   fused_ssim (autograd)
// on top of a fastgs backend chosen at LINK time (oracle/Makefile):
//   ref_fastgs_torch   <- the reference's own fastgs objects (forward.cu, backward.cu, rasterization_api.cu, adam*.cu)
//   b200_fastgs_torch  <- oracle/_ref/libgsplat_backend_b200.so (this project's host layer, which exports the
//                         same mangled fast_gs::rasterization::{forward,backward}_wrapper / fast_gs::optimizer symbols)
// Both modules are the same object code above the backend boundary, so (a) the first is the "reference fastgs build"
// training step timed beside ours, (b) the second proves that the reference's callers link and run against our
// boundary unchanged (VERDICT r1 item 6).
//
// The same for the 3DGUT (--gut) path: src/training/rasterization/rasterizer_autograd.cpp (SphericalHarmonicsFunction,
// fully_fused_projection_with_ut, GUTRasterizationFunction) compiled UNCHANGED (oracle/ref_stubs/core/*.hpp stand in for
// the two application headers it includes but does not use) on top of a gsplat backend chosen at link time: the
// reference's own gsplat objects (glm shim build) or this project's host layer.  GutHarness::render restates
// gs::training::rasterize (src/training/rasterization/rasterizer.cpp:46-437, RGB / RGB_D / D modes, no bounding box) and
// the SplatData getters (src/core/splat_data.cpp:267-286).
//
// What is restated here (20 lines, because gs::Camera / gs::SplatData need the whole application):
//   fast_rasterize()            src/training/rasterization/fast_rasterizer.cpp:12-67  -> Harness::render
//   compute_photometric_loss()  src/training/trainer.cpp:103-131                      -> Harness::photometric_loss
//   create_optimizer()          src/training/strategies/strategy_utils.cpp:21-49      -> Harness::Harness
//   the step structure          src/training/trainer.cpp:579-757 (render, loss, backward, optimizer step, zero_grad)
#include "Ops.h"
#include "adam_api.h"
#include "fast_rasterizer_autograd.hpp"
#include "rasterization/rasterizer_autograd.hpp"
#include "fused_adam.hpp"
#include "kernels/fused_ssim.cuh"
#include "rasterization_api.h"
#ifdef LFS_B200_LEGACY_OPS
#include "gsplat_legacy_ops.h" // lichtfeld-studio_b200/host: the legacy 2-D ops exist on this project's backend only
#endif

#include <ATen/cuda/CUDAContext.h>
#include <torch/extension.h>

namespace {
    using torch::Tensor;

    struct Harness {
        Tensor means, sh0, shN, scales, rot, op, densification_info;
        std::unique_ptr<gs::training::FusedAdam> opt;

        Harness(Tensor means_, Tensor sh0_, Tensor shN_, Tensor scales_, Tensor rot_, Tensor op_, std::vector<double> lrs) {
            auto prep = [](Tensor t) { return t.to(torch::kCUDA).contiguous().clone().set_requires_grad(true); };
            means = prep(means_), sh0 = prep(sh0_), shN = prep(shN_), scales = prep(scales_), rot = prep(rot_), op = prep(op_);
            densification_info = torch::zeros({2, means.size(0)}, means.options()).set_requires_grad(false);
            using Options = gs::training::FusedAdam::Options;
            std::vector<torch::optim::OptimizerParamGroup> groups;
            auto add = [&groups](const Tensor& p, double lr) {
                auto o = std::make_unique<Options>(lr);
                o->eps(1e-15).betas(std::make_tuple(0.9, 0.999));
                groups.emplace_back(std::vector<Tensor>{p}, std::unique_ptr<torch::optim::OptimizerOptions>(std::move(o)));
            };
            add(means, lrs[0]), add(sh0, lrs[1]), add(shN, lrs[2]), add(scales, lrs[3]), add(rot, lrs[4]), add(op, lrs[5]);
            auto g = std::make_unique<Options>(0.f);
            g->eps(1e-15);
            opt = std::make_unique<gs::training::FusedAdam>(std::move(groups), std::move(g));
        }

        // fast_rasterize (fast_rasterizer.cpp:12-67)
        std::pair<Tensor, Tensor> render(const Tensor& w2c, const Tensor& cam_position, int active_sh_bases, int width,
                                         int height, float fx, float fy, float cx, float cy, Tensor& bg) {
            fast_gs::rasterization::FastGSSettings s;
            s.cam_position = cam_position;
            s.active_sh_bases = active_sh_bases;
            s.width = width, s.height = height;
            s.focal_x = fx, s.focal_y = fy, s.center_x = cx, s.center_y = cy;
            s.near_plane = 0.01f, s.far_plane = 1e10f;
            auto out = gs::training::FastGSRasterize::apply(means, scales, rot, op, sh0, shN, w2c, densification_info, s);
            Tensor image = out[0] + (1.0f - out[1]) * bg.unsqueeze(-1).unsqueeze(-1);
            return {image, out[1]};
        }

        // compute_photometric_loss (trainer.cpp:103-131)
        static Tensor photometric_loss(Tensor rendered, Tensor gt, float lambda_dssim) {
            rendered = rendered.dim() == 3 ? rendered.unsqueeze(0) : rendered;
            gt = gt.dim() == 3 ? gt.unsqueeze(0) : gt;
            auto l1 = torch::l1_loss(rendered, gt);
            auto ssim_loss = 1.f - fused_ssim(rendered, gt, "valid", true);
            return (1.f - lambda_dssim) * l1 + lambda_dssim * ssim_loss;
        }

        // one batch of views -> one optimizer step; returns the summed loss when read_loss
        double train_step(int iteration, std::vector<Tensor> w2cs, std::vector<Tensor> cam_positions,
                          std::vector<std::vector<double>> intrinsics, std::vector<Tensor> gts, Tensor bg,
                          double lambda_dssim, int active_sh_bases, int width, int height, bool read_loss) {
            Tensor total;
            for (size_t v = 0; v < w2cs.size(); ++v) {
                const auto& k = intrinsics[v];
                auto [image, alpha] = render(w2cs[v], cam_positions[v], active_sh_bases, width, height, (float)k[0],
                                             (float)k[1], (float)k[2], (float)k[3], bg);
                Tensor loss = photometric_loss(image, gts[v], (float)lambda_dssim);
                loss.backward();
                if (read_loss)
                    total = total.defined() ? total + loss.detach() : loss.detach();
            }
            opt->step(iteration);
            opt->zero_grad(true, iteration);
            return read_loss ? total.item<double>() : 0.0;
        }

        // forward + loss + backward of ONE view without the optimizer: returns (image, alpha, loss, grads[6]) for parity
        std::vector<Tensor> view_grads(Tensor w2c, Tensor cam_position, std::vector<double> k, Tensor gt, Tensor bg,
                                       double lambda_dssim, int active_sh_bases, int width, int height) {
            opt->zero_grad(true, 0);
            auto [image, alpha] = render(w2c, cam_position, active_sh_bases, width, height, (float)k[0], (float)k[1],
                                         (float)k[2], (float)k[3], bg);
            Tensor loss = photometric_loss(image, gt, (float)lambda_dssim);
            loss.backward();
            return {image.detach(), alpha.detach(), loss.detach(), means.grad(), sh0.grad(), shN.grad(), scales.grad(),
                    rot.grad(), op.grad()};
        }

        std::vector<Tensor> params() { return {means.detach(), sh0.detach(), shN.detach(), scales.detach(), rot.detach(), op.detach()}; }
    };
    // ------------------------------------------------------------------------------------------------ 3DGUT path
    struct GutHarness {
        Tensor means, sh0, shN, scales, rot, op;
        std::unique_ptr<gs::training::FusedAdam> opt;
        int64_t last_n_isects = 0;

        GutHarness(Tensor means_, Tensor sh0_, Tensor shN_, Tensor scales_, Tensor rot_, Tensor op_, std::vector<double> lrs) {
            auto prep = [](Tensor t) { return t.to(torch::kCUDA).contiguous().clone().set_requires_grad(true); };
            means = prep(means_), sh0 = prep(sh0_), shN = prep(shN_), scales = prep(scales_), rot = prep(rot_), op = prep(op_);
            using Options = gs::training::FusedAdam::Options;
            std::vector<torch::optim::OptimizerParamGroup> groups;
            auto add = [&groups](const Tensor& p, double lr) {
                auto o = std::make_unique<Options>(lr);
                o->eps(1e-15).betas(std::make_tuple(0.9, 0.999));
                groups.emplace_back(std::vector<Tensor>{p}, std::unique_ptr<torch::optim::OptimizerOptions>(std::move(o)));
            };
            add(means, lrs[0]), add(sh0, lrs[1]), add(shN, lrs[2]), add(scales, lrs[3]), add(rot, lrs[4]), add(op, lrs[5]);
            auto g = std::make_unique<Options>(0.f);
            g->eps(1e-15);
            opt = std::make_unique<gs::training::FusedAdam>(std::move(groups), std::move(g));
        }

        // gs::training::rasterize (rasterizer.cpp:46-437); mode: 0 RGB, 1 RGB_D, 2 D.  Returns (image [ch,H,W] clamped for
        // RGB, alpha [1,H,W], depth or undefined).
        std::vector<Tensor> render(const Tensor& viewmat, const Tensor& K, Tensor bg_color, int sh_degree, int image_width,
                                   int image_height, int mode) {
            using torch::indexing::None;
            using torch::indexing::Slice;
            // SplatData getters (splat_data.cpp:267-286)
            Tensor means3D = means;
            Tensor opacities = torch::sigmoid(op).squeeze(-1);
            Tensor scales_a = torch::exp(scales);
            Tensor rotations = torch::nn::functional::normalize(rot, torch::nn::functional::NormalizeFuncOptions().dim(-1));
            Tensor sh_coeffs = torch::cat({sh0, shN}, 1);
            Tensor prepared_bg = bg_color.defined() && bg_color.numel() ? bg_color.view({1, -1}).to(torch::kCUDA) : Tensor();
            const float eps2d = 0.3f, near_plane = 0.01f, far_plane = 10000.0f, radius_clip = 0.0f;
            const int tile_size = 16;
            auto proj_settings = gs::training::GUTProjectionSettings{image_width, image_height, eps2d, near_plane, far_plane,
                                                                      radius_clip, 1.0f, gsplat::CameraModelType::PINHOLE};
            auto proj = gs::training::fully_fused_projection_with_ut(means3D, rotations, scales_a, opacities, viewmat, K,
                                                                     std::nullopt, std::nullopt, std::nullopt, proj_settings,
                                                                     UnscentedTransformParameters());
            Tensor radii = proj[0], means2d = proj[1], depths = proj[2];
            auto means2d_with_grad = means2d.contiguous();
            means2d_with_grad.set_requires_grad(true);
            means2d_with_grad.retain_grad();
            auto viewmat_inv = torch::inverse(viewmat);
            auto campos = viewmat_inv.index({Slice(), Slice(None, 3), 3});
            auto dirs = means3D.unsqueeze(0) - campos.unsqueeze(1);
            auto masks = (radii > 0).all(-1);
            auto shs = sh_coeffs.unsqueeze(0);
            auto sh_degree_tensor = torch::tensor({sh_degree}, torch::TensorOptions().dtype(torch::kInt32).device(dirs.device()));
            auto colors = gs::training::SphericalHarmonicsFunction::apply(sh_degree_tensor, dirs.contiguous(), shs.contiguous(),
                                                                          masks.contiguous())[0];
            colors = torch::clamp_min(colors + 0.5f, 0.0f);
            Tensor render_colors, final_bg;
            if (mode == 0) {
                render_colors = colors, final_bg = prepared_bg;
            } else if (mode == 2) {
                render_colors = depths.unsqueeze(-1);
                if (prepared_bg.defined())
                    final_bg = torch::zeros({1, 1}, prepared_bg.options());
            } else {
                render_colors = torch::cat({colors, depths.unsqueeze(-1)}, -1);
                if (prepared_bg.defined())
                    final_bg = torch::cat({prepared_bg, torch::zeros({1, 1}, prepared_bg.options())}, -1);
            }
            if (!final_bg.defined())
                final_bg = at::empty({0}, colors.options().dtype(torch::kFloat32));
            Tensor final_opacities = opacities.unsqueeze(0);
            const int tile_width = (image_width + tile_size - 1) / tile_size, tile_height = (image_height + tile_size - 1) / tile_size;
            const auto isect = gsplat::intersect_tile(means2d_with_grad, radii, depths, {}, {}, 1, tile_size, tile_width,
                                                      tile_height, true);
            const auto isect_ids = std::get<1>(isect);
            const auto flatten_ids = std::get<2>(isect);
            last_n_isects = flatten_ids.numel();
            auto isect_offsets = gsplat::intersect_offset(isect_ids, 1, tile_width, tile_height);
            isect_offsets = isect_offsets.reshape({1, tile_height, tile_width});
            auto raster_settings = gs::training::GUTRasterizationSettings{image_width, image_height, tile_size, 1.0f,
                                                                           gsplat::CameraModelType::PINHOLE};
            auto out = gs::training::GUTRasterizationFunction::apply(means3D, rotations, scales_a, render_colors, final_opacities,
                                                                     final_bg, std::nullopt, viewmat, K, std::nullopt,
                                                                     std::nullopt, std::nullopt, isect_offsets, flatten_ids,
                                                                     raster_settings, UnscentedTransformParameters{});
            Tensor rendered_image = out[0], rendered_alpha = out[1], image, depth;
            if (mode == 0) {
                image = rendered_image;
            } else if (mode == 2) {
                depth = rendered_image;
            } else {
                image = rendered_image.index({Slice(), Slice(), Slice(), Slice(None, -1)});
                depth = rendered_image.index({Slice(), Slice(), Slice(), Slice(-1, None)});
            }
            std::vector<Tensor> r(3);
            if (image.defined())
                r[0] = torch::clamp(image.squeeze(0).permute({2, 0, 1}), 0.0f, 1.0f);
            r[1] = rendered_alpha.squeeze(0).permute({2, 0, 1});
            if (depth.defined())
                r[2] = depth.squeeze(0).permute({2, 0, 1});
            return r;
        }

        double train_step(int iteration, std::vector<Tensor> viewmats, std::vector<Tensor> Ks, std::vector<Tensor> gts,
                          Tensor bg, double lambda_dssim, int sh_degree, int width, int height, bool read_loss) {
            Tensor total;
            for (size_t v = 0; v < viewmats.size(); ++v) {
                auto r = render(viewmats[v], Ks[v], bg, sh_degree, width, height, 0);
                Tensor loss = Harness::photometric_loss(r[0], gts[v], (float)lambda_dssim);
                loss.backward();
                if (read_loss)
                    total = total.defined() ? total + loss.detach() : loss.detach();
            }
            opt->step(iteration);
            opt->zero_grad(true, iteration);
            return read_loss ? total.item<double>() : 0.0;
        }

        // one view, no optimiser: (image, alpha, depth|empty, loss, grads[6])
        std::vector<Tensor> view_grads(Tensor viewmat, Tensor K, Tensor gt, Tensor bg, double lambda_dssim, int sh_degree,
                                       int width, int height, int mode) {
            opt->zero_grad(true, 0);
            auto r = render(viewmat, K, bg, sh_degree, width, height, mode);
            Tensor loss = mode == 2 ? r[2].mean() : Harness::photometric_loss(r[0], gt, (float)lambda_dssim);
            if (mode == 1)
                loss = loss + 0.1f * r[2].mean(); // make the depth channel carry gradient
            loss.backward();
            return {r[0].defined() ? r[0].detach() : Tensor(), r[1].detach(), r[2].defined() ? r[2].detach() : Tensor(),
                    loss.detach(), means.grad(), sh0.grad(), shN.grad(), scales.grad(), rot.grad(), op.grad()};
        }
    };
} // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    m.def("forward_wrapper", &fast_gs::rasterization::forward_wrapper);
    m.def("backward_wrapper", &fast_gs::rasterization::backward_wrapper);
    m.def("adam_step_wrapper", &fast_gs::optimizer::adam_step_wrapper);
    m.def("fused_ssim", [](Tensor a, Tensor b, std::string padding, bool train) { return fused_ssim(a, b, padding, train); });
    // the remaining gsplat:: operators of gsplat/Ops.h, called directly (the autograd classes above cover the other seven)
    // gsplat::projection_ut_3dgs_fused with every camera model / shutter / distortion argument (enums as ints)
    m.def("projection_ut", [](Tensor means, Tensor quats, Tensor scales, std::optional<Tensor> opacities, Tensor viewmats0,
                              std::optional<Tensor> viewmats1, Tensor Ks, int width, int height, double eps2d, double near_plane,
                              double far_plane, double radius_clip, bool calc_compensations, int camera_model, int rs_type,
                              std::optional<Tensor> radial, std::optional<Tensor> tangential, std::optional<Tensor> prism) {
        return gsplat::projection_ut_3dgs_fused(means, quats, scales, opacities, viewmats0, viewmats1, Ks, width, height,
                                                (float)eps2d, (float)near_plane, (float)far_plane, (float)radius_clip,
                                                calc_compensations, static_cast<gsplat::CameraModelType>(camera_model),
                                                UnscentedTransformParameters{}, static_cast<ShutterType>(rs_type), radial,
                                                tangential, prism);
    });
    m.def("raster_fwd", [](Tensor means, Tensor quats, Tensor scales, Tensor colors, Tensor opacities,
                           std::optional<Tensor> backgrounds, int width, int height, Tensor viewmats0,
                           std::optional<Tensor> viewmats1, Tensor Ks, int camera_model, int rs_type,
                           std::optional<Tensor> radial, std::optional<Tensor> tangential, std::optional<Tensor> prism,
                           Tensor tile_offsets, Tensor flatten_ids) {
        return gsplat::rasterize_to_pixels_from_world_3dgs_fwd(
            means, quats, scales, colors, opacities, backgrounds, std::nullopt, width, height, 16, viewmats0, viewmats1, Ks,
            static_cast<gsplat::CameraModelType>(camera_model), UnscentedTransformParameters{},
            static_cast<ShutterType>(rs_type), radial, tangential, prism, tile_offsets, flatten_ids);
    });
    m.def("raster_bwd", [](Tensor means, Tensor quats, Tensor scales, Tensor colors, Tensor opacities,
                           std::optional<Tensor> backgrounds, int width, int height, Tensor viewmats0,
                           std::optional<Tensor> viewmats1, Tensor Ks, int camera_model, int rs_type,
                           std::optional<Tensor> radial, std::optional<Tensor> tangential, std::optional<Tensor> prism,
                           Tensor tile_offsets, Tensor flatten_ids, Tensor render_alphas, Tensor last_ids,
                           Tensor v_render_colors, Tensor v_render_alphas) {
        return gsplat::rasterize_to_pixels_from_world_3dgs_bwd(
            means, quats, scales, colors, opacities, backgrounds, std::nullopt, width, height, 16, viewmats0, viewmats1, Ks,
            static_cast<gsplat::CameraModelType>(camera_model), UnscentedTransformParameters{},
            static_cast<ShutterType>(rs_type), radial, tangential, prism, tile_offsets, flatten_ids, render_alphas, last_ids,
            v_render_colors, v_render_alphas);
    });
    m.def("quats_to_rotmats", &gsplat::quats_to_rotmats);
    m.def("relocation", &gsplat::relocation);
    m.def("add_noise", &gsplat::add_noise);
    m.def("intersect_tile", [](Tensor means2d, Tensor radii, Tensor depths, int C, int tile_size, int tw, int th, bool sort) {
        return gsplat::intersect_tile(means2d, radii, depths, {}, {}, C, tile_size, tw, th, sort);
    });
    m.def("intersect_tile_packed", [](Tensor means2d, Tensor radii, Tensor depths, Tensor camera_ids, Tensor gaussian_ids, int C,
                                      int tile_size, int tw, int th, bool sort) {
        return gsplat::intersect_tile(means2d, radii, depths, camera_ids, gaussian_ids, C, tile_size, tw, th, sort);
    });
    m.def("intersect_offset", &gsplat::intersect_offset);
#ifdef LFS_B200_LEGACY_OPS
    // legacy 2-D op surface of the reference's gtests (SURVEY F5): host layer -> C ABI -> csrc/legacy2d.cu
    m.def("quat_scale_to_covar_preci_fwd", &gsplat::quat_scale_to_covar_preci_fwd);
    m.def("quat_scale_to_covar_preci_bwd", &gsplat::quat_scale_to_covar_preci_bwd);
    m.def("projection_ewa_3dgs_fused_fwd",
          [](Tensor means, std::optional<Tensor> covars, std::optional<Tensor> quats, std::optional<Tensor> scales,
             std::optional<Tensor> opacities, Tensor viewmats, Tensor Ks, int w, int h, double eps2d, double near_p,
             double far_p, double clip, bool comp) {
              return gsplat::projection_ewa_3dgs_fused_fwd(means, covars, quats, scales, opacities, viewmats, Ks, (uint32_t)w,
                                                           (uint32_t)h, (float)eps2d, (float)near_p, (float)far_p, (float)clip,
                                                           comp, gsplat::CameraModelType::PINHOLE);
          });
    m.def("rasterize_to_pixels_3dgs_fwd", &gsplat::rasterize_to_pixels_3dgs_fwd);
    m.def("rasterize_to_pixels_3dgs_bwd", &gsplat::rasterize_to_pixels_3dgs_bwd);
#endif
    py::class_<GutHarness>(m, "GutHarness")
        .def(py::init<Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, std::vector<double>>())
        // the autograd engine must not be entered with the GIL held
        .def("render", &GutHarness::render, py::call_guard<py::gil_scoped_release>())
        .def("train_step", &GutHarness::train_step, py::call_guard<py::gil_scoped_release>())
        .def("view_grads", &GutHarness::view_grads, py::call_guard<py::gil_scoped_release>())
        .def_readonly("last_n_isects", &GutHarness::last_n_isects);
    py::class_<Harness>(m, "Harness")
        .def(py::init<Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, std::vector<double>>())
        .def("train_step", &Harness::train_step, py::call_guard<py::gil_scoped_release>())
        .def("view_grads", &Harness::view_grads, py::call_guard<py::gil_scoped_release>())
        .def("params", &Harness::params)
        .def_readwrite("densification_info", &Harness::densification_info);
}

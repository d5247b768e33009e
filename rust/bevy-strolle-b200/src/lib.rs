//! `bevy_strolle::StrollePlugin` for the B200 engine.
//!
//! Same shape as the reference plugin (`/bevy-strolle/src/lib.rs:29-84`, `stages.rs`, `rendering_node.rs`): the main world's meshes,
//! materials, images, instances, lights, sun and cameras are mirrored into the engine once per frame (extract in `ExtractSchedule`, apply
//! in `Render::Prepare`), and a render-graph node on the camera's view renders through the engine.  The CUDA engine composes into host
//! memory in the view's own format (`Rgba16Float`, the HDR main texture the reference requires), so the node ends with one
//! `write_texture` into that texture at the viewport's position where the reference records compute passes; FXAA, tonemapping and
//! upscaling follow as in the reference's graph.
//!
//! `STROLLE_B200_DEVICES=0,1,2,3` selects the GPUs (default `0`); several devices = row strips of every camera's frame.
pub mod prelude {
    pub use crate::{StrolleCamera, StrollePlugin, StrolleSun};
}

mod sync;

use bevy::core_pipeline::fxaa::FxaaNode;
use bevy::core_pipeline::tonemapping::TonemappingNode;
use bevy::core_pipeline::upscaling::UpscalingNode;
use bevy::prelude::*;
use bevy::render::render_graph::{NodeRunError, RenderGraphApp, RenderGraphContext, ViewNode, ViewNodeRunner};
use bevy::render::renderer::{RenderContext, RenderQueue};
use bevy::render::view::ViewTarget;
use bevy::render::RenderApp;
pub use strolle as st;

/// Name of the render graph a camera selects with `CameraRenderGraph::new(bevy_strolle::graph::NAME)` (`/bevy-strolle/src/graph.rs`).
pub mod graph {
    pub const NAME: &str = "strolle";
    pub mod node {
        pub const RENDERING: &str = "strolle_rendering";
        pub const TONEMAPPING: &str = "strolle_tonemapping";
        pub const FXAA: &str = "strolle_fxaa";
        pub const UPSCALING: &str = "strolle_upscaling";
    }
}

/// Per-camera settings (`/bevy-strolle/src/camera.rs`)
#[derive(Clone, Debug, Default, Component)]
pub struct StrolleCamera {
    pub mode: st::CameraMode,
}

/// The sun (`/bevy-strolle/src/sun.rs`)
#[derive(Clone, Debug, Default, Resource, Deref, DerefMut)]
pub struct StrolleSun {
    sun: st::Sun,
}

#[derive(Clone, Debug)]
pub struct EngineParams;

impl st::Params for EngineParams {
    type ImageHandle = AssetId<Image>;
    type InstanceHandle = Entity;
    type LightHandle = Entity;
    type MaterialHandle = AssetId<StandardMaterial>;
    type MeshHandle = AssetId<Mesh>;
}

#[derive(Resource, Deref, DerefMut)]
pub(crate) struct EngineResource(pub st::Engine<EngineParams>);

pub struct StrollePlugin;

impl Plugin for StrollePlugin {
    fn build(&self, app: &mut App) {
        app.insert_resource(StrolleSun::default());
        let Ok(render_app) = app.get_sub_app_mut(RenderApp) else { return };
        render_app.insert_resource(sync::Synced::default());
        sync::setup(render_app);
        // the reference's graph (`/bevy-strolle/src/graph.rs`): the HDR frame is anti-aliased and tonemapped by Bevy's own nodes
        render_app
            .add_render_sub_graph(graph::NAME)
            .add_render_graph_node::<ViewNodeRunner<RenderingNode>>(graph::NAME, graph::node::RENDERING)
            .add_render_graph_node::<ViewNodeRunner<TonemappingNode>>(graph::NAME, graph::node::TONEMAPPING)
            .add_render_graph_node::<ViewNodeRunner<UpscalingNode>>(graph::NAME, graph::node::UPSCALING)
            .add_render_graph_node::<ViewNodeRunner<FxaaNode>>(graph::NAME, graph::node::FXAA)
            .add_render_graph_edges(graph::NAME, &[graph::node::RENDERING, graph::node::FXAA, graph::node::TONEMAPPING, graph::node::UPSCALING]);
    }

    fn finish(&self, app: &mut App) {
        let Ok(render_app) = app.get_sub_app_mut(RenderApp) else { return };
        let devices: Vec<i32> = std::env::var("STROLLE_B200_DEVICES")
            .ok()
            .map(|v| v.split(',').filter_map(|d| d.trim().parse().ok()).collect())
            .filter(|v: &Vec<i32>| !v.is_empty())
            .unwrap_or_else(|| vec![0]);
        let engine = st::Engine::new(&devices).expect("strolle_b200: no usable CUDA device (this engine has no CPU fallback)");
        render_app.insert_resource(EngineResource(engine));
    }
}

/// `RenderingNode` (`/bevy-strolle/src/rendering_node.rs:14-36`)
#[derive(Default)]
pub(crate) struct RenderingNode;

impl ViewNode for RenderingNode {
    type ViewQuery = &'static ViewTarget;

    fn run(&self, graph: &mut RenderGraphContext, _render_context: &mut RenderContext, target: &ViewTarget, world: &World) -> Result<(), NodeRunError> {
        let entity = graph.view_entity();
        let engine = world.resource::<EngineResource>();
        let synced = world.resource::<sync::Synced>();
        let Some(camera) = synced.cameras.get(&entity) else { return Ok(()) };
        let mut frame = camera.frame.lock().unwrap();
        if let Err(err) = engine.render_camera(camera.handle, &mut frame) {
            error!("strolle: {err}");
            return Ok(());
        }
        let size = wgpu::Extent3d { width: frame.size.x, height: frame.size.y, depth_or_array_layers: 1 };
        let layout = wgpu::ImageDataLayout { offset: 0, bytes_per_row: Some(frame.size.x * frame.format.bytes_per_pixel() as u32), rows_per_image: Some(frame.size.y) };
        let copy = wgpu::ImageCopyTexture { texture: target.main_texture(), mip_level: 0, origin: wgpu::Origin3d { x: camera.position.x, y: camera.position.y, z: 0 }, aspect: wgpu::TextureAspect::All };
        world.resource::<RenderQueue>().write_texture(copy, &frame.pixels, layout, size);
        Ok(())
    }
}

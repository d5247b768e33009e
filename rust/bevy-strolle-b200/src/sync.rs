//! World -> engine synchronisation: what `/bevy-strolle/src/stages/{extract,prepare}.rs` and `state.rs` do, in one module.
//! `ExtractSchedule` systems copy what changed out of the main world into `Pending`; one `Render::Prepare` system replays it on the
//! engine in the order the reference uses (meshes, materials, images, instances, lights, sun, cameras, then `tick`).
use std::f32::consts::PI;
use std::sync::Mutex;

use bevy::prelude::*;
use bevy::render::camera::{CameraProjection, CameraRenderGraph, ExtractedCamera};
use bevy::render::mesh::VertexAttributeValues;
use bevy::render::render_resource::{PrimitiveTopology, TextureFormat};
use bevy::render::view::{RenderLayers, ViewTarget};
use bevy::render::{Extract, ExtractSchedule, Render, RenderSet};
use bevy::utils::{HashMap, HashSet};

use crate::{st, EngineParams, EngineResource, StrolleCamera, StrolleSun};

pub(crate) struct SyncedCamera {
    pub handle: st::CameraHandle,
    pub position: UVec2,
    pub frame: Mutex<st::Frame>,
}

#[derive(Default, Resource)]
pub(crate) struct Synced {
    pub cameras: HashMap<Entity, SyncedCamera>,
}

struct PendingCamera {
    entity: Entity,
    transform: Mat4,
    projection: Mat4,
    mode: Option<st::CameraMode>,
}

#[derive(Default, Resource)]
struct Pending {
    meshes: Vec<(AssetId<Mesh>, Mesh)>,
    meshes_removed: Vec<AssetId<Mesh>>,
    materials: Vec<(AssetId<StandardMaterial>, StandardMaterial)>,
    materials_removed: Vec<AssetId<StandardMaterial>>,
    images: Vec<(AssetId<Image>, UVec2, Vec<u8>)>,
    images_removed: Vec<AssetId<Image>>,
    instances: Vec<(Entity, AssetId<Mesh>, AssetId<StandardMaterial>, bevy::math::Affine3A)>,
    instances_removed: Vec<Entity>,
    lights: Vec<(Entity, st::Light)>,
    lights_removed: Vec<Entity>,
    sun: Option<st::Sun>,
    cameras: Vec<PendingCamera>,
}

pub(crate) fn setup(render_app: &mut App) {
    render_app.insert_resource(Pending::default());
    render_app.add_systems(ExtractSchedule, (extract_assets, extract_instances, extract_lights, extract_cameras));
    render_app.add_systems(Render, apply.in_set(RenderSet::Prepare));
}

fn asset_changes<A: Asset + Clone>(events: &mut EventReader<AssetEvent<A>>, assets: &Assets<A>, changed: &mut Vec<(AssetId<A>, A)>, removed: &mut Vec<AssetId<A>>) {
    let mut touched = HashSet::new();
    for event in events.read() {
        match event {
            AssetEvent::Added { id } | AssetEvent::Modified { id } => {
                touched.insert(*id);
            }
            AssetEvent::Removed { id } => {
                touched.remove(id);
                removed.push(*id);
            }
            AssetEvent::LoadedWithDependencies { .. } => {}
        }
    }
    for id in touched {
        match assets.get(id) {
            Some(asset) => changed.push((id, asset.clone())),
            None => removed.push(id),
        }
    }
}

#[allow(clippy::too_many_arguments)]
fn extract_assets(
    mut pending: ResMut<Pending>,
    mut mesh_events: Extract<EventReader<AssetEvent<Mesh>>>,
    meshes: Extract<Res<Assets<Mesh>>>,
    mut material_events: Extract<EventReader<AssetEvent<StandardMaterial>>>,
    materials: Extract<Res<Assets<StandardMaterial>>>,
    mut image_events: Extract<EventReader<AssetEvent<Image>>>,
    images: Extract<Res<Assets<Image>>>,
    sun: Extract<Res<StrolleSun>>,
) {
    let pending = &mut *pending;
    asset_changes(&mut mesh_events, &meshes, &mut pending.meshes, &mut pending.meshes_removed);
    asset_changes(&mut material_events, &materials, &mut pending.materials, &mut pending.materials_removed);
    let mut changed = Vec::new();
    asset_changes(&mut image_events, &images, &mut changed, &mut pending.images_removed);
    for (id, image) in changed {
        // the atlas holds Rgba8UnormSrgb texels (`/strolle/src/images.rs:38-43`); other formats are not sampled by the reference either
        if image.texture_descriptor.dimension == wgpu::TextureDimension::D2 && image.texture_descriptor.format.block_size(None) == Some(4) {
            let size = UVec2::new(image.texture_descriptor.size.width, image.texture_descriptor.size.height);
            pending.images.push((id, size, image.data));
        }
    }
    pending.sun = Some(***sun);
}

#[allow(clippy::type_complexity)]
fn extract_instances(
    mut pending: ResMut<Pending>,
    changed: Extract<
        Query<
            (Entity, &Handle<Mesh>, &Handle<StandardMaterial>, &GlobalTransform, &InheritedVisibility, Option<&RenderLayers>),
            Or<(Changed<Handle<Mesh>>, Changed<Handle<StandardMaterial>>, Changed<GlobalTransform>, Changed<InheritedVisibility>, Changed<RenderLayers>)>,
        >,
    >,
    mut removed: Extract<RemovedComponents<Handle<Mesh>>>,
) {
    pending.instances_removed.extend(removed.read());
    for (entity, mesh, material, transform, visibility, layers) in changed.iter() {
        let hidden = !visibility.get() || layers.is_some_and(|l| *l != RenderLayers::all());
        if hidden {
            pending.instances_removed.push(entity);
        } else {
            pending.instances.push((entity, mesh.id(), material.id(), transform.affine()));
        }
    }
}

#[allow(clippy::type_complexity)]
fn extract_lights(
    mut pending: ResMut<Pending>,
    points: Extract<Query<(Entity, &PointLight, &GlobalTransform), Or<(Changed<PointLight>, Changed<GlobalTransform>)>>>,
    spots: Extract<Query<(Entity, &SpotLight, &GlobalTransform), Or<(Changed<SpotLight>, Changed<GlobalTransform>)>>>,
    mut removed_points: Extract<RemovedComponents<PointLight>>,
    mut removed_spots: Extract<RemovedComponents<SpotLight>>,
) {
    pending.lights_removed.extend(removed_points.read().chain(removed_spots.read()));
    let rgb = |c: Color| {
        let [r, g, b, _] = c.as_linear_rgba_f32();
        Vec3::new(r, g, b)
    };
    for (entity, light, transform) in points.iter() {
        let intensity = light.intensity / (4.0 * PI);   // candela-ish, as `/bevy-strolle/src/stages/extract.rs:285`
        if intensity < 0.0001 {
            pending.lights_removed.push(entity);
            continue;
        }
        pending.lights.push((entity, st::Light::Point { position: transform.translation(), radius: light.radius, color: rgb(light.color) * intensity, range: light.range }));
    }
    for (entity, light, transform) in spots.iter() {
        let intensity = light.intensity / (4.0 * PI);
        if intensity < 0.0001 {
            pending.lights_removed.push(entity);
            continue;
        }
        let (_, rotation, translation) = transform.to_scale_rotation_translation();
        pending.lights.push((
            entity,
            st::Light::Spot { position: translation, radius: light.radius, color: rgb(light.color) * intensity, range: light.range, direction: -(rotation * Vec3::Z).normalize(), angle: light.outer_angle },
        ));
    }
}

fn extract_cameras(mut pending: ResMut<Pending>, cameras: Extract<Query<(Entity, &Camera, &CameraRenderGraph, &Projection, &GlobalTransform, Option<&StrolleCamera>)>>) {
    for (entity, camera, render_graph, projection, transform, settings) in cameras.iter() {
        if !camera.is_active || **render_graph != crate::graph::NAME {
            continue;
        }
        assert!(camera.hdr, "Strolle requires an HDR camera");
        pending.cameras.push(PendingCamera { entity, transform: transform.compute_matrix(), projection: projection.get_projection_matrix(), mode: settings.map(|s| s.mode) });
    }
}

fn triangles_of(mesh: &Mesh) -> Option<Vec<st::MeshTriangle>> {
    if mesh.primitive_topology() != PrimitiveTopology::TriangleList {
        return None;
    }
    let positions = mesh.attribute(Mesh::ATTRIBUTE_POSITION).and_then(VertexAttributeValues::as_float3)?;
    let normals = mesh.attribute(Mesh::ATTRIBUTE_NORMAL).and_then(VertexAttributeValues::as_float3)?;
    let uvs: &[[f32; 2]] = match mesh.attribute(Mesh::ATTRIBUTE_UV_0) {
        Some(VertexAttributeValues::Float32x2(v)) => v,
        _ => &[],
    };
    let tangents: &[[f32; 4]] = match mesh.attribute(Mesh::ATTRIBUTE_TANGENT) {
        Some(VertexAttributeValues::Float32x4(v)) => v,
        _ => &[],
    };
    let indices: Vec<usize> = mesh.indices()?.iter().collect();
    let corner = |i: usize| (positions[i], normals[i], uvs.get(i).copied().unwrap_or_default(), tangents.get(i).copied().unwrap_or_default());
    Some(
        indices
            .chunks_exact(3)
            .map(|v| {
                let (a, b, c) = (corner(v[0]), corner(v[1]), corner(v[2]));
                st::MeshTriangle::default().with_positions([a.0, b.0, c.0]).with_normals([a.1, b.1, c.1]).with_uvs([a.2, b.2, c.2]).with_tangents([a.3, b.3, c.3])
            })
            .collect(),
    )
}

fn material_of(mat: &StandardMaterial) -> st::Material<EngineParams> {
    let [r, g, b, a] = mat.base_color.as_linear_rgba_f32();
    let alpha = match mat.alpha_mode {
        AlphaMode::Opaque => 1.0,
        AlphaMode::Mask(cutoff) => (a >= cutoff) as u32 as f32,
        _ => a,
    };
    st::Material {
        base_color: Vec4::new(r, g, b, alpha),
        base_color_texture: mat.base_color_texture.as_ref().map(|h| h.id()),
        emissive: Vec4::from_array(mat.emissive.as_linear_rgba_f32()),
        emissive_texture: mat.emissive_texture.as_ref().map(|h| h.id()),
        perceptual_roughness: mat.perceptual_roughness,
        metallic: mat.metallic,
        metallic_roughness_texture: mat.metallic_roughness_texture.as_ref().map(|h| h.id()),
        reflectance: mat.reflectance,
        ior: if mat.thickness > 0.0 { mat.ior } else { 1.0 },
        normal_map_texture: mat.normal_map_texture.as_ref().map(|h| h.id()),
        alpha_mode: if matches!(mat.alpha_mode, AlphaMode::Opaque) { st::AlphaMode::Opaque } else { st::AlphaMode::Blend },
    }
}

/// The engine's format for a view's main texture: the reference composes into `view_target.main_texture_format()`
/// (`/bevy-strolle/src/stages/prepare.rs:297`), which for the HDR cameras it requires is `Rgba16Float`.
fn viewport_format(format: TextureFormat) -> Option<st::ViewportFormat> {
    match format {
        TextureFormat::Rgba16Float => Some(st::ViewportFormat::Rgba16Float),
        _ => None,
    }
}

fn apply(mut engine: ResMut<EngineResource>, mut pending: ResMut<Pending>, mut synced: ResMut<Synced>, views: Query<(Entity, &ExtractedCamera, &ViewTarget)>) {
    let engine = &mut engine.0;
    let p = std::mem::take(&mut *pending);
    for id in p.meshes_removed.iter().copied().chain(p.meshes.iter().map(|(id, _)| *id)) {
        engine.remove_mesh(id);
    }
    for (id, mesh) in &p.meshes {
        if let Some(triangles) = triangles_of(mesh) {
            engine.insert_mesh(*id, st::Mesh::new(triangles));
        }
    }
    for id in p.materials_removed {
        engine.remove_material(id);
    }
    for (id, material) in &p.materials {
        engine.insert_material(*id, material_of(material));
    }
    for id in p.images_removed {
        engine.remove_image(id);
    }
    for (id, size, data) in p.images {
        engine.insert_image(id, st::Image::new(st::ImageData::Raw { data }, size));
    }
    for entity in p.instances_removed {
        engine.remove_instance(entity);
    }
    for (entity, mesh, material, transform) in p.instances {
        engine.insert_instance(entity, st::Instance::new(mesh, material, transform));
    }
    for entity in p.lights_removed {
        engine.remove_light(entity);
    }
    for (entity, light) in p.lights {
        engine.insert_light(entity, light);
    }
    if let Some(sun) = p.sun {
        engine.update_sun(sun);
    }
    // cameras: create / update the ones seen this frame, delete the rest (`/bevy-strolle/src/stages/prepare.rs:283-347`)
    let mut alive = HashSet::new();
    for cam in p.cameras {
        let Some((_, view, target)) = views.iter().find(|(e, _, _)| *e == cam.entity) else { continue };
        let Some(size) = view.physical_viewport_size else { continue };
        let Some(format) = viewport_format(target.main_texture_format()) else {
            error!("strolle: the view's main texture is {:?}; Strolle requires an HDR camera (Rgba16Float)", target.main_texture_format());
            continue;
        };
        let position = view.viewport.as_ref().map(|v| v.physical_position).unwrap_or_default();
        let viewport = st::CameraViewport { format, size, position };
        let camera = st::Camera { mode: cam.mode.unwrap_or_default(), viewport: viewport.clone(), transform: cam.transform, projection: cam.projection };
        alive.insert(cam.entity);
        match synced.cameras.get_mut(&cam.entity) {
            Some(known) => {
                if let Err(err) = engine.update_camera(known.handle, camera) {
                    error!("strolle: {err}");
                    continue;
                }
                known.position = position;
                let mut frame = known.frame.lock().unwrap();
                if frame.size != viewport.size || frame.format != viewport.format {
                    *frame = st::Frame::new(&viewport);
                }
            }
            None => match engine.create_camera(camera) {
                Ok(handle) => {
                    synced.cameras.insert(cam.entity, SyncedCamera { handle, position, frame: Mutex::new(st::Frame::new(&viewport)) });
                }
                Err(err) => error!("strolle: {err}"),
            },
        }
    }
    let dead: Vec<Entity> = synced.cameras.keys().copied().filter(|e| !alive.contains(e)).collect();
    for entity in dead {
        if let Some(cam) = synced.cameras.remove(&entity) {
            let _ = engine.delete_camera(cam.handle);
        }
    }
    if let Err(err) = engine.tick() {
        error!("strolle: {err}");
    }
}
